"""The conviqt sampler on one GPU (cmdr_sht_conviqt_sampler / cmdr_sht_conviqt_interp through comm_conviqt.make_sampler):
bit for bit the mirror comm_conviqt.interp (commander3/src/comm_conviqt_mod.f90:155-205) on the same cube, from host
and from device arrays, for both optim values; the table of a double cube; pixels outside the sky; and the real size
(nside 1024, bmax 8: an 805 MB table)."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _defined(psi, bmax):
    """Samples the reference can evaluate: those whose modulo(-psi, 2 pi) does not round up to 2 pi (where it would
    read one row past its cube and the mirror raises IndexError)."""
    f = np.float32
    twopi, psires = f(2.0 * math.pi), f(2.0 * math.pi / (2 * bmax))
    u = np.fmod(-psi.astype(f), twopi)
    u = np.where(u < 0, u + twopi, u).astype(f)
    return (u / psires).astype(np.int64) < 2 * bmax


def _samples(rng, npix, bmax, n):
    pix = rng.integers(0, npix, n).astype(np.int32)
    psi = rng.uniform(-3 * math.pi, 3 * math.pi, n).astype(np.float32)
    psi[:8] = [0.0, -0.0, 2 * math.pi, -2 * math.pi, -1e-30, 1e5, -7.5e6, math.pi / bmax]
    ok = _defined(psi, bmax)
    return pix[ok], psi[ok]


def table(s, npix, bmax):
    """The sampler's whole table, read back through interp with optim 2 at the bin centres psi = -k psires."""
    import torch
    f = np.float32
    psires = f(2.0 * math.pi / (2 * bmax))
    k = np.arange(2 * bmax)
    psi = -(k.astype(f) * psires).astype(f)
    pix = torch.arange(npix, dtype=torch.int32, device=s.device).repeat(2 * bmax)
    q = torch.as_tensor(psi, device=s.device).repeat_interleave(npix)
    optim, s.optim = s.optim, 2
    try:
        return s.interp(pix, q).reshape(2 * bmax, npix).cpu().numpy()
    finally:
        s.optim = optim


def _conviqt(nside, lmax, bmax, seed, device):
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    rng = np.random.default_rng(seed)
    info = comm_mapinfo(None, nside, lmax, 3, True)
    sky, beam = comm_map(info), comm_map(info)
    sky.alm[...] = rng.standard_normal(sky.alm.shape)
    beam.alm[...] = rng.standard_normal(beam.alm.shape) / (1.0 + info.lm[0])
    return comm_conviqt(nside, lmax, 3, bmax, beam, sky, device=device), sky


def _bits(a):
    return np.asarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("optim", [0, 2])
def test_sampler_matches_mirror(shtlib, optim):
    import torch
    dev = torch.device("cuda", 0)
    nside, lmax, bmax = 128, 256, 6
    cv, sky = _conviqt(nside, lmax, bmax, 31, dev)
    cvh, _ = _conviqt(nside, lmax, bmax, 31, None)          # the same cube in host memory
    assert np.array_equal(_bits(cvh.c), _bits(cv.c.cpu().numpy()))
    cv.optim = cvh.optim = optim
    pix, psi = _samples(np.random.default_rng(32 + optim), cv.npix, bmax, 1_000_000)
    ref = cv.interp(pix, psi)
    with cv.make_sampler() as s, cvh.make_sampler() as sh:
        assert np.array_equal(_bits(table(s, cv.npix, bmax)), _bits(cv.c.cpu().numpy()))
        n0 = shtlib.launch_count()
        out = s.interp(pix, psi)                            # host arrays
        assert shtlib.launch_count() > n0
        assert isinstance(out, np.ndarray) and out.dtype == np.float32
        assert np.array_equal(_bits(out), _bits(ref))
        outd = s.interp(torch.as_tensor(pix, device=dev), torch.as_tensor(psi, device=dev))   # device arrays
        assert isinstance(outd, torch.Tensor) and outd.is_cuda
        assert np.array_equal(_bits(outd.cpu().numpy()), _bits(ref))
        # int64 pixels and float64 angles are converted as the mirror converts them
        out64 = sh.interp(pix.astype(np.int64), psi.astype(np.float64))
        assert np.array_equal(_bits(out64), _bits(ref))
        # into a caller's buffer, with broadcasting of one angle over many pixels
        buf = torch.empty(1000, dtype=torch.float32, device=dev)
        r = s.interp(torch.as_tensor(pix[:1000], device=dev), torch.tensor(0.25, device=dev), out=buf)
        assert r is buf and np.array_equal(_bits(buf.cpu().numpy()), _bits(cv.interp(pix[:1000], np.float32(0.25))))


def test_double_cube_gives_its_float_rounding(shtlib):
    import torch
    from commander_b200.comm_conviqt import conviqt_sampler
    dev = torch.device("cuda", 0)
    nside, lmax, bmax = 32, 64, 4
    cv, sky = _conviqt(nside, lmax, bmax, 41, dev)
    c64 = torch.zeros((2 * bmax, cv.info.np), dtype=torch.float64, device=dev)
    cv.precompute_sky(sky, cube=c64)
    want = c64.cpu().numpy().astype(np.float32)
    with conviqt_sampler(c64, bmax, cv.npix, 0, cv.info.geom_info_T) as s:
        assert np.array_equal(_bits(table(s, cv.npix, bmax)), _bits(want))
    with conviqt_sampler(c64.cpu().numpy(), bmax, cv.npix, 0, cv.info.geom_info_T) as s:
        assert np.array_equal(_bits(table(s, cv.npix, bmax)), _bits(want))


def test_bits_are_copied_exactly(shtlib):
    """-0.0, denormals, infinities and NaN payloads of the cube reach the table unchanged (no arithmetic on the way)."""
    import torch
    from commander_b200.comm_map import comm_mapinfo
    from commander_b200.comm_conviqt import conviqt_sampler
    nside, bmax = 8, 2
    info = comm_mapinfo(None, nside, 16, 1, False)
    c = np.random.default_rng(5).standard_normal((2 * bmax, info.np)).astype(np.float32)
    c.view(np.uint32)[:, :4] = [0x80000000, 0x00000001, 0x7f800000, 0x7fc01234]
    with conviqt_sampler(c, bmax, info.npix, 0, info.geom_info_T) as s:
        assert np.array_equal(table(s, info.npix, bmax).view(np.uint32), c.view(np.uint32))
        assert s.device == torch.device("cuda", torch.cuda.current_device())


def test_pixels_outside_the_sky(shtlib):
    import torch
    dev = torch.device("cuda", 0)
    nside, bmax = 16, 3
    cv, _ = _conviqt(nside, 32, bmax, 51, dev)
    npix = cv.npix
    pix = np.array([5, -1, npix, npix - 1, -2 ** 31, 2 ** 31 - 1, 0], dtype=np.int32)
    psi = np.full(pix.size, 0.3, dtype=np.float32)
    bad = np.array([False, True, True, False, True, True, False])
    with cv.make_sampler() as s:
        for on_dev in (False, True):
            if on_dev:
                p, q = torch.as_tensor(pix, device=dev), torch.as_tensor(psi, device=dev)
                out, st = torch.empty(pix.size, dtype=torch.float32, device=dev), torch.cuda.current_stream().cuda_stream
            else:
                p, q, out, st = pix, psi, np.empty(pix.size, dtype=np.float32), None
            nbad = shtlib.conviqt_interp(s.handle, p, q, 0, out, stream=st)
            o = out.cpu().numpy() if on_dev else out
            assert nbad == int(bad.sum()) and np.array_equal(np.isnan(o), bad)
            assert np.array_equal(_bits(o[~bad]), _bits(cv.interp(pix[~bad], psi[~bad])))
        with pytest.raises(IndexError, match="4 pixel"):
            s.interp(pix, psi)
        with pytest.raises(IndexError, match="1 pixel"):
            s.interp(np.array([2 ** 40, 3], dtype=np.int64), np.zeros(2))      # beyond int32: refused, not wrapped
        with pytest.raises(IndexError):
            s.interp(torch.tensor([3, -7], device=dev), torch.zeros(2, device=dev))
        assert s.interp(np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.float32)).size == 0


def test_real_size(shtlib):
    """nside 1024 / bmax 8 (an 805 MB table, the size a TOD run samples): the table and a 1e5-sample subset of 1e7
    device samples, both optim values, bit for bit the mirror."""
    import torch
    dev = torch.device("cuda", 0)
    nside, lmax, bmax = 1024, 1500, 8
    cv, _ = _conviqt(nside, lmax, bmax, 61, dev)
    pix, psi = _samples(np.random.default_rng(62), cv.npix, bmax, 10_000_000)
    pd, qd = torch.as_tensor(pix, device=dev), torch.as_tensor(psi, device=dev)
    sub = np.random.default_rng(63).choice(pix.size, 100_000, replace=False)
    with cv.make_sampler() as s:
        assert np.array_equal(_bits(table(s, cv.npix, bmax)), _bits(cv.c.cpu().numpy()))
        for optim in (0, 2):
            s.optim = cv.optim = optim
            out = s.interp(pd, qd).cpu().numpy()
            assert np.array_equal(_bits(out[sub]), _bits(cv.interp(pix[sub], psi[sub])))
