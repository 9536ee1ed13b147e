"""GPU parity tests of cmdr_sht_conviqt_cube and its mirror commander_b200/comm_conviqt.py against the CPU
restatement oracle/conviqt.py (commander3/src/comm_conviqt_mod.f90:207-357).
Tolerances: double-precision cube, relative L2 <= 1e-10; the single-precision cube (what the reference stores,
:281) must equal the rounded oracle value to within one float32 ulp of the cube's largest entry."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-10


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _setup(nside, lmax, lmax_beam, nmaps, seed):
    from commander_b200 import comm_map, comm_mapinfo
    rng = np.random.default_rng(seed)
    info = comm_mapinfo(None, nside, lmax, nmaps, nmaps == 3)
    binfo = comm_mapinfo(None, nside, lmax_beam, nmaps, nmaps == 3)
    sky, beam = comm_map(info), comm_map(binfo)
    sky.alm[...] = rng.standard_normal(sky.alm.shape)
    beam.alm[...] = rng.standard_normal(beam.alm.shape) / (1.0 + binfo.lm[0])
    return info, sky, beam


@pytest.mark.parametrize("nside,lmax,lmax_beam,bmax,nmaps", [(8, 16, 16, 1, 3), (8, 16, 12, 3, 3), (16, 32, 32, 4, 1),
                                                             (32, 64, 48, 6, 3), (16, 40, 40, 9, 3),
                                                             # up to CMDR_MAX_SPIN: 64 psi planes at bmax 32
                                                             (16, 48, 48, 16, 3), (16, 48, 40, 31, 1),
                                                             (16, 48, 48, 32, 3)])
def test_cube_vs_oracle(shtlib, cpu_oracle, nside, lmax, lmax_beam, bmax, nmaps):
    import torch
    from commander_b200 import comm_map
    from commander_b200.comm_conviqt import comm_conviqt
    from oracle import conviqt as O
    info, sky, beam = _setup(nside, lmax, lmax_beam, nmaps, 11 * nside + bmax)
    n0 = shtlib.launch_count()
    cv = comm_conviqt(nside, lmax, nmaps, bmax, beam, sky)           # host buffers, float32 cube
    assert shtlib.launch_count() > n0
    ref = O.precompute_sky(cpu_oracle, nside, lmax, bmax, sky.alm, cv.alm_beam)
    c64 = np.zeros((2 * bmax, info.np))
    cv.precompute_sky(sky, cube=c64)
    assert rel(c64, ref) <= TOL, rel(c64, ref)
    ulp = np.abs(ref).max() * 2.0 ** -23
    assert cv.c.dtype == np.float32 and np.abs(cv.c.astype(np.float64) - ref).max() <= ulp
    # device-resident: sky a_lm, beam table and cube in HBM
    dev = torch.device("cuda", 0)
    skyd = comm_map(info, device=dev)
    skyd.alm.copy_(torch.as_tensor(sky.alm))
    cvd = comm_conviqt(nside, lmax, nmaps, bmax, beam, skyd, device=dev)
    assert np.array_equal(cvd.c.cpu().numpy(), cv.c)
    c64d = torch.zeros((2 * bmax, info.np), dtype=torch.float64, device=dev)
    cvd.precompute_sky(skyd, cube=c64d)
    assert np.array_equal(c64d.cpu().numpy(), c64)


def test_axisymmetric_beam_known_answer(shtlib):
    """nside 256 / lmax 512 (no oracle needed): a beam with only b_l0 = sqrt((2l+1)/4pi) B_l gives, in every psi
    plane, the sky smoothed with B_l -- the convolution theorem, checked against comm_map%Y."""
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    nside, lmax, bmax = 256, 512, 4
    rng = np.random.default_rng(5)
    info = comm_mapinfo(None, nside, lmax, 1, False)
    sky, beam = comm_map(info), comm_map(info)
    sky.alm[...] = rng.standard_normal(sky.alm.shape)
    l, m = info.lm[0].astype(np.float64), info.lm[1]
    B = np.exp(-0.5 * l * (l + 1) * math.radians(1.0) ** 2)
    beam.alm[0, m == 0] = (np.sqrt((2 * l + 1) / (4 * math.pi)) * B)[m == 0]
    cv = comm_conviqt(nside, lmax, 1, bmax, beam, sky)
    c64 = np.zeros((2 * bmax, info.np))
    cv.precompute_sky(sky, cube=c64)
    b32 = np.zeros(lmax + 1)
    b32[info.lm[0][m == 0]] = cv.alm_beam[:, 0].real.astype(np.float64)[(info.lm[0] * (info.lm[0] + 1) // 2)[m == 0]]
    ref = comm_map(info)
    ref.alm[0] = sky.alm[0] * (b32 / np.sqrt((2 * np.arange(lmax + 1) + 1) / (4 * math.pi)))[info.lm[0]]
    ref.Y()
    for k in range(2 * bmax):
        assert rel(c64[k], ref.map[0]) <= 1e-12


def test_beam_rotation_shifts_psi(shtlib):
    """nside 512 / lmax 1000, IQU, bmax 8: turning the beam by a quarter turn about its axis (b_lm -> i^m b_lm,
    exact in single precision) shifts the cube by psisteps/4 planes.  A size-independent property of the whole
    chain get_alms -> spin-j synthesis -> psi transform."""
    import torch
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    dev = torch.device("cuda", 0)
    nside, lmax, bmax = 512, 1000, 8
    info = comm_mapinfo(None, nside, lmax, 3, True)
    rng = np.random.default_rng(6)
    sky = comm_map(info, device=dev)
    sky.alm.copy_(torch.as_tensor(rng.standard_normal((3, info.nalm))))
    beam = comm_map(info)
    beam.alm[...] = rng.standard_normal(beam.alm.shape) / (1.0 + info.lm[0])
    cv = comm_conviqt(nside, lmax, 3, bmax, beam, sky, device=dev)
    c0 = torch.zeros((2 * bmax, info.np), dtype=torch.float64, device=dev)
    cv.precompute_sky(sky, cube=c0)
    # (re, im) of b_lm times i^m in the real-packed layout: m odd swaps the pair with a sign
    l, m = info.lm[0], info.lm[1]
    rot = beam.alm.copy()
    pos = np.nonzero(m > 0)[0]
    re, im = beam.alm[:, pos], beam.alm[:, pos + 1]
    q = m[pos] % 4
    rot[:, pos] = np.where(q == 0, re, np.where(q == 1, -im, np.where(q == 2, -re, im)))
    rot[:, pos + 1] = np.where(q == 0, im, np.where(q == 1, re, np.where(q == 2, -im, -re)))
    beam2 = comm_map(info)
    beam2.alm[...] = rot
    cv2 = comm_conviqt(nside, lmax, 3, bmax, beam2, sky, device=dev)
    c1 = torch.zeros_like(c0)
    cv2.precompute_sky(sky, cube=c1)
    shift = (2 * bmax) // 4
    want = torch.roll(c0, -shift, dims=0)
    assert float((c1 - want).norm() / want.norm()) <= 1e-12
    assert float(c0.norm()) > 0 and float((c1 - c0).norm() / c0.norm()) > 1e-3


def test_cube_vs_golden(shtlib):
    """The committed conviqt cubes (dense definitional spin-j matrices, tests/golden/make_golden.py) through the C ABI."""
    import glob
    import os
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    paths = sorted(glob.glob(os.path.join(gold, "conviqt_*.npz")))
    assert paths
    for path in paths:
        g = np.load(path)
        nside, lmax, bmax = int(g["nside"]), int(g["lmax"]), int(g["bmax"])
        info = comm_mapinfo(None, nside, lmax, 3, True)
        sky, beam = comm_map(info), comm_map(info)
        sky.alm[...] = g["sky_alm"]
        beam.alm[...] = g["beam_alm"]
        cv = comm_conviqt(nside, lmax, 3, bmax, beam, sky, precompute=False)
        c64 = np.zeros((2 * bmax, info.np))
        cv.precompute_sky(sky, cube=c64)
        assert rel(c64, g["cube"]) <= TOL, (path, rel(c64, g["cube"]))
