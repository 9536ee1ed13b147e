"""The conviqt sampler without a GPU: the per-sample psi lookup of commander_b200/csrc/conviqt_interp.cuh (what
conviqt_interp_kernel runs) compiled with g++ against oracle/conviqt.py interp (commander3/src/comm_conviqt_mod.f90:
155-205) bit for bit, and the local -> RING placement of the full-sky table against comm_mapinfo's pixel lists
(tests/host_emul/emul_conviqt_interp.cpp)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_conviqt_interp.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_conviqt_interp.so")
    deps = [src, os.path.join(ROOT, "commander_b200", "csrc", "conviqt_interp.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror",
                               "-ffp-contract=off", "-o", so, src])
    L = C.CDLL(so)
    vp = C.c_void_p
    L.emul_conviqt_interp.argtypes = [vp, C.c_longlong, C.c_int, C.c_int, C.c_longlong, vp, vp, vp]
    L.emul_conviqt_psires.argtypes = [C.c_int]
    L.emul_conviqt_psires.restype = C.c_float
    L.emul_conviqt_check_rings.argtypes = [C.c_int, C.c_int, vp, vp, C.c_int, C.c_char_p, C.c_int]
    L.emul_conviqt_check_rings.restype = C.c_int
    L.emul_conviqt_scatter.argtypes = [C.c_int, C.c_int, vp, vp, C.c_longlong, vp, vp]
    L.emul_conviqt_scatter.restype = C.c_longlong
    return L


def _interp(L, tab, bmax, optim, pix, psi):
    tab = np.ascontiguousarray(tab, dtype=np.float32)
    pix = np.ascontiguousarray(pix, dtype=np.int32)
    psi = np.ascontiguousarray(psi, dtype=np.float32)
    out = np.empty(pix.size, dtype=np.float32)
    L.emul_conviqt_interp(tab.ctypes.data, tab.shape[1], bmax, optim, pix.size, pix.ctypes.data, psi.ctypes.data,
                          out.ctypes.data)
    return out


def _angles(rng, bmax, n):
    """n float32 angles: uniform over a few turns, plus the special ones -- 0, -0, +-2 pi (float32 and float64), exact
    multiples of psires (in float32 and as float64 products), tiny negatives and positives, |psi| >> 2 pi."""
    f = np.float32
    psisteps = 2 * bmax
    psires = f(2.0 * math.pi / psisteps)
    special = [0.0, -0.0, f(2 * math.pi), -f(2 * math.pi), 2 * math.pi, -2 * math.pi, f(4 * math.pi), -f(6 * math.pi)]
    k = np.arange(-3 * psisteps, 3 * psisteps + 1)
    special += list((k.astype(f) * psires).astype(f)) + list(k * (2.0 * math.pi / psisteps))
    tiny = [-1e-38, -1e-30, -1e-12, -1e-7, -2.4e-7, -5e-7, -np.float32(1.4e-45), 1e-38, 1e-30, 1e-12, 1e-7, 2e-7, 2.4e-7,
            5e-7]
    big = [1e3, -1e3, 12345.678, -98765.4, 1e6, -1e6, 3.3e7, -3.3e7, 1e10, -1e20]
    special += tiny + big
    s = np.array(special, dtype=np.float64).astype(f)
    m = n - s.size
    u = rng.uniform(-4 * math.pi, 4 * math.pi, m // 2)
    near = (rng.integers(-4 * psisteps, 4 * psisteps, m // 4) * (2 * math.pi / psisteps)
            + rng.standard_normal(m // 4) * 1e-6)                              # next to the bin edges
    wide = np.exp(rng.uniform(-20, 25, m - m // 2 - m // 4)) * rng.choice([-1.0, 1.0], m - m // 2 - m // 4)
    return np.concatenate([s, u.astype(f), near.astype(f), wide.astype(f)])


@pytest.mark.parametrize("bmax", [1, 3, 8, 32])
@pytest.mark.parametrize("optim", [0, 2])
def test_interp_matches_oracle_bitwise(emul, bmax, optim):
    from oracle import conviqt as O
    rng = np.random.default_rng(1000 * bmax + optim)
    psisteps, npix, n = 2 * bmax, 12 * 4 ** 2, 100_000
    c = rng.standard_normal((psisteps, npix)).astype(np.float32)
    c[:, 0] = -0.0
    c[0, 1] = 3.0e38
    pix = rng.integers(0, npix, n).astype(np.int32)
    psi = _angles(rng, bmax, n)
    assert emul.emul_conviqt_psires(psisteps) == np.float32(2.0 * math.pi / psisteps)
    out = _interp(emul, c, bmax, optim, pix, psi)
    # where modulo(-psi, 2 pi) rounds up to 2 pi the reference reads row psisteps, one past the cube: the sampler reads
    # row 0 there, i.e. the oracle on the cube with row 0 repeated after the last row
    c_ext = np.concatenate([c, c[:1]])
    ref = np.empty(n, dtype=np.float32)
    edge = []
    with np.errstate(over="ignore"):                       # the weights of pixel 1 overflow to inf, in both
        for i in range(n):
            try:
                ref[i] = O.interp(c, psisteps, int(pix[i]), psi[i], optim)
            except IndexError:
                edge.append(i)
                ref[i] = O.interp(c_ext, psisteps, int(pix[i]), psi[i], optim)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), np.nonzero(out.view(np.uint32) != ref.view(np.uint32))
    assert optim == 2 or psisteps & (psisteps - 1) or edge     # tiny positive psi hits the edge for powers of two
    assert all(0.0 < psi[i] < 1e-6 for i in edge), psi[edge]
    e = np.array([i for i in edge if pix[i] != 1], dtype=np.int64)       # (pixel 1 overflows in the weights)
    assert np.all(np.abs(out[e] - c[0, pix[e]]) <= 1e-6 * np.abs(c[0, pix[e]]))


def test_interp_outside_the_sky_and_non_finite_angles(emul):
    bmax, npix = 2, 48
    c = np.arange(4 * npix, dtype=np.float32).reshape(4, npix)
    pix = np.array([-1, npix, -2 ** 31, 2 ** 31 - 1, 0, 5, 5, 5], dtype=np.int32)
    psi = np.array([0.5, 0.5, 0.5, 0.5, 0.5, np.nan, np.inf, -np.inf], dtype=np.float32)
    for optim in (0, 2):
        out = _interp(emul, c, bmax, optim, pix, psi)
        assert np.all(np.isnan(out[[0, 1, 2, 3, 5, 6, 7]])) and np.isfinite(out[4])


def _rings(info):
    return [int(r) for r in info.rings]


def _check(emul, nside, rings_of, whole=True):
    nr = np.array([len(r) for r in rings_of], dtype=np.int32)
    flat = np.array([x for r in rings_of for x in r] or [0], dtype=np.int32)
    err = C.create_string_buffer(512)
    ok = emul.emul_conviqt_check_rings(nside, len(rings_of), nr.ctypes.data, flat.ctypes.data, int(whole), err, len(err))
    return bool(ok), err.value.decode()


@pytest.mark.parametrize("nside", [1, 2, 16, 64])
def test_scatter_reproduces_comm_mapinfo_pixels(shtlib, emul, nside):
    from commander_b200.comm_map import comm_mapinfo
    from commander_b200.dist import Comm
    npix = 12 * nside ** 2
    for P in range(1, 9):
        infos = [comm_mapinfo(Comm(r, P, 900 + P), nside, 2 * nside, 1, False) for r in range(P)]
        rings_of = [_rings(i) for i in infos]
        assert _check(emul, nside, rings_of) == (True, "")
        stride = max(max(i.np for i in infos), 1) + 3          # padded blocks of the all-gather
        nr = np.array([len(r) for r in rings_of], dtype=np.int32)
        flat = np.array([x for r in rings_of for x in r], dtype=np.int32)
        owner = np.empty(npix, dtype=np.int32)
        local = np.empty(npix, dtype=np.int64)
        nruns = emul.emul_conviqt_scatter(nside, P, nr.ctypes.data, flat.ctypes.data, stride, owner.ctypes.data,
                                          local.ctypes.data)
        assert nruns >= 4 * nside - 1
        assert owner.min() >= 0                                  # every global pixel receives exactly one local pixel
        for r, info in enumerate(infos):
            assert np.array_equal(owner[info.pix], np.full(info.np, r))
            assert np.array_equal(local[info.pix], np.arange(info.np))
        for i in infos:
            i.dealloc()


def test_scatter_follows_the_geometry_ring_order(emul):
    """A full-sky geometry given in another ring order: the local pixels follow that order (running sum of nph)."""
    from commander_b200.comm_map import _in_ring_count, _ring_start
    nside = 4
    rings = list(range(4 * nside - 1, 0, -1))
    pix = np.concatenate([np.arange(_ring_start(nside, r), _ring_start(nside, r) + _in_ring_count(nside, r)) for r in rings])
    owner = np.empty(12 * nside ** 2, dtype=np.int32)
    local = np.empty(12 * nside ** 2, dtype=np.int64)
    nr = np.array([len(rings)], dtype=np.int32)
    flat = np.array(rings, dtype=np.int32)
    emul.emul_conviqt_scatter(nside, 1, nr.ctypes.data, flat.ctypes.data, pix.size, owner.ctypes.data, local.ctypes.data)
    assert np.array_equal(local[pix], np.arange(pix.size)) and np.all(owner == 0)


@pytest.mark.parametrize("rings_of,whole,msg", [
    ([[1, 2], [3]], True, ""),
    ([[1, 2], []], True, "ring 3 held by no rank"),
    ([[1, 2], [2, 3]], True, "ring 2 held twice"),
    ([[1, 1]], False, "ring 1 held twice"),
    ([[0]], False, "ring 0 outside 1..3"),
    ([[4]], False, "ring 4 outside 1..3"),
    ([[1]], False, ""),
])
def test_ring_checks(emul, rings_of, whole, msg):
    ok, err = _check(emul, 1, rings_of, whole)
    assert ok == (msg == "") and err.startswith(msg)


def test_nside_beyond_32bit_pixels_is_refused(emul):
    ok, err = _check(emul, 13378, [[1]], False)
    assert not ok and "32-bit" in err
    assert _check(emul, 13377, [[1]], False)[0]


def test_symbols_exported(shtlib):
    L = shtlib.lib()
    for sym in ("cmdr_sht_conviqt_sampler", "cmdr_sht_conviqt_interp", "cmdr_sht_conviqt_sampler_destroy"):
        assert sym in shtlib.ABI_SYMBOLS
        getattr(L, sym)


def test_python_argument_checks(shtlib):
    geom = shtlib.sharp_make_healpix_geom_info(2)
    try:
        with pytest.raises(ValueError, match="cube must be"):
            shtlib.conviqt_sampler(np.zeros((4, 48), dtype=np.float32), 3, geom)
        with pytest.raises(ValueError, match="cube must be"):
            shtlib.conviqt_sampler(np.zeros((6, 48), dtype=np.float16), 3, geom)
        with pytest.raises(ValueError, match="pix must be"):
            shtlib.conviqt_interp(None, np.zeros(4, dtype=np.int64), np.zeros(4, dtype=np.float32), 0,
                                  np.zeros(4, dtype=np.float32))
        with pytest.raises(ValueError, match="same length"):
            shtlib.conviqt_interp(None, np.zeros(4, dtype=np.int32), np.zeros(3, dtype=np.float32), 0,
                                  np.zeros(4, dtype=np.float32))
    finally:
        shtlib.sharp_destroy_geom_info(geom)
