"""SHARP_ALM2MAP_DERIV1 without a GPU: the gradient reference (tests/deriv_ref.py) against mpmath.diff and against the
spin-1 identity, the kernels' parity-split accumulate (legendre_core.cuh) in host emulation against the plain spin-1
form, and the argument checks of sharp.alm2map_der1."""
import ctypes as C
import math
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

from oracle import sht_def as D

import deriv_ref as G
import slam_ref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (l, m, theta): m = 0, near-pole theta, the equator, l = m
CASES = [(1, 0, 0.7), (5, 0, 1e-3), (6, 3, 0.4), (6, 6, 2.9), (12, 1, 1e-4), (40, 17, math.pi / 2), (80, 2, 3.1),
         (25, 25, 0.05)]


def _lam(l, m, theta):
    sgn = -1 if m % 2 else 1
    return sgn * mp.sqrt(mp.mpf(2 * l + 1) / (4 * mp.pi)) * D.wigner_d(l, -m, 0, mp.cos(theta / 2), mp.sin(theta / 2))


@pytest.mark.parametrize("l,m,theta", CASES)
def test_gradient_relation_matches_mpmath_diff(l, m, theta):
    cth, sth = math.cos(theta), math.sin(theta)
    g = G.grad_columns(l, m, cth, sth)
    with mp.workdps(40):
        th = mp.atan2(mp.mpf(sth), mp.mpf(cth))
        dref = float(mp.diff(lambda t: _lam(l, m, t), th))
        mref = float(m * _lam(l, m, th) / mp.sin(th))
    scale = max(abs(dref), abs(mref), 1e-300)
    assert abs(g[0, l] - dref) <= 1e-13 * scale, (g[0, l], dref)
    assert abs(g[1, l] - mref) <= 1e-13 * scale, (g[1, l], mref)


@pytest.mark.parametrize("nside,ring,lmax,m", [(64, 1, 150, 0), (64, 1, 150, 3), (64, 40, 150, 0), (64, 100, 150, 77),
                                               (512, 2, 300, 1), (512, 1023, 300, 150), (512, 2047, 300, 12)])
def test_gradient_relation_matches_spin1_identity(nside, ring, lmax, m):
    cth, sth = R.ring_trig(nside, ring)
    g = G.grad_columns(lmax, m, cth, sth)
    p = R.slam_column(lmax, m, 1, cth, sth)
    q = R.slam_column(lmax, m, -1, cth, sth)
    l = np.arange(lmax + 1, dtype=np.float64)
    f = np.sqrt(l * (l + 1))
    d_id, m_id = -f * (p - q) / 2, f * (p + q) / 2
    for got, want in ((g[0], d_id), (g[1], m_id)):
        scale = max(float(np.abs(want).max()), 1e-300)
        assert float(np.abs(got - want).max()) <= 1e-12 * scale
    assert g[0, 0] == 0.0 and g[1, 0] == 0.0


@pytest.fixture(scope="module")
def emul_d1():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_deriv1.cpp")
    coef = os.path.join(ROOT, "commander_b200", "csrc", "coef.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_deriv1.so")
    deps = [src, coef, os.path.join(ROOT, "commander_b200", "csrc", "legendre_core.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src, coef, "-lpthread"])
    L = C.CDLL(so)
    L.emul_d1_phases.argtypes = [C.c_int] * 4 + [C.c_void_p] * 4
    return L


def test_parity_split_accumulate_on_host(emul_d1):
    """Random sweep over (nside <= 2048, lmax <= 4000, m, ring): the 4-FMA parity-split sums and their epilogue give the
    phases of the 8-FMA spin-1 (cp, cm) form to 1e-13 of the largest phase."""
    rng = np.random.default_rng(11)
    worst, n = 0.0, 0
    for _ in range(300):
        nside = int(2 ** rng.integers(2, 12))
        lmax = int(rng.integers(2, min(4000, 4 * nside) + 1))
        m = int(rng.integers(0, lmax + 1)) if rng.random() < 0.8 else int(rng.integers(0, 3))
        north = int(rng.integers(1, 2 * nside + 1))
        c = rng.standard_normal(2 * (lmax + 1))
        d1, ref, ab = np.zeros(8), np.zeros(8), np.zeros(1)
        emul_d1.emul_d1_phases(lmax, m, nside, north, c.ctypes.data, d1.ctypes.data, ref.ctypes.data, ab.ctypes.data)
        assert np.all(np.isfinite(d1))
        scale = float(np.abs(ref).max())
        err = float(np.abs(d1 - ref).max())
        assert err <= 1e-13 * scale + 1e-16 * ab[0], (nside, lmax, m, north, err, scale)
        if scale > 0:
            worst = max(worst, err / scale)
            n += 1
    assert n > 100
    print(f"\nparity-split accumulate: worst {worst:.2e} of the largest phase over {n} (ring, m)")


def test_alm2map_der1_rejects_wrong_shapes(shtlib):
    sharp = shtlib
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(8)
    gi = sharp.sharp_make_healpix_geom_info(4)
    try:
        alm = np.zeros((1, ai.n_local))
        mp2 = np.zeros((2, gi.n_local))
        for a, m in ((np.zeros((2, ai.n_local)), mp2),                 # two a_lm columns
                     (np.zeros(ai.n_local), mp2),                       # 1-d a_lm
                     (alm, np.zeros((1, gi.n_local))),                  # one map
                     (alm, np.zeros((3, gi.n_local))),
                     (alm.astype(np.float32), mp2),                     # dtypes
                     (alm, mp2.astype(np.float32)),
                     (alm, np.zeros((2, gi.n_local + 1))),              # sizes
                     (np.zeros((1, ai.n_local - 1)), mp2),
                     (alm, np.zeros((gi.n_local, 2)).T)):               # not C-contiguous
            with pytest.raises(ValueError):
                sharp.alm2map_der1(a, ai, m, gi)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_iqu_entry_points_reject_deriv1(shtlib):
    """The fused IQU calls carry three-column pointer tables; DERIV1 (one a_lm column, two maps) is refused before the
    library is called, as the library itself aborts on it."""
    sharp = shtlib
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(8)
    gi = sharp.sharp_make_healpix_geom_info(4)
    try:
        alm, mp3 = np.zeros((3, ai.n_local)), np.zeros((3, gi.n_local))
        for t in (sharp.SHARP_ALM2MAP_DERIV1, -1, 5):
            with pytest.raises(ValueError):
                sharp.execute_iqu(t, alm, mp3, gi, gi, ai)
            with pytest.raises(ValueError):
                sharp.execute_iqu(t, alm, mp3, gi, gi, ai, comm=7)
            with pytest.raises(ValueError):
                sharp.execute_iqu_batch(t, [alm], [mp3], gi, gi, ai)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)
