"""Spin 2 as scalar sums, on the host (tests/host_emul/emul_s2scalar.cpp, built from the product's legendre_core.cuh and
coef.cpp): the banded map from (E, B) to the two scalar coefficient sequences reproduces the spin-2 recurrences of the
synthesis kernel, north and south, at lmax 4000 / nside 2048 on rings with sin(theta) >= S2S_MIN_STH for small m, m near
the ring's cut-off and m near lmax; and the analysis map is its exact transpose."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NSIDE, LMAX = 2048, 4000
S2S_MIN_STH = 0.05   # legendre_core.cuh


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_s2scalar.cpp")
    coef = os.path.join(ROOT, "commander_b200", "csrc", "coef.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_s2scalar.so")
    hdrs = [os.path.join(ROOT, "commander_b200", "csrc", h) for h in ("legendre_core.cuh", "sht_internal.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src, coef] + hdrs):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src, coef, "-lpthread"])
    L = C.CDLL(so)
    L.emul_s2s_synth.argtypes = [C.c_int] * 4 + [C.c_void_p] * 3
    L.emul_s2s_adjoint.argtypes = [C.c_int] * 2 + [C.c_void_p] * 4
    return L


def ring_sth_cth(nside, north):
    if north < nside:
        omc = north * north / (3.0 * nside * nside)
    else:
        omc = 1.0 - (2.0 * nside - north) * 2.0 / (3.0 * nside)
    return math.sqrt(omc * (2.0 - omc)), 1.0 - omc


def mlim(lmax, spin, sth, cth):   # legendre_core.cuh mlim_for_ring
    ofs = max(lmax * 0.01, 100.0)
    b = -2 * spin * abs(cth)
    t1 = lmax * sth + ofs
    c = spin * spin - t1 * t1
    discr = b * b - 4 * c
    if discr <= 0:
        return lmax
    return int(min((-b + math.sqrt(discr)) / 2.0, lmax) + 0.5)


def first_nonpolar_ring(nside):
    north = 1
    while ring_sth_cth(nside, north)[0] < S2S_MIN_STH:
        north += 1
    return north


@pytest.mark.parametrize("north", ["first", 160, 400, 1000, 1800, 2 * NSIDE])
def test_scalar_route_matches_spin2_recurrence(emul, north):
    if north == "first":
        north = first_nonpolar_ring(NSIDE)
    sth, cth = ring_sth_cth(NSIDE, north)
    assert sth >= S2S_MIN_STH
    ml = mlim(LMAX, 2, sth, cth)
    ms = sorted({0, 1, 2, 3, ml, max(ml - 7, 4)} | ({LMAX - 3, LMAX} if ml >= LMAX else set()))
    rng = np.random.default_rng(north)
    errs, vals = [], []
    for m in ms:
        E = rng.standard_normal(2 * (LMAX + 1))
        B = rng.standard_normal(2 * (LMAX + 1))
        if m == 0:
            E[1::2] = 0.0
            B[1::2] = 0.0
        out = np.zeros(16)
        emul.emul_s2s_synth(NSIDE, LMAX, m, north, E.ctypes.data, B.ctypes.data, out.ctypes.data)
        direct, route = out[:8], out[8:]
        errs.append(np.max(np.abs(route - direct)))
        vals.append(np.max(np.abs(direct)))
    top = max(vals)
    assert top > 0
    worst = max(errs) / top
    assert worst <= 1e-12, f"ring {north} (sin {sth:.4f}): max error {worst:.2e} of the largest value, m = {ms}"


@pytest.mark.parametrize("m", [0, 1, 2, 3, 57, 1000, 3998])
def test_analysis_map_is_the_transpose(emul, m):
    rng = np.random.default_rng(m + 1)
    E = rng.standard_normal(2 * (LMAX + 1))
    B = rng.standard_normal(2 * (LMAX + 1))
    T = rng.standard_normal(4 * (LMAX + 3 - m))
    out = np.zeros(2)
    emul.emul_s2s_adjoint(LMAX, m, E.ctypes.data, B.ctypes.data, T.ctypes.data, out.ctypes.data)
    assert abs(out[0] - out[1]) <= 1e-13 * abs(out[0]), out
