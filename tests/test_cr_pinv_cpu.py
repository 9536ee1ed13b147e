"""The host side of the pseudo-inverse preconditioner of the native multi-component constrained-realisation system without
a GPU (commander_b200/csrc/cr_pinv.h and check_cr_pseudoinv in cr_plan.h, compiled with g++ through
tests/host_emul/emul_crpinv.cpp): the one-sided Jacobi pseudo-inverse, the U+ / alpha^2 U+ / P P^t tables against the
V of comm_cr.cr_system.initDiffPrecond_pseudoinv written in numpy, and the refusals of cmdr_cr_set_pseudoinv."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "commander_b200", "csrc")
EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_crpinv.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_crpinv.so")
    deps = [src] + [os.path.join(CSRC, h) for h in ("cr_pinv.h", "cr_plan.h", "cr_block.cuh", "sht_internal.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = C.CDLL(so)
    L.emul_cr_pinv_check.restype = C.c_int
    L.emul_cr_pinv_check.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double, C.c_char_p, C.c_int]
    return L


def pinv(L, V):
    V = np.ascontiguousarray(V, dtype=np.float64)
    out = np.zeros(V.shape[::-1])
    L.emul_cr_pinv(V.shape[0], V.shape[1], V.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def shapes():
    for npre in range(1, 17):
        for nb in range(1, 31):
            yield nb, npre


def test_pinv_random(emul):
    rng = np.random.default_rng(1)
    for nb, npre in shapes():
        V = rng.standard_normal((nb + npre, npre))
        assert rel(pinv(emul, V), np.linalg.pinv(V, rcond=max(V.shape) * EPS)) <= 1e-12, (nb, npre)


def test_pinv_zero_and_duplicated_columns(emul):
    rng = np.random.default_rng(2)
    for nb, npre in shapes():
        V = rng.standard_normal((nb + npre, npre))
        z = []
        if npre > 1:
            z = list(rng.choice(npre, size=min(2, npre - 1), replace=False))
            V[:, z] = 0.0
        if npre > 3:
            a, b = [k for k in range(npre) if k not in z][:2]
            V[:, a] = V[:, b]
        got = pinv(emul, V)
        assert rel(got, np.linalg.pinv(V, rcond=max(V.shape) * EPS)) <= 1e-12, (nb, npre)
        assert np.all(got[z] == 0.0)           # a component beyond its lmax gets exactly zero rows
    assert np.all(pinv(emul, np.zeros((5, 3))) == 0.0)


def test_pinv_scaled(emul):
    """The whole matrix scaled by 1e-8 .. 1e8: against numpy.  Columns of their own scales (1e-8 .. 1e8) under an identity
    block, the shape of V: against a 60-digit reference, which numpy's bidiagonalising SVD does not reach."""
    rng = np.random.default_rng(3)
    for (nb, npre), s in zip(shapes(), np.tile(10.0 ** np.arange(-8, 9), 40)):
        V = s * rng.standard_normal((nb + npre, npre))
        assert rel(pinv(emul, V), np.linalg.pinv(V, rcond=max(V.shape) * EPS)) <= 1e-12, (nb, npre, s)
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 60
    worst_np = 0.0
    for t in range(40):
        nb, npre = int(rng.integers(1, 31)), int(rng.integers(1, 17))
        V = np.zeros((nb + npre, npre))
        V[:nb] = rng.standard_normal((nb, npre)) * 10.0 ** rng.uniform(-8, 8, size=npre)
        for k in range(npre):
            if t % 4 or k % 3:
                V[nb + k, k] = 1.0
        sv = np.linalg.svd(V, compute_uv=False)
        if sv.min() <= 100.0 * max(V.shape) * EPS * sv.max():
            continue                                    # a singular value near the cut-off: either choice is right
        M = mp.matrix(V.tolist())
        ref = np.array(((M.T * M) ** -1 * M.T).tolist(), dtype=np.float64)
        assert rel(pinv(emul, V), ref) <= 1e-12, (nb, npre)
        worst_np = max(worst_np, rel(np.linalg.pinv(V, rcond=max(V.shape) * EPS), ref))
    print("numpy.linalg.pinv on graded columns, worst relative error:", worst_np)


def _dp(a):
    return C.cast(a.ctypes.data, C.c_void_p)


def _tables(L, comps, bands, F_mean, alpha):
    nc, nb = len(comps), len(bands)
    lmax_pre = max(c["lmax"] for c in comps)
    nl = max(lmax_pre, max(b["lmax"] for b in bands)) + 1
    nmaps_pre = max(c["nmaps"] for c in comps)
    keep = []

    def arr(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        keep.append(a)
        return a
    Cl = (C.c_void_p * nc)(*[None if c["Cl"] is None else _dp(arr(c["Cl"])) for c in comps])
    bl = (C.c_void_p * nb)(*[_dp(arr(b["b_l"])) for b in bands])
    U = np.zeros((nc, nb, 3, nl))
    UA = np.zeros_like(U)
    PP = np.zeros((nmaps_pre, lmax_pre + 1, nc * (nc + 1) // 2))
    ints = lambda v: (C.c_int * len(v))(*v)   # noqa: E731
    L.emul_cr_pinv_tables(nc, ints([c["nmaps"] for c in comps]), ints([c["lmax"] for c in comps]), Cl, nb,
                          ints([b["nmaps"] for b in bands]), ints([b["lmax"] for b in bands]), bl, _dp(arr(F_mean)),
                          _dp(arr(alpha)), _dp(U), _dp(UA), _dp(PP))
    return U, UA, PP


def _numpy_tables(comps, bands, F_mean, alpha):
    """The V loop of cr_system.initDiffPrecond_pseudoinv (and tests/test_gpu_cr_multi.py::_oracle_pseudoinv), per band
    nmaps, then numpy's pinv."""
    nc, nb = len(comps), len(bands)
    lmax_pre = max(c["lmax"] for c in comps)
    nmaps_pre = max(c["nmaps"] for c in comps)
    M = np.zeros((nmaps_pre, lmax_pre + 1, nc, nb + nc))
    for j in range(nmaps_pre):
        for l in range(lmax_pre + 1):
            V = np.zeros((nb + nc, nc))
            for q, b in enumerate(bands):
                if l > b["lmax"] or j >= b["nmaps"]:
                    continue
                for k, c in enumerate(comps):
                    if l > c["lmax"] or j >= c["nmaps"]:
                        continue
                    V[q, k] = alpha[q, j] * b["b_l"][l, j] * F_mean[q, k, j]
                    if c["Cl"] is not None:
                        V[q, k] *= 0.0 if (j > 0 and l < 2) else np.sqrt(c["Cl"][l, j])
            for k, c in enumerate(comps):
                if c["Cl"] is not None and l <= c["lmax"] and j < c["nmaps"]:
                    V[nb + k, k] = 1.0
            M[j, l] = np.linalg.pinv(V, rcond=max(V.shape) * EPS)
    return M


def test_tables_against_numpy(emul):
    """Components: 3 maps / lmax 40 with prior; 3 maps / lmax 24 with prior; 1 map / lmax 8 without prior.  Bands: 3 maps
    / lmax 32; 1 map / lmax 20; 3 maps / lmax 48 (beyond every component).  Covers polarisation l < 2, l beyond lmax_k or
    lmax_q, 1-map bands and components, and a component without prior."""
    rng = np.random.default_rng(4)
    l = np.arange(49, dtype=np.float64)
    comps = [dict(nmaps=3, lmax=40, Cl=np.stack([40.0 / (l * (l + 1) + 1.0)] * 3, axis=1)[:41]),
             dict(nmaps=3, lmax=24, Cl=np.stack([8.0 / (l + 1.0) ** 2.5] * 3, axis=1)[:25]),
             dict(nmaps=1, lmax=8, Cl=None)]
    bands = []
    for nm, lmax, fwhm in ((3, 32, 600.0), (1, 20, 700.0), (3, 48, 300.0)):
        sigma = fwhm * np.pi / 180.0 / 60.0 / np.sqrt(8.0 * np.log(2.0))
        bl = np.exp(-0.5 * l[:lmax + 1, None] * (l[:lmax + 1, None] + 1) * sigma ** 2) * np.array([1.0, 1.02, 1.02])
        bands.append(dict(nmaps=nm, lmax=lmax, b_l=bl))
    F_mean = rng.uniform(0.3, 2.5, size=(3, 3, 3))
    alpha = rng.uniform(0.5, 3.0, size=(3, 3))
    alpha[1, 1:] = 0.0                                   # what compute_alpha_nu leaves for a 1-map band
    U, UA, PP = _tables(emul, comps, bands, F_mean, alpha)
    M = _numpy_tables(comps, bands, F_mean, alpha)
    nc, nb, lmax_pre = 3, 3, 40
    for j in range(3):
        for q in range(nb):
            ref = M[j, :, :, q].T                          # (k, l)
            assert rel(U[:, q, j, :lmax_pre + 1], ref) <= 1e-12 or np.abs(ref).max() == 0.0
            assert np.abs(U[:, q, j, :lmax_pre + 1] - ref).max() <= 1e-12 * np.abs(M).max()
            np.testing.assert_allclose(UA[:, q, j, :lmax_pre + 1], alpha[q, j] ** 2 * U[:, q, j, :lmax_pre + 1], rtol=1e-15)
        for ll in range(lmax_pre + 1):
            P = M[j, ll][:, nb:]
            ref = P @ P.T
            got = np.array([[PP[j, ll, (min(a, b) * nc - min(a, b) * (min(a, b) - 1) // 2 + abs(a - b))] for b in range(nc)]
                            for a in range(nc)])
            assert np.abs(got - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()), (j, ll)
    assert np.all(U[:, :, :, lmax_pre + 1:] == 0.0)
    assert np.all(U[2, :, 1:] == 0.0)                     # the 1-map component has no Q, U rows
    assert np.all(U[:, 1, 1:] == 0.0)                     # nor the 1-map band Q, U columns
    assert np.all(U[1, :, :, 25:] == 0.0) and np.all(U[2, :, :, 9:] == 0.0)   # beyond lmax_k: exactly zero
    assert np.all(U[:, 1, :, 21:] == 0.0)                 # beyond lmax_q
    assert np.all(U[:2, :, 1:, :2] == 0.0)                # polarisation l < 2 carries no signal, only the prior row
    assert np.all(PP[1:, :, 5] == 0.0)                    # the component without prior has no Q, U


def check(L, multi, ncomp, need=0.0, free=1e12):
    err = C.create_string_buffer(512)
    ok = L.emul_cr_pinv_check(multi, ncomp, need, free, err, len(err))
    return bool(ok), err.value.decode()


def test_refusals(emul):
    assert check(emul, 1, 3) == (True, "")
    assert check(emul, 1, 16, 1e9, 1e9) == (True, "")
    assert check(emul, 0, 1) == (
        False, "needs a handle of cmdr_cr_setup_multi (give a one-component system to cmdr_cr_setup_multi with ncomp = 1)")
    assert check(emul, 1, 17) == (False, "ncomp 17 above the pseudo-inverse preconditioner's limit of 16")
    assert check(emul, 1, 3, 2048.0, 1024.0) == (
        False, "the pseudo-inverse preconditioner needs 2048 bytes of device memory, 1024 are free")


def test_symbol_exported(shtlib):
    assert "cmdr_cr_set_pseudoinv" in shtlib.ABI_SYMBOLS
    getattr(shtlib.lib(), "cmdr_cr_set_pseudoinv")
