"""CPU tests of the host-side logic: the C ABI library loads and exports every symbol the
header declares (no compute calls without a GPU), descriptor arithmetic, the comm_mapinfo
layout mirror, and a host emulation of the device Legendre math."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from oracle import sht_def as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol(shtlib):
    hdr = open(os.path.join(ROOT, "include", "cmdr_sht.h")).read()
    declared = set(re.findall(r"\b((?:sharp|cmdr_sht|cmdr_cr)_[a-zA-Z0-9_]+)\s*\(", hdr))
    declared -= {"sharp_alm_info", "sharp_geom_info"}
    assert len(declared) >= 23
    L = shtlib.lib()
    for sym in sorted(declared):
        assert hasattr(L, sym), f"libcmdr_sht.so does not export {sym}"
    assert set(shtlib.ABI_SYMBOLS) == declared
    assert L.cmdr_sht_version() >= 100


def test_library_is_sm100a_only():
    lib = os.path.join(ROOT, "commander_b200", "lib", "libcmdr_sht.so")
    if not os.path.exists(lib):
        pytest.skip("library not built")
    # the toolkit commander_b200/csrc/Makefile builds with when it is not on PATH
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-lelf", lib], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_descriptor_counts(shtlib):
    sharp = shtlib
    for lmax, ms in ((0, None), (5, None), (12, [0, 3, 6, 9, 12]), (12, [1, 4, 7, 10]), (7, [])):
        ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
        assert ai.n_local == D.alm_count(lmax, range(lmax + 1) if ms is None else ms)
        sharp.sharp_destroy_alm_info(ai)
    for nside, rings in ((1, None), (2, None), (8, None), (8, [1, 31, 16]), (4, D.mapinfo_rings(4, 2, 5)), (4, [])):
        gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
        assert gi.n_local == D.map_size(nside, range(1, 4 * nside) if rings is None else rings)
        sharp.sharp_destroy_geom_info(gi)


def test_comm_mapinfo_layout_matches_reference_rules(shtlib):
    """commander3/src/comm_map_mod.f90:193-261, 1213-1262."""
    from commander_b200.comm_map import comm_mapinfo

    class FakeComm:
        handle = None

        def __init__(self, rank, size):
            self.rank, self.size = rank, size
    nside, lmax, P = 8, 21, 3
    seen_pix, seen_lm = [], set()
    for r in range(P):
        info = comm_mapinfo(FakeComm(r, P), nside, lmax, 3, True)
        assert list(info.rings) == D.mapinfo_rings(nside, r, P)
        assert list(info.ms) == D.mapinfo_ms(lmax, r, P)
        assert info.np == D.map_size(nside, info.rings) and info.nalm == D.alm_count(lmax, info.ms)
        assert np.all(np.diff(info.pix) > 0)
        seen_pix.append(info.pix)
        idx = D.alm_index(lmax, info.ms)
        for i, (l, m) in enumerate(idx):
            assert info.i2lm(i) == (l, m) and info.lm2i(l, m) == i
            seen_lm.add((l, m))
        assert info.lm2i(lmax + 1, 0) == -1 and info.lm2i(3, 4) == -1
        other_m = (r + 1) % P
        assert info.lm2i(max(other_m, 1) + P * 0 + (0 if other_m else P), other_m if other_m else 0) in (-1, info.lm2i(P, 0))
        li, mi = info.lm[0], info.lm[1]
        assert np.array_equal(info.lm2i_vec(li, mi), np.arange(info.nalm))
        info.dealloc()
    assert np.array_equal(np.sort(np.concatenate(seen_pix)), np.arange(12 * nside ** 2))
    assert len(seen_lm) == (lmax + 1) ** 2


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_legendre.cpp")
    coef = os.path.join(ROOT, "commander_b200", "csrc", "coef.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul.so")
    hdrs = [os.path.join(ROOT, "commander_b200", "csrc", h) for h in ("legendre_core.cuh", "sht_internal.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src, coef] + hdrs):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src, coef, "-lpthread"])
    L = C.CDLL(so)
    L.emul_lambda.argtypes = [C.c_int] * 5 + [C.c_void_p, C.c_void_p]
    L.emul_lambda_front.argtypes = [C.c_int] * 5 + [C.c_void_p, C.c_void_p]

    def front(lmax, m, nside, north, force_row):
        P = np.zeros(lmax + 1); M = np.zeros(lmax + 1)
        lb = L.emul_lambda_front(lmax, m, nside, north, force_row, P.ctypes.data, M.ctypes.data)
        return lb, P, M

    def run(spin, lmax, m, nside, north):
        P = np.zeros(lmax + 1); M = np.zeros(lmax + 1)
        L.emul_lambda(spin, lmax, m, nside, north, P.ctypes.data, M.ctypes.data)
        return P, M
    run.front = front
    return run


def test_device_recurrence_math_spin0(emul):
    """The product's g-scaled recurrence + 2^512 scale bookkeeping (legendre_core.cuh, coef.cpp),
    executed on the host, against the reference's recurrence (math_tools.f90:926-1028)."""
    for nside, lmax in ((64, 200), (256, 700)):
        for m in (0, 1, 2, 3, 17, 100, 199, lmax):
            for north in (1, 2, nside // 2, nside, nside + 1, 2 * nside - 1, 2 * nside):
                cth, sth, *_ = D.healpix_ring(nside, north)
                ref = D.comp_normalised_Plm(lmax, m, math.atan2(sth, cth))
                P, _ = emul(0, lmax, m, nside, north)
                # values whose scaled recurrence variable is below 2^-70 are (deliberately) not accumulated
                # by the product (libsharp2 starts at 2^-60): absolute floor 1e-19
                assert np.max(np.abs(P - ref)) <= 2e-12 * max(np.max(np.abs(ref)), 1e-30) + 1e-19


def test_device_recurrence_math_spin0_two_l_per_step(emul):
    """The transform kernels' spin-0 form -- recurrence in x^2, two l per step, lambda of both parities rebuilt
    from the mix rows (coef.cpp fill_spin0_x2, legendre_core.cuh step0x2; the scheme libsharp2 uses for scalar
    transforms) -- against the reference's recurrence (math_tools.f90:926-1028).  Near the equator the even-l values
    are differences of O(l) larger numbers, hence the looser relative bound than the one-step form."""
    for nside, lmax in ((64, 200), (256, 700), (256, 701)):
        for m in (0, 1, 2, 3, 17, 100, 199, lmax - 1, lmax):
            for north in (1, 2, nside // 2, nside, nside + 1, 2 * nside - 1, 2 * nside):
                cth, sth, *_ = D.healpix_ring(nside, north)
                ref = D.comp_normalised_Plm(lmax, m, math.atan2(sth, cth))
                P, _ = emul(-1, lmax, m, nside, north)
                assert np.max(np.abs(P - ref)) <= 2e-11 * max(np.max(np.abs(ref)), 1e-30) + 1e-19, (nside, lmax, m, north)


def test_device_recurrence_math_spin2(emul):
    import mpmath as mp
    mp.mp.dps = 400
    nside, lmax = 32, 150
    for m in (0, 1, 2, 3, 40, 120, 150):
        for north in (1, 3, 20, 32, 50, 64):
            cth, sth, *_ = D.healpix_ring(nside, north)
            P, M = emul(2, lmax, m, nside, north)
            for l in (max(m, 2), max(m, 2) + 1, max(m, 2) + 7, 100, 149, 150):
                if l > lmax or l < max(m, 2):
                    continue
                rp, rm = float(D.slam(l, m, 2, cth, sth)), float(D.slam(l, m, -2, cth, sth))
                sc = max(abs(rp), abs(rm))
                assert abs(P[l] - rp) <= 1e-11 * sc + 1e-19 and abs(M[l] - rm) <= 1e-11 * sc + 1e-19


def test_spin2_scalar_front_on_host(emul):
    """The scalar front phase of the spin-2 kernels (legendre_core.cuh spin2_from_scalar / spin2_front_convert,
    legendre.cu spin2_front_phase): scalar two-l-per-step recurrence, conversion to the two spin-2 recurrences at a tile
    boundary -- natural hand-over and forced early ones (another ring of the warp got there first) -- against the plain
    spin-2 recurrence for rings with sin(theta) >= 0.15 (the kernels' FRONT_MIN_STH), and against the definitional
    Wigner-d values."""
    import mpmath as mp
    mp.mp.dps = 60
    nside, lmax = 512, 1000
    used = 0
    for m in (4, 7, 35, 120, 300, 600, 900):
        for north in (100, 128, 200, 400, 512, 700, 1000):
            cth, sth, *_ = D.healpix_ring(nside, north)
            if sth < 0.15:
                continue
            P, M = emul(2, lmax, m, nside, north)
            for force in (-1, 0, 8, 64, 200):
                lb, Pf, Mf = emul.front(lmax, m, nside, north, force)
                if lb < 0:          # ring starts above the threshold: the kernels take the plain path
                    continue
                both = (P != 0) & (Pf != 0)
                if not both.any():
                    continue
                used += 1
                sc = max(np.abs(P[both]).max(), np.abs(M[both]).max())
                assert np.abs(P - Pf)[both].max() <= 2e-11 * sc and np.abs(M - Mf)[both].max() <= 2e-11 * sc, (m, north, force)
                if force == -1 and north in (128, 512):
                    l = int(np.nonzero(both)[0][0]) + 3
                    rp, rm = float(D.slam(l, m, 2, cth, sth)), float(D.slam(l, m, -2, cth, sth))
                    assert abs(Pf[l] - rp) <= 1e-10 * max(abs(rp), abs(rm)) and abs(Mf[l] - rm) <= 1e-10 * max(abs(rp), abs(rm))
    assert used > 40


def test_recurrence_variants_random_sweep(emul):
    """Random (nside, lmax, m, ring) up to nside 2048 / lmax 4000: the two-l-per-step spin-0 form against the one-step
    form (which the tests above pin to the reference's recurrence), and the scalar front phase of the spin-2 kernels
    against the plain spin-2 recurrence, natural and forced hand-over points.  Absolute floor 3e-15: a ring joins the
    accumulation at a group boundary (8 l), and near l = m the functions grow by up to 2^20 per group, so both forms
    drop values of that size around the joining point -- each in its own way."""
    rng = np.random.default_rng(20261018)
    n0 = n2 = 0
    for _ in range(500):
        nside = int(rng.choice([16, 64, 256, 1024, 2048]))
        lmax = min(4000, int(rng.integers(4, 3 * nside + 1)))
        m = int(rng.integers(0, lmax + 1))
        north = int(rng.integers(1, 2 * nside + 1)) if rng.random() < 0.8 else int(2 * nside - rng.integers(0, 4))
        P, _ = emul(0, lmax, m, nside, north)
        Q, _ = emul(-1, lmax, m, nside, north)
        assert np.isfinite(Q).all()
        both = (P != 0) & (Q != 0)
        if both.any():
            n0 += 1
            assert np.abs(P - Q)[both].max() <= 2e-11 * np.abs(P[both]).max() + 3e-15, (nside, lmax, m, north)
        cth, sth, *_ = D.healpix_ring(nside, north)
        if m < 4 or sth < 0.15:
            continue
        P, M = emul(2, lmax, m, nside, north)
        force = int(rng.choice([-1, -1, 0, 2, 8, int(rng.integers(0, (lmax - m) // 2 + 1))]))
        lb, Pf, Mf = emul.front(lmax, m, nside, north, force)
        if lb < 0:
            continue
        assert np.isfinite(Pf).all() and np.isfinite(Mf).all()
        both = (P != 0) & (Pf != 0)
        if both.any():
            n2 += 1
            sc = max(np.abs(P[both]).max(), np.abs(M[both]).max())
            assert max(np.abs(P - Pf)[both].max(), np.abs(M - Mf)[both].max()) <= 2e-11 * sc + 3e-15, (nside, lmax, m, north, force)
            if force == -1:     # the seeded path must not join later than the plain one by more than a group
                assert np.nonzero(Pf)[0][0] <= np.nonzero(P)[0][0] + 8
    assert n0 > 300 and n2 > 40


@pytest.mark.parametrize("spin", [1, 3, 5])
def test_device_recurrence_math_arbitrary_spin(emul, spin):
    """start_spin_s + the spin-s coefficient tables (conviqt, commander3/src/comm_conviqt_mod.f90:234-239)
    against the definitional (+-s)lambda_lm of the oracle (mpmath Wigner d)."""
    import mpmath as mp
    mp.mp.dps = 400
    nside, lmax = 32, 120
    for m in (0, 1, spin - 1, spin, spin + 1, 40, 119):
        for north in (1, 3, 20, 32, 50, 64):
            cth, sth, *_ = D.healpix_ring(nside, north)
            P, M = emul(spin, lmax, m, nside, north)
            l0 = max(m, spin)
            for l in (l0, l0 + 1, l0 + 6, 90, 119, 120):
                if l > lmax or l < l0:
                    continue
                rp, rm = float(D.slam(l, m, spin, cth, sth)), float(D.slam(l, m, -spin, cth, sth))
                sc = max(abs(rp), abs(rm))
                assert abs(P[l] - rp) <= 1e-11 * sc + 1e-19 and abs(M[l] - rm) <= 1e-11 * sc + 1e-19, (m, north, l)


@pytest.mark.parametrize("spin", [8, 17, 31, 32])
def test_device_recurrence_math_high_spin(emul, spin):
    """start_spin_s (plain powers of sin / cos(theta/2) for m < s) and the spin-s coefficient tables up to
    CMDR_MAX_SPIN = 32 at lmax 1000, every l, against the independent mpmath reference of tests/slam_ref.py."""
    import slam_ref as R
    nside, lmax = 512, 1000
    worst = 0.0
    for m in sorted({0, 1, spin - 1, spin, spin + 1, 40, 500, 999, lmax}):
        for north in (1, 3, 40, 256, 512, 700, 1024):
            cth, sth = R.ring_trig(nside, north)
            P, M = emul(spin, lmax, m, nside, north)
            rp = R.slam_column(lmax, m, spin, cth, sth)
            rm = R.slam_column(lmax, m, -spin, cth, sth)
            sc = max(np.abs(rp).max(), np.abs(rm).max())
            if sc == 0:
                assert not P.any() and not M.any()
                continue
            l0 = max(m, spin)
            assert not P[:l0].any() and not M[:l0].any()
            err = max(np.abs(P - rp).max(), np.abs(M - rm).max())
            # ring 1 (sin theta = 0.003): the start values use sin / cos(theta/2) of the exact ring, the recurrence the
            # float64 z = cos(theta), whose rounding moves theta by up to 2^-53 / (1 - z) / 2 relative, i.e. up to
            # ~(m + s) * 4e-11 here; the reference is evaluated at arccos(z)
            eps = 2e-9 if sth < 0.01 else 1e-11
            worst = max(worst, (err - 1e-19) / sc)
            assert err <= eps * sc + 1e-19, (m, north, err / sc)
    print(f"spin {spin}: worst |delta| / max|lambda| {worst:.2e}")


@pytest.mark.parametrize("spin,m,north", [(31, 193, 63), (31, 199, 64), (16, 193, 63), (32, 200, 63)])
def test_high_spin_start_above_threshold_joins(emul, spin, m, north):
    """m >= s with fewer than 8 l left: Ksm (which carries 2^s) lifts the start values over the join threshold although
    sin^(m-s) alone is below it.  start_spin_s must join at once -- the recurrences check only every 8 l, so these
    values (up to 4e-11 at nside 64 / lmax 200) came out as 0 before."""
    import slam_ref as R
    nside, lmax = 64, 200
    cth, sth = R.ring_trig(nside, north)
    P, M = emul(spin, lmax, m, nside, north)
    rp, rm = R.slam_column(lmax, m, spin, cth, sth), R.slam_column(lmax, m, -spin, cth, sth)
    sc = max(np.abs(rp).max(), np.abs(rm).max())
    assert sc > 1e-17
    assert max(np.abs(P - rp).max(), np.abs(M - rm).max()) <= 1e-11 * sc + 1e-19


@pytest.fixture(scope="module")
def emul_fft():
    """tests/host_emul/emul_bluefft.cpp: the product's blue_fft.cuh executed on the host."""
    src = os.path.join(ROOT, "tests", "host_emul", "emul_bluefft.cpp")
    hdr = os.path.join(ROOT, "commander_b200", "csrc", "blue_fft.cuh")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_bluefft.so")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    L = C.CDLL(so)
    L.emul_fft.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.emul_fft2.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.emul_conv2.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.emul_bitrev.argtypes = [C.c_uint, C.c_int]
    L.emul_bitrev.restype = C.c_uint
    return L


@pytest.mark.parametrize("M", [4, 8, 16, 32, 1024, 2048, 4096, 8192])
def test_blue_fft_pair_on_host(emul_fft, M):
    """DIF forward = numpy FFT in bit-reversed order; DIT inverse of a bit-reversed spectrum = M * ifft; and the
    circular convolution u -> DIT(DIF(u) .* V_bitrev) the fused Bluestein kernels rely on."""
    rng = np.random.default_rng(M)
    bits = M.bit_length() - 1
    br = np.array([emul_fft.emul_bitrev(i, bits) for i in range(M)])
    assert np.array_equal(br[br], np.arange(M))
    x = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    for nthreads in (1, 7, 256):
        y = x.copy()
        emul_fft.emul_fft(y.ctypes.data, M, 0, nthreads)
        ref = np.fft.fft(x)
        assert np.abs(y - ref[br]).max() <= 1e-12 * np.abs(ref).max()
        z = y.copy()
        emul_fft.emul_fft(z.ctypes.data, M, 1, nthreads)
        assert np.abs(z - M * x).max() <= 1e-12 * M * np.abs(x).max()
    v = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    V = np.fft.fft(v)
    u = x.copy()
    emul_fft.emul_fft(u.ctypes.data, M, 0, 64)
    u *= V[br]
    emul_fft.emul_fft(u.ctypes.data, M, 1, 64)
    conv = np.fft.ifft(np.fft.fft(x) * V) * M
    assert np.abs(u - conv).max() <= 1e-11 * np.abs(conv).max()


def test_chain_order_round_trip(shtlib):
    """alm <-> chain-file order l^2+l+m (commander3/src/comm_map_mod.f90:712-739, 860-889), one rank and the two ranks of a
    round-robin split: the ranks' arrays add up to the single-rank one."""
    from commander_b200.comm_map import comm_map, comm_mapinfo
    from commander_b200.dist import Comm
    lmax, nside = 11, 4
    rng = np.random.default_rng(0)
    info = comm_mapinfo(None, nside, lmax, 3, True)
    m = comm_map(info)
    m.alm[...] = rng.standard_normal(m.alm.shape)
    full = m.alm_to_chain_order(dtype=np.float64)
    assert full.shape == ((lmax + 1) ** 2, 3)
    for i in range(info.nalm):
        l, mm = info.i2lm(i)
        assert np.array_equal(full[l * l + l + mm], m.alm[:, i])
    assert m.alm_to_chain_order().dtype == np.float32
    parts = []
    for r in range(2):
        ir = comm_mapinfo(Comm(r, 2, 9), nside, lmax, 3, True)
        mr = comm_map(ir)
        mr.alm_from_chain_order(full)
        for i in range(ir.nalm):
            l, mm = ir.i2lm(i)
            assert np.array_equal(mr.alm[:, i], full[l * l + l + mm])
        parts.append(mr.alm_to_chain_order(dtype=np.float64))
    assert np.array_equal(parts[0] + parts[1], full)
    back = comm_map(info)
    back.alm_from_chain_order(full)
    assert np.array_equal(back.alm, m.alm)


def test_empty_and_single_ring_handles(shtlib):
    """A rank may own no m or no ring at all (sharp_execute is then called with null pointers, SURVEY 8b); handles for
    empty lists and for a single unpaired ring are valid and report their sizes.  Host only: no compute call."""
    sharp = shtlib
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(10, ms=np.zeros(0, dtype=np.int32))
    gi = sharp.sharp_make_healpix_geom_info(4, rings=np.zeros(0, dtype=np.int32))
    assert ai.n_local == 0 and gi.n_local == 0
    eq = sharp.sharp_make_healpix_geom_info(4, rings=np.array([8], dtype=np.int32))      # the equator alone
    cap = sharp.sharp_make_healpix_geom_info(4, rings=np.array([1, 15], dtype=np.int32))  # the two polar rings
    assert eq.n_local == 16 and cap.n_local == 8
    one_m = sharp.sharp_make_mmajor_real_packed_alm_info(10, ms=np.array([10], dtype=np.int32))
    assert one_m.n_local == 2
    for h in (ai, one_m):
        sharp.sharp_destroy_alm_info(h)
    for h in (gi, eq, cap):
        sharp.sharp_destroy_geom_info(h)


@pytest.mark.parametrize("M", [1024, 2048, 4096, 8192])
def test_blue_fft_register_blocked_variant_on_host(emul_fft, M):
    """The register-blocked, padded FFT pair (3-4 stages per pass, bf2_* schedule) computes the same bit-reversed
    spectrum and the same inverse as numpy; slots i + (i >> 4) + (i >> 8) hold element i, the pad slots are never touched."""
    rng = np.random.default_rng(M + 1)
    bits = M.bit_length() - 1
    br = np.array([emul_fft.emul_bitrev(i, bits) for i in range(M)])
    idx = np.arange(M) + (np.arange(M) >> 4) + (np.arange(M) >> 8)
    nslots = M + M // 16 + M // 256 + 1                       # bf_padded(M)
    x = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    for nthreads in (1, 5, 512):
        buf = np.full(nslots, 7.0 + 3.0j)
        buf[idx] = x
        emul_fft.emul_fft2(buf.ctypes.data, M, 0, nthreads)
        ref = np.fft.fft(x)
        assert np.abs(buf[idx] - ref[br]).max() <= 1e-12 * np.abs(ref).max()
        emul_fft.emul_fft2(buf.ctypes.data, M, 1, nthreads)
        assert np.abs(buf[idx] - M * x).max() <= 1e-12 * M * np.abs(x).max()
        pad = np.setdiff1d(np.arange(nslots), idx)
        assert np.all(buf[pad] == 7.0 + 3.0j)
    # the whole convolution as the kernel sequences it (strided DIF passes, in-register middle with the bit-reversed
    # filter spectrum, strided DIT passes)
    v = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    V = np.fft.fft(v)
    vbr = np.ascontiguousarray(V[br])
    buf = np.full(nslots, 7.0 + 3.0j)
    buf[idx] = x
    emul_fft.emul_conv2(buf.ctypes.data, vbr.ctypes.data, M, 33)
    conv = np.fft.ifft(np.fft.fft(x) * V) * M
    assert np.abs(buf[idx] - conv).max() <= 1e-11 * np.abs(conv).max()


def test_add_alm_set_alm_loops(shtlib):
    """add_alm / set_alm (commander3/src/comm_map_mod.f90:1167-1211) against the Fortran loops written out:
    for i in info: (l,m) = info%i2lm(i); j = self%info%lm2i(l,m); skip j == -1; q <= min(nmaps)."""
    from commander_b200 import comm_map, comm_mapinfo
    rng = np.random.default_rng(17)
    big = comm_mapinfo(None, 4, 11, 3, True)
    small = comm_mapinfo(None, 4, 6, 1, False)
    for self_info, other in ((big, small), (small, big)):
        m = comm_map(self_info)
        m.alm[:] = rng.standard_normal(m.alm.shape)
        alm = rng.standard_normal((other.nmaps, other.nalm))
        q = min(self_info.nmaps, other.nmaps)
        want_add, want_set = m.alm.copy(), m.alm.copy()
        for i in range(other.nalm):
            l, mm = other.i2lm(i)
            j = self_info.lm2i(l, mm)
            if j == -1:
                continue
            want_add[:q, j] += alm[:q, i]
            want_set[:q, j] = alm[:q, i]
        a = comm_map(self_info); a.alm[:] = m.alm
        a.add_alm(alm, other)
        assert np.array_equal(a.alm, want_add)
        s = comm_map(self_info); s.alm[:] = m.alm
        s.set_alm(alm, other)
        assert np.array_equal(s.alm, want_set)
        # alm_equal, :1148-1165
        o = comm_map(other)
        o.alm[:] = 7.0
        m.alm_equal(o)
        want = np.zeros_like(o.alm)
        for i in range(other.nalm):
            l, mm = other.i2lm(i)
            j = self_info.lm2i(l, mm)
            if j != -1:
                want[:q, i] = m.alm[:q, j]
        assert np.array_equal(o.alm, want)


@pytest.fixture(scope="module")
def emul_ring():
    """tests/host_emul/emul_ringsplit.cpp: ring_split.cuh + blue_fft.cuh sequenced as ring_split_kernel / ring_pow2_kernel do."""
    src = os.path.join(ROOT, "tests", "host_emul", "emul_ringsplit.cpp")
    hdrs = [os.path.join(ROOT, "commander_b200", "csrc", h) for h in ("blue_fft.cuh", "ring_split.cuh")]
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_ringsplit.so")
    if not os.path.exists(so) or os.path.getmtime(so) < max([os.path.getmtime(src)] + [os.path.getmtime(h) for h in hdrs]):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src])
    L = C.CDLL(so)
    L.emul_ring_split.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.emul_ring_pow2.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.emul_ring_half.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    return L


@pytest.mark.parametrize("i,M", [(1, 1024), (3, 1024), (129, 1024), (512, 1024), (513, 2048), (1000, 2048), (1025, 4096),
                                 (1531, 4096), (2047, 4096)])
def test_ring_split_transform_on_host(emul_ring, i, M):
    """A cap ring of n = 4 i points through four length-i chirp-z transforms of work length M and one radix-4 pass:
    both directions against numpy's FFT of the whole ring (every i of the classes the kernel serves, incl. primes)."""
    n = 4 * i
    rng = np.random.default_rng(i)
    Z = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    x = np.empty(n, dtype=np.complex128)
    emul_ring.emul_ring_split(Z.ctypes.data, x.ctypes.data, n, M, 0)
    ref = np.fft.ifft(Z) * n
    assert np.abs(x - ref).max() <= 2e-12 * np.abs(ref).max()
    F = np.empty(n, dtype=np.complex128)
    emul_ring.emul_ring_split(Z.ctypes.data, F.ctypes.data, n, M, 1)
    ref = np.fft.fft(Z)
    assert np.abs(F - ref).max() <= 2e-12 * np.abs(ref).max()


@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192])
def test_ring_pow2_transform_on_host(emul_ring, n):
    rng = np.random.default_rng(n)
    Z = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    x = np.empty(n, dtype=np.complex128)
    emul_ring.emul_ring_pow2(Z.ctypes.data, x.ctypes.data, n, 0)
    ref = np.fft.ifft(Z) * n
    assert np.abs(x - ref).max() <= 1e-12 * np.abs(ref).max()
    emul_ring.emul_ring_pow2(Z.ctypes.data, x.ctypes.data, n, 1)
    ref = np.fft.fft(Z)
    assert np.abs(x - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("n", [2048, 4096, 8192, 16384])
def test_ring_half_transform_on_host(emul_ring, n):
    """One ring of n real samples through one complex transform of length n / 2 (ring_half_kernel: even / odd sample
    packing, ring_split.cuh rh_pack / rh_unpack) against numpy's real FFTs, both directions."""
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n)
    X = np.fft.fft(x)                       # Hermitian spectrum, e^{-} convention
    out = np.empty(n)
    Xs = np.ascontiguousarray(X / 1.0)
    emul_ring.emul_ring_half(Xs.ctypes.data, out.ctypes.data, n, 0)
    assert np.abs(out - n * x).max() <= 1e-12 * n * np.abs(x).max()
    F = np.empty(n, dtype=np.complex128)
    emul_ring.emul_ring_half(x.ctypes.data, F.ctypes.data, n, 1)
    assert np.abs(F - X).max() <= 1e-12 * np.abs(X).max()
