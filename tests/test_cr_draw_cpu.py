"""The draw stream of the constrained-realisation fluctuation terms without a GPU: commander_b200/csrc/rng.cuh compiled
with g++ against its known answers and against the numpy restatement oracle/rng.py, the local -> global ring table of
cr_draw.h against comm_mapinfo's pixel lists, and the argument checks of cmdr_cr_compute_rhs_draw
(tests/host_emul/emul_rng.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "commander_b200", "csrc")

# Philox4x32-10 known answers: (counter, key) -> output words
KAT = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_rng.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_rng.so")
    deps = [src] + [os.path.join(CSRC, f) for f in ("rng.cuh", "cr_draw.h", "conviqt_interp.cuh", "sht_internal.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror",
                               "-ffp-contract=off", "-o", so, src])
    L = C.CDLL(so)
    vp, ull, u32 = C.c_void_p, C.c_ulonglong, C.c_uint32
    L.emul_philox.argtypes = [C.c_longlong, vp, u32, u32, vp]
    L.emul_gauss.argtypes = [C.c_longlong, vp, vp]
    L.emul_eta_pix.argtypes = [ull, ull, C.c_uint, C.c_uint, C.c_longlong, vp, vp]
    L.emul_eta_alm.argtypes = [ull, ull, C.c_uint, C.c_uint, C.c_longlong, vp, vp, vp]
    L.emul_ring_table.argtypes = [C.c_int, C.c_int, vp, vp, vp, vp]
    L.emul_ring_table.restype = C.c_int
    L.emul_check_draw.argtypes = [C.c_int, C.c_char_p, C.c_int]
    L.emul_check_draw.restype = C.c_int
    L.emul_draw_words.argtypes = [ull, ull, C.c_int, C.c_int, vp]
    return L


def _philox(L, ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    out = np.empty_like(ctr)
    L.emul_philox(ctr.shape[0], ctr.ctypes.data, key[0], key[1], out.ctypes.data)
    return out


def test_philox_known_answers(emul):
    from oracle import rng
    for ctr, key, want in KAT:
        assert tuple(int(w) for w in _philox(emul, [ctr], key)[0]) == want
        assert tuple(int(w) for w in rng.philox4x32_10(ctr, key)) == want


def test_words_and_gaussians_match_the_oracle(emul):
    """10^6 counters: every Philox word equal; the Gaussians within 1e-13 (libm cos against numpy cos)."""
    from oracle import rng
    r = np.random.default_rng(5)
    n = 1_000_000
    ctr = r.integers(0, 2 ** 32, size=(n, 4), dtype=np.uint64).astype(np.uint32)
    ctr[:4] = [[0, 0, 0, 0], [0xffffffff] * 4, [1, 2, 3, 4], [0x80000000, 0, 0, 0]]
    key = (0x9e3779b9, 0x12345678)
    w = _philox(emul, ctr, key)
    wo = np.stack(rng.philox4x32_10(tuple(ctr[:, i] for i in range(4)), key), axis=1).astype(np.uint32)
    assert np.array_equal(w, wo)
    g = np.empty(n)
    emul.emul_gauss(n, np.ascontiguousarray(w).ctypes.data, g.ctypes.data)
    go = rng.gauss(tuple(wo[:, i].astype(np.uint64) for i in range(4)))
    assert np.all(np.isfinite(g))
    assert np.max(np.abs(g - go)) < 1e-13
    # the extreme words: u1 = 2^-53 (largest |eta|) and u1 = 1 (eta = 0)
    ext = np.array([[0, 0, 0, 0], [0xffffffff, 0xffffffff, 0, 0]], dtype=np.uint32)
    emul.emul_gauss(2, ext.ctypes.data, g.ctypes.data)
    assert g[0] == pytest.approx(np.sqrt(2 * 53 * np.log(2.0)), rel=1e-15) and g[1] == 0.0


@pytest.mark.parametrize("seed,draw", [(0, 0), (1234, 7), (2 ** 64 - 1, 2 ** 63 + 5), (0xdeadbeef00000001, 2 ** 32)])
def test_pixel_and_prior_draws_match_the_oracle(emul, seed, draw):
    from oracle import rng
    pix = np.concatenate([np.arange(5000), [12 * 8192 ** 2 - 1, 2 ** 31, 2 ** 32 - 1]]).astype(np.uint32)
    out = np.empty(pix.size)
    for q, j in [(0, 0), (0, 2), (29, 1), (2 ** 20, 2)]:
        emul.emul_eta_pix(seed, draw, q, j, pix.size, pix.ctypes.data, out.ctypes.data)
        assert np.max(np.abs(out - rng.eta_pix(seed, draw, q, j, pix))) < 1e-13
    lmax = 60
    ls = np.concatenate([np.full(2 * l + 1, l) for l in range(lmax + 1)]).astype(np.int32)
    ms = np.concatenate([np.arange(-l, l + 1) for l in range(lmax + 1)]).astype(np.int32)
    out = np.empty(ls.size)
    for k, j in [(0, 0), (1, 2), (15, 1)]:
        emul.emul_eta_alm(seed, draw, k, j, ls.size, ls.ctypes.data, ms.ctypes.data, out.ctypes.data)
        assert np.max(np.abs(out - rng.eta_alm(seed, draw, k, j, ls, ms))) < 1e-13


def test_columns_are_distinct_streams():
    """The pixel column of (q, j), the prior column of (k, j) and the draw index each select a different stream."""
    from oracle import rng
    idx = np.arange(4096)
    streams = [rng.eta_pix(1, 0, 0, 0, idx), rng.eta_pix(1, 0, 0, 1, idx), rng.eta_pix(1, 0, 1, 0, idx),
               rng.eta_pix(1, 1, 0, 0, idx), rng.eta_pix(2, 0, 0, 0, idx),
               rng.eta_alm(1, 0, 0, 0, np.zeros(4096, dtype=np.int64), idx)]   # l = 0, m_s = idx: index idx
    for a in range(len(streams)):
        for b in range(a):
            assert abs(np.corrcoef(streams[a], streams[b])[0, 1]) < 6 / np.sqrt(idx.size)


def _rings(info):
    return [int(r) for r in info.rings]


@pytest.mark.parametrize("nside", [1, 2, 16, 64])
def test_ring_table_reproduces_comm_mapinfo_pixels(shtlib, emul, nside):
    """Every rank's table (one row per local ring) expands to exactly comm_mapinfo's pixel list, in storage order."""
    from commander_b200.comm_map import comm_mapinfo
    from commander_b200.dist import Comm
    for P in (1, 3, 8):
        infos = [comm_mapinfo(Comm(r, P, 700 + P), nside, 2 * nside, 1, False) for r in range(P)]
        for info in infos:
            rr = np.array(_rings(info), dtype=np.int32)
            n = rr.size
            loc, glob, nph = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int32)
            assert emul.emul_ring_table(nside, n, rr.ctypes.data, loc.ctypes.data, glob.ctypes.data, nph.ctypes.data) == n
            pix = np.full(info.np, -1, dtype=np.int64)
            for a, g, k in zip(loc, glob, nph):
                pix[a:a + k] = g + np.arange(k)
            assert np.array_equal(pix, info.pix)
            assert int(nph.sum()) == info.np
        assert sorted(np.concatenate([i.pix for i in infos]).tolist()) == list(range(12 * nside ** 2))
        for i in infos:
            i.dealloc()


def test_ring_table_follows_the_given_ring_order(emul):
    """A geometry given in another ring order: local pixels follow that order (running sum of nph)."""
    nside = 4
    rr = np.array([9, 1, 15, 4], dtype=np.int32)
    loc, glob, nph = np.empty(4, dtype=np.int64), np.empty(4, dtype=np.int64), np.empty(4, dtype=np.int32)
    emul.emul_ring_table(nside, 4, rr.ctypes.data, loc.ctypes.data, glob.ctypes.data, nph.ctypes.data)
    from commander_b200.comm_map import _in_ring_count, _ring_start
    want_n = [_in_ring_count(nside, int(r)) for r in rr]
    assert nph.tolist() == want_n
    assert loc.tolist() == [0] + list(np.cumsum(want_n)[:-1])
    assert glob.tolist() == [_ring_start(nside, int(r)) for r in rr]


def _check(L, terms):
    err = C.create_string_buffer(256)
    ok = L.emul_check_draw(terms, err, len(err))
    return bool(ok), err.value.decode()


@pytest.mark.parametrize("terms", [-1, 4, 5, 1 << 30, -(1 << 31)])
def test_bad_terms_are_refused(emul, terms):
    ok, msg = _check(emul, terms)
    assert not ok and "terms" in msg and "0..3" in msg


@pytest.mark.parametrize("terms", [0, 1, 2, 3])
def test_good_terms_are_accepted(emul, terms):
    assert _check(emul, terms) == (True, "")


def test_rank_comparison_words(emul):
    """The words the ranks compare: non-negative, different whenever seed, draw or terms differ, all -1 on a refusal."""
    def words(seed, draw, terms, ok=1):
        w = np.empty(7, dtype=np.int32)
        emul.emul_draw_words(seed, draw, terms, ok, w.ctypes.data)
        return tuple(int(x) for x in w)
    cases = [(0, 0, 3), (1, 0, 3), (0, 1, 3), (0, 0, 1), (2 ** 64 - 1, 0, 3), (0, 2 ** 64 - 1, 3), (2 ** 63, 0, 3),
             (2 ** 30, 0, 3), (2 ** 60, 0, 3), (0, 2 ** 31, 3), (0x80000000, 0x80000000, 2)]
    seen = {}
    for c in cases:
        w = words(*c)
        assert all(x >= 0 for x in w)
        assert w not in seen, (c, seen.get(w))
        seen[w] = c
    assert words(5, 6, 3, ok=0) == (-1,) * 7
