"""Deterministic analysis without a GPU: the partials indexing, the ordered reduce and the warp-block cut of pipelined
launches of commander_b200/csrc/det.h, compiled with g++ (tests/host_emul/emul_det.cpp).  Every a_lm slot must be
reduced over every block that stored it exactly once, in ascending block order, on the layouts and geometries the
transforms take; every work slot must fall into exactly one launch of a chunked analysis."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DET_EMPTY = 0x7FFFFFFF


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_det.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_det.so")
    deps = [src, os.path.join(ROOT, "commander_b200", "csrc", "det.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror", "-o", so, src])
    L = C.CDLL(so)
    L.emul_det_check.restype = C.c_int
    return L


def _layout(ms, lmax, kind):
    """(mvstart, ndst in doubles) of a real-packed, complex (with gaps, as sharp_make_general_alm_info allows) or
    scalar-sum scratch layout"""
    mvs, pos = [], 0
    for i, m in enumerate(ms):
        if kind == "real":
            mvs.append(pos if m == 0 else pos - 2 * m)
            pos += (lmax + 1) if m == 0 else 2 * (lmax + 1 - m)
        elif kind == "complex":
            mvs.append(pos - m)
            pos += lmax + 1 - m + (i % 3)       # gaps between the m columns
        else:
            mvs.append(0)
            pos += 2 * 2 * ((lmax - m) // 2 + 1)
    ndst = 2 * pos if kind == "complex" else pos
    return mvs, ndst


def _check(L, nslots, bs, ms, lmax, spin, kind, ncomp, seed):
    rng = np.random.default_rng(seed)
    nb = (nslots + bs - 1) // bs
    first = np.empty((nb, len(ms)), dtype=np.int32)
    for b in range(nb):
        for i, m in enumerate(ms):
            l0 = max(m, spin)
            first[b, i] = DET_EMPTY if rng.uniform() < 0.25 else rng.integers(l0, lmax + 1)
    mvs, ndst = _layout(ms, lmax, kind)
    ms_c = np.ascontiguousarray(ms, dtype=np.int32)
    mvs_c = np.ascontiguousarray(mvs, dtype=np.int64)
    r = L.emul_det_check(nslots, bs, len(ms), ms_c.ctypes.data_as(C.c_void_p), mvs_c.ctypes.data_as(C.c_void_p),
                         int(kind == "real"), int(kind == "s2s"), lmax, spin, ncomp,
                         np.ascontiguousarray(first).ctypes.data_as(C.c_void_p), C.c_longlong(ndst))
    assert r == 0, f"check {r}"


CASES = [  # (name, nslots, ms, lmax)
    ("full sky nside 64", 128, list(range(0, 129)), 128),
    ("ring subset with and without mirrors", 37, list(range(0, 61)), 60),
    ("m subset without m = 0", 300, list(range(1, 90, 3)), 90),
    ("single ring", 1, list(range(0, 20)), 19),
    ("single m", 700, [7], 50),
    ("lmax > 3 nside - 1", 16, list(range(0, 41)), 40),
]


@pytest.mark.parametrize("name,nslots,ms,lmax", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("kind", ["real", "complex"])
def test_every_slot_reduced_once_in_order(emul, name, nslots, ms, lmax, kind):
    _check(emul, nslots, 256, ms, lmax, 0, kind, 1, 1)        # anal0_kernel: 8 ring pairs per lane
    _check(emul, nslots, 128, ms, lmax, 2, kind, 2, 2)        # anal2_kernel: 4 per lane, E and B


@pytest.mark.parametrize("name,nslots,ms,lmax", CASES, ids=[c[0] for c in CASES])
def test_scalar_sum_scratch(emul, name, nslots, ms, lmax):
    _check(emul, nslots, 256, ms, lmax + 2, 0, "s2s", 2, 3)   # spin 2 as two scalar sums up to lmax + 2


def _cuts(L, nslots, bs, wcut):
    nch = len(wcut) - 1
    w = np.ascontiguousarray(wcut, dtype=np.int32)
    owner = np.empty(nslots, dtype=np.int32)
    b = np.empty(nch, dtype=np.int32)
    e = np.empty(nch, dtype=np.int32)
    L.emul_det_cut(nslots, bs, nch, w.ctypes.data_as(C.c_void_p), owner.ctypes.data_as(C.c_void_p),
                   b.ctypes.data_as(C.c_void_p), e.ctypes.data_as(C.c_void_p))
    return owner, b, e


def _check_cuts(L, nslots, bs, wcut):
    owner, b, e = _cuts(L, nslots, bs, wcut)
    assert np.all(owner >= 0), "a slot in no launch or in two"
    assert np.all((b % bs == 0) | (b == e))
    chunk_of = np.searchsorted(wcut, np.arange(nslots), side="right") - 1
    for s0 in range(0, nslots, bs):
        last = min(s0 + bs, nslots) - 1
        blk = owner[s0:last + 1]
        assert np.all(blk == blk[0]), "a block split between launches"
        assert blk[0] == chunk_of[last] or (chunk_of[last] < len(wcut) - 2 and blk[0] > chunk_of[last]), \
            "a straddling block not in the later launch"


@pytest.mark.parametrize("bs", [128, 256])
@pytest.mark.parametrize("seed", range(8))
def test_pipelined_cuts(emul, bs, seed):
    """Work-slot chunk cuts like those of the distributed pipeline (chunks of a few slots to a few thousand, some empty,
    the last ones empty too): every slot in exactly one launch, launches on block boundaries, a block that straddles two
    chunks in the later launch only."""
    rng = np.random.default_rng(seed)
    nslots = int(rng.integers(1, 5000))
    k = int(rng.integers(1, 9))
    inner = np.sort(rng.integers(0, nslots + 1, size=k - 1))
    if seed % 2:
        inner[-(k // 2 + 1):] = nslots if k > 1 else inner[-1:]   # empty final chunks
    _check_cuts(emul, nslots, bs, np.concatenate([[0], inner, [nslots]]))


@pytest.mark.parametrize("wcut", [[0, 300, 1000, 1000], [0, 1000, 1000, 1000], [0, 0, 0, 1000], [0, 1000]])
def test_empty_final_chunk(emul, wcut):
    """nslots not a multiple of the block: the tail block is launched once, by the last chunk, even when that is empty."""
    owner, b, e = _cuts(emul, 1000, 256, wcut)
    assert np.all(owner >= 0)
    assert e[-1] == 1000 and np.all(e[:-1] % 256 == 0)
    _check_cuts(emul, 1000, 256, wcut)
