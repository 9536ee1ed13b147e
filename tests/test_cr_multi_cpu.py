"""The multi-component constrained-realisation system without a GPU: the input checks and slot maps of
cmdr_cr_setup_multi (commander_b200/csrc/cr_plan.h) and the per-slot block arithmetic of its preconditioner
(cr_block.cuh), both compiled with g++ (tests/host_emul/emul_crmulti.cpp), and the argument checks of
comm_cr.cr_native_multi_system."""
import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "commander_b200", "csrc")


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_crmulti.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_crmulti.so")
    deps = [src, os.path.join(CSRC, "cr_plan.h"), os.path.join(CSRC, "cr_block.cuh"), os.path.join(CSRC, "sht_internal.h"),
            os.path.join(ROOT, "include", "cmdr_sht.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = C.CDLL(so)
    L.emul_cr_plan.restype = C.c_int
    L.emul_cr_block.restype = None
    return L


def _ints(v):
    v = [int(x) for x in v]
    return (C.c_int * max(len(v), 1))(*v)


def plan(L, comps, bands, precond=1, device_bytes=1e15):
    """comps: dicts lmax, nmaps, ms [, rp, prior]; bands: dicts lmax, nmaps, ms [, rp, hasP].  Returns (result, error)."""
    cms = [m for c in comps for m in c["ms"]]
    bms = [m for b in bands for m in b["ms"]]
    lmax_all = max([c["lmax"] for c in comps] + [b["lmax"] for b in bands] + [0])
    nl = len(comps) + 2 * len(bands) + 1
    bstart = (C.c_longlong * (nl * (lmax_all + 2)))()
    nalm = (C.c_longlong * nl)()
    lmax = (C.c_int * nl)()
    Ls = (C.c_int * max(len(bands), 1))()
    misc = (C.c_int * 4)()
    nbytes = C.c_double()
    err = C.create_string_buffer(512)
    ok = L.emul_cr_plan(
        len(comps), _ints(c["lmax"] for c in comps), _ints(c["nmaps"] for c in comps), _ints(c.get("rp", 1) for c in comps),
        _ints(len(c["ms"]) for c in comps), _ints(cms), _ints(c.get("prior", 1) for c in comps),
        len(bands), _ints(b["lmax"] for b in bands), _ints(b["nmaps"] for b in bands), _ints(b.get("rp", 1) for b in bands),
        _ints(len(b["ms"]) for b in bands), _ints(bms), _ints(b.get("hasP", 1) for b in bands),
        precond, C.c_double(device_bytes), bstart, nalm, lmax, Ls, misc, C.byref(nbytes), err, len(err))
    if not ok:
        return None, err.value.decode()
    nm = misc[0]
    return dict(nm=nm, lmax_pre=misc[1], nmaps_pre=misc[2], lmax_all=misc[3], L=list(Ls)[:len(bands)],
                bstart=np.array(bstart[:nl * nm]).reshape(nl, nm), nalm=list(nalm), lmax=list(lmax),
                bytes=nbytes.value), ""


def _ms(lmax, rank=0, size=1):
    return list(range(rank, lmax + 1, size))


# ------------------------------------------------------------------ slot maps

@pytest.mark.parametrize("rank,size", [(0, 1), (0, 3), (2, 3), (1, 4)])
def test_slot_maps_match_comm_mapinfo(emul, shtlib, rank, size):
    """Every slot of every layout (components, bands as given, bands at their transform lmax, preconditioner) against
    comm_mapinfo.lm2i_vec of the same layout, for components and bands of differing lmax and m's distributed
    round-robin over `size` ranks."""
    from commander_b200 import comm_mapinfo
    comm = SimpleNamespace(rank=rank, size=size, handle=None)
    comps = [dict(lmax=40, nmaps=3), dict(lmax=32, nmaps=3), dict(lmax=8, nmaps=1)]
    bands = [dict(lmax=32, nmaps=3), dict(lmax=48, nmaps=1), dict(lmax=24, nmaps=3)]
    for d in comps + bands:
        d["ms"] = _ms(d["lmax"], rank, size)
    p, err = plan(emul, comps, bands)
    assert err == "" and p["lmax_pre"] == 40 and p["nmaps_pre"] == 3 and p["lmax_all"] == 48
    assert p["L"] == [32, 40, 24]
    nc, nb = len(comps), len(bands)
    mval = _ms(48, rank, size)
    assert p["nm"] == len(mval)
    layouts = [c["lmax"] for c in comps] + [b["lmax"] for b in bands] + p["L"] + [p["lmax_pre"]]
    assert p["lmax"] == layouts
    for lay, lmax in enumerate(layouts):
        info = comm_mapinfo(comm, 4, lmax, 1, False)
        assert p["nalm"][lay] == info.nalm
        ls, ms, got = [], [], []
        for im, m in enumerate(mval):
            if m > lmax:
                assert p["bstart"][lay, im] == -1
                continue
            for l in range(m, lmax + 1):
                for sgn in ((1,) if m == 0 else (1, -1)):
                    t = l if m == 0 else 2 * (l - m) + (sgn < 0)
                    ls.append(l); ms.append(sgn * m); got.append(p["bstart"][lay, im] + t)
        ref = info.lm2i_vec(np.array(ls), np.array(ms))
        assert (ref >= 0).all() and np.array_equal(np.array(got), ref), lay
    # a band layout at L_q < lmax_q is dense over the band's m's up to L_q
    assert p["nalm"][nc + nb + 1] == comm_mapinfo(comm, 4, 40, 1, False).nalm


def test_block_table_bytes(emul):
    comps = [dict(lmax=20, nmaps=3, ms=_ms(20)), dict(lmax=10, nmaps=1, ms=_ms(10))]
    bands = [dict(lmax=30, nmaps=3, ms=_ms(30))]
    p, _ = plan(emul, comps, bands)
    assert p["bytes"] == 8 * 3 * 3 * 21 * 21          # 3 triangle entries, 3 maps, (lmax_pre + 1)^2 slots
    assert plan(emul, comps, bands, precond=0)[0]["bytes"] == 0


# ------------------------------------------------------------------ refusals

def _ok():
    return [dict(lmax=16, nmaps=3, ms=_ms(16)), dict(lmax=8, nmaps=1, ms=_ms(8), prior=0)], \
           [dict(lmax=12, nmaps=3, ms=_ms(12)), dict(lmax=20, nmaps=1, ms=_ms(20), hasP=0)]


def _refuse(emul, comps, bands, **kw):
    p, err = plan(emul, comps, bands, **kw)
    assert p is None
    return err


def test_valid_input_is_accepted(emul):
    comps, bands = _ok()
    assert plan(emul, comps, bands)[1] == ""
    assert plan(emul, comps, bands, precond=0)[1] == ""


def test_refusals(emul):
    comps, bands = _ok()
    assert _refuse(emul, [], bands) == "ncomp 0 (at least 1)"
    assert _refuse(emul, comps, []) == "nbands 0 (at least 1)"
    assert _refuse(emul, comps, bands, precond=2) == "precond 2 unsupported (0 = none, 1 = block diagonal)"
    assert _refuse(emul, comps, bands, precond=-1) == "precond -1 unsupported (0 = none, 1 = block diagonal)"
    c = [dict(comps[0], nmaps=2)] + comps[1:]
    assert _refuse(emul, c, bands) == "component 0: nmaps 2 unsupported (1 or 3)"
    b = bands[:1] + [dict(bands[1], nmaps=0)]
    assert _refuse(emul, comps, b) == "band 1: nmaps 0 unsupported (1 or 3)"
    c = comps[:1] + [dict(comps[1], rp=0)]
    assert _refuse(emul, c, bands) == "component 1: needs the real-packed a_lm layout of comm_mapinfo"
    b = [dict(bands[0], rp=0)] + bands[1:]
    assert _refuse(emul, comps, b) == "band 0: needs the real-packed a_lm layout of comm_mapinfo"
    c = [dict(comps[0], lmax=-1)] + comps[1:]
    assert _refuse(emul, c, bands) == "component 0: alm_info is NULL"
    b = [dict(bands[0], hasP=0)] + bands[1:]
    assert _refuse(emul, comps, b) == "band 0: geom_P is NULL with nmaps 3"
    c = [dict(comps[0], prior=2)] + comps[1:]
    assert _refuse(emul, c, bands) == "component 0: sqrtS columns must be all NULL (no prior) or all given"


def test_npre_limit(emul):
    _, bands = _ok()
    comps = [dict(lmax=8, nmaps=1, ms=_ms(8)) for _ in range(17)]
    assert _refuse(emul, comps, bands) == "ncomp 17 above the block preconditioner's limit of 16"
    assert plan(emul, comps, bands, precond=0)[1] == ""          # no blocks, no limit
    assert plan(emul, comps[:16], bands)[1] == ""


def test_table_must_fit_device_memory(emul):
    comps, bands = _ok()
    p, _ = plan(emul, comps, bands)
    assert plan(emul, comps, bands, device_bytes=p["bytes"])[1] == ""
    err = _refuse(emul, comps, bands, device_bytes=p["bytes"] - 1)
    assert err == f"the block preconditioner needs {int(p['bytes'])} bytes of device memory, {int(p['bytes']) - 1} are free"
    assert plan(emul, comps, bands, precond=0, device_bytes=0)[1] == ""


def test_mismatched_m_sets(emul):
    comps, bands = _ok()
    # a band from another rank's share of the m's
    b = [dict(bands[0], ms=_ms(12, 1, 2))] + bands[1:]
    assert _refuse(emul, comps, b) == ("band 0: its local m's differ from those of band 1 truncated at lmax 12 (every handle "
                                      "must list this rank's m's in comm_mapinfo's order)")
    # same m's, other order
    c = [dict(comps[0], ms=_ms(16)[::-1])] + comps[1:]
    assert _refuse(emul, c, bands).startswith("component 0: its local m's differ from those of band 1 truncated at lmax 16")
    # one m missing
    c = comps[:1] + [dict(comps[1], ms=_ms(8)[:-1])]
    assert _refuse(emul, c, bands).startswith("component 1: its local m's differ")
    # a rank with no m's at all is fine when every handle agrees
    c = [dict(x, ms=[]) for x in comps]
    b = [dict(x, ms=[]) for x in bands]
    p, err = plan(emul, c, b)
    assert err == "" and p["nm"] == 0 and all(n == 0 for n in p["nalm"])


# ------------------------------------------------------------------ block finish / invert / apply

def _block_ref(M, sS, prior):
    """cr_system.initDiffPrecond_diagonal's per-slot steps in numpy: active set, sqrt(S) both sides, unit prior,
    inverse on the active set, identity elsewhere."""
    n = M.shape[0]
    act = np.diag(M) > 0
    s = np.where(prior, sS, 1.0)
    A = M * s[:, None] * s[None, :]
    A = A + np.diag((act & prior).astype(float))
    full = np.where(act[:, None] & act[None, :], A, 0.0) + np.diag((~act).astype(float))
    return np.linalg.inv(full)


@pytest.mark.parametrize("n", list(range(1, 17)))
def test_block_against_numpy(emul, n):
    rng = np.random.default_rng(100 + n)
    tri = [(a, b) for a in range(n) for b in range(a, n)]
    assert [emul.emul_cr_tri(a, b, n) for a, b in tri] == list(range(len(tri)))
    for trial in range(6):
        G = rng.standard_normal((n, n + 2))
        M = G @ G.T                                   # SPD, like sum_nu N_lm b^2 F F^t over enough bands
        inactive = rng.uniform(size=n) < (0.3 if trial else 0.0)
        if trial == 5:
            inactive[:] = True                        # nothing observed at this slot: identity
        M[inactive, :] = 0.0
        M[:, inactive] = 0.0
        prior = rng.uniform(size=n) < 0.6
        sS = rng.uniform(0.1, 3.0, size=n)
        sS[rng.uniform(size=n) < 0.15] = 0.0          # C_l = 0 (or an l < 2 polarisation mode)
        ref = _block_ref(M, sS, prior)
        t = np.array([M[a, b] for a, b in tri])
        r = rng.standard_normal(n)
        z = np.zeros(n)
        pr = (C.c_int * n)(*prior.astype(int))
        emul.emul_cr_block(n, t.ctypes.data_as(C.c_void_p), sS.ctypes.data_as(C.c_void_p), pr,
                           r.ctypes.data_as(C.c_void_p), z.ctypes.data_as(C.c_void_p))
        got = np.zeros((n, n))
        for e, (a, b) in enumerate(tri):
            got[a, b] = got[b, a] = t[e]
        scale = np.abs(ref).max()
        assert np.abs(got - ref).max() <= 1e-10 * scale, (n, trial)
        assert np.abs(z - ref @ r).max() <= 1e-10 * scale * np.abs(r).sum()
        assert np.array_equal(got[inactive][:, inactive], np.eye(int(inactive.sum())))


# ------------------------------------------------------------------ Python front end

def _pyproblem():
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, gaussian_beam
    b = cr_band(comm_mapinfo(None, 4, 8, 3, True), np.ones((3, 192)), gaussian_beam(8, 600.0, 3))
    c = cr_component(comm_mapinfo(None, 4, 6, 3, True), Cl=np.ones((7, 3)), F_mean=np.ones((1, 3)))
    return c, b


def test_front_end_argument_checks(shtlib):
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system
    c, b = _pyproblem()
    with pytest.raises(ValueError, match="Preconditioner type not supported: pseudoinv"):
        cr_native_multi_system([c], [b], precond="pseudoinv")
    with pytest.raises(ValueError, match="per-pixel mixing"):
        cr_native_multi_system([cr_component(c.x_info, Cl=c.Cl, F_mean=c.F_mean, F=[np.ones((3, 192))])], [b])
    with pytest.raises(ValueError, match="F_mean has shape"):
        cr_native_multi_system([cr_component(c.x_info, Cl=c.Cl, F_mean=np.ones((2, 3)))], [b])
    with pytest.raises(ValueError, match="invN has shape"):
        cr_native_multi_system([c], [cr_band(b.info, np.ones((3, 100)), b.b_l)])
    with pytest.raises(ValueError, match="b_l has shape"):
        cr_native_multi_system([c], [cr_band(b.info, b.invN, b.b_l[:5])])
    with pytest.raises(ValueError, match="Cl has shape"):
        cr_native_multi_system([cr_component(c.x_info, Cl=np.ones((3, 3)), F_mean=c.F_mean)], [b])
    with pytest.raises(ValueError, match="cr_band"):
        cr_native_multi_system([c], [object()])
    with pytest.raises(ValueError, match="at least one"):
        cr_native_multi_system([], [b])
