"""Per-pixel mixing on the native multi-component constrained-realisation system without a GPU: the argument checks of
cmdr_cr_set_mixing_map (check_cr_mixing in commander_b200/csrc/cr_plan.h, compiled with g++ through
tests/host_emul/emul_crmix.cpp) and those of comm_cr.cr_native_multi_system's pixel_mixing / set_mixing_map."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "commander_b200", "csrc")


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_crmix.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_crmix.so")
    deps = [src, os.path.join(CSRC, "cr_plan.h"), os.path.join(CSRC, "sht_internal.h"), os.path.join(ROOT, "include", "cmdr_sht.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror",
                               "-Wno-unknown-pragmas", "-o", so, src])
    L = C.CDLL(so)
    L.emul_cr_mix_check.restype = C.c_int
    return L


# components: 3 maps, 1 map; bands: 3 maps, 1 map
CNM, BNM = [3, 1], [3, 1]


def check(L, band, comp, F_given=1, null_col=-1, multi=1, cnm=CNM, bnm=BNM):
    err = C.create_string_buffer(512)
    ok = L.emul_cr_mix_check(multi, len(cnm), len(bnm), (C.c_int * len(cnm))(*cnm), (C.c_int * len(bnm))(*bnm), band, comp,
                             F_given, null_col, err, len(err))
    return bool(ok), err.value.decode()


def test_valid_calls_are_accepted(emul):
    for q in range(2):
        for k in range(2):
            assert check(emul, q, k) == (True, "")
            assert check(emul, q, k, F_given=0) == (True, "")
    # columns beyond min(nmaps_band, nmaps_comp) are never read
    assert check(emul, 1, 0, null_col=1) == (True, "")
    assert check(emul, 0, 1, null_col=2) == (True, "")


def test_refusals(emul):
    assert check(emul, 0, 0, multi=0) == (
        False, "needs a handle of cmdr_cr_setup_multi (a cmdr_cr_setup handle has one component and no mixing)")
    assert check(emul, 0, 0, F_given=0, multi=0)[0] is False
    assert check(emul, 2, 0) == (False, "band 2 out of range (nbands 2)")
    assert check(emul, -1, 0) == (False, "band -1 out of range (nbands 2)")
    assert check(emul, 0, 2) == (False, "comp 2 out of range (ncomp 2)")
    assert check(emul, 0, -1, F_given=0) == (False, "comp -1 out of range (ncomp 2)")
    for j in range(3):
        assert check(emul, 0, 0, null_col=j) == (
            False, f"F[{j}] is NULL: give all 3 columns (min(nmaps_band, nmaps_comp)), or F = NULL for F_mean mixing")
    assert check(emul, 1, 0, null_col=0) == (
        False, "F[0] is NULL: give all 1 columns (min(nmaps_band, nmaps_comp)), or F = NULL for F_mean mixing")


# ------------------------------------------------------------------ Python front end

def _pyproblem(F):
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, gaussian_beam
    b = cr_band(comm_mapinfo(None, 4, 8, 3, True), np.ones((3, 192)), gaussian_beam(8, 600.0, 3))
    c = cr_component(comm_mapinfo(None, 4, 6, 3, True), Cl=np.ones((7, 3)), F_mean=np.ones((1, 3)), F=F)
    return c, b


def test_front_end_pixel_mixing_checks(shtlib):
    from commander_b200.comm_cr import cr_native_multi_system
    c, b = _pyproblem([np.ones((3, 192))])
    with pytest.raises(ValueError, match="per-pixel mixing F is not supported by the native system"):
        cr_native_multi_system([c], [b])
    with pytest.raises(ValueError, match="per-pixel mixing F is not supported by the native system"):
        cr_native_multi_system([c], [b], pixel_mixing=False)
    for bad in (np.ones((2, 192)), np.ones((3, 191)), np.ones(192), np.ones((3, 192, 1))):
        c, b = _pyproblem([bad])
        with pytest.raises(ValueError, match=r"F of component 0 in band 0 has shape .*, expected \(3 or more, 192\)"):
            cr_native_multi_system([c], [b], pixel_mixing=True)
    c, b = _pyproblem([np.ones((3, 192)), None])
    with pytest.raises(ValueError, match="component F has 2 entries, expected one per band"):
        cr_native_multi_system([c], [b], pixel_mixing=True)


def test_set_mixing_map_checks(shtlib):
    """set_mixing_map's own checks run before the library is called: an object without a handle is enough."""
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_component, cr_native_multi_system
    c, b = _pyproblem(None)
    t = cr_component(comm_mapinfo(None, 4, 4, 1, False), F_mean=np.ones((1, 1)))
    nat = cr_native_multi_system.__new__(cr_native_multi_system)
    nat.comps, nat.bands = [c, t], [b]
    for q, k in ((1, 0), (-1, 0)):
        with pytest.raises(ValueError, match=f"band {q} out of range"):
            nat.set_mixing_map(q, k, np.ones((3, 192)))
    with pytest.raises(ValueError, match="component 2 out of range"):
        nat.set_mixing_map(0, 2, None)
    with pytest.raises(ValueError, match=r"has shape \(3, 100\), expected \(3 or more, 192\)"):
        nat.set_mixing_map(0, 0, np.ones((3, 100)))
    with pytest.raises(ValueError, match=r"has shape \(0, 192\), expected \(1 or more, 192\)"):
        nat.set_mixing_map(0, 1, np.ones((0, 192)))
    # accepted shapes: the first min(nmaps_q, nmaps_k) rows as contiguous float64 columns, extra rows ignored
    cols = nat._mixing_cols(0, 1, np.arange(3 * 192, dtype=np.float32).reshape(3, 192))
    assert len(cols) == 1 and cols[0].dtype == np.float64 and cols[0].flags.c_contiguous
    assert np.array_equal(cols[0], np.arange(192))
    assert len(nat._mixing_cols(0, 0, np.ones((4, 192)))) == 3
