"""Seed tables of the spin-0 Legendre kernels, on the host (tests/host_emul/emul_seed.cpp, built from the product's
legendre_core.cuh and coef.cpp): a warp started from the seeded state at its first accumulating row ends with the same
synthesis sums and recurrence state, bit for bit, as the warp that runs the recurrence up from l = m, for polar and
non-polar blocks, with and without invalid slots (beyond the m cut-off) in the warp."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def seed0():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_seed.cpp")
    coef = os.path.join(ROOT, "commander_b200", "csrc", "coef.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_seed.so")
    hdrs = [os.path.join(ROOT, "commander_b200", "csrc", h) for h in ("legendre_core.cuh", "sht_internal.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src, coef] + hdrs):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", so, src, coef, "-lpthread"])
    L = C.CDLL(so)
    L.emul_seed0.argtypes = [C.c_int] * 4 + [C.c_void_p, C.c_void_p]

    def run(nside, lmax, m, north):
        n = np.ascontiguousarray(north, dtype=np.int32)
        same = C.c_int(0)
        j0 = L.emul_seed0(nside, lmax, m, len(n), n.ctypes.data, C.byref(same))
        return j0, bool(same.value)
    return run


@pytest.mark.parametrize("m", [0, 5, 40, 150, 300, 600])
def test_seeded_warp_matches_unseeded(seed0, m):
    nside, lmax = 256, 700
    blocks = {
        "polar": np.arange(1, 33),                               # sin(theta) from 0.007 to 0.2
        "polar_with_invalid": np.where(np.arange(1, 33) < 9, -1, np.arange(1, 33)),
        "mid": np.arange(100, 132),
        "equator": np.arange(2 * nside - 31, 2 * nside + 1),
    }
    skipped = 0
    for name, north in blocks.items():
        j0, same = seed0(nside, lmax, m, north)
        assert same, f"{name}, m = {m}: seeded warp differs (seeded start row {j0})"
        assert j0 % 4 == 0
        skipped += j0
    if m >= 150:
        assert skipped > 0    # the polar blocks start well above l = m at these m
