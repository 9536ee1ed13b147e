"""What a transform call runs, without a GPU: commander_b200/csrc/job.h, the resolution every entry point does before it
touches data, compiled with g++ (tests/host_emul/emul_job.cpp).  Refused jobs come back as a message here; the library
prints it and aborts."""
import ctypes as C
import os
import subprocess

import pytest

from commander_b200.sharp import SHARP_ADD, SHARP_ALM2MAP_DERIV1, SHARP_DP, SHARP_NO_FFT, SHARP_WY, SHARP_Y, SHARP_Yt, SHARP_YtW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAP_JOBS = (SHARP_YtW, SHARP_Y, SHARP_Yt, SHARP_WY)


@pytest.fixture(scope="module")
def resolve():
    src = os.path.join(ROOT, "tests", "host_emul", "emul_job.cpp")
    out = os.path.join(ROOT, "tests", "host_emul", "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libemul_job.so")
    deps = [src, os.path.join(ROOT, "commander_b200", "csrc", "job.h"), os.path.join(ROOT, "include", "cmdr_sht.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror", "-o", so, src])
    L = C.CDLL(so)
    L.emul_resolve_job.argtypes = [C.c_int] * 4 + [C.c_void_p, C.c_char_p, C.c_int]
    L.emul_resolve_job.restype = C.c_int

    def run(type, spin, flags=SHARP_DP, iqu=False):
        out = (C.c_int * 7)()
        err = C.create_string_buffer(256)
        ok = L.emul_resolve_job(type, spin, flags, int(iqu), out, err, len(err))
        keys = ("spin", "alm_cols", "map_cols", "synth", "weighted", "add", "deriv1")
        return (dict(zip(keys, out)) if ok else None), err.value.decode()
    return run


@pytest.mark.parametrize("spin", [0, 1, 2, 32])
@pytest.mark.parametrize("type", MAP_JOBS)
def test_map_jobs(resolve, type, spin):
    job, err = resolve(type, spin)
    assert job is not None and err == ""
    cols = 1 if spin == 0 else 2
    assert job == {"spin": spin, "alm_cols": cols, "map_cols": cols, "synth": int(type in (SHARP_Y, SHARP_WY)),
                   "weighted": int(type in (SHARP_WY, SHARP_YtW)), "add": 0, "deriv1": 0}
    assert resolve(type, spin, SHARP_DP | SHARP_ADD)[0]["add"] == 1
    assert resolve(type, spin, iqu=True)[0] == job


@pytest.mark.parametrize("spin", [0, 1, 2, 32, -1, 33])
def test_deriv1_is_one_alm_column_to_two_maps_on_the_spin1_tables(resolve, spin):
    job, err = resolve(SHARP_ALM2MAP_DERIV1, spin)
    assert err == ""
    assert job == {"spin": 1, "alm_cols": 1, "map_cols": 2, "synth": 1, "weighted": 0, "add": 0, "deriv1": 1}
    assert resolve(SHARP_ALM2MAP_DERIV1, spin, SHARP_DP | SHARP_ADD)[0]["add"] == 1


@pytest.mark.parametrize("type,spin,flags,msg", [
    (-1, 0, SHARP_DP, "job type -1 unsupported"),
    (5, 0, SHARP_DP, "job type 5 unsupported"),
    (SHARP_Y, -1, SHARP_DP, "spin -1 unsupported (0..32)"),
    (SHARP_YtW, 33, SHARP_DP, "spin 33 unsupported (0..32)"),
    (SHARP_Y, 0, SHARP_DP | SHARP_NO_FFT, "SHARP_NO_FFT unsupported"),
    (SHARP_Yt, 2, SHARP_NO_FFT | SHARP_ADD, "SHARP_NO_FFT unsupported"),
    (SHARP_ALM2MAP_DERIV1, 0, SHARP_DP | SHARP_NO_FFT, "SHARP_NO_FFT unsupported"),
])
def test_refused_jobs(resolve, type, spin, flags, msg):
    for iqu in (False, True):
        job, err = resolve(type, spin, flags, iqu)
        assert job is None and err == (msg if not (iqu and type == SHARP_ALM2MAP_DERIV1) else "job type 4 unsupported")


def test_iqu_entry_points_run_the_map_jobs_only(resolve):
    for spin in (0, 2):
        for t in MAP_JOBS:
            assert resolve(t, spin, iqu=True)[0] is not None
        job, err = resolve(SHARP_ALM2MAP_DERIV1, spin, iqu=True)
        assert job is None and err == "job type 4 unsupported"
