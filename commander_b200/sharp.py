"""ctypes binding of libcmdr_sht.so that mirrors `module sharp` of the reference
(commander3/src/sharp.f90): same constant names, same wrapper procedures, same
argument meaning.  Arrays are laid out as the Fortran side has them: alm(0:n_alm-1, nmaps)
and map(0:n_pix-1, nmaps) column-major, i.e. shape (nmaps, n) C-contiguous here.

Inputs may be numpy arrays (host memory, as Fortran passes) or torch CUDA tensors
(device memory; the library detects this with cudaPointerGetAttributes).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

# job types, commander3/src/sharp.f90:8-14
SHARP_YtW, SHARP_Y, SHARP_Yt, SHARP_WY, SHARP_ALM2MAP_DERIV1 = 0, 1, 2, 3, 4
# alm_info flags, commander3/src/sharp.f90:5
SHARP_PACKED = 1
# job flags, commander3/src/sharp.f90:17-20
SHARP_DP = 1 << 4
SHARP_ADD = 1 << 5
SHARP_REAL_HARMONICS = 1 << 6
SHARP_NO_FFT = 1 << 7

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libcmdr_sht.so")
_lib = None

ABI_SYMBOLS = [
    # part 1: what commander3/src/sharp.f90 binds
    "sharp_make_general_alm_info", "sharp_make_mmajor_real_packed_alm_info", "sharp_alm_count",
    "sharp_destroy_alm_info", "sharp_make_subset_healpix_geom_info", "sharp_destroy_geom_info",
    "sharp_map_size", "sharp_execute", "sharp_execute_mpi_fortran",
    # part 2: additive
    "cmdr_sht_version", "cmdr_sht_execute_dev", "cmdr_sht_execute_iqu", "cmdr_sht_execute_iqu_batch", "cmdr_sht_get_unique_id",
    "cmdr_sht_comm_register", "cmdr_sht_comm_destroy", "cmdr_sht_comm_set_exchange", "cmdr_sht_execute_dist",
    "cmdr_sht_execute_iqu_dist", "cmdr_sht_mix", "cmdr_sht_invn_diag", "cmdr_sht_conviqt_cube", "cmdr_sht_allreduce_sum", "cmdr_sht_launch_count",
    "cmdr_sht_set_profiling", "cmdr_sht_last_legendre_ms", "cmdr_sht_nominal_flops",
    "cmdr_sht_release_caches", "cmdr_sht_measure_fp64_tflops", "cmdr_sht_measure_fp64_tflops_3op",
    "cmdr_sht_measure_host_copy", "cmdr_sht_host_copy_threads",
    "cmdr_cr_setup", "cmdr_cr_destroy", "cmdr_cr_matmulA", "cmdr_cr_invM", "cmdr_cr_set_precond_diag",
    "cmdr_cr_get_precond_diag", "cmdr_cr_compute_rhs", "cmdr_cr_solve", "cmdr_cr_matmul_count",
]


def lib() -> C.CDLL:
    """Loads libcmdr_sht.so.  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C commander_b200/csrc).  There is no CPU fallback.")
    L = C.CDLL(_LIB_PATH)
    vp, ci, dp = C.c_void_p, C.c_int, C.POINTER(C.c_double)
    L.sharp_make_general_alm_info.argtypes = [ci, ci, ci, vp, vp, ci, C.POINTER(vp)]
    L.sharp_make_mmajor_real_packed_alm_info.argtypes = [ci, ci, ci, vp, C.POINTER(vp)]
    L.sharp_alm_count.argtypes = [vp]
    L.sharp_alm_count.restype = C.c_ssize_t
    L.sharp_destroy_alm_info.argtypes = [vp]
    L.sharp_make_subset_healpix_geom_info.argtypes = [ci, ci, ci, vp, vp, C.POINTER(vp)]
    L.sharp_destroy_geom_info.argtypes = [vp]
    L.sharp_map_size.argtypes = [vp]
    L.sharp_map_size.restype = C.c_ssize_t
    L.sharp_execute.argtypes = [ci, ci, vp, vp, vp, vp, ci, dp, C.POINTER(C.c_ulonglong)]
    L.sharp_execute_mpi_fortran.argtypes = [ci, ci, ci, vp, vp, vp, vp, ci, dp, C.POINTER(C.c_ulonglong)]
    L.cmdr_sht_version.restype = ci
    L.cmdr_sht_execute_dev.argtypes = [ci, ci, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_execute_iqu.argtypes = [ci, vp, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_execute_iqu_batch.argtypes = [ci, ci, vp, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_get_unique_id.argtypes = [vp]
    L.cmdr_sht_comm_register.argtypes = [ci, ci, ci, vp]
    L.cmdr_sht_comm_register.restype = ci
    L.cmdr_sht_comm_destroy.argtypes = [ci]
    L.cmdr_sht_comm_set_exchange.argtypes = [ci, ci]
    L.cmdr_sht_execute_dist.argtypes = [ci, ci, ci, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_execute_iqu_dist.argtypes = [ci, ci, vp, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_mix.argtypes = [ci, ci, vp, vp, vp, vp, vp, vp]
    L.cmdr_sht_invn_diag.argtypes = [ci, vp, C.c_double, vp, vp, vp]
    L.cmdr_sht_conviqt_cube.argtypes = [ci, ci, ci, vp, vp, vp, vp, vp, ci, vp]
    L.cmdr_sht_allreduce_sum.argtypes = [ci, vp, ci, vp]
    L.cmdr_sht_launch_count.restype = C.c_ulonglong
    L.cmdr_sht_set_profiling.argtypes = [ci]
    L.cmdr_sht_last_legendre_ms.argtypes = [vp, ci]
    L.cmdr_sht_last_legendre_ms.restype = ci
    L.cmdr_sht_nominal_flops.argtypes = [vp, vp, ci]
    L.cmdr_sht_nominal_flops.restype = C.c_ulonglong
    L.cmdr_sht_measure_fp64_tflops.argtypes = [ci, ci]
    L.cmdr_sht_measure_fp64_tflops.restype = C.c_double
    L.cmdr_sht_measure_fp64_tflops_3op.argtypes = [ci, ci]
    L.cmdr_sht_measure_fp64_tflops_3op.restype = C.c_double
    L.cmdr_sht_measure_host_copy.argtypes = [C.c_size_t, ci, ci, ci]
    L.cmdr_sht_measure_host_copy.restype = C.c_double
    L.cmdr_sht_host_copy_threads.restype = ci
    L.cmdr_cr_setup.argtypes = [ci, ci, ci, vp, vp, vp, vp, vp, vp, ci]
    L.cmdr_cr_setup.restype = vp
    L.cmdr_cr_destroy.argtypes = [vp]
    L.cmdr_cr_matmulA.argtypes = [vp, vp, vp, vp]
    L.cmdr_cr_invM.argtypes = [vp, vp, vp, vp]
    L.cmdr_cr_set_precond_diag.argtypes = [vp, vp]
    L.cmdr_cr_get_precond_diag.argtypes = [vp, vp]
    L.cmdr_cr_compute_rhs.argtypes = [vp, vp, vp, vp, vp, vp]
    L.cmdr_cr_solve.argtypes = [vp, vp, vp, ci, ci, C.c_double, ci, ci, ci, vp, vp]
    L.cmdr_cr_solve.restype = ci
    L.cmdr_cr_matmul_count.argtypes = [vp]
    L.cmdr_cr_matmul_count.restype = C.c_ulonglong
    _lib = L
    return L


class sharp_alm_info:
    """type sharp_alm_info, commander3/src/sharp.f90:27-30"""

    def __init__(self):
        self.handle = C.c_void_p(None)
        self.n_local = 0


class sharp_geom_info:
    """type sharp_geom_info, commander3/src/sharp.f90:22-25"""

    def __init__(self):
        self.handle = C.c_void_p(None)
        self.n_local = 0


def sharp_make_mmajor_real_packed_alm_info(lmax, ms=None) -> sharp_alm_info:
    """commander3/src/sharp.f90:115-134 (ms absent -> m = 0..lmax)."""
    L = lib()
    info = sharp_alm_info()
    if ms is not None:
        ms_copy = np.ascontiguousarray(ms, dtype=np.int32)
        L.sharp_make_mmajor_real_packed_alm_info(lmax, 1, len(ms_copy), ms_copy.ctypes.data, C.byref(info.handle))
    else:
        L.sharp_make_mmajor_real_packed_alm_info(lmax, 1, lmax + 1, None, C.byref(info.handle))
    info.n_local = int(L.sharp_alm_count(info.handle))
    return info


def sharp_destroy_alm_info(info: sharp_alm_info) -> None:
    """commander3/src/sharp.f90:136-141"""
    if info.handle:
        lib().sharp_destroy_alm_info(info.handle)
    info.handle = C.c_void_p(None)


def sharp_make_healpix_geom_info(nside, rings=None, weight=None) -> sharp_geom_info:
    """commander3/src/sharp.f90:145-166 (rings absent -> all 4*nside-1 rings)."""
    L = lib()
    info = sharp_geom_info()
    w = None if weight is None else np.ascontiguousarray(weight, dtype=np.float64)
    if w is not None and w.shape != (2 * nside,):
        raise ValueError("weight must have 2*nside entries")
    wp = None if w is None else w.ctypes.data
    if rings is not None:
        r = np.ascontiguousarray(rings, dtype=np.int32)
        L.sharp_make_subset_healpix_geom_info(nside, 1, len(r), r.ctypes.data, wp, C.byref(info.handle))
    else:
        L.sharp_make_subset_healpix_geom_info(nside, 1, 4 * nside - 1, None, wp, C.byref(info.handle))
    info.n_local = int(L.sharp_map_size(info.handle))
    return info


def sharp_destroy_geom_info(info: sharp_geom_info) -> None:
    """commander3/src/sharp.f90:168-173"""
    if info.handle:
        lib().sharp_destroy_geom_info(info.handle)
    info.handle = C.c_void_p(None)


def _col_ptrs(arr, nmaps, n_local):
    """Pointer table over the columns, commander3/src/sharp.f90:219-224."""
    ptrs = (C.c_void_p * nmaps)()
    if n_local == 0:
        return ptrs, None
    if isinstance(arr, np.ndarray):
        if arr.dtype != np.float64 or not arr.flags.c_contiguous or arr.shape != (nmaps, n_local):
            raise ValueError(f"expected C-contiguous float64 array of shape ({nmaps}, {n_local}), got {arr.shape} {arr.dtype}")
        base, step = arr.ctypes.data, arr.strides[0]
    else:  # torch tensor (host or CUDA)
        import torch
        if arr.dtype != torch.float64 or not arr.is_contiguous() or tuple(arr.shape) != (nmaps, n_local):
            raise ValueError(f"expected contiguous float64 tensor of shape ({nmaps}, {n_local}), got {tuple(arr.shape)} {arr.dtype}")
        base, step = arr.data_ptr(), arr.stride(0) * 8
    for k in range(nmaps):
        ptrs[k] = base + k * step
    return ptrs, arr


def sharp_execute(type, spin, nmaps, alm, alm_info: sharp_alm_info, map, geom_info: sharp_geom_info,
                  add=False, time=False, opcnt=False, comm=None):
    """commander3/src/sharp.f90:186-241 (`sharp_execute_d`).

    alm has shape (nmaps, alm_info.n_local), map (nmaps, geom_info.n_local).
    Returns (time, opcnt) when requested, else None."""
    L = lib()
    mod_flags = SHARP_DP
    if add:
        mod_flags |= SHARP_ADD
    ntrans = nmaps if spin == 0 else nmaps // 2
    if ntrans != 1:
        print("ERROR: ntrans /= 1")   # commander3/src/sharp.f90:216
    alm_ptr, _a = _col_ptrs(alm, nmaps, alm_info.n_local)
    map_ptr, _m = _col_ptrs(map, nmaps, geom_info.n_local)
    t = C.c_double(0.0) if time else None
    oc = C.c_ulonglong(0) if opcnt else None
    tp = C.byref(t) if time else None
    op = C.byref(oc) if opcnt else None
    if comm is not None:
        L.sharp_execute_mpi_fortran(int(comm), type, spin, alm_ptr, map_ptr, geom_info.handle,
                                    alm_info.handle, mod_flags, tp, op)
    else:
        L.sharp_execute(type, spin, alm_ptr, map_ptr, geom_info.handle, alm_info.handle, mod_flags, tp, op)
    if time or opcnt:
        return (t.value if time else None, oc.value if opcnt else None)
    return None


def alm2map_der1(alm, alm_info: sharp_alm_info, map, geom_info: sharp_geom_info, add=False, comm=None):
    """Gradient maps of one spin-0 a_lm column (SHARP_ALM2MAP_DERIV1, healpy's alm2map_der1):
    map[0] = dT/dtheta and map[1] = (1/sin theta) dT/dphi, where T is what SHARP_Y (spin 0) makes from
    the same a_lm.  alm has shape (1, alm_info.n_local), map (2, geom_info.n_local); numpy or torch,
    host or device.  No ring weights; `add` accumulates into both maps."""
    L = lib()
    flags = SHARP_DP | (SHARP_ADD if add else 0)
    alm_ptr, _a = _col_ptrs(alm, 1, alm_info.n_local)
    map_ptr, _m = _col_ptrs(map, 2, geom_info.n_local)
    if comm is not None:
        L.sharp_execute_mpi_fortran(int(comm), SHARP_ALM2MAP_DERIV1, 1, alm_ptr, map_ptr, geom_info.handle,
                                    alm_info.handle, flags, None, None)
    else:
        L.sharp_execute(SHARP_ALM2MAP_DERIV1, 1, alm_ptr, map_ptr, geom_info.handle, alm_info.handle, flags,
                        None, None)


# ---- additive entry points (include/cmdr_sht.h part 2)

def _check_iqu_job(type):
    if type not in (SHARP_YtW, SHARP_Y, SHARP_Yt, SHARP_WY):
        raise ValueError(f"job type {type} has no fused IQU form (SHARP_YtW, SHARP_Y, SHARP_Yt, SHARP_WY only)")


def execute_iqu(type, alm, map, geom_T: sharp_geom_info, geom_P: sharp_geom_info, alm_info: sharp_alm_info,
                add=False, stream=None, comm=None):
    """Fused T + (Q,U) transform: one call for what comm_map%Y etc. do in two
    (commander3/src/comm_map_mod.f90:444-447).  alm (3, n_alm), map (3, n_pix).  SHARP_YtW, SHARP_Y, SHARP_Yt or
    SHARP_WY: the gradient job has no IQU form (use alm2map_der1)."""
    _check_iqu_job(type)
    L = lib()
    flags = SHARP_DP | (SHARP_ADD if add else 0)
    alm_ptr, _a = _col_ptrs(alm, 3, alm_info.n_local)
    map_ptr, _m = _col_ptrs(map, 3, geom_T.n_local)
    st = C.c_void_p(stream) if stream else None
    if comm is not None:
        L.cmdr_sht_execute_iqu_dist(int(comm), type, alm_ptr, map_ptr, geom_T.handle, geom_P.handle,
                                    alm_info.handle, flags, st)
    else:
        L.cmdr_sht_execute_iqu(type, alm_ptr, map_ptr, geom_T.handle, geom_P.handle, alm_info.handle, flags, st)


def execute_iqu_batch(type, alms, maps, geom_T: sharp_geom_info, geom_P: sharp_geom_info, alm_info: sharp_alm_info,
                      add=False, stream=None):
    """nbatch fused IQU transforms with shared handles (one per frequency band); alms / maps are
    sequences of (3, n_alm) / (3, n_pix) arrays.  Host arrays are pipelined band against band."""
    _check_iqu_job(type)
    L = lib()
    nb = len(alms)
    if nb != len(maps):
        raise ValueError("alms and maps must have the same length")
    flags = SHARP_DP | (SHARP_ADD if add else 0)
    aptr = (C.c_void_p * (3 * nb))()
    mptr = (C.c_void_p * (3 * nb))()
    keep = []
    for b in range(nb):
        pa, ka = _col_ptrs(alms[b], 3, alm_info.n_local)
        pm, km = _col_ptrs(maps[b], 3, geom_T.n_local)
        keep += [ka, km]
        for c in range(3):
            aptr[3 * b + c] = pa[c]
            mptr[3 * b + c] = pm[c]
    st = C.c_void_p(stream) if stream else None
    L.cmdr_sht_execute_iqu_batch(type, nb, aptr, mptr, geom_T.handle, geom_P.handle, alm_info.handle, flags, st)


def mix(alm, F, geom_T: sharp_geom_info, geom_P: sharp_geom_info, alm_info: sharp_alm_info, nmaps=3,
        stream=None, comm=None):
    """alm <- YtW(F .* Y(alm)) with the map kept on the device (cmdr_sht_mix; the mixing step of
    commander3/src/comm_diffuse_comp_mod.f90:2078-2080, 2148-2150).  alm (nmaps, n_alm) is updated
    in place, F (nmaps, n_pix); host (numpy) or device (torch) arrays."""
    L = lib()
    alm_ptr, _a = _col_ptrs(alm, nmaps, alm_info.n_local)
    f_ptr, _f = _col_ptrs(F, nmaps, geom_T.n_local)
    st = C.c_void_p(stream) if stream else None
    gp = geom_P.handle if geom_P is not None else None
    L.cmdr_sht_mix(int(comm) if comm is not None else -1, nmaps, alm_ptr, f_ptr, geom_T.handle, gp,
                   alm_info.handle, st)


def invN_diag(a_l0, npix, alm_info: sharp_alm_info, out, stream=None) -> None:
    """N_lm of compute_invN_lm (commander3/src/comm_N_mod.f90:127-197) from the m=0 coefficients a_l0
    (nmaps, lmax+1; numpy, host) of YtW(N^-1 map); out (nmaps, n_alm), numpy or torch (device)."""
    L = lib()
    a_l0 = np.ascontiguousarray(a_l0, dtype=np.float64)
    nmaps = a_l0.shape[0]
    a_ptr, _a = _col_ptrs(a_l0, nmaps, a_l0.shape[1])
    o_ptr, _o = _col_ptrs(out, nmaps, alm_info.n_local)
    st = C.c_void_p(stream) if stream else None
    L.cmdr_sht_invn_diag(nmaps, a_ptr, float(npix), alm_info.handle, o_ptr, st)


def conviqt_cube(sky_alm, beam, bmax, geom_T: sharp_geom_info, alm_info: sharp_alm_info, cube, stream=None,
                 comm=None) -> None:
    """cube <- the psi cube of comm_conviqt%precompute_sky (commander3/src/comm_conviqt_mod.f90:207-292).
    sky_alm (nmaps, n_alm) float64; beam (ntri, nmaps) complex64 (alm_beam of the reference, transposed
    into memory order); cube (2*bmax, n_pix) float32 or float64.  numpy (host) or torch (device) arrays."""
    L = lib()
    nmaps = sky_alm.shape[0]
    alm_ptr, _a = _col_ptrs(sky_alm, nmaps, alm_info.n_local)
    ntri = beam.shape[0]
    if isinstance(beam, np.ndarray):
        if beam.dtype != np.complex64 or not beam.flags.c_contiguous or beam.shape != (ntri, nmaps):
            raise ValueError("beam must be a C-contiguous complex64 array of shape (ntri, nmaps)")
        bptr = beam.ctypes.data
    else:
        import torch
        if beam.dtype != torch.complex64 or not beam.is_contiguous() or tuple(beam.shape) != (ntri, nmaps):
            raise ValueError("beam must be a contiguous complex64 tensor of shape (ntri, nmaps)")
        bptr = beam.data_ptr()
    shape = (2 * bmax, geom_T.n_local)
    if isinstance(cube, np.ndarray):
        if cube.dtype not in (np.float32, np.float64) or not cube.flags.c_contiguous or cube.shape != shape:
            raise ValueError(f"cube must be a C-contiguous float32/float64 array of shape {shape}")
        cptr, f64 = cube.ctypes.data, cube.dtype == np.float64
    else:
        import torch
        if cube.dtype not in (torch.float32, torch.float64) or not cube.is_contiguous() or tuple(cube.shape) != shape:
            raise ValueError(f"cube must be a contiguous float32/float64 tensor of shape {shape}")
        cptr, f64 = cube.data_ptr(), cube.dtype == torch.float64
    st = C.c_void_p(stream) if stream else None
    L.cmdr_sht_conviqt_cube(int(comm) if comm is not None else -1, nmaps, int(bmax), alm_ptr, bptr,
                            geom_T.handle, alm_info.handle, cptr, 1 if f64 else 0, st)


def launch_count() -> int:
    return int(lib().cmdr_sht_launch_count())


def set_profiling(on: bool) -> None:
    lib().cmdr_sht_set_profiling(1 if on else 0)


def last_legendre_ms():
    buf = (C.c_double * (3 * 4096))()
    n = lib().cmdr_sht_last_legendre_ms(buf, 4096)
    return [(int(buf[3 * i]), int(buf[3 * i + 1]), float(buf[3 * i + 2])) for i in range(n)]


def nominal_flops(geom_info: sharp_geom_info, alm_info: sharp_alm_info, spin: int) -> int:
    return int(lib().cmdr_sht_nominal_flops(geom_info.handle, alm_info.handle, spin))


def measure_fp64_tflops(iters: int = 4096, reps: int = 5) -> float:
    return float(lib().cmdr_sht_measure_fp64_tflops(iters, reps))


def measure_fp64_tflops_3op(iters: int = 4096, reps: int = 3) -> float:
    return float(lib().cmdr_sht_measure_fp64_tflops_3op(iters, reps))
