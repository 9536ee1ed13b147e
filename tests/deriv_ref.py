"""Independent high-precision reference for the gradient job SHARP_ALM2MAP_DERIV1 (test helper, not a conftest).

From the spin-0 functions lambda_lm of slam_ref (mpmath, Wigner-d start values and recurrence) alone:

    sin(theta) d_theta lambda_lm = l z lambda_lm - sqrt((2l+1)/(2l-1) (l^2 - m^2)) lambda_{l-1,m},   z = cos(theta)
    (1/sin theta) d_phi of lambda_lm e^{i m phi} = i m lambda_lm / sin(theta) e^{i m phi}

evaluated in mpmath (the difference cancels near the poles) and rounded at the end.  Nothing here touches the spin-1
functions: the tests check the relation against mpmath.diff and, separately, against the spin-1 identity
    d_theta lambda = -sqrt(l(l+1)) ((+1)lambda - (-1)lambda) / 2,  m lambda / sin = sqrt(l(l+1)) ((+1)lambda + (-1)lambda) / 2.
"""
from __future__ import annotations

import math

import mpmath as mp
import numpy as np

from oracle import sht_def as D

import slam_ref as R

_CACHE: dict = {}


def _grad_mpf(lmax: int, m: int, cth: float, sth: float, dps: int = 40):
    """(d_theta lambda_lm, m lambda_lm / sin theta) for l = 0..lmax, mpf lists."""
    lam = R._column_mpf(lmax, m, 0, cth, sth, dps)
    with mp.workdps(dps):
        theta = mp.atan2(mp.mpf(sth), mp.mpf(cth))      # the angle slam_ref evaluates lambda at
        z, s = mp.cos(theta), mp.sin(theta)
        dth = [mp.mpf(0)] * (lmax + 1)
        mph = [mp.mpf(0)] * (lmax + 1)
        for l in range(max(m, 1), lmax + 1):
            prev = lam[l - 1] if l - 1 >= m else mp.mpf(0)
            c = mp.sqrt(mp.mpf(2 * l + 1) / (2 * l - 1) * (l * l - m * m))
            dth[l] = (l * z * lam[l] - c * prev) / s
            mph[l] = m * lam[l] / s
    return dth, mph


def grad_columns(lmax: int, m: int, cth: float, sth: float) -> np.ndarray:
    """(2, lmax+1) float64: d_theta lambda_lm and m lambda_lm / sin theta at the ring (cth, sth of slam_ref.ring_trig)."""
    key = (lmax, m, float(cth), float(sth))
    col = _CACHE.get(key)
    if col is None:
        dth, mph = _grad_mpf(lmax, m, cth, sth)
        col = np.array([[float(v) for v in dth], [float(v) for v in mph]])
        _CACHE[key] = col
    return col.copy()


def _task(args):
    lmax, m, trig = args
    return [(lmax, m, c, s, grad_columns(lmax, m, c, s)) for c, s in trig]


def prefetch(nside: int, lmax: int, pairs, workers: int = 0) -> None:
    """Computes grad_columns for every (ring, m) of pairs in worker processes and caches them here."""
    import concurrent.futures as cf
    import multiprocessing as mpc
    import os
    by_m = {}
    for r, m in pairs:
        by_m.setdefault(m, set()).add(R.ring_trig(nside, r))
    tasks = [(lmax, m, sorted(t)) for m, t in by_m.items()]
    tasks = [t for t in tasks if any((lmax, t[1], c, s) not in _CACHE for c, s in t[2])]
    if not tasks:
        return
    tasks.sort(key=lambda t: -(lmax - t[1]) * len(t[2]))
    workers = workers or max(1, min(len(tasks), os.cpu_count() or 1))
    with cf.ProcessPoolExecutor(workers, mp_context=mpc.get_context("fork")) as ex:
        for res in ex.map(_task, tasks):
            for L, m, c, s, col in res:
                _CACHE[(L, m, c, s)] = col


def expected_gradient(nside: int, ring: int, lmax: int, m: int, a: np.ndarray) -> np.ndarray:
    """{d_theta T, d_phi T / sin theta} on `ring` (shape (2, nph)) of the real-packed coefficients a (nslot, lmax+1) at
    order m alone (slot 0: +m, slot 1: -m; T as SHARP_Y spin 0 makes it).  Sums over l in math.fsum."""
    _, _, nph, phi0, _ = D.healpix_ring(nside, ring)
    phi = phi0 + 2.0 * np.pi * np.arange(nph) / nph
    cth, sth = R.ring_trig(nside, ring)
    g = grad_columns(lmax, m, cth, sth)
    out = np.zeros((2, nph))
    if m == 0:
        out[0] = math.fsum(a[0] * g[0])
        return out
    e = np.exp(1j * m * phi)
    rt2 = math.sqrt(2.0)
    for k, c in enumerate((1.0 / rt2 + 0j, 1j / rt2)):
        out[0] += math.fsum(a[k] * g[0]) * 2.0 * (c * e).real
        out[1] += math.fsum(a[k] * g[1]) * 2.0 * (1j * c * e).real
    return out


def e_of_alm(alm: np.ndarray, lmax: int, ms) -> np.ndarray:
    """E = -sqrt(l(l+1)) a over a real-packed m-major a_lm row (or rows): the spin-1 input that gives DERIV1."""
    l = np.array([l for l, _ in D.alm_index(lmax, ms)], dtype=np.float64)
    return -np.sqrt(l * (l + 1)) * alm
