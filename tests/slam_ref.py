"""Independent high-precision reference for the spin-weighted harmonics (test helper, not a conftest).

    s-lambda_lm(theta) = (-1)^m sqrt((2l+1)/4pi) d^l_{-m,s}(theta)          (oracle/sht_def.py slam)

computed for l = 0..lmax in mpmath: the first two values (l0 = max(|m|,|s|) and l0 + 1) come from the explicit
Wigner-d sum of oracle/sht_def.py (one and two terms there, so cheap at any l), the rest from the three-term
recurrence of the Wigner d functions in l (Edmonds 1957, eq. 4.1.20 form)

    j sqrt(((j+1)^2 - m1^2)((j+1)^2 - m2^2)) d^{j+1}
        = (2j+1) (j(j+1) cos(beta) - m1 m2) d^j - (j+1) sqrt((j^2 - m1^2)(j^2 - m2^2)) d^{j-1}.

mpmath numbers have an unbounded exponent, so there is no scaling, no start-value table, no underflow floor and no
m cut-off: none of the devices the kernels (commander_b200/csrc/legendre_core.cuh) and the CPU oracle
(oracle/sht_cpu.c) share.  Values below the float64 range come back as 0.

Columns are cached per process: the GPU and oracle tests ask for the same (ring, m, s) many times.
"""
from __future__ import annotations

import math

import mpmath as mp
import numpy as np

from oracle import sht_def as D

_CACHE: dict = {}
_COEF: dict = {}


def _coefs(lmax: int, m1: int, m2: int, dps: int):
    """Recurrence coefficients in lambda = sqrt((2l+1)/4pi) d form (theta-independent, cached):
    lam_{j+1} = alpha_j (cos(beta) - beta_j) lam_j - gamma_j lam_{j-1}."""
    key = (m1, m2, dps)
    c = _COEF.get(key)
    if c is not None and len(c[0]) >= lmax + 1:
        return c
    with mp.workdps(dps + 10):
        al, be, ga = [None] * (lmax + 1), [None] * (lmax + 1), [None] * (lmax + 1)
        for j in range(max(abs(m1), abs(m2)) + 1, lmax):
            jp = j + 1
            d1 = mp.sqrt(mp.mpf((jp * jp - m1 * m1) * (jp * jp - m2 * m2)))
            d0 = mp.sqrt(mp.mpf((j * j - m1 * m1) * (j * j - m2 * m2)))
            # N_{j+1} / N_j and N_{j+1} / N_{j-1}, N_l = sqrt(2l+1)
            r1 = mp.sqrt(mp.mpf(2 * j + 3) / (2 * j + 1))
            r2 = mp.sqrt(mp.mpf(2 * j + 3) / (2 * j - 1))
            al[j] = (2 * j + 1) * jp * r1 / d1
            be[j] = mp.mpf(m1 * m2) / (j * jp)
            ga[j] = jp * d0 * r2 / (j * d1)
    _COEF[key] = (al, be, ga)
    return al, be, ga


def _column_mpf(lmax: int, m: int, s: int, cth, sth, dps: int):
    """List of mpf values s-lambda_{l,m} for l = 0..lmax (zeros below l0)."""
    with mp.workdps(dps):
        out = [mp.mpf(0)] * (lmax + 1)
        l0 = max(abs(m), abs(s))
        if l0 > lmax:
            return out
        theta = mp.atan2(mp.mpf(sth), mp.mpf(cth))
        ch, sh = mp.cos(theta / 2), mp.sin(theta / 2)
        cb = mp.cos(theta)
        m1, m2 = -m, s
        sgn = -1 if (m % 2) else 1
        four_pi = 4 * mp.pi
        out[l0] = sgn * mp.sqrt(mp.mpf(2 * l0 + 1) / four_pi) * D.wigner_d(l0, m1, m2, ch, sh)
        if l0 + 1 > lmax:
            return out
        out[l0 + 1] = sgn * mp.sqrt(mp.mpf(2 * l0 + 3) / four_pi) * D.wigner_d(l0 + 1, m1, m2, ch, sh)
        al, be, ga = _coefs(lmax, m1, m2, dps)
        prev, cur = out[l0], out[l0 + 1]
        for j in range(l0 + 1, lmax):
            prev, cur = cur, al[j] * (cb - be[j]) * cur - ga[j] * prev
            out[j + 1] = cur
        return out


def slam_column(lmax: int, m: int, s: int, cth: float, sth: float, dps: int = 40) -> np.ndarray:
    """s-lambda_{l,m}(theta) for l = 0..lmax as float64 (m and s may be negative); 0 for l < max(|m|, |s|)."""
    key = (lmax, m, s, float(cth), float(sth), dps)
    col = _CACHE.get(key)
    if col is None:
        # a longer cached column of the same (m, s, theta) serves a shorter request
        for (L, mm, ss, c, sn, dd), v in _CACHE.items():
            if (mm, ss, c, sn, dd) == key[1:] and L >= lmax:
                return v[:lmax + 1].copy()
        col = np.array([float(v) for v in _column_mpf(lmax, m, s, cth, sth, dps)])
        col.setflags(write=False)
        _CACHE[key] = col
    return col.copy()


def ring_trig(nside: int, ring: int):
    """(cos theta, sin theta) of a HEALPix ring as the transforms see it: z = cos theta correctly rounded to float64
    (what commander_b200/csrc/abi.cu computes in long double and rounds), sin theta = sqrt(1 - z^2) of that float64 z.

    The reference is evaluated at theta = arccos(z) of the rounded z.  The rounding of z itself moves theta by up to
    2^-53 / sin(theta) -- at ring 1 of nside 2048 that changes lambda at l = 4000 by up to ~1e-9 -- which is a property
    of the float64 geometry every FP64 transform starts from, not an error of any of them."""
    from fractions import Fraction
    north = 4 * nside - ring if ring > 2 * nside else ring
    if north < nside:
        z = 1 - Fraction(north * north, 3 * nside * nside)
    else:
        z = Fraction(2 * (2 * nside - north), 3 * nside)
    cth = float(z)
    with mp.workdps(40):
        sth = float(mp.sqrt((1 - mp.mpf(cth)) * (1 + mp.mpf(cth))))
    return (cth if north == ring else -cth), sth


def ring_columns(nside: int, ring: int, lmax: int, m: int, spin: int, dps: int = 40) -> np.ndarray:
    """The functions a transform of spin `spin` reads at (ring, m): shape (1, lmax+1) for spin 0 (lambda_lm),
    (2, lmax+1) for spin s > 0 ((+s)lambda_lm, (-s)lambda_lm)."""
    cth, sth = ring_trig(nside, ring)
    if spin == 0:
        return slam_column(lmax, m, 0, cth, sth, dps)[None, :]
    return np.stack([slam_column(lmax, m, spin, cth, sth, dps), slam_column(lmax, m, -spin, cth, sth, dps)])


def pixel_basis(nside: int, ring: int, m: int, spin: int) -> np.ndarray:
    """Map values on `ring` of one unit real-packed coefficient at degree l, as linear forms in ring_columns(l).

    Returns B of shape (ncomp_in, nslot, ncomp_out, nfun, nph): component c_out of the map at pixel j is
    sum_f B[c_in, slot, c_out, f, j] * ring_columns[f, l] for a unit coefficient (component c_in, slot) at degree l.
    slot 0 is +m (the cos part), slot 1 is -m (the sin part; only when m > 0): the real-packed layout of
    oracle/sht_def.py alm_index.  The same definition Y_matrix uses, with lambda_{l,-m} taken from
    s-lambda_{l,-m} = (-1)^(s+m) (-s)-lambda_{l,m}."""
    _, _, nph, phi0, _ = D.healpix_ring(nside, ring)
    phi = phi0 + 2.0 * np.pi * np.arange(nph) / nph
    e = np.exp(1j * m * phi)
    nslot = 1 if m == 0 else 2
    rt2 = math.sqrt(2.0)
    cs = [1.0 + 0j] if m == 0 else [1.0 / rt2 + 0j, 1j / rt2]
    if spin == 0:
        B = np.zeros((1, nslot, 1, 1, nph))
        for k, c in enumerate(cs):
            B[0, k, 0, 0] = (c * e).real * (1.0 if m == 0 else 2.0)
        return B
    B = np.zeros((2, nslot, 2, 2, nph))
    ssg = 1.0 if (spin & 1) else -1.0
    sg = (-1) ** (m % 2)
    sym = (-1) ** ((spin + m) % 2)
    for ci in range(2):
        for k, c in enumerate(cs):
            cE, cB = (c, 0.0) if ci == 0 else (0.0, c)
            for f, (lpp, lmp) in enumerate(((1.0, 0.0), (0.0, 1.0))):
                lpn, lmn = sym * lmp, sym * lpp
                P = ssg * (cE + 1j * cB) * lpp * e
                M = -(cE - 1j * cB) * lmp * e
                if m > 0:
                    cEn, cBn = sg * np.conj(cE), sg * np.conj(cB)
                    P = P + ssg * (cEn + 1j * cBn) * lpn * np.conj(e)
                    M = M - (cEn - 1j * cBn) * lmn * np.conj(e)
                B[ci, k, 0, f] = (0.5 * (P + M)).real
                B[ci, k, 1, f] = ((P - M) / 2j).real
    return B


def expected_analysis(nside: int, ring: int, lmax: int, m: int, spin: int, x: np.ndarray, dps: int = 40):
    """Y^T of a map that is zero except x (ncomp, nph) on `ring`, at order m: shape (ncomp, nslot, lmax+1), in
    the transform's own normalisation (no ring weight).  Sums over pixels in numpy, no FFT."""
    B = pixel_basis(nside, ring, m, spin)
    lam = ring_columns(nside, ring, lmax, m, spin, dps)
    coef = np.einsum("iocfj,cj->iof", B, x)           # (ncomp_in, nslot, nfun)
    return np.einsum("iof,fl->iol", coef, lam)


def expected_synthesis(nside: int, ring: int, lmax: int, m: int, spin: int, a: np.ndarray, dps: int = 40):
    """Y of coefficients a (ncomp, nslot, lmax+1) at order m only, on `ring`: shape (ncomp, nph).  The sums over l are
    exact (math.fsum)."""
    B = pixel_basis(nside, ring, m, spin)
    lam = ring_columns(nside, ring, lmax, m, spin, dps)
    ci, ns = B.shape[0], B.shape[1]
    sums = np.array([[[math.fsum(a[i, k] * lam[f]) for f in range(lam.shape[0])] for k in range(ns)] for i in range(ci)])
    return np.einsum("iocfj,iof->cj", B, sums)


def mlim_for_ring(lmax: int, spin: int, sth: float, cth: float) -> int:
    """The per-ring m cut-off of the kernels and of the oracle (libsharp2's form), restated."""
    ofs = max(lmax * 0.01, 100.0)
    b = -2 * spin * abs(cth)
    t1 = lmax * sth + ofs
    c = float(spin * spin) - t1 * t1
    discr = b * b - 4 * c
    if discr <= 0:
        return lmax
    return int(min((-b + math.sqrt(discr)) / 2.0, lmax) + 0.5)


# ---------------------------------------------------------------------------------------------------------------------
# The probe set of the value-by-value tests (tests/test_oracle_deep.py, tests/test_gpu_deep_parity.py)
# ---------------------------------------------------------------------------------------------------------------------
FRONT_MIN_STH = 0.15      # sin(theta) below which the spin-2 kernels do not run the scalar front phase (legendre.cu)
POLAR_STH = 0.01          # rings nearer the pole than this have a bound of their own (see the tests)


def _first_ring(nside, pred):
    """Smallest northern ring number r for which pred(sin theta_r) holds."""
    for r in range(1, 2 * nside + 1):
        if pred(ring_trig(nside, r)[1]):
            return r
    return 2 * nside


def probe_set(nside: int, lmax: int, spin: int, full: bool = True):
    """{(ring, m): class} -- the (ring, m) pairs a value-by-value test reads, each with the name of its ring class.

    Rings (northern ring number r, southern mirrors 4 nside - r):
      polar      1, 2, 3, 4 (4 to 16 pixels: heavy aliasing of m onto few pixels) and the mirrors of 1 and 2
      front      either side of sin(theta) = FRONT_MIN_STH, and one ring at sin(theta) ~ 0.04 below it
      mlim       either side of the ring where the m cut-off mlim_for_ring(theta) reaches lmax / 2
      capbelt    nside - 1, nside, nside + 1 (last cap ring, first two belt rings) and the mirror of nside
      split      1024 and 1025 at nside 2048 (4096 / 4100 pixels: whole-ring chirp-z / radix-4 split ring kernels)
      equator    2 nside - 1 and 2 nside (the unpaired equator ring) and the mirror of 2 nside - 1
    m, on every ring:
      0..5; 30, 300, 1000, 2000, 3000 (where <= lmax; the spin-2 scalar front phase needs the start value below the
      threshold, i.e. m large enough); every m with lmax - m + 1 in {1, 2, 7, 8, 9, 127, 128, 129} (8-l groups,
      128-l tiles, parity of the l pairing; m = lmax among them); for spin s > 0 also s - 1, s, s + 1.
    m, per ring, around that ring's cut-off mc = mlim_for_ring: mc - 90, mc - 50, mc - 20, mc, mc + 1 (when mc < lmax),
      and lmax / 2 on the two mlim rings.
    With full=False (the arbitrary-spin runs) the rings are polar, front, capbelt and equator only."""
    rf = _first_ring(nside, lambda s: s >= FRONT_MIN_STH)
    r04 = _first_ring(nside, lambda s: s >= 0.04)
    mhalf = lmax // 2
    rm = _first_ring(nside, lambda s: mlim_for_ring(lmax, spin, s, math.sqrt(1 - s * s)) >= mhalf)
    cls = {}

    def add(r, c):
        if 1 <= r < 4 * nside and r not in cls:
            cls[r] = c
    for r in (1, 2, 3, 4, 4 * nside - 1, 4 * nside - 2):
        add(r, "polar")
    for r in (rf - 1, rf, r04, 4 * nside - rf):
        add(r, "front")
    if full:
        for r in (rm - 1, rm):
            add(r, "mlim")
    for r in (nside - 1, nside, nside + 1, 3 * nside):
        add(r, "capbelt")
    if full and nside == 2048:
        for r in (1024, 1025):
            add(r, "split")
    for r in (2 * nside - 1, 2 * nside, 2 * nside + 1):
        add(r, "equator")
    ms = set(range(6)) | {m for m in (30, 300, 1000, 2000, 3000) if m <= lmax}
    ms |= {lmax + 1 - n for n in (1, 2, 7, 8, 9, 127, 128, 129) if lmax + 1 - n >= 0}
    if spin > 0:
        ms |= {m for m in (spin - 1, spin, spin + 1) if 0 <= m <= lmax}
    out = {}
    for r, c in cls.items():
        cth, sth = ring_trig(nside, r)
        mc = mlim_for_ring(lmax, spin, sth, cth)
        mr = set(ms)
        if mc < lmax:
            mr |= {m for m in (mc - 90, mc - 50, mc - 20, mc, mc + 1) if 0 <= m <= lmax}
        if c == "mlim":
            mr.add(mhalf)
        for m in mr:
            out[(r, m)] = c
    return out


def _columns_task(args):
    lmax, m, s, trig = args
    return [(lmax, m, s, c, sn, slam_column(lmax, m, s, c, sn)) for c, sn in trig]


def prefetch(nside: int, lmax: int, spin: int, pairs, workers: int = 0) -> None:
    """Computes the ring_columns of every (ring, m) in pairs in worker processes and caches them here."""
    import concurrent.futures as cf
    import multiprocessing as mpc
    import os
    by_ms = {}
    for r, m in pairs:
        for s in ((0,) if spin == 0 else (spin, -spin)):
            by_ms.setdefault((m, s), []).append(ring_trig(nside, r))
    tasks = [(lmax, m, s, sorted(set(t))) for (m, s), t in by_ms.items()]
    tasks = [t for t in tasks if any((lmax, t[1], t[2], c, sn, 40) not in _CACHE for c, sn in t[3])]
    if not tasks:
        return
    workers = workers or max(1, min(len(tasks), os.cpu_count() or 1))
    # longest columns first
    tasks.sort(key=lambda t: -(lmax - max(abs(t[1]), abs(t[2]))) * len(t[3]))
    with cf.ProcessPoolExecutor(workers, mp_context=mpc.get_context("fork")) as ex:
        for res in ex.map(_columns_task, tasks):
            for L, m, s, c, sn, col in res:
                col.setflags(write=False)
                _CACHE[(L, m, s, c, sn, 40)] = col


# ---------------------------------------------------------------------------------------------------------------------
# Running the probes against a transform
# ---------------------------------------------------------------------------------------------------------------------
# absolute floor per unit of sum |input|: the kernels join the accumulation once |mu| >= 2^-70, checked at 8-l group
# boundaries, and near l = m the functions grow by up to 2^20 over a group, so values up to ~2^-50 can be left out
# (the floor of the random sweep in tests/test_host.py, 3e-15 on lambda, has the same origin)
FLOOR = 1e-15


def pack(a: dict, lmax: int, ms) -> np.ndarray:
    """{m: (nc, nslot, lmax+1)} -> real-packed m-major alm (nc, nalm) over ms."""
    return np.concatenate([a[m][:, :, m:].transpose(0, 2, 1).reshape(a[m].shape[0], -1) for m in ms], axis=1)


def unpack(alm: np.ndarray, lmax: int, ms) -> dict:
    out, i = {}, 0
    for m in ms:
        ns = 1 if m == 0 else 2
        n = ns * (lmax + 1 - m)
        v = np.zeros((alm.shape[0], ns, lmax + 1))
        v[:, :, m:] = alm[:, i:i + n].reshape(alm.shape[0], lmax + 1 - m, ns).transpose(0, 2, 1)
        out[m] = v
        i += n
    return out


def run_probes(nside: int, lmax: int, spin: int, pairs: dict, analyse, synthesise, seed: int = 0,
               weighted_rings=(), analyse_w=None, weight=None):
    """Reads every probe of `pairs` ({(ring, m): class}) through a transform and compares it value by value.

    analyse(ring, ms, x) -> real-packed alm over ms of Y^T of the map that is x (nc, nph) on `ring`, zero elsewhere;
    synthesise(m, rings, a) -> {ring: (nc, nph)} of Y of the packed coefficients a (nc, nalm) at order m alone;
    analyse_w(ring, ms, x), when given, is Y^T W for the rings in weighted_rings (ring weights 4 pi / npix weight[r-1]).
    Spin s > 0 is read with a Q-only and a U-only map so that both functions of every coefficient are seen.

    The scale S of a reading is its largest expected magnitude, but at least the size a sum of random terms has
    (max |lambda| times the 2-norm of the ring's input for analysis, the 2-norm of a_l lambda_l for synthesis): a
    reading whose pixel sums happen to cancel is not held to a tighter absolute bound than its neighbours.
    Returns one record per reading: dict(kind, ring, m, cls, err = max |delta| / S, S,
    floor = FLOOR * sum |input|, excess = max(|delta| - floor) / S, cut = m is past the ring's m cut-off,
    zero_ok = values the definition makes zero, and every value past the cut-off, are exactly 0)."""
    rng = np.random.default_rng(seed)
    nc = 1 if spin == 0 else 2
    rings = sorted({r for r, _ in pairs})
    ms_all = sorted({m for _, m in pairs})
    recs = []

    def record(kind, r, m, got, ex, inp, typ):
        cth, sth = ring_trig(nside, r)
        cut = m > mlim_for_ring(lmax, spin, sth, cth)
        fl = FLOOR * float(np.abs(inp).sum())
        d = np.abs(got - ex)
        zero_ok = bool(np.all(got == 0)) if cut else True
        if got.ndim == 3:
            zero_ok &= bool(np.all(got[:, :, :max(m, spin)] == 0))
        recs.append(dict(kind=kind, ring=r, m=m, cls=pairs[(r, m)], S=max(float(np.abs(ex).max()), typ), cut=cut,
                         dmax=float(d.max()), exabs=max(float((d - fl).max()), 0.0), floor=fl, zero_ok=zero_ok))

    for r in rings:
        ms = sorted(m for rr, m in pairs if rr == r)
        nph = D.healpix_ring(nside, r)[2]
        jobs = [("Yt", analyse, 1.0)]
        if r in weighted_rings and analyse_w is not None:
            jobs.append(("YtW", analyse_w, D.ring_weight(nside, r, weight)))
        for kind, fn, w in jobs:
            for comp in range(nc):
                x = np.zeros((nc, nph))
                x[comp] = rng.standard_normal(nph)
                got = unpack(fn(r, ms, x), lmax, ms)
                for m in ms:
                    ex = w * expected_analysis(nside, r, lmax, m, spin, x)
                    typ = w * float(np.abs(ring_columns(nside, r, lmax, m, spin)).max() * np.linalg.norm(x))
                    record(kind + ("" if spin == 0 else "QU"[comp]), r, m, got[m], ex, x, typ)
    for m in ms_all:
        rs = sorted(r for r, mm in pairs if mm == m)
        ns = 1 if m == 0 else 2
        a = rng.standard_normal((nc, ns, lmax + 1))
        a[:, :, :m] = 0.0
        out = synthesise(m, rs, pack({m: a}, lmax, [m]))
        for r in rs:
            lam = ring_columns(nside, r, lmax, m, spin)
            typ = float(np.sqrt(max(np.sum((a[i, k] * lam[f]) ** 2) for i in range(nc) for k in range(ns)
                                    for f in range(lam.shape[0]))))
            record("Y", r, m, out[r], expected_synthesis(nside, r, lmax, m, spin, a), a, typ)
    # scale: the probe's own largest expected value; for m past the ring's cut-off (where the transform returns
    # exactly 0 and the error is the dropped value itself) the ring's largest over all probed m of the same reading
    ring_scale = {}
    for q in recs:
        k = (q["kind"], q["ring"])
        ring_scale[k] = max(ring_scale.get(k, 0.0), q["S"])
    for q in recs:
        S = ring_scale[(q["kind"], q["ring"])] if q["cut"] else q["S"]
        q["S_eff"] = S
        q["err"] = q["dmax"] / S if S > 0 else q["dmax"]
        q["excess"] = q["exabs"] / S if S > 0 else q["exabs"]
    return recs


def summarize(recs, label: str) -> str:
    """Worst error per (reading, ring class), one line each: the numbers the tests' bounds are set from."""
    worst = {}
    for q in recs:
        k = (q["kind"], q["cls"])
        if k not in worst or q["excess"] > worst[k]["excess"]:
            worst[k] = q
    lines = [f"{label}: worst max(|delta| - floor) / S per reading and ring class"]
    for (kind, cls), q in sorted(worst.items()):
        lines.append(f"  {kind:5s} {cls:8s} {q['excess']:.2e}  (ring {q['ring']}, m {q['m']}, S {q['S']:.2e}, "
                     f"max|delta|/S {q['err']:.2e}{', past cut-off' if q['cut'] else ''})")
    return "\n".join(lines)
