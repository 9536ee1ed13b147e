"""The CPU oracle (oracle/sht_cpu.c) value by value against the independent reference of tests/slam_ref.py at the
target size -- the same probes as tests/test_gpu_deep_parity.py, one ring and an m subset per call.  The oracle is what
every whole-map parity test compares the kernels with, and it runs the same kind of scaled three-term recurrence; these
bounds make "how good is the oracle" a measured number (worst values, x86-64 with AVX-512, written beside each bound)."""
import numpy as np
import pytest

from oracle import sht_def as D

import slam_ref as R

# worst max(|delta| - floor) / S measured: 4.4e-12 (spin 0 and 2, nside 2048 / lmax 4000 and 1024 / 2048; spins 3, 17,
# 32 at 1024 / 2048 below that)
EPS = 1e-11
# sin(theta) < 0.01: measured 2.75e-9 (ring 1, m 12, nside 2048).  The oracle computes z = 1 - r^2 / (3 nside^2) in
# float64 arithmetic, not correctly rounded, so its ring 1 sits up to an ulp of z away from the reference's
# arccos(round(z)) -- 7e-10 of theta at nside 2048, times m + s for lambda ~ theta^(m+s).
EPS_POLAR = 5e-9

CASES = [(2048, 4000, 0, True), (2048, 4000, 2, True), (1024, 2048, 0, True), (1024, 2048, 2, True),
         (1024, 2048, 3, False), (1024, 2048, 17, False), (1024, 2048, 32, False)]


def _oracle(S, nside, lmax, spin):
    def analyse(r, ms, x):
        return S.execute(S.Yt, spin, nside, lmax, map=x, rings=[r], ms=ms, mlim_skip=True)

    def analyse_w(weight):
        def f(r, ms, x):
            return S.execute(S.YtW, spin, nside, lmax, map=x, rings=[r], ms=ms, weight=weight, mlim_skip=True)
        return f

    def synthesise(m, rings, a):
        out = S.execute(S.Y, spin, nside, lmax, alm=a, rings=rings, ms=[m], mlim_skip=True)
        res, o = {}, 0
        for r in rings:
            n = D.healpix_ring(nside, r)[2]
            res[r] = out[:, o:o + n]
            o += n
        return res
    return analyse, analyse_w, synthesise


@pytest.mark.parametrize("nside,lmax,spin,full", CASES)
def test_oracle_value_by_value(cpu_oracle, nside, lmax, spin, full):
    pairs = R.probe_set(nside, lmax, spin, full=full)
    R.prefetch(nside, lmax, spin, pairs)
    w = np.random.default_rng(nside + spin).uniform(0.5, 1.5, 2 * nside)
    an, anw, sy = _oracle(cpu_oracle, nside, lmax, spin)
    recs = R.run_probes(nside, lmax, spin, pairs, an, sy, seed=spin + 3, weighted_rings=(1, nside, 2 * nside),
                        analyse_w=anw(w), weight=w)
    print("\n" + R.summarize(recs, f"oracle nside {nside} lmax {lmax} spin {spin}"))
    for q in recs:
        eps = EPS_POLAR if R.ring_trig(nside, q["ring"])[1] < R.POLAR_STH else EPS
        assert q["zero_ok"] and q["excess"] <= eps, q


@pytest.mark.parametrize("spin,ring,m", [(0, 1, 14), (0, 101, 100), (0, 1000, 1200), (2, 101, 100), (2, 1000, 1200),
                                         (2, 377, 650)])
def test_oracle_floor_is_applied_consistently(cpu_oracle, spin, ring, m):
    """The oracle does not accumulate |lambda| < 2^-100 (TBITS) and joins the accumulation at the first l where the
    larger of its functions reaches it: readouts before the first l with max|lambda| >= 2^-101 are exactly 0, readouts
    from the first l with max|lambda| >= 2^-99 on are not (the recurrence is checked every l)."""
    S = cpu_oracle
    nside, lmax = 2048, 4000
    nc = 1 if spin == 0 else 2
    nph = D.healpix_ring(nside, ring)[2]
    x = np.random.default_rng(ring).standard_normal((nc, nph))
    got = R.unpack(S.execute(S.Yt, spin, nside, lmax, map=x, rings=[ring], ms=[m]), lmax, [m])[m]
    lam = np.abs(R.ring_columns(nside, ring, lmax, m, spin)).max(axis=0)
    lo = int(np.argmax(lam >= 2.0 ** -101))
    hi = int(np.argmax(lam >= 2.0 ** -99))
    assert m < lo < hi < lmax
    assert not got[:, :, :lo].any()
    assert np.all(np.abs(got[:, :, hi:]).max(axis=(0, 1))[lam[hi:] > 0] > 0)
