"""CPU self-tests of tests/slam_ref.py, the high-precision reference the deep parity tests compare with: against the
explicit Wigner-d sum of the definitional oracle, against scipy's spin-0 harmonics, and dps 40 against dps 80 at the
target size."""
import math

import mpmath as mp
import numpy as np
import pytest

from oracle import sht_def as D

import slam_ref as R

# polar, mid-latitude and equator rings of nside 64
RINGS = (1, 2, 40, 128)


@pytest.mark.parametrize("s", [0, 1, 2, 3, 8, 17, 31, 32])
def test_against_wigner_sum(s):
    """Every l <= 100 against the explicit sum (dps 60), both signs of the spin, m on either side of |s|."""
    lmax = 100
    mp.mp.dps = 60
    for sgn in ((1,) if s == 0 else (1, -1)):
        for m in sorted({0, 1, max(s - 1, 0), s, s + 1, 40, lmax}):
            for r in RINGS:
                cth, sth = R.ring_trig(64, r)
                col = R.slam_column(lmax, m, sgn * s, cth, sth)
                ref = np.array([float(D.slam(l, m, sgn * s, cth, sth)) for l in range(lmax + 1)])
                assert np.all(col[:max(m, s)] == 0)
                sc = np.abs(ref).max()
                if sc == 0:
                    assert np.all(col == 0)
                    continue
                # relative to each value; values that cancel to zero (equator, odd l + m) to 1e-30 of the column
                err = np.abs(col - ref) - 1e-13 * np.abs(ref)
                assert err.max() <= 1e-30 * sc, (s * sgn, m, r, err.max() / sc)


def test_negative_m_symmetry():
    """s-lambda_{l,-m} = (-1)^(s+m) (-s)-lambda_{l,m}, which the probe helpers use for the -m half of a real-packed
    coefficient."""
    for s, m, r in ((2, 3, 5), (3, 7, 40), (32, 5, 90), (1, 1, 128)):
        cth, sth = R.ring_trig(64, r)
        a = R.slam_column(60, -m, s, cth, sth)
        b = R.slam_column(60, m, -s, cth, sth)
        assert np.abs(a - (-1) ** ((s + m) % 2) * b).max() <= 1e-15 * np.abs(b).max()


def test_against_scipy_spin0():
    from scipy.special import sph_harm_y
    lmax = 500
    for m in (0, 1, 7, 250, 499):
        for th in (1e-3, 0.3, 1.2, math.pi / 2, 2.5):
            # scipy works from x = cos(theta) rounded to float64, which near the pole moves P_l by l^2 ulp: give the
            # reference the same x
            cth = math.cos(th)
            col = R.slam_column(lmax, m, 0, cth, math.sqrt((1.0 - cth) * (1.0 + cth)))
            ls = np.arange(m, lmax + 1)
            ref = sph_harm_y(ls, m, th, 0.0).real
            sc = np.abs(ref).max()
            # scipy's own values 1 mrad from the pole carry up to 6e-11 (its recurrence runs in x = cos(theta))
            tol = 1e-12 if th > 0.01 else 1e-10
            assert np.abs(col[m:] - ref).max() <= tol * sc + 1e-300, (m, th)


@pytest.mark.parametrize("s,m,ring", [(0, 0, 1), (0, 1200, 700), (2, 5, 1), (2, 3000, 2048), (-2, 40, 3),
                                      (32, 3, 900), (-31, 2000, 1500), (17, 17, 2)])
def test_stable_in_precision(s, m, ring):
    """dps 40 and dps 80 agree to 1e-25 of the column's largest value at nside 2048 / lmax 4000."""
    cth, sth = R.ring_trig(2048, ring)
    a = R._column_mpf(4000, m, s, cth, sth, 40)
    b = R._column_mpf(4000, m, s, cth, sth, 80)
    with mp.workdps(80):
        sc = max(abs(v) for v in b)
        assert sc > 0
        worst = max(abs(x - y) for x, y in zip(a, b)) / sc
    assert worst <= 1e-25, float(worst)
