"""The transforms on the GPU value by value against an independent high-precision reference (tests/slam_ref.py), at
the target size and for every spin the library accepts.

The parity tests of test_gpu_parity.py compare whole maps / a_lm sets with the CPU oracle in one relative L2 norm;
that cannot see an error confined to one ring, one m or one of the two spin-s functions, and the oracle runs the same
kind of recurrence as the kernels.  Here every probe (ring r, order m) is read on its own, through the C ABI with
device-resident arrays and the FULL HEALPix geometry (the kernels take their skip / mixed / all-on, spin-2 front phase
and m cut-off decisions per warp of 128 adjacent ring pairs, so a one-ring geometry would bypass them):

  analysis   Y^T (and once Y^T W) of a map that is random on ring r and zero elsewhere, over an m subset: each a_lm
             column is ring r's lambda readout for every l; expected = reference lambda times the exact pixel sums
             sum_j x_j cos(m phi_j), sum_j x_j sin(m phi_j) (no FFT, aliasing on short rings included).  Spin s > 0 is
             run with a Q-only and a U-only map so that both (+-s) functions are read.
  synthesis  Y with ms = [m] and random a_l for every l; the probed rings pixel by pixel against
             sum_l a_l lambda_l(theta_r) (sqrt2 cos / sin of m phi) with the sums over l in math.fsum.

Bounds per value, S = the probe's largest expected magnitude (for m past the ring's cut-off, where the transform must
return exactly 0, the ring's largest over the probed m; at least the size of a random sum, see slam_ref.run_probes):
|delta| <= eps S + 1e-15 sum|input| (slam_ref.FLOOR: the 2^-70 join threshold of the kernels, checked every 8 l).  Front-phase rings
(sin theta >= 0.15, spin 2) are held to eps = 1e-11, inside the 2e-11 of the larger function DESIGN 3.1 states.
Values the definition makes zero (l < max(m, s)) must be exactly 0.
The probe set is slam_ref.probe_set (rings 1-4, the sin(theta) = 0.15 front-phase edge, the m cut-off, cap/belt,
chirp-z / split ring kernels at 4096 / 4100 pixels, the equator; m 0-5, the 8-l group and 128-l tile edges near lmax,
m around each ring's cut-off, m on both sides of s).
Run with -s to see the worst error per probe class."""
import numpy as np
import pytest

from oracle import sht_def as D

import slam_ref as R

pytestmark = pytest.mark.gpu

# per value, relative to S: the host-emulation bounds of the recurrences (tests/test_host.py), 1e-11 for the spin-s
# recurrences and 2e-11 for the two-l-per-step spin-0 form (its even-l values are differences of O(l) larger numbers)
EPS = 1e-11
EPS_SPIN0 = 2e-11
# Rings with sin(theta) < 0.01 (rings 1..12 at nside 2048, 1..6 at nside 1024).  The kernels take the start values from
# sin / cos(theta/2) of the exact ring and run the recurrence in z = cos(theta) rounded to float64; that rounding moves
# theta by up to 2^-53 / (1 - z) / 2 relative (7e-10 at ring 1 of nside 2048), and lambda ~ theta^(m+s) near the pole
# by (m + s) times that.  Measured on one B200 (1000 W) worst 2.4e-9 (ring 1, m 12-14, nside 2048); the CPU oracle on
# the same probes 2.75e-9 (tests/test_oracle_deep.py), host emulation 1.2e-10 at ring 1 of nside 512 (test_host.py).
EPS_POLAR = 5e-9

TARGET = [(2048, 4000, 0), (2048, 4000, 2), (1024, 2048, 0), (1024, 2048, 2)]
SPINS = (1, 3, 8, 9, 16, 17, 31, 32)
ARBITRARY = [(1024, 2048, s) for s in SPINS] + [(64, 200, s) for s in SPINS]


def _transforms(sharp, nside, lmax, spin, weight):
    import torch
    nc = 1 if spin == 0 else 2
    gi = sharp.sharp_make_healpix_geom_info(nside)
    gw = sharp.sharp_make_healpix_geom_info(nside, weight=weight)
    mapbuf = torch.zeros((nc, gi.n_local), dtype=torch.float64, device="cuda")

    def analyse(job, geom):
        def f(r, ms, x):
            _, _, nph, _, ofs = D.healpix_ring(nside, r)
            ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
            alm = torch.full((nc, ai.n_local), float("nan"), dtype=torch.float64, device="cuda")
            mapbuf.zero_()
            mapbuf[:, ofs:ofs + nph] = torch.from_numpy(x).cuda()
            sharp.sharp_execute(job, spin, nc, alm, ai, mapbuf, geom)
            torch.cuda.synchronize()
            sharp.sharp_destroy_alm_info(ai)
            return alm.cpu().numpy()
        return f

    def synthesise(m, rings, a):
        ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=[m])
        alm = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        mapbuf.fill_(float("nan"))
        sharp.sharp_execute(sharp.SHARP_Y, spin, nc, alm, ai, mapbuf, gi)
        torch.cuda.synchronize()
        sharp.sharp_destroy_alm_info(ai)
        out = {}
        for r in rings:
            _, _, nph, _, ofs = D.healpix_ring(nside, r)
            out[r] = mapbuf[:, ofs:ofs + nph].cpu().numpy()
        return out

    def close():
        sharp.sharp_destroy_geom_info(gi)
        sharp.sharp_destroy_geom_info(gw)
    return analyse(sharp.SHARP_Yt, gi), analyse(sharp.SHARP_YtW, gw), synthesise, close


def _check(shtlib, nside, lmax, spin, full):
    pairs = R.probe_set(nside, lmax, spin, full=full)
    R.prefetch(nside, lmax, spin, pairs)
    rng = np.random.default_rng(nside + lmax + 100 * spin)
    w = rng.uniform(0.5, 1.5, 2 * nside)
    an, anw, sy, close = _transforms(shtlib, nside, lmax, spin, w)
    wr = (1, nside, 2 * nside, 4 * nside - 1)
    try:
        recs = R.run_probes(nside, lmax, spin, pairs, an, sy, seed=spin + 7, weighted_rings=wr, analyse_w=anw,
                            weight=w)
    finally:
        close()
    print("\n" + R.summarize(recs, f"GPU nside {nside} lmax {lmax} spin {spin}"))
    bad = []
    for q in recs:
        polar = R.ring_trig(nside, q["ring"])[1] < R.POLAR_STH
        eps = EPS_POLAR if polar else (EPS_SPIN0 if spin == 0 else EPS)
        if not q["zero_ok"] or not (q["excess"] <= eps):
            bad.append(q)
    assert not bad, f"{len(bad)} of {len(recs)} readings out of bounds, e.g. " + "; ".join(
        f"{q['kind']} ring {q['ring']} m {q['m']}: {q['excess']:.2e} zero_ok={q['zero_ok']}" for q in bad[:8])
    assert sum(q["kind"].startswith("YtW") for q in recs) > 0


@pytest.mark.parametrize("nside,lmax,spin", TARGET)
def test_deep_parity_target_size(shtlib, nside, lmax, spin):
    _check(shtlib, nside, lmax, spin, full=True)


@pytest.mark.parametrize("nside,lmax,spin", ARBITRARY)
def test_deep_parity_arbitrary_spin(shtlib, nside, lmax, spin):
    _check(shtlib, nside, lmax, spin, full=False)
