"""Spin 2 as scalar sums on the inputs the full-sphere comparison (test_gpu_s2scalar.py) does not reach.

The synthesis runs one scalar kernel for both map components (Q and U share the recurrence; synth0_kernel<2>).  Here the
route is compared against the spin-2 kernels on an m subset with a ring subset (unpaired rings, some of them polar), at
small lmax (row counts of an m that are not a multiple of the 4-row group, ring-pair counts that are not a multiple of
the 128 of a warp), and for SHARP_Yt with SHARP_ADD on a ring subset; and the launch count of a synthesis shows that the
route issues one Legendre launch for both components."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL = 1e-11


def _run(sharp, type, alm, mp, ai, gi, add=False):
    import torch
    n0 = sharp.launch_count()
    sharp.sharp_execute(type, 2, 2, alm, ai, mp, gi, add=add)
    torch.cuda.synchronize()
    return sharp.launch_count() - n0


def _both_routes(sharp, ai, gi, seed):
    """Y, Yt, YtW and Yt + SHARP_ADD with the route off and on; returns ({route: outputs}, {route: launches of Y})."""
    import torch
    rng = np.random.default_rng(seed)
    alm = torch.from_numpy(rng.standard_normal((2, ai.n_local))).cuda()
    mp_in = torch.from_numpy(rng.standard_normal((2, gi.n_local))).cuda()
    alm_add = torch.from_numpy(rng.standard_normal((2, ai.n_local))).cuda()
    out, launches = {}, {}
    for on in (False, True):
        sharp.set_spin2_scalar(on)
        mp = torch.empty((2, gi.n_local), dtype=torch.float64, device="cuda")
        _run(sharp, sharp.SHARP_Y, alm, mp, ai, gi)   # builds this route's seed table (a launch of its own)
        launches[on] = _run(sharp, sharp.SHARP_Y, alm, mp, ai, gi)
        res = {"Y": mp}
        for name, type in (("Yt", sharp.SHARP_Yt), ("YtW", sharp.SHARP_YtW)):
            a = torch.empty_like(alm)
            _run(sharp, type, a, mp_in, ai, gi)
            res[name] = a
        a = alm_add.clone()
        _run(sharp, sharp.SHARP_Yt, a, mp_in, ai, gi, add=True)
        res["Yt_add"] = a
        out[on] = res
    return out, launches


def _check(out, what):
    import torch
    for name in out[False]:
        ref, new = out[False][name], out[True][name]
        assert torch.isfinite(new).all(), (what, name)
        err = float((new - ref).abs().max() / ref.abs().max())
        assert err <= TOL, f"{name} ({what}): {err:.2e} of the largest value"


@pytest.mark.parametrize("nside,lmax", [(64, 10), (64, 37), (128, 253)])
def test_scalar_route_small_lmax(nside, lmax):
    from commander_b200 import sharp
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    try:
        out, launches = _both_routes(sharp, ai, gi, lmax)
        _check(out, f"nside {nside}, lmax {lmax}")
        # route on: prep_s2s_kernel and one synth0_kernel for Q and U, then prep_s2_kernel and synth2_kernel for the
        # polar ring pairs; route off: prep_s2_kernel and synth2_kernel.  The ring FFTs are the same on both.
        assert launches[True] - launches[False] == 2, launches
    finally:
        sharp.set_spin2_scalar(True)
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


@pytest.mark.parametrize("nside,lmax", [(256, 500), (512, 1000)])
def test_scalar_route_m_and_ring_subset(nside, lmax):
    from commander_b200 import sharp
    rng = np.random.default_rng(nside + 1)
    ms = np.sort(rng.choice(lmax + 1, size=(lmax + 1) // 3, replace=False))
    rings = np.sort(rng.choice(np.arange(2, 4 * nside), size=(4 * nside - 1) * 2 // 5, replace=False))
    rings = np.concatenate([[1], rings])   # the northernmost ring: a polar slot, without its mirror
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
    gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
    try:
        out, launches = _both_routes(sharp, ai, gi, nside)
        _check(out, f"m and ring subset, nside {nside}, lmax {lmax}")
        assert launches[True] - launches[False] == 2, launches
    finally:
        sharp.set_spin2_scalar(True)
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)
