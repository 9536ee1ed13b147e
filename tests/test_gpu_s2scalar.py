"""Spin 2 as scalar sums (cmdr_sht_set_spin2_scalar): the route against the spin-2 kernels on the same inputs.

With the route on, a single-GPU spin-2 transform runs the scalar Legendre kernels on the two premixed coefficient
sequences (phases scaled by 1 / sin^2) and keeps the spin-2 kernels for the polar ring pairs only.  For SHARP_Y, SHARP_Yt,
SHARP_YtW and SHARP_Yt with SHARP_ADD (onto non-zero a_lm) the outputs of both routes must agree to 1e-11 of the largest
value, at nside 512, 1024 and 2048; the launch count shows that the route ran."""
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


@pytest.mark.parametrize("nside,lmax", [(512, 1000), (1024, 2000), (2048, 4000)])
def test_scalar_route_matches_spin2_kernels(nside, lmax):
    import torch
    from commander_b200 import sharp
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    rng = np.random.default_rng(nside)
    alm = torch.from_numpy(rng.standard_normal((2, ai.n_local))).cuda()
    mp_in = torch.from_numpy(rng.standard_normal((2, gi.n_local))).cuda()
    alm_add = torch.from_numpy(rng.standard_normal((2, ai.n_local))).cuda()
    try:
        out, launches = {}, {}
        for on in (False, True):
            sharp.set_spin2_scalar(on)
            mp = torch.empty((2, gi.n_local), dtype=torch.float64, device="cuda")
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
        assert launches[True] != launches[False], "the scalar route did not run"
        for name in out[False]:
            ref, new = out[False][name], out[True][name]
            assert torch.isfinite(new).all(), name
            err = float((new - ref).abs().max() / ref.abs().max())
            assert err <= TOL, f"{name} at nside {nside}: {err:.2e} of the largest value"
    finally:
        sharp.set_spin2_scalar(True)
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)
