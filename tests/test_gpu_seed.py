"""Seed tables of the Legendre kernels: the seeded kernels against the unseeded ones on the same inputs.

With the tables on, every warp of synth0 / anal0 / synth2 / anal2 starts at its first accumulating l from state built
once per plan instead of from the closed-form start values.  The skipped part adds exact zeros, so
  synthesis  the maps are bit-for-bit those of the unseeded kernels;
  analysis   the a_lm agree to the order of the atomic additions (<= 1e-13 relative L2 per component).
Checked at the benchmark size, on a ring subset with an m subset, and through comm_mapinfo; the tables must have been
built (non-zero byte count), i.e. the seeded path was the one that ran."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TOL_ANAL = 1e-13


def _pair(sharp, spin, alm, ai, gi):
    """Y then YtW of `alm` (device, 1 or 2 columns): the map and the a_lm that came back."""
    import torch
    nc = alm.shape[0]
    mp = torch.full((nc, gi.n_local), float("nan"), dtype=torch.float64, device="cuda")
    back = torch.full_like(alm, float("nan"))
    sharp.sharp_execute(sharp.SHARP_Y, spin, nc, alm, ai, mp, gi)
    sharp.sharp_execute(sharp.SHARP_YtW, spin, nc, back, ai, mp, gi)
    torch.cuda.synchronize()
    return mp, back


def _compare(sharp, ai, gi, seed):
    import torch
    rng = np.random.default_rng(seed)
    try:
        for spin in (0, 2):
            alm = torch.from_numpy(rng.standard_normal((1 if spin == 0 else 2, ai.n_local))).cuda()
            sharp.set_legendre_seeds(False)
            m0, a0 = _pair(sharp, spin, alm, ai, gi)
            sharp.set_legendre_seeds(True)
            m1, a1 = _pair(sharp, spin, alm, ai, gi)
            assert torch.equal(m0, m1), f"spin {spin}: seeded synthesis differs"
            for c in range(a0.shape[0]):
                rel = float(torch.linalg.norm(a1[c] - a0[c]) / torch.linalg.norm(a0[c]))
                assert rel <= TOL_ANAL, f"spin {spin} component {c}: seeded analysis rel L2 {rel:.3e}"
    finally:
        sharp.set_legendre_seeds(True)
    assert sharp.legendre_seed_bytes() > 0


def test_seeded_at_benchmark_size(shtlib):
    sharp = shtlib
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(4000)
    gi = sharp.sharp_make_healpix_geom_info(2048)
    try:
        _compare(sharp, ai, gi, 1)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


@pytest.mark.parametrize("nside,lmax", [(256, 700), (512, 1000)])
def test_seeded_on_ring_and_m_subsets(shtlib, nside, lmax):
    sharp = shtlib
    ms = np.arange(1, lmax + 1, 3, dtype=np.int32)             # every third m, m = 0 absent
    rings = np.arange(1, 4 * nside, 2, dtype=np.int32)          # every other ring: pairs with and without a mirror
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
    gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
    try:
        _compare(sharp, ai, gi, 2)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_seeded_through_comm_mapinfo(shtlib):
    import torch
    sharp = shtlib
    from commander_b200 import comm_map, comm_mapinfo
    info = comm_mapinfo(None, 1024, 2000, 3, True)
    m = comm_map(info, device=torch.device("cuda", 0))
    rng = np.random.default_rng(3)
    m.alm.copy_(torch.from_numpy(rng.standard_normal(tuple(m.alm.shape))))
    alm_in = m.alm.clone()
    out = {}
    try:
        for seeds in (False, True):
            sharp.set_legendre_seeds(seeds)
            m.alm.copy_(alm_in)
            m.Y()
            mp = m.map.clone()
            m.YtW()
            torch.cuda.synchronize()
            out[seeds] = (mp, m.alm.clone())
    finally:
        sharp.set_legendre_seeds(True)
    assert torch.equal(out[False][0], out[True][0])
    for c in range(3):
        a0, a1 = out[False][1][c], out[True][1][c]
        assert float(torch.linalg.norm(a1 - a0) / torch.linalg.norm(a0)) <= TOL_ANAL
    assert sharp.legendre_seed_bytes() > 0
