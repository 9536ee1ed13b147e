"""The bookkeeping of tests/dist_deep_check.py without a GPU: its rank layouts, the union each one is compared on, and
the slicing that maps every rank's local pixels and local packed a_lm onto the single-GPU arrays.  The CPU oracle
stands in for the per-rank engine: the rank slices of its result on the reference handles must equal its result on
each rank's own handles, and the rank sums of the exchange (every rank's m's onto my rings, every rank's rings onto
my m's) must reproduce the reference."""
import numpy as np
import pytest

import dist_deep_check as K
from oracle import sht_def as D

WORLDS = (2, 3, 8)


def _check_structure(name, nside, lmax, world):
    lay = K.layout(name, nside, lmax, world)
    assert len(lay) == world
    assert [(r.tolist(), m.tolist()) for r, m in lay] == \
        [(r.tolist(), m.tolist()) for r, m in K.layout(name, nside, lmax, world)], "not reproducible from the seed"
    all_r = np.concatenate([r for r, _ in lay])
    all_m = np.concatenate([m for _, m in lay])
    assert len(set(all_r.tolist())) == len(all_r), "a ring on two ranks"
    assert len(set(all_m.tolist())) == len(all_m), "an m on two ranks"
    ref_r, ref_m = K.union(lay)
    assert ref_r.tolist() == sorted(all_r.tolist()) and ref_m.tolist() == sorted(all_m.tolist())
    every_r, every_m = list(range(1, 4 * nside)), list(range(lmax + 1))
    pair = {r: min(r, 4 * nside - r) for r in every_r}
    owner = {int(x): k for k, (r, _) in enumerate(lay) for x in r}
    if name == "mapinfo":
        for k, (r, m) in enumerate(lay):
            assert r.tolist() == D.mapinfo_rings(nside, k, world) and m.tolist() == D.mapinfo_ms(lmax, k, world)
    if name in ("mapinfo", "lopsided", "blocks"):
        assert ref_r.tolist() == every_r and ref_m.tolist() == every_m
    if name in ("mapinfo", "lopsided", "subset"):
        # every ring pair on one rank: the distributed work order is the single-GPU order
        for r in owner:
            assert owner[4 * nside - r if r != 2 * nside else r] == owner[r]
    if name == "lopsided":
        assert len(lay[0][0]) == 0 and len(lay[-1][1]) == 0
        assert 2 * nside in lay[-1][0].tolist()
        assert set(range(lmax // 2 + 1)) <= set(lay[0][1].tolist())
        if world == 2:
            assert len(lay[0][1]) == lmax + 1 and len(lay[1][0]) == 4 * nside - 1
        else:
            npairs = [len({pair[int(x)] for x in r}) for r, _ in lay]
            assert len(set(npairs[1:])) > 1, "the pairs are not spread unevenly"
    if name == "subset":
        missing = sorted(set(every_r) - set(ref_r.tolist()))
        assert 0.2 < len({pair[r] for r in missing}) / (2 * nside) < 0.5
        assert all(pair[r] not in {pair[x] for x in ref_r.tolist()} for r in missing), "half a pair left out"
        gap = sorted(set(every_m) - set(ref_m.tolist()))
        assert gap and gap == list(range(gap[0], gap[-1] + 1)), "the m's left out are not one band"
        assert any(r.tolist() != sorted(r.tolist()) for r, _ in lay), "no ring list out of order"
    if name == "blocks":
        for r, m in lay:
            assert r.tolist() == list(range(r[0], r[-1] + 1)) and m.tolist() == list(range(m[0], m[-1] + 1))
        split = sum(owner[r] != owner[4 * nside - r] for r in range(1, 2 * nside))
        assert split > nside, "most pairs must be split between two ranks"
        pix = [int(K.ring_nph(nside, r).sum()) for r, _ in lay]
        assert max(pix) < 1.5 * 12 * nside ** 2 / world
    return lay, ref_r, ref_m


def _check_slicing(nside, lmax, lay, ref_r, ref_m):
    npix, nalm = int(K.ring_nph(nside, ref_r).sum()), int(K.m_count(lmax, ref_m).sum())
    assert npix == D.map_size(nside, ref_r) and nalm == D.alm_count(lmax, ref_m)
    pidx = [K.pix_index(nside, ref_r, r) for r, _ in lay]
    aidx = [K.alm_index(lmax, ref_m, m) for _, m in lay]
    # every reference pixel / coefficient exactly once over the ranks
    assert np.array_equal(np.sort(np.concatenate(pidx)), np.arange(npix))
    assert np.array_equal(np.sort(np.concatenate(aidx)), np.arange(nalm))
    full = ref_r.tolist() == list(range(1, 4 * nside))
    for (r, m), pi, ai in zip(lay, pidx, aidx):
        assert len(pi) == D.map_size(nside, r) and len(ai) == D.alm_count(lmax, m)
        # in list order: the local map is the rank's rings one after the other as listed
        if full:   # the reference is the full sphere: positions are RING pixel numbers
            want = [np.arange(D.healpix_ring(nside, int(x))[4], D.healpix_ring(nside, int(x))[4]
                              + D.healpix_ring(nside, int(x))[2]) for x in r]
            assert np.array_equal(pi, np.concatenate(want) if want else np.zeros(0, dtype=np.int64))
        lm_ref = D.alm_index(lmax, ref_m.tolist())
        assert [lm_ref[i] for i in ai] == D.alm_index(lmax, m.tolist())
        seg = K.segments(K.ring_nph(nside, r))
        assert len(seg) == len(pi) and (len(seg) == 0 or seg[-1] == len(r) - 1)


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", K.LAYOUTS)
def test_layouts_and_slicing(name, world):
    for nside, lmax in ((8, 20), (64, 150), (256, 1100)):
        lay, ref_r, ref_m = _check_structure(name, nside, lmax, world)
        _check_slicing(nside, lmax, lay, ref_r, ref_m)


def test_sizes_and_pipeline_threshold():
    # the smallest nside that takes the chunked host pipeline: 12 nside^2 >= 2^20 ranks (W = 3 exactly on it)
    assert [K.pipeline_nside(w) for w in (2, 3, 4, 8, 12)] == [512, 512, 1024, 1024, 1024]
    assert K.sizes(8, True)[-2:] == [(1024, 1536), (2048, 4000)] and K.sizes(3, False)[-1] == (512, 768)
    # dist.cu get_plan: slots per chunk a multiple of 128, at least 128
    assert K.pipeline_chunks(1024, "8") == 8 and K.pipeline_chunks(2048, "8") == 8
    assert K.pipeline_chunks(2048, "3") == 3 and K.pipeline_chunks(300, "8") == 3 and K.pipeline_chunks(2048, "0") == 8


@pytest.mark.parametrize("world", WORLDS)
@pytest.mark.parametrize("name", K.LAYOUTS)
def test_oracle_as_rank_engine(cpu_oracle, name, world):
    S = cpu_oracle
    nside, lmax = 8, 20
    lay = K.layout(name, nside, lmax, world)
    ref_r, ref_m = K.union(lay)
    rng = np.random.default_rng(5)
    for spin in (0, 2):
        nc = 1 if spin == 0 else 2
        alm = rng.standard_normal((nc, D.alm_count(lmax, ref_m)))
        mp = rng.standard_normal((nc, D.map_size(nside, ref_r)))
        Y = S.execute(S.Y, spin, nside, lmax, alm=alm, rings=ref_r, ms=ref_m)
        Yt = S.execute(S.Yt, spin, nside, lmax, map=mp, rings=ref_r, ms=ref_m)
        pidx = [K.pix_index(nside, ref_r, r) for r, _ in lay]
        aidx = [K.alm_index(lmax, ref_m, m) for _, m in lay]
        for k, (r, m) in enumerate(lay):
            # the rank's slices of the reference == the engine on the rank's own handles
            own = S.execute(S.Y, spin, nside, lmax, alm=alm, rings=r, ms=ref_m) if len(r) else np.zeros((nc, 0))
            assert np.array_equal(own, Y[:, pidx[k]])
            own = S.execute(S.Yt, spin, nside, lmax, map=mp, rings=ref_r, ms=m) if len(m) else np.zeros((nc, 0))
            assert np.array_equal(own, Yt[:, aidx[k]])
            # the exchange: the other ranks' m's (their a_lm slices) onto my rings, my m's from their rings' map slices
            if len(r):
                got = sum(S.execute(S.Y, spin, nside, lmax, alm=np.ascontiguousarray(alm[:, aidx[j]]), rings=r, ms=mj)
                          for j, (_, mj) in enumerate(lay) if len(mj))
                assert np.allclose(got, Y[:, pidx[k]], rtol=0, atol=1e-12 * np.abs(Y).max())
            if len(m):
                got = sum(S.execute(S.Yt, spin, nside, lmax, map=np.ascontiguousarray(mp[:, pidx[j]]), rings=rj, ms=m)
                          for j, (rj, _) in enumerate(lay) if len(rj))
                assert np.allclose(got, Yt[:, aidx[k]], rtol=0, atol=1e-12 * np.abs(Yt).max())
