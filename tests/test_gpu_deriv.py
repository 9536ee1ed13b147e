"""SHARP_ALM2MAP_DERIV1 on one GPU: {d_theta T, d_phi T / sin theta} of a spin-0 a_lm set.

  closed forms     a_10 = 1, a dipole d.n, zonal a_l0 (the phi map vanishes)
  value by value   synthesis probes of slam_ref.probe_set, one m at a time, against the mpmath gradient reference of
                   tests/deriv_ref.py (built from the spin-0 functions only), with the bounds of test_gpu_deep_parity.py
  spin-1 identity  against the general spin-1 SHARP_Y with E = -sqrt(l(l+1)) a, B = 0 built through the public API, and
                   against the CPU oracle's spin-1 synthesis of the same E (also on comm_mapinfo ring / m subsets)
  entry points     device pointers, cmdr_sht_execute_dev on a side stream, pinned and pageable host arrays (chunked
                   pipeline at nside 512), SHARP_ADD, empty m lists, a NULL second a_lm pointer, opcnt."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import sht_def as D

import deriv_ref as G
import slam_ref as R

pytestmark = pytest.mark.gpu

EPS = 1e-11          # per value, relative to the probe's scale, off the pole
EPS_POLAR = 5e-9     # sin(theta) < 0.01: the rounded-z effect of DESIGN 8 (test_gpu_deep_parity.py EPS_POLAR)


def _der1(sharp, alm, ai, gi, out=None, add=False):
    import torch
    if out is None:
        out = torch.full((2, gi.n_local), float("nan"), dtype=torch.float64, device="cuda")
    sharp.alm2map_der1(alm, ai, out, gi, add=add)
    torch.cuda.synchronize()
    return out


def _pix_angles(nside, rings=None):
    rings = range(1, 4 * nside) if rings is None else rings
    th, ph = [], []
    for r in rings:
        cth, sth, nph, phi0, _ = D.healpix_ring(nside, r)
        th.append(np.full(nph, math.atan2(sth, cth)))
        ph.append(phi0 + 2 * np.pi * np.arange(nph) / nph)
    return np.concatenate(th), np.concatenate(ph)


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def test_closed_forms(shtlib):
    import torch
    sharp = shtlib
    nside, lmax = 64, 20
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    th, ph = _pix_angles(nside)
    st, ct = np.sin(th), np.cos(th)
    idx = {lm: i for i, lm in enumerate(D.alm_index(lmax, range(lmax + 1)))}
    try:
        # a_10 = 1: T = sqrt(3/4pi) cos(theta)
        alm = torch.zeros((1, ai.n_local), dtype=torch.float64, device="cuda")
        alm[0, idx[(1, 0)]] = 1.0
        g = _der1(sharp, alm, ai, gi).cpu().numpy()
        assert np.abs(g[0] + math.sqrt(3 / (4 * math.pi)) * st).max() <= 1e-14
        assert np.abs(g[1]).max() <= 1e-15
        # dipole T = d.n in the real-packed basis: a_10 = sqrt(4pi/3) d_z, a_11 = -sqrt(4pi/3) d_x, a_1-1 = sqrt(4pi/3) d_y
        d = np.array([0.3, -1.7, 0.9])
        f = math.sqrt(4 * math.pi / 3)
        alm.zero_()
        alm[0, idx[(1, 0)]] = f * d[2]
        alm[0, idx[(1, 1)]] = -f * d[0]
        alm[0, idx[(1, -1)]] = f * d[1]
        T = torch.zeros((1, gi.n_local), dtype=torch.float64, device="cuda")
        sharp.sharp_execute(sharp.SHARP_Y, 0, 1, alm, ai, T, gi)
        T = T.cpu().numpy()[0]
        assert np.abs(T - (d[0] * st * np.cos(ph) + d[1] * st * np.sin(ph) + d[2] * ct)).max() <= 1e-14
        g = _der1(sharp, alm, ai, gi).cpu().numpy()
        assert np.abs(g[0] - (d[0] * ct * np.cos(ph) + d[1] * ct * np.sin(ph) - d[2] * st)).max() <= 1e-14
        assert np.abs(g[1] - (-d[0] * np.sin(ph) + d[1] * np.cos(ph))).max() <= 1e-14
        # zonal a_l0 only: no phi dependence
        rng = np.random.default_rng(3)
        alm.zero_()
        a0 = rng.standard_normal(lmax + 1)
        alm[0, :lmax + 1] = torch.from_numpy(a0)
        g = _der1(sharp, alm, ai, gi).cpu().numpy()
        assert np.abs(g[1]).max() <= 1e-15 * np.abs(a0).sum()
        assert np.abs(g[0]).max() > 0
        # l = 0 contributes nothing: exactly zero maps
        alm.zero_()
        alm[0, 0] = 1.0
        g = _der1(sharp, alm, ai, gi).cpu().numpy()
        assert np.all(g == 0.0)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


@pytest.mark.parametrize("nside,lmax", [(2048, 4000), (1024, 2048)])
def test_deriv1_value_by_value(shtlib, nside, lmax):
    import torch
    sharp = shtlib
    pairs = R.probe_set(nside, lmax, 1, full=True)
    G.prefetch(nside, lmax, pairs)
    rng = np.random.default_rng(nside + lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    out = torch.empty((2, gi.n_local), dtype=torch.float64, device="cuda")
    recs = []
    try:
        for m in sorted({m for _, m in pairs}):
            rs = sorted(r for r, mm in pairs if mm == m)
            ns = 1 if m == 0 else 2
            a = rng.standard_normal((1, ns, lmax + 1))
            a[:, :, :m] = 0.0
            if m == 0:
                a[0, 0, 0] = 5.0                      # l = 0 must contribute nothing
            ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=[m])
            alm = torch.from_numpy(np.ascontiguousarray(R.pack({m: a}, lmax, [m]))).cuda()
            out.fill_(float("nan"))
            _der1(sharp, alm, ai, gi, out)
            sharp.sharp_destroy_alm_info(ai)
            for r in rs:
                _, _, nph, _, ofs = D.healpix_ring(nside, r)
                got = out[:, ofs:ofs + nph].cpu().numpy()
                ex = G.expected_gradient(nside, r, lmax, m, a[0])
                cth, sth = R.ring_trig(nside, r)
                g = G.grad_columns(lmax, m, cth, sth)
                typ = float(np.sqrt(max(np.sum((a[0, k] * g[f]) ** 2) for k in range(ns) for f in range(2))))
                cut = m > R.mlim_for_ring(lmax, 1, sth, cth)
                fl = R.FLOOR * float(np.abs(a).sum())
                d = np.abs(got - ex)
                recs.append(dict(ring=r, m=m, cut=cut, S=max(float(np.abs(ex).max()), typ), polar=sth < R.POLAR_STH,
                                 exabs=max(float((d - fl).max()), 0.0), zero_ok=bool(np.all(got == 0)) if cut else True))
    finally:
        sharp.sharp_destroy_geom_info(gi)
    ring_scale = {}
    for q in recs:
        ring_scale[q["ring"]] = max(ring_scale.get(q["ring"], 0.0), q["S"])
    bad, worst = [], {}
    for q in recs:
        S = ring_scale[q["ring"]] if q["cut"] else q["S"]
        q["excess"] = q["exabs"] / S if S > 0 else q["exabs"]
        k = "polar" if q["polar"] else "other"
        worst[k] = max(worst.get(k, 0.0), q["excess"])
        if not q["zero_ok"] or not q["excess"] <= (EPS_POLAR if q["polar"] else EPS):
            bad.append(q)
    print(f"\nDERIV1 nside {nside} lmax {lmax}: {len(recs)} readings, worst excess {worst}")
    assert not bad, f"{len(bad)} of {len(recs)} out of bounds, e.g. " + "; ".join(
        f"ring {q['ring']} m {q['m']}: {q['excess']:.2e} zero_ok={q['zero_ok']}" for q in bad[:8])


def test_deriv1_matches_general_spin1(shtlib):
    import torch
    sharp = shtlib
    nside, lmax = 2048, 4000
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    try:
        rng = np.random.default_rng(5)
        a = rng.standard_normal((1, ai.n_local))
        alm = torch.from_numpy(a).cuda()
        got = _der1(sharp, alm, ai, gi)
        eb = torch.zeros((2, ai.n_local), dtype=torch.float64, device="cuda")
        eb[0] = torch.from_numpy(G.e_of_alm(a[0], lmax, range(lmax + 1))).cuda()
        ref = torch.zeros((2, gi.n_local), dtype=torch.float64, device="cuda")
        sharp.sharp_execute(sharp.SHARP_Y, 1, 2, eb, ai, ref, gi)
        torch.cuda.synchronize()
        for c in range(2):
            e = float(torch.linalg.norm(got[c] - ref[c]) / torch.linalg.norm(ref[c]))
            print(f"\nDERIV1 vs spin-1 Y, map {c}: {e:.2e}")
            assert e <= 1e-12
        assert torch.equal(alm, torch.from_numpy(a).cuda())
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


@pytest.mark.parametrize("nside,lmax,rank", [(1024, 2048, None), (512, 1024, 0), (512, 1024, 2)])
def test_deriv1_matches_oracle_composition(shtlib, cpu_oracle, nside, lmax, rank):
    """DERIV1 = the oracle's spin-1 synthesis of E = -sqrt(l(l+1)) a, B = 0 (full sphere, or the rings and m's of
    comm_mapinfo rank `rank` of 3)."""
    sharp, S = shtlib, cpu_oracle
    rings = None if rank is None else D.mapinfo_rings(nside, rank, 3)
    ms = list(range(lmax + 1)) if rank is None else D.mapinfo_ms(lmax, rank, 3)
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
    gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
    try:
        rng = np.random.default_rng(nside + (rank or 0))
        a = rng.standard_normal((1, ai.n_local))
        got = np.zeros((2, gi.n_local))
        sharp.alm2map_der1(a, ai, got, gi)
        eb = np.zeros((2, ai.n_local))
        eb[0] = G.e_of_alm(a[0], lmax, ms)
        ref = S.execute(S.Y, 1, nside, lmax, alm=eb, rings=rings, ms=None if rank is None else ms)
        for c in range(2):
            assert _rel(got[c], ref[c]) <= 1e-10, (c, _rel(got[c], ref[c]))
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_deriv1_entry_points(shtlib):
    import torch
    sharp = shtlib
    L = sharp.lib()
    nside, lmax = 512, 1024                       # 3.1 M pixels: the chunked host pipeline runs
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    try:
        rng = np.random.default_rng(9)
        a = rng.standard_normal((1, ai.n_local))
        a_keep = a.copy()
        alm_d = torch.from_numpy(a).cuda()
        ref = _der1(sharp, alm_d, ai, gi).cpu().numpy()
        assert np.all(np.isfinite(ref))
        outs = {}
        # cmdr_sht_execute_dev on a side stream, a_lm table with a NULL second entry
        s = torch.cuda.Stream()
        md = torch.full((2, gi.n_local), float("nan"), dtype=torch.float64, device="cuda")
        ap = (C.c_void_p * 2)(alm_d.data_ptr(), None)
        mp_ = (C.c_void_p * 2)(md[0].data_ptr(), md[1].data_ptr())
        torch.cuda.synchronize()
        L.cmdr_sht_execute_dev(sharp.SHARP_ALM2MAP_DERIV1, 0, ap, mp_, gi.handle, ai.handle, sharp.SHARP_DP,
                               C.c_void_p(s.cuda_stream))
        s.synchronize()
        outs["execute_dev"] = md.cpu().numpy()
        # pinned host arrays (chunked pipeline)
        ah = torch.from_numpy(a).pin_memory()
        mh = torch.full((2, gi.n_local), float("nan"), dtype=torch.float64).pin_memory()
        sharp.alm2map_der1(ah.numpy(), ai, mh.numpy(), gi)
        outs["pinned"] = mh.numpy().copy()
        assert np.array_equal(ah.numpy(), a_keep)
        # pageable numpy arrays, through sharp_execute with a NULL second a_lm pointer and opcnt
        mn = np.full((2, gi.n_local), np.nan)
        ap = (C.c_void_p * 2)(a.ctypes.data, None)
        mp_ = (C.c_void_p * 2)(mn[0].ctypes.data, mn[1].ctypes.data)
        oc = C.c_ulonglong(0)
        L.sharp_execute(sharp.SHARP_ALM2MAP_DERIV1, 7, ap, mp_, gi.handle, ai.handle, sharp.SHARP_DP, None, C.byref(oc))
        outs["pageable"] = mn
        nlm = sum(lmax + 1 - m for m in range(lmax + 1))
        assert oc.value == int(nlm * (2 * nside - 0.5) * 20.0)
        assert np.array_equal(a, a_keep)
        for k, v in outs.items():
            assert _rel(v, ref) <= 1e-14, (k, _rel(v, ref))
        # SHARP_ADD onto non-zero maps, device and host
        base = rng.standard_normal((2, gi.n_local))
        md = torch.from_numpy(base.copy()).cuda()
        _der1(sharp, alm_d, ai, gi, md, add=True)
        assert _rel(md.cpu().numpy(), base + ref) <= 1e-14
        mn = base.copy()
        sharp.alm2map_der1(a, ai, mn, gi, add=True)
        assert _rel(mn, base + ref) <= 1e-14
        assert torch.equal(alm_d.cpu(), torch.from_numpy(a_keep))
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_deriv1_empty_lists(shtlib):
    import torch
    sharp = shtlib
    nside, lmax = 32, 40
    a0 = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=[])
    gi = sharp.sharp_make_healpix_geom_info(nside)
    g0 = sharp.sharp_make_healpix_geom_info(nside, rings=[])
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    try:
        out = _der1(sharp, torch.zeros((1, 0), dtype=torch.float64, device="cuda"), a0, gi).cpu().numpy()
        assert np.all(out == 0.0)
        host = np.full((2, gi.n_local), np.nan)
        sharp.alm2map_der1(np.zeros((1, 0)), a0, host, gi)
        assert np.all(host == 0.0)
        alm = torch.ones((1, ai.n_local), dtype=torch.float64, device="cuda")
        out = _der1(sharp, alm, ai, g0)
        assert out.shape == (2, 0)
    finally:
        for h in (a0, ai):
            sharp.sharp_destroy_alm_info(h)
        for h in (gi, g0):
            sharp.sharp_destroy_geom_info(h)
