"""Deterministic mode (cmdr_sht_set_deterministic / CMDR_SHT_DETERMINISTIC=1): the analysis kernels store per-warp-block
partials and an ordered reduce adds them to the a_lm (commander_b200/csrc/det.h), so an analysis gives the same bits on
every call, on every host path, with the seed tables on or off, and SHARP_ADD adds exactly the plain result.  The mode is
switched on inside each test and restored afterwards; the end-to-end checks run in fresh processes with the variable set."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def det(shtlib):
    prev = shtlib.deterministic()
    shtlib.set_deterministic(True)
    try:
        yield shtlib
    finally:
        shtlib.set_deterministic(prev)
        shtlib.set_spin2_scalar(True)
        shtlib.set_legendre_seeds(True)


def _rel(a, b):
    import torch
    return float(torch.linalg.norm(a - b) / torch.linalg.norm(b))


def _anal(sharp, job, spin, mp, ai, gi, out=None, add=False):
    """Analysis of the device map `mp` (1 or 2 columns) into a fresh a_lm tensor (or into `out`)."""
    import torch
    nc = mp.shape[0]
    if out is None:
        out = torch.full((nc, ai.n_local), float("nan"), dtype=torch.float64, device="cuda")
    sharp.sharp_execute(job, spin, nc, out, ai, mp, gi, add=add)
    torch.cuda.synchronize()
    return out


def _unrelated(sharp):
    """A transform on other handles, then every cached buffer dropped: the next call starts from fresh scratch."""
    import torch
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(100)
    gi = sharp.sharp_make_healpix_geom_info(64)
    try:
        mp = torch.ones((2, gi.n_local), dtype=torch.float64, device="cuda")
        _anal(sharp, sharp.SHARP_YtW, 2, mp, ai, gi)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)
    torch.cuda.synchronize()
    sharp.lib().cmdr_sht_release_caches()


@pytest.mark.parametrize("spin,s2s", [(0, True), (2, True), (2, False), (3, True)])
def test_repeatable(det, spin, s2s):
    import torch
    sharp = det
    sharp.set_spin2_scalar(s2s)
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(2000)
    gi = sharp.sharp_make_healpix_geom_info(1024)
    try:
        rng = np.random.default_rng(10 + spin)
        mp = torch.from_numpy(rng.standard_normal((1 if spin == 0 else 2, gi.n_local))).cuda()
        for job in (sharp.SHARP_YtW, sharp.SHARP_Yt):
            runs = []
            for _ in range(3):
                runs.append(_anal(sharp, job, spin, mp, ai, gi))
                _unrelated(sharp)
            assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2]), f"spin {spin} job {job}"
        # the default mode agrees to the rounding of its atomic additions
        sharp.set_deterministic(False)
        ref = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi)
        sharp.set_deterministic(True)
        got = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi)
        for c in range(ref.shape[0]):
            assert _rel(got[c], ref[c]) <= 1e-13, (spin, c)
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_iqu_target_size_and_host_paths(det):
    """IQU at nside 2048 / lmax 4000: repeatable, and the same bits from device, pinned and pageable arrays, through
    sharp_execute (the chunked host path's size), cmdr_sht_execute_iqu, _iqu_batch and comm_map.YtW."""
    import torch
    sharp = det
    from commander_b200 import comm_map, comm_mapinfo
    info = comm_mapinfo(None, 2048, 4000, 3, True)
    gT, gP, ai = info.geom_info_T, info.geom_info_P, info.alm_info
    rng = np.random.default_rng(20)
    mp_h = rng.standard_normal((3, gT.n_local))
    mp = torch.from_numpy(mp_h).cuda()
    dev = []
    for _ in range(3):
        a = torch.full((3, ai.n_local), float("nan"), dtype=torch.float64, device="cuda")
        sharp.execute_iqu(sharp.SHARP_YtW, a, mp, gT, gP, ai)
        torch.cuda.synchronize()
        dev.append(a)
        _unrelated(sharp)
    assert torch.equal(dev[0], dev[1]) and torch.equal(dev[0], dev[2])
    ref = dev[0].cpu()
    # sharp_execute per spin, device / pinned / pageable
    mp_pin = torch.from_numpy(mp_h).pin_memory()
    for kind in ("device", "pinned", "pageable"):
        for spin, cols in ((0, slice(0, 1)), (2, slice(1, 3))):
            g = gT if spin == 0 else gP
            if kind == "device":
                a = torch.empty((cols.stop - cols.start, ai.n_local), dtype=torch.float64, device="cuda")
                m = mp[cols].contiguous()
            elif kind == "pinned":
                a = torch.empty((cols.stop - cols.start, ai.n_local), dtype=torch.float64).pin_memory()
                m = mp_pin[cols].contiguous().pin_memory()
            else:
                a = np.empty((cols.stop - cols.start, ai.n_local))
                m = np.ascontiguousarray(mp_h[cols])
            sharp.sharp_execute(sharp.SHARP_YtW, spin, cols.stop - cols.start, a, ai, m, g)
            torch.cuda.synchronize()
            got = torch.as_tensor(a).cpu()
            assert torch.equal(got, ref[cols]), f"sharp_execute {kind} spin {spin}"
    # fused IQU from host arrays, the batch entry point, comm_map
    a = np.empty((3, ai.n_local))
    sharp.execute_iqu(sharp.SHARP_YtW, a, mp_h, gT, gP, ai)
    assert torch.equal(torch.from_numpy(a), ref)
    outs = [np.empty((3, ai.n_local)) for _ in range(2)]
    sharp.execute_iqu_batch(sharp.SHARP_YtW, outs, [mp_h, mp_h], gT, gP, ai)
    for o in outs:
        assert torch.equal(torch.from_numpy(o), ref)
    cm = comm_map(info, device=torch.device("cuda", 0))
    cm.map.copy_(mp)
    cm.YtW()
    torch.cuda.synchronize()
    assert torch.equal(cm.alm.cpu(), ref)


@pytest.mark.parametrize("nside,lmax,subset", [(1024, 2000, False), (256, 700, True), (512, 1000, True)])
def test_seed_tables_on_and_off(det, nside, lmax, subset):
    import torch
    sharp = det
    ms = np.arange(1, lmax + 1, 3, dtype=np.int32) if subset else None
    rings = np.arange(1, 4 * nside, 2, dtype=np.int32) if subset else None
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
    gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
    try:
        rng = np.random.default_rng(30)
        for spin in (0, 2):
            mp = torch.from_numpy(rng.standard_normal((1 if spin == 0 else 2, gi.n_local))).cuda()
            sharp.set_legendre_seeds(False)
            a0 = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi)
            sharp.set_legendre_seeds(True)
            a1 = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi)
            assert torch.equal(a0, a1), f"spin {spin}"
        assert sharp.legendre_seed_bytes() > 0
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_add_is_prior_plus_plain(det):
    import torch
    sharp = det
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(700)
    gi = sharp.sharp_make_healpix_geom_info(256)
    try:
        rng = np.random.default_rng(40)
        for spin in (0, 2):
            nc = 1 if spin == 0 else 2
            mp = torch.from_numpy(rng.standard_normal((nc, gi.n_local))).cuda()
            prior = torch.from_numpy(rng.standard_normal((nc, ai.n_local))).cuda()
            plain = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi)
            acc = _anal(sharp, sharp.SHARP_YtW, spin, mp, ai, gi, out=prior.clone(), add=True)
            assert torch.equal(acc, prior + plain), f"spin {spin}"
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_against_oracle(det, cpu_oracle):
    import torch
    sharp = det
    S = cpu_oracle
    nside, lmax = 64, 128
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    try:
        rng = np.random.default_rng(50)
        for spin in (0, 2):
            mp_h = rng.standard_normal((1 if spin == 0 else 2, gi.n_local))
            got = _anal(sharp, sharp.SHARP_YtW, spin, torch.from_numpy(mp_h).cuda(), ai, gi).cpu().numpy()
            ref = S.execute(S.YtW, spin, nside, lmax, map=mp_h)
            assert np.linalg.norm(got - ref) / np.linalg.norm(ref) <= 1e-10, spin
    finally:
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def test_mix_and_invn_diag(det):
    import torch
    sharp = det
    from commander_b200 import comm_mapinfo
    info = comm_mapinfo(None, 512, 1000, 3, True)
    gT, gP, ai = info.geom_info_T, info.geom_info_P, info.alm_info
    rng = np.random.default_rng(60)
    alm0 = torch.from_numpy(rng.standard_normal((3, ai.n_local))).cuda()
    F = torch.from_numpy(1.0 + 0.3 * rng.uniform(size=(3, gT.n_local))).cuda()
    mixed = []
    for _ in range(3):
        a = alm0.clone()
        sharp.mix(a, F, gT, gP, ai, nmaps=3)
        torch.cuda.synchronize()
        mixed.append(a)
        _unrelated(sharp)
    assert torch.equal(mixed[0], mixed[1]) and torch.equal(mixed[0], mixed[2])
    a_l0 = rng.standard_normal((3, 1001)) * 1e-3
    a_l0[:, 0] = 1.0
    outs = []
    for _ in range(3):
        o = torch.zeros((3, ai.n_local), dtype=torch.float64, device="cuda")
        sharp.invN_diag(a_l0, 12 * 512 ** 2, ai, o)
        outs.append(o)
        _unrelated(sharp)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    sharp.set_deterministic(False)
    ref = torch.zeros((3, ai.n_local), dtype=torch.float64, device="cuda")
    sharp.invN_diag(a_l0, 12 * 512 ** 2, ai, ref)
    sharp.set_deterministic(True)
    for c in range(3):
        assert _rel(outs[0][c], ref[c]) <= 1e-12


_E2E = r"""
import sys
import numpy as np
import torch
sys.path[:0] = [{root!r}, {tests!r}]
from commander_b200 import comm_mapinfo, sharp
from commander_b200.comm_cr import cr_native_system
from test_gpu_cr_mix_native import _mixed, _systems
assert sharp.deterministic()
dev = torch.device("cuda", 0)
# 3-band x 3-component system with per-pixel mixing and the pseudo-inverse preconditioner
bands, comps, rng = _mixed(70)
nat, _ = _systems(bands, comps, dev)
nat.set_pseudoinv(True)
data = [torch.as_tensor(rng.standard_normal((b.get("nmaps", 3), 12 * b["nside"] ** 2)) / np.sqrt(b["invN"]), device=dev)
        for b in bands]
b = nat.computeRHS_draw(data, 11, 4)
x, it, hist = nat.solve(b, maxiter=30, cg_conv_crit="fixed_iter")
# one-component handle with the diagonal preconditioner
info = comm_mapinfo(None, 32, 64, 3, True)
npix = 12 * 32 ** 2
invN = [torch.as_tensor(1.0 + rng.uniform(size=(3, npix)), device=dev) for _ in range(2)]
b_l = [np.ones((65, 3)) * f for f in (1.0, 0.8)]
l = np.arange(65, dtype=np.float64)
one = cr_native_system(info, invN, b_l, Cl=np.stack([20.0 / (l * (l + 1) + 1.0)] * 3, axis=1), precond="diagonal")
d1 = [torch.as_tensor(rng.standard_normal((3, npix)), device=dev) for _ in range(2)]
b1 = one.computeRHS_draw(d1, 11, 4)
x1, it1, hist1 = one.solve(b1, maxiter=30, cg_conv_crit="fixed_iter")
np.savez({out!r}, x=x.cpu().numpy(), hist=np.array(hist), x1=x1.cpu().numpy(), hist1=np.array(hist1), it=[it, it1])
"""


def _fresh(tmp_path, name, det_env):
    out = str(tmp_path / f"{name}.npz")
    env = dict(os.environ)
    env.pop("CMDR_SHT_DETERMINISTIC", None)
    if det_env:
        env["CMDR_SHT_DETERMINISTIC"] = "1"
    code = _E2E.format(root=ROOT, tests=os.path.join(ROOT, "tests"), out=out)
    subprocess.run([sys.executable, "-c", code], check=True, env=env, cwd=ROOT, timeout=900)
    return np.load(out)


def test_draw_and_solve_in_fresh_processes(shtlib, tmp_path):
    r1 = _fresh(tmp_path, "a", True)
    r2 = _fresh(tmp_path, "b", True)
    assert list(r1["it"]) == [30, 30]
    for k in ("x", "hist", "x1", "hist1"):
        assert np.array_equal(r1[k], r2[k]), k
    assert np.all(np.isfinite(r1["hist"])) and r1["hist"][-1] < r1["hist"][0]


def test_off_without_the_variable(shtlib):
    env = dict(os.environ)
    env.pop("CMDR_SHT_DETERMINISTIC", None)
    code = f"import sys; sys.path.insert(0, {ROOT!r}); from commander_b200 import sharp; print(int(sharp.deterministic()))"
    out = subprocess.run([sys.executable, "-c", code], check=True, env=env, capture_output=True, text=True, timeout=300)
    assert out.stdout.strip() == "0"
