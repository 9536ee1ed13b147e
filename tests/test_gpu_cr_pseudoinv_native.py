"""GPU tests of the pseudo-inverse preconditioner on the native multi-component constrained-realisation system
(cmdr_cr_set_pseudoinv, commander_b200/csrc/cr_multi.cu, through comm_cr.cr_native_multi_system.set_pseudoinv): against
the torch mirror comm_cr.cr_system with precond = 'pseudoinv' and against the same preconditioner composed from
CPU-oracle transforms (tests/test_gpu_cr_multi.py::_oracle_pseudoinv)."""
import numpy as np
import pytest

from test_gpu_cr_multi import _oracle_pseudoinv, _problem
from test_gpu_cr_multi_native import _np, _parts, _problem4, _systems, real_size_problem, rel

pytestmark = pytest.mark.gpu


def _pinv_systems(bands, comps, dev, precond="diagonal"):
    nat, mir = _systems(bands, comps, dev, precond=precond)
    nat.set_pseudoinv(True)
    mir.precond = "pseudoinv"
    return nat, mir


@pytest.mark.parametrize("where", ["host", "device"])
def test_invM_against_mirror_and_oracle(shtlib, cpu_oracle, where):
    """_problem4 (3 IQU bands and a 1-map band; CMB, dust, a 1-map component without prior) against the mirror; the
    3-band _problem, whose bands the oracle composition takes, against the oracle."""
    import torch
    dev = torch.device("cuda", 0)
    conv = (lambda a: a) if where == "host" else (lambda a: torch.as_tensor(a, device=dev))
    bands, comps, rng = _problem4(41)
    nat, mir = _pinv_systems(bands, comps, dev)
    r = rng.standard_normal(nat.ncr)
    got = nat.invM(conv(r))
    assert isinstance(got, np.ndarray) == (where == "host")
    got = _np(got)
    ref = mir.invM(torch.as_tensor(r, device=dev)).cpu().numpy()
    assert rel(got, ref) <= 1e-10, rel(got, ref)
    r2 = rng.standard_normal(nat.ncr)
    a, b = float(r2 @ got), float(r @ _np(nat.invM(conv(r2))))
    assert abs(a - b) <= 1e-11 * max(abs(a), abs(b))
    bands3, comps3, rng3 = _problem(42, False)
    nat3, _ = _pinv_systems(bands3, comps3, dev)
    r3 = rng3.standard_normal(nat3.ncr)
    got3 = _np(nat3.invM(conv(r3)))
    ref3 = np.concatenate([v.ravel() for v in _oracle_pseudoinv(cpu_oracle, bands3, comps3, _parts(comps3, r3))])
    assert rel(got3, ref3) <= 1e-9, rel(got3, ref3)


def test_switch(shtlib):
    """Off gives bit for bit the block preconditioner of a handle that never switched; a handle built without a
    preconditioner switches on (the mirror's result) and back to the identity."""
    import torch
    dev = torch.device("cuda", 0)
    bands, comps, rng = _problem4(43)
    plain, _ = _systems(bands, comps, dev)
    nat, mir = _pinv_systems(bands, comps, dev)
    r = torch.as_tensor(rng.standard_normal(nat.ncr), device=dev)
    zp = nat.invM(r)
    nat.set_pseudoinv(False)
    assert torch.equal(nat.invM(r), plain.invM(r))
    nat.set_pseudoinv(True)                                # the tables are kept: the same result again
    assert rel(nat.invM(r).cpu().numpy(), zp.cpu().numpy()) <= 1e-14
    none, _ = _systems(bands, comps, dev, precond="none")
    assert torch.equal(none.invM(r), r)
    none.set_pseudoinv(True)
    ref = mir.invM(r).cpu().numpy()
    assert rel(none.invM(r).cpu().numpy(), ref) <= 1e-10
    data = [torch.as_tensor(rng.standard_normal((b.get("nmaps", 3), 12 * b["nside"] ** 2)), device=dev) for b in bands]
    b = none.computeRHS(data)
    _, it, h = none.solve(b, maxiter=4, cg_conv_crit="fixed_iter")
    assert it == 4 and len(h) == 5
    none.set_pseudoinv(False)
    assert torch.equal(none.invM(r), r)


def test_with_pixel_mixing(shtlib):
    """Per-pixel mixing maps installed: the pseudo-inverse keeps F_mean, as the mirror's does."""
    import torch
    from test_gpu_cr_mix_native import _mixed
    from test_gpu_cr_mix_native import _systems as _mix_systems
    dev = torch.device("cuda", 0)
    bands, comps, rng = _mixed(44)
    nat, mir = _mix_systems(bands, comps, dev)
    nat.set_pseudoinv(True)
    mir.precond = "pseudoinv"
    r = torch.as_tensor(rng.standard_normal(nat.ncr), device=dev)
    assert rel(nat.invM(r).cpu().numpy(), mir.invM(r).cpu().numpy()) <= 1e-10
    x = torch.as_tensor(rng.standard_normal(nat.ncr), device=dev)
    assert rel(nat.matmulA(x).cpu().numpy(), mir.matmulA(x).cpu().numpy()) <= 1e-12   # the scratch reuse leaves A intact


def test_solve(shtlib):
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps, rng = _problem4(45)
    nat, mir = _pinv_systems(bands, comps, dev)
    data = [torch.as_tensor(rng.standard_normal((b.get("nmaps", 3), 12 * b["nside"] ** 2)) / np.sqrt(b["invN"]), device=dev)
            for b in bands]
    b = nat.computeRHS(data)
    x, it, hist = nat.solve(b, maxiter=500, cg_tol=1e-10)
    xr, itr, histr = solve_cr_eqn_by_CG(mir, b.clone(), maxiter=500, cg_tol=1e-10)
    assert abs(it - itr) <= 1 and 3 < it < 500, (it, itr)
    assert float((x - xr).norm() / xr.norm()) <= 1e-6
    np.testing.assert_allclose(hist[:10], histr[:10], rtol=1e-8)
    n0 = nat.n_matmul
    _, it5, h5 = nat.solve(b, maxiter=5, cg_conv_crit="fixed_iter")
    assert it5 == 5 and len(h5) == 6 and nat.n_matmul - n0 == 6
    # the solution is that of the block-diagonal run
    plain, _ = _systems(bands, comps, dev)
    xd, itd, _ = plain.solve(b, maxiter=500, cg_tol=1e-10)
    assert float((x - xd).norm() / xd.norm()) <= 1e-4
    print("CG iterations to 1e-10: block diagonal", itd, "pseudo-inverse", it)


def test_real_size(shtlib):
    """The real-size sampling group of test_gpu_cr_multi_native: three fixed_iter iterations with the pseudo-inverse,
    native against the mirror."""
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps = real_size_problem(np.random.default_rng(15))
    nat, mir = _pinv_systems(bands, comps, dev)
    rng = np.random.default_rng(46)
    data = [torch.as_tensor(rng.standard_normal((3, 12 * b["nside"] ** 2)), device=dev) for b in bands]
    b = nat.computeRHS(data)
    x, it, h = nat.solve(b, maxiter=3, cg_conv_crit="fixed_iter")
    xr, itr, hr = solve_cr_eqn_by_CG(mir, b.clone(), maxiter=3, cg_conv_crit="fixed_iter")
    assert it == itr == 3
    np.testing.assert_allclose(h, hr, rtol=1e-9)
    assert float((x - xr).norm() / xr.norm()) <= 1e-9
