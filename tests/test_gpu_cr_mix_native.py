"""GPU tests of per-pixel mixing on the native multi-component constrained-realisation system (cmdr_cr_set_mixing_map,
commander_b200/csrc/cr_multi.cu, through comm_cr.cr_native_multi_system(pixel_mixing=True) / set_mixing_map): against the
operator composed from CPU-oracle transforms and against the torch mirror comm_cr.cr_system with the same F."""
import numpy as np
import pytest

from test_gpu_cr_multi import _oracle_A
from test_gpu_cr_multi_native import _np, _oracle_bands, _parts, _problem4, real_size_problem, rel

pytestmark = pytest.mark.gpu


def _mixed(seed):
    """_problem4 (components CMB 3 maps / lmax 40, dust 3 / 32, low-l 1 / 8; bands 16 / 32, 16 / 40, 32 / 48 in IQU and
    8 / 20 in T) with mixed pairs of every shape:
      dust in bands 1 and 2 (IQU, lmax_k < lmax_q: the component's own layout);
      the 1-map component in band 0 (a T-only mix in an IQU band);
      CMB in band 3 (a 3-map component in the 1-map band, lmax_k > lmax_q: the re-pack path);
      CMB in band 0 (IQU, lmax_k > lmax_q: the re-pack path)."""
    bands, comps, rng = _problem4(seed)

    def F(q, scale, nm=3):
        return scale * (1.0 + 0.3 * rng.uniform(size=(nm, 12 * bands[q]["nside"] ** 2)))
    for c in comps:
        c["F"] = [None] * len(bands)
    comps[1]["F"][1] = F(1, 1.0)
    comps[1]["F"][2] = F(2, 2.5)
    comps[2]["F"][0] = F(0, 1.5, 1)
    comps[0]["F"][3] = F(3, 0.8)
    comps[0]["F"][0] = F(0, 1.1)
    return bands, comps, rng


def _systems(bands, comps, dev, F_dev=False, precond="diagonal"):
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, cr_system
    cb = []
    for b in bands:
        nm = b.get("nmaps", 3)
        cb.append(cr_band(comm_mapinfo(None, b["nside"], b["lmax"], nm, nm == 3), torch.as_tensor(b["invN"], device=dev), b["b_l"]))
    def conv(f, nm):      # the mirror uses a map as given: only the rows the pair mixes
        if f is None or hasattr(f, "data_ptr"):
            return None if f is None else f[:nm]
        return torch.as_tensor(f[:nm], device=dev) if F_dev else np.ascontiguousarray(f[:nm])
    cc = [cr_component(comm_mapinfo(None, c["nside"], c["lmax"], c["nmaps"], c["nmaps"] == 3), Cl=c["Cl"], F_mean=c["F_mean"],
                       F=None if c.get("F") is None else [conv(f, min(c["nmaps"], b.get("nmaps", 3))) for f, b in zip(c["F"], bands)])
          for c in comps]
    return cr_native_multi_system(cc, cb, precond=precond, pixel_mixing=True), cr_system(cc, cb, dev)


@pytest.mark.parametrize("F_where", ["host", "device"])
@pytest.mark.parametrize("where", ["host", "device"])
def test_operator_and_rhs(shtlib, cpu_oracle, where, F_where):
    import torch
    dev = torch.device("cuda", 0)
    bands, comps, rng = _mixed(31)
    nat, mir = _systems(bands, comps, dev, F_dev=F_where == "device")
    conv = (lambda a: a) if where == "host" else (lambda a: torch.as_tensor(a, device=dev))
    x = rng.standard_normal(nat.ncr)
    got = nat.matmulA(conv(x))
    assert isinstance(got, np.ndarray) == (where == "host")
    got = _np(got)
    ref = np.concatenate([v.ravel() for v in _oracle_A(cpu_oracle, _oracle_bands(bands), comps, _parts(comps, x))])
    assert rel(got, ref) <= 1e-10, rel(got, ref)
    mref = mir.matmulA(torch.as_tensor(x, device=dev)).cpu().numpy()
    assert rel(got, mref) <= 1e-12, rel(got, mref)
    y = rng.standard_normal(nat.ncr)
    a, b = float(y @ got), float(x @ _np(nat.matmulA(conv(y))))
    assert abs(a - b) <= 1e-11 * max(abs(a), abs(b))
    # right-hand side with both fluctuation terms
    data = [rng.standard_normal((b.get("nmaps", 3), 12 * b["nside"] ** 2)) for b in bands]
    eta = [rng.standard_normal(d.shape) for d in data]
    eta_alm = rng.standard_normal(nat.ncr)
    rhs = _np(nat.computeRHS([conv(d) for d in data], [conv(e) for e in eta], conv(eta_alm)))
    T = lambda a: torch.as_tensor(a, device=dev)   # noqa: E731
    rref = mir.computeRHS([T(d) for d in data], [T(e) for e in eta], T(eta_alm)).cpu().numpy()
    assert rel(rhs, rref) <= 1e-12, rel(rhs, rref)


def test_setter(shtlib):
    """Clearing every map gives the F_mean operator bit for bit, with the launches of a handle that never had one;
    replacing a map gives the mirror built with the new one."""
    import torch
    from commander_b200 import sharp
    dev = torch.device("cuda", 0)
    bands, comps, rng = _mixed(32)
    plain = [dict(c, F=None) for c in comps]
    fresh, _ = _systems(bands, plain, dev)
    nat, _ = _systems(bands, comps, dev)
    x = torch.as_tensor(rng.standard_normal(nat.ncr), device=dev)
    fresh.matmulA(x)                                # first calls build each plan's seed tables
    y_mixed = nat.matmulA(x)
    for k, c in enumerate(comps):
        for q, f in enumerate(c["F"]):
            if f is not None:
                nat.set_mixing_map(q, k, None)
    nat.set_mixing_map(1, 2, None)                  # clearing a pair that has no map is a no-op

    def launches(s):
        n0 = sharp.launch_count()
        y = s.matmulA(x)
        torch.cuda.synchronize()
        return y, sharp.launch_count() - n0
    y0, n_fresh = launches(fresh)
    y1, n_cleared = launches(nat)
    assert n_fresh == n_cleared
    # bit for bit wherever the fresh handle reproduces itself (the analysis kernels sum ring chunks with atomics)
    if torch.equal(y0, fresh.matmulA(x)):
        assert torch.equal(y0, y1)
    assert rel(y1.cpu().numpy(), y0.cpu().numpy()) <= 1e-14
    assert rel(y_mixed.cpu().numpy(), y0.cpu().numpy()) > 1e-3
    # set again, then replace one map: the mirror built with the new maps
    for k, c in enumerate(comps):
        for q, f in enumerate(c["F"]):
            if f is not None:
                nat.set_mixing_map(q, k, f)
    assert rel(nat.matmulA(x).cpu().numpy(), y_mixed.cpu().numpy()) <= 1e-14
    comps[1]["F"][2] = 0.5 * (1.0 + rng.uniform(size=(3, 12 * bands[2]["nside"] ** 2)))
    nat.set_mixing_map(2, 1, torch.as_tensor(comps[1]["F"][2], device=dev))
    comps[2]["F"][3] = 2.0 + rng.uniform(size=(1, 12 * bands[3]["nside"] ** 2))   # a new pair
    nat.set_mixing_map(3, 2, comps[2]["F"][3])
    _, mir = _systems(bands, comps, dev)
    assert rel(nat.matmulA(x).cpu().numpy(), mir.matmulA(x).cpu().numpy()) <= 1e-12


def test_solve(shtlib):
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps, rng = _mixed(33)
    nat, mir = _systems(bands, comps, dev)
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


def test_real_size(shtlib):
    """The real-size sampling group of test_gpu_cr_multi_native with dust mixed per pixel in all three bands: three
    fixed_iter iterations, native against the mirror."""
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps = real_size_problem(np.random.default_rng(15))
    rng = np.random.default_rng(34)
    comps[1]["F"] = [torch.as_tensor(f * (1.0 + 0.3 * rng.uniform(size=(3, 12 * b["nside"] ** 2))), device=dev)
                     for f, b in zip((0.2, 0.9, 2.8), bands)]
    nat, mir = _systems(bands, comps, dev)
    data = [torch.as_tensor(rng.standard_normal((3, 12 * b["nside"] ** 2)), device=dev) for b in bands]
    b = nat.computeRHS(data)
    assert rel(b.cpu().numpy(), mir.computeRHS(data).cpu().numpy()) <= 1e-12
    x, it, h = nat.solve(b, maxiter=3, cg_conv_crit="fixed_iter")
    xr, itr, hr = solve_cr_eqn_by_CG(mir, b.clone(), maxiter=3, cg_conv_crit="fixed_iter")
    assert it == itr == 3
    np.testing.assert_allclose(h, hr, rtol=1e-9)
    assert float((x - xr).norm() / xr.norm()) <= 1e-9
