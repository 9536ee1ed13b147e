"""GPU tests of the native multi-component constrained-realisation system (cmdr_cr_setup_multi, commander_b200/csrc/
cr_multi.cu, through comm_cr.cr_native_multi_system): against the operator composed from CPU-oracle transforms, against
the torch mirror comm_cr.cr_system, and, for one component, against the fused one-component system cr_native_system."""
import numpy as np
import pytest

from test_gpu_cr_multi import _lm, _oracle_A, _problem

pytestmark = pytest.mark.gpu


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _np(v):
    return v if isinstance(v, np.ndarray) else v.cpu().numpy()


def _problem4(seed):
    """_problem's 3 bands / 3 components plus a temperature-only band (nmaps 1, its own nside / lmax / beam)."""
    from commander_b200.comm_cr import gaussian_beam
    bands, comps, rng = _problem(seed, False)
    npix = 12 * 8 ** 2
    bands.append(dict(nside=8, lmax=20, fwhm=700.0, sig=0.8, nmaps=1, b_l=gaussian_beam(20, 700.0, 3),
                      invN=(1.0 / (0.8 * (1.0 + 0.5 * rng.uniform(size=(1, npix))))) ** 2))
    for c in comps:
        c["F_mean"] = np.vstack([c["F_mean"], c["F_mean"][-1:] * 0.8])
    return bands, comps, rng


def _oracle_bands(bands):
    """A band of one map is a band of three whose Q, U maps carry no weight (N^-1 = 0): same operator."""
    out = []
    for b in bands:
        if b.get("nmaps", 3) == 1:
            b = dict(b, invN=np.vstack([b["invN"], np.zeros((2, b["invN"].shape[1]))]))
        out.append(b)
    return out


def _systems(bands, comps, dev, precond="diagonal"):
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, cr_system
    cb = []
    for b in bands:
        nm = b.get("nmaps", 3)
        cb.append(cr_band(comm_mapinfo(None, b["nside"], b["lmax"], nm, nm == 3), torch.as_tensor(b["invN"], device=dev), b["b_l"]))
    cc = [cr_component(comm_mapinfo(None, c["nside"], c["lmax"], c["nmaps"], c["nmaps"] == 3), Cl=c["Cl"], F_mean=c["F_mean"])
          for c in comps]
    return cr_native_multi_system(cc, cb, precond=precond), cr_system(cc, cb, dev)


def _parts(comps, v):
    out, o = [], 0
    for c in comps:
        n = c["nmaps"] * _lm(c["lmax"])[0].size
        out.append(v[o:o + n].reshape(c["nmaps"], -1)); o += n
    return out


@pytest.mark.parametrize("where", ["host", "device"])
def test_operator_and_rhs(shtlib, cpu_oracle, where):
    import torch
    dev = torch.device("cuda", 0)
    bands, comps, rng = _problem4(11)
    nat, mir = _systems(bands, comps, dev)
    assert nat.ncr == mir.ncr
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
    rhs0 = _np(nat.computeRHS([conv(d) for d in data]))
    assert rel(rhs0, mir.computeRHS([T(d) for d in data]).cpu().numpy()) <= 1e-12


def test_block_preconditioner(shtlib):
    import torch
    dev = torch.device("cuda", 0)
    bands, comps, rng = _problem4(12)
    nat, mir = _systems(bands, comps, dev)
    r = torch.as_tensor(rng.standard_normal(nat.ncr), device=dev)
    got = nat.invM(r).cpu().numpy()
    ref = mir.invM(r).cpu().numpy()
    assert rel(got, ref) <= 1e-10, rel(got, ref)
    r2 = rng.standard_normal(nat.ncr)
    a, b = float(r2 @ got), float(r.cpu().numpy() @ nat.invM(r2))
    assert abs(a - b) <= 1e-11 * max(abs(a), abs(b))
    none, _ = _systems(bands, comps, dev, precond="none")
    assert np.array_equal(none.invM(r2), r2)


def test_solve(shtlib):
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps, rng = _problem4(13)
    nat, mir = _systems(bands, comps, dev)
    data = [torch.as_tensor(rng.standard_normal((b.get("nmaps", 3), 12 * b["nside"] ** 2)) / np.sqrt(b["invN"]), device=dev)
            for b in bands]
    b = nat.computeRHS(data)
    x, it, hist = nat.solve(b, maxiter=500, cg_tol=1e-10)
    xr, itr, histr = solve_cr_eqn_by_CG(mir, b.clone(), maxiter=500, cg_tol=1e-10)
    assert abs(it - itr) <= 1 and 3 < it < 500, (it, itr)
    assert float((x - xr).norm() / xr.norm()) <= 1e-6
    np.testing.assert_allclose(hist[:10], histr[:10], rtol=1e-8)
    # fixed_iter: exactly maxiter iterations and maxiter + 1 applications of A
    n0 = nat.n_matmul
    _, it5, h5 = nat.solve(b, maxiter=5, cg_conv_crit="fixed_iter")
    assert it5 == 5 and len(h5) == 6 and nat.n_matmul - n0 == 6
    # x0 is honoured: the same history as the mirror started from the same point
    x0 = x * 0.9
    _, _, hx = nat.solve(b, x0=x0, maxiter=4, cg_conv_crit="fixed_iter")
    _, _, hxr = solve_cr_eqn_by_CG(mir, b.clone(), x0=x0.clone(), maxiter=4, cg_conv_crit="fixed_iter")
    np.testing.assert_allclose(hx, hxr, rtol=1e-8)
    assert hx[0] < 0.1 * hist[0]
    # the block preconditioner needs no more iterations than none
    none, _ = _systems(bands, comps, dev, precond="none")
    xn, itn, _ = none.solve(b, maxiter=3000, cg_tol=1e-10)
    assert it <= itn, (it, itn)
    assert float((x - xn).norm() / x.norm()) <= 1e-4


def test_one_component_agrees_with_the_fused_system(shtlib):
    """One component and bands that share its comm_mapinfo: the general path against cr_native_system, with F_mean folded
    back into b_l for the latter."""
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, cr_native_system, gaussian_beam
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(14)
    nside, lmax = 32, 64
    info = comm_mapinfo(None, nside, lmax, 3, True)
    l = np.arange(lmax + 1, dtype=np.float64)
    Cl = np.stack([30.0 / (l * (l + 1) + 1.0)] * 3, axis=1)
    F = np.array([[1.0, 1.0, 1.0], [0.7, 0.6, 0.6]])
    invN = [rng.uniform(0.5, 2.0, size=(3, info.np)) for _ in range(2)]
    bl = [gaussian_beam(lmax, 300.0, 3), gaussian_beam(lmax, 450.0, 3)]
    fused = cr_native_system(info, invN, [bl[q] * F[q][None, :] for q in range(2)], Cl=Cl)
    gen = cr_native_multi_system([cr_component(info, Cl=Cl, F_mean=F)], [cr_band(info, invN[q], bl[q]) for q in range(2)])
    n = 3 * info.nalm
    x = rng.standard_normal(n)
    assert rel(gen.matmulA(x), fused.matmulA(x.reshape(3, -1)).ravel()) <= 1e-12
    assert rel(gen.invM(x), fused.invM(x.reshape(3, -1)).ravel()) <= 1e-12
    data = [rng.standard_normal((3, info.np)) for _ in range(2)]
    bg = gen.computeRHS(data)
    bf = fused.computeRHS(data)
    assert rel(bg, bf.ravel()) <= 1e-12
    xg, itg, hg = gen.solve(bg, maxiter=40, cg_tol=1e-9)
    xf, itf, hf = fused.solve(bf, maxiter=40, cg_tol=1e-9)
    assert itg == itf
    np.testing.assert_allclose(hg, hf, rtol=1e-12)
    assert rel(xg, xf.ravel()) <= 1e-12


def test_real_size(shtlib):
    """Bands 512 / 1500, 1024 / 2000, 1024 / 2000; CMB (3 maps, lmax 2000, prior), dust (3, 1500, prior), a 1-map
    low-l component without prior: three fixed_iter iterations, native against the mirror."""
    import torch
    from commander_b200.comm_cr import solve_cr_eqn_by_CG
    dev = torch.device("cuda", 0)
    bands, comps = real_size_problem(np.random.default_rng(15))
    nat, mir = _systems(bands, comps, dev)
    rng = np.random.default_rng(16)
    data = [torch.as_tensor(rng.standard_normal((3, 12 * b["nside"] ** 2)), device=dev) for b in bands]
    b = nat.computeRHS(data)
    assert rel(b.cpu().numpy(), mir.computeRHS(data).cpu().numpy()) <= 1e-12
    x, it, h = nat.solve(b, maxiter=3, cg_conv_crit="fixed_iter")
    xr, itr, hr = solve_cr_eqn_by_CG(mir, b.clone(), maxiter=3, cg_conv_crit="fixed_iter")
    assert it == itr == 3
    np.testing.assert_allclose(h, hr, rtol=1e-9)
    assert float((x - xr).norm() / xr.norm()) <= 1e-9


def real_size_problem(rng):
    """The sampling group of tools/cr_multi_bench.py: bands (nside / lmax) 512 / 1500, 1024 / 2000, 1024 / 2000;
    components CMB (3 maps, lmax 2000, prior), dust (3 maps, lmax 1500, prior), a 1-map low-l component (lmax 200,
    no prior)."""
    from commander_b200.comm_cr import gaussian_beam
    bands = []
    for nside, lmax, fwhm, sig in ((512, 1500, 20.0, 1.0), (1024, 2000, 10.0, 0.7), (1024, 2000, 7.0, 1.3)):
        bands.append(dict(nside=nside, lmax=lmax, b_l=gaussian_beam(lmax, fwhm, 3),
                          invN=(1.0 / (sig * (1.0 + 0.5 * rng.uniform(size=(3, 12 * nside ** 2))))) ** 2))
    l = np.arange(2001, dtype=np.float64)
    comps = [dict(nside=1024, lmax=2000, nmaps=3, Cl=np.stack([1e3 / (l * (l + 1) + 1.0)] * 3, axis=1), F_mean=np.ones((3, 3))),
             dict(nside=1024, lmax=1500, nmaps=3, Cl=np.stack([50.0 / (l[:1501] + 1.0) ** 2.4] * 3, axis=1),
                  F_mean=np.array([[0.2] * 3, [0.9] * 3, [2.8] * 3])),
             dict(nside=64, lmax=200, nmaps=1, Cl=None, F_mean=np.array([[1.4], [1.0], [0.6]]))]
    return bands, comps
