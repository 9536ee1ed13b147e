"""The constrained-realisation fluctuation terms drawn on the device (cmdr_cr_compute_rhs_draw / cmdr_cr_draw_eta,
commander_b200/csrc/cr_draw.cu, stream of rng.cuh) on both handle kinds:
  * draw_eta equals the numpy restatement oracle/rng.py at every local pixel and amplitude (1e-13 absolute: a wrong
    Philox word would move eta by O(1));
  * computeRHS fed with those draws equals computeRHS_draw bit for bit, with and without data, for every `terms`;
  * the one-dimensional law at nside 1024 IQU (mean, variance, Kolmogorov-Smirnov) and the independence of seeds and
    draws;
  * Cov(b) = A for F_mean systems with data = NULL: 10^4 right-hand sides whitened by the Cholesky factor of A."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _single(nside=4, lmax=8, prior=True, nbands=2, seed=3):
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_native_system, gaussian_beam
    rng = np.random.default_rng(seed)
    info = comm_mapinfo(None, nside, lmax, 3, True)
    invN = [torch.as_tensor((1.0 / (0.8 + 0.4 * q + 0.5 * rng.uniform(size=(3, info.np)))) ** 2, device="cuda")
            for q in range(nbands)]
    bls = [gaussian_beam(lmax, 700.0 - 150.0 * q) * (1.0 + 0.2 * q) for q in range(nbands)]
    l = np.arange(lmax + 1, dtype=np.float64)
    Cl = np.stack([10.0 / (l * (l + 1) + 1.0)] * 3, axis=1) if prior else None
    return cr_native_system(info, invN, bls, Cl, precond="none"), info


def _multi(seed=11):
    """2 bands of different nside and lmax; a CMB-like IQU component with a prior and a temperature-only component
    without one"""
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, gaussian_beam
    rng = np.random.default_rng(seed)
    bands = []
    for nside, lmax, fwhm, sig in [(4, 8, 700.0, 1.0), (8, 10, 500.0, 0.7)]:
        info = comm_mapinfo(None, nside, lmax, 3, True)
        invN = (1.0 / (sig * (1.0 + 0.5 * rng.uniform(size=(3, info.np))))) ** 2
        bands.append(cr_band(info, torch.as_tensor(invN, device="cuda"), gaussian_beam(lmax, fwhm, 3)))
    l = np.arange(9, dtype=np.float64)
    comps = [cr_component(comm_mapinfo(None, 8, 8, 3, True), Cl=np.stack([10.0 / (l * (l + 1) + 1.0)] * 3, axis=1),
                          F_mean=np.ones((2, 3))),
             cr_component(comm_mapinfo(None, 8, 6, 1, False), Cl=None, F_mean=np.array([[1.5], [0.6]]))]
    return cr_native_multi_system(comps, bands, precond="none"), bands, comps


def _oracle_single(sysn, info, seed, draw, prior):
    from oracle import rng
    pix = [np.stack([rng.eta_pix(seed, draw, q, j, info.pix) for j in range(3)]) for q in range(sysn.nbands)]
    alm = np.zeros((3, info.nalm))
    if prior:
        alm = np.stack([rng.eta_alm(seed, draw, 0, j, info.lm[0], info.lm[1]) for j in range(3)])
    return pix, alm


def _oracle_multi(bands, comps, seed, draw):
    from oracle import rng
    pix = [np.stack([rng.eta_pix(seed, draw, q, j, b.info.pix) for j in range(b.info.nmaps)]) for q, b in enumerate(bands)]
    alm = []
    for k, c in enumerate(comps):
        if c.Cl is None:
            alm.append(np.zeros(c.nmaps * c.x_info.nalm))
        else:
            alm.append(np.concatenate([rng.eta_alm(seed, draw, k, j, c.x_info.lm[0], c.x_info.lm[1]) for j in range(c.nmaps)]))
    return pix, np.concatenate(alm)


@pytest.mark.parametrize("seed,draw", [(0, 0), (20260101, 17), (2 ** 64 - 1, 2 ** 40 + 3)])
def test_draw_eta_matches_oracle(shtlib, seed, draw):
    for prior in (True, False):
        sysn, info = _single(nside=8, lmax=12, prior=prior)
        pix, alm = sysn.draw_eta(seed, draw)
        want_pix, want_alm = _oracle_single(sysn, info, seed, draw, prior)
        for p, w in zip(pix, want_pix):
            assert np.max(np.abs(p.cpu().numpy() - w)) < 1e-13
        assert np.max(np.abs(alm.cpu().numpy() - want_alm)) < 1e-13
        if not prior:
            assert not alm.any()
    nat, bands, comps = _multi()
    pix, alm = nat.draw_eta(seed, draw)
    want_pix, want_alm = _oracle_multi(bands, comps, seed, draw)
    for p, w in zip(pix, want_pix):
        assert np.max(np.abs(p.cpu().numpy() - w)) < 1e-13
    assert np.max(np.abs(alm.cpu().numpy() - want_alm)) < 1e-13


def _data(shapes, seed):
    import torch
    rng = np.random.default_rng(seed)
    return [torch.as_tensor(rng.standard_normal(s), device="cuda") for s in shapes]


@pytest.mark.parametrize("kind", ["single_prior", "single_noprior", "multi"])
def test_both_entries_agree_bitwise(shtlib, kind):
    """computeRHS(data, *draw_eta(s, d)) == computeRHS_draw(data, s, d), with and without data, for every `terms`"""
    import torch
    if kind == "multi":
        sysn, bands, _ = _multi()
        shapes = [(b.info.nmaps, b.info.np) for b in bands]
    else:
        sysn, info = _single(prior=kind == "single_prior")
        shapes = [(3, info.np)] * sysn.nbands
    s, d = 987654321, 5
    eta_pix, eta_alm = sysn.draw_eta(s, d)
    for data in (_data(shapes, 1), None):
        given = data if data is not None else [torch.zeros(sh, dtype=torch.float64, device="cuda") for sh in shapes]
        for pixel in (True, False):
            for prior in (True, False):
                want = sysn.computeRHS(given, eta_pix if pixel else None, eta_alm if prior else None)
                got = sysn.computeRHS_draw(data, s, d, pixel=pixel, prior=prior)
                assert torch.equal(got, want), (kind, data is None, pixel, prior)
                assert got.abs().max() > 0 or (data is None and not pixel and (not prior or kind == "single_noprior"))


def test_python_refuses_bad_seed_and_draw(shtlib):
    sysn, _ = _single()
    for bad in (-1, 2 ** 64, 1.5):
        with pytest.raises(ValueError):
            sysn.computeRHS_draw(None, bad, 0)
        with pytest.raises(ValueError):
            sysn.draw_eta(0, bad)


def test_one_dimensional_law_and_independence(shtlib):
    """nside 1024 IQU: 37.7 M draws of one band against N(0, 1); other seeds and draws uncorrelated; repeatable"""
    import torch
    from scipy import stats
    sysn, info = _single(nside=1024, lmax=8, prior=True, nbands=1)
    seed, draw = 424242, 9
    e = sysn.draw_eta(seed, draw)[0][0]
    n = e.numel()
    assert n == 3 * 12 * 1024 ** 2
    mean = float(e.mean())
    var = float(e.var(unbiased=False))
    assert abs(mean) < 6 / np.sqrt(n), mean
    assert abs(var - 1.0) < 6 * np.sqrt(2.0 / n), var
    p = stats.kstest(e.cpu().numpy().ravel(), "norm").pvalue
    assert p > 1e-4, p
    for other in ((seed + 1, draw), (seed, draw + 1), (seed ^ (1 << 63), draw), (seed, draw + (1 << 32))):
        f = sysn.draw_eta(*other)[0][0]
        corr = float(((e - e.mean()) * (f - f.mean())).mean() / (e.std(unbiased=False) * f.std(unbiased=False)))
        assert abs(corr) < 6 / np.sqrt(n), (other, corr)
    again = sysn.draw_eta(seed, draw)[0][0]
    assert torch.equal(again, e)
    # the draws of the three maps are different streams too
    for a, b in ((0, 1), (0, 2), (1, 2)):
        c = float(torch.corrcoef(torch.stack([e[a], e[b]]))[0, 1])
        assert abs(c) < 6 / np.sqrt(e[a].numel()), (a, b, c)


def _dense_A(sysn, n, flat):
    """A built column by column with matmulA on unit vectors, symmetrised"""
    import torch
    A = np.empty((n, n))
    for i in range(n):
        x = torch.zeros(n, dtype=torch.float64, device="cuda")
        x[i] = 1.0
        y = sysn.matmulA(x if flat else x.view(3, -1))
        A[:, i] = y.reshape(-1).cpu().numpy()
    return 0.5 * (A + A.T)


def _check_covariance(sysn, n, flat, N=10_000, seed=77):
    import torch
    A = _dense_A(sysn, n, flat)
    sel = np.diag(A) > 1e-12 * np.max(np.diag(A))
    B = torch.empty((N, n), dtype=torch.float64, device="cuda")
    for i in range(N):
        B[i] = sysn.computeRHS_draw(None, seed, i).reshape(-1)
    B = B.cpu().numpy()
    assert not np.any(B[:, ~sel]), "a coordinate A does not reach received a draw"
    L = np.linalg.cholesky(A[np.ix_(sel, sel)])
    W = np.linalg.solve(L, B[:, sel].T)                    # whitened draws, (n_sel, N)
    C = W @ W.T / N
    dev_cov = np.max(np.abs(C - np.eye(C.shape[0])))
    dev_mean = np.max(np.abs(W.mean(axis=1)))
    assert dev_cov < 6 * np.sqrt(2.0 / N), dev_cov
    assert dev_mean < 6 / np.sqrt(N), dev_mean
    return int(sel.sum())


@pytest.mark.parametrize("prior", [True, False])
def test_covariance_is_A_single(shtlib, prior):
    sysn, info = _single(nside=4, lmax=8, prior=prior, nbands=2)
    nsel = _check_covariance(sysn, 3 * info.nalm, flat=False)
    assert nsel == (3 * info.nalm if prior else 3 * info.nalm - 2 * 4)    # without a prior A is 0 on l < 2 of E and B


def test_covariance_is_A_multi(shtlib):
    nat, bands, comps = _multi()
    assert _check_covariance(nat, nat.ncr, flat=True) == nat.ncr
