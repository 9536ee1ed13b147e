"""Constrained-realisation CG for a CMB-only signal model: the mirror of the part of
`comm_cr_mod` that drives the SHT hot path (commander3/src/comm_cr_mod.f90).

    A = 1 + sqrt(S) B^T Y^T N^-1 Y B sqrt(S)            cr_matmulA, :771-1024 (one band, F = 1)
    b = sqrt(S) B^T Y^T N^-1 d  [+ sqrt(S) B^T Y^T N^-1/2 eta1 + eta0]   cr_computeRHS, :542-769
    PCG with M^-1 = diag                                  solve_cr_eqn_by_CG, :201-348; cr_invM :1026-1077

with N^-1 = siN^2 per pixel (commander3/src/comm_N_rms_mod.f90:264-273), B = b_l per l and
component (commander3/src/comm_B_bl_mod.f90:108-127), S = diagonal C_l (TT, EE, BB;
commander3/src/comm_Cl_mod.f90:588-637), and the diagonal preconditioner of
commander3/src/comm_diffuse_comp_mod.f90:2186-2235 for npre = 1.

All vectors live on the GPU as torch tensors of shape (nmaps, nalm) in the real-packed basis; the
two SHTs per A application are `comm_map%Y` and `comm_map%Yt` on device pointers; the two dot products
per iteration go through `mpi_dot_product` = local dot + NCCL all-reduce
(commander3/src/comm_utils.f90:599-614).

The preconditioner's N^-1_{lm,lm} is `compute_invN_lm` (commander3/src/comm_N_mod.f90:127-197), on the GPU
(`cmdr_sht_invn_diag`: the Wigner-3j sum of the reference evaluated as an exact quadrature).  `invN_lm="monopole"`
keeps only its L = 0 term, the sky mean of siN^2 times npix/4pi (what round 1 started with).  Any SPD
preconditioner gives the same solution; only the iteration count differs.
"""
from __future__ import annotations

import math

import numpy as np

from .comm_map import comm_map, comm_mapinfo


def gaussian_beam(lmax: int, fwhm_arcmin: float, nmaps: int = 3) -> np.ndarray:
    """b_l(l, j): Gaussian beam with the spin-2 factor of commander3/src/comm_map_mod.f90:1122-1135."""
    sigma = fwhm_arcmin * math.pi / 180.0 / 60.0 / math.sqrt(8.0 * math.log(2.0))
    l = np.arange(lmax + 1, dtype=np.float64)
    bl = np.empty((lmax + 1, nmaps))
    bl[:, 0] = np.exp(-0.5 * l * (l + 1) * sigma ** 2)
    for j in range(1, nmaps):
        bl[:, j] = np.exp(-0.5 * l * (l + 1) * sigma ** 2) * math.exp(2.0 * sigma ** 2)
    return bl


def compute_invN_lm(invN_diag: comm_map) -> None:
    """commander3/src/comm_N_mod.f90:127-197.  On entry invN_diag%map holds N^-1 per pixel (all columns treated
    as scalars, :146); on exit invN_diag%alm holds N_lm: `YtW_scalar`, the m = 0 coefficients from the rank that
    owns them to everybody (:147-152), then the 3j sum per local (l,m) (:154-184) -- here one GPU kernel."""
    from . import sharp
    info = invN_diag.info
    invN_diag.YtW_scalar()
    lmax, nm = info.lmax, info.nmaps
    i0 = info.lm2i(0, 0)
    if invN_diag.device is None:
        a_l0 = np.zeros((nm, lmax + 1))
        if i0 >= 0:
            a_l0[:] = invN_diag.alm[:, i0:i0 + lmax + 1]
        if info.dist and info.comm.size > 1:
            raise NotImplementedError("host-resident comm_map on several ranks: use device maps")
    else:
        import torch
        a = torch.zeros((nm, lmax + 1), dtype=torch.float64, device=invN_diag.alm.device)
        if i0 >= 0:
            a.copy_(invN_diag.alm[:, i0:i0 + lmax + 1])
        if info.dist and info.comm.size > 1:
            info.comm.allreduce_sum_(a)          # mpi_bcast from the owner of m = 0: zero everywhere else
        a_l0 = a.cpu().numpy()
    sharp.invN_diag(a_l0, float(info.npix), info.alm_info, invN_diag.alm)


class cr_cmb_system:
    """One band, one component (CMB, F = 1) constrained-realisation system."""

    def __init__(self, info: comm_mapinfo, siN, b_l: np.ndarray, Cl: np.ndarray, mask=None, mb_eff: float = 1.0,
                 precond: str = "diagonal", invN_lm: str = "wigner"):
        import torch
        self.torch = torch
        self.info = info
        dev = siN.device
        self.dev = dev
        self.siN = siN
        self.invN = siN * siN
        if mask is not None:
            self.invN = self.invN * mask      # samp_group mask, comm_N_rms_mod.f90:270-272
        l = info.lm[0].astype(np.int64)
        nm = info.nmaps
        # per-(alm slot, component) factors
        bl = np.stack([b_l[l, j] for j in range(nm)]) * mb_eff                 # matmulB
        sS = np.stack([np.sqrt(np.maximum(Cl[l, j], 0.0)) for j in range(nm)])  # sqrtS, diagonal C_l
        for j in range(1, nm):
            sS[j, l < 2] = 0.0
        self.bl = torch.as_tensor(bl, device=dev)
        self.sqrtS = torch.as_tensor(sS, device=dev)
        self.sSbl = self.sqrtS * self.bl      # sqrt(S) and the beam act on the same slots: one pass instead of two
        self.buf = comm_map(info, device=dev)
        # diagonal preconditioner: 1 + C_l b_l^2 N^-1_{lm,lm}, monopole term of compute_invN_lm
        mean_invN = self.invN.sum(dim=1)
        self._allreduce(mean_invN)
        mean_invN = mean_invN / float(info.npix)
        invN_diag = mean_invN * float(info.npix) / (4.0 * math.pi)
        if invN_lm == "wigner":
            # P_cr%invM_diff for npre = 1 with the full N_lm (comm_diffuse_comp_mod.f90:1167-1252)
            self.buf.map.copy_(self.invN)
            compute_invN_lm(self.buf)
            self.invN_lm = self.buf.alm.clone()
            self.Minv = 1.0 / (1.0 + (self.sqrtS * self.bl) ** 2 * self.invN_lm)
        elif invN_lm == "monopole":
            self.invN_lm = None
            self.Minv = 1.0 / (1.0 + (self.sqrtS * self.bl) ** 2 * invN_diag[:, None])
        else:
            raise ValueError("invN_lm must be 'wigner' or 'monopole'")
        # pseudo-inverse preconditioner (precond_type = 'pseudoinv')
        if precond not in ("diagonal", "pseudoinv"):
            raise ValueError("Preconditioner type not supported: " + precond)
        self.precond = precond
        # alpha_nu^2 = mean inverse noise variance in harmonic units (N%alpha_nu, :2293-2295): with it T / alpha^2 is
        # O(1), which the pseudo-inverse needs (V = [alpha U; 1])
        self.alpha2 = invN_diag[:, None]
        U = self.sqrtS * self.bl * torch.sqrt(self.alpha2)
        self.Uplus = U / (U * U + 1.0)
        self.Pplus2 = 1.0 / (U * U + 1.0) ** 2
        # N%N: sigma^2 per pixel; masked / unobserved pixels (N^-1 = 0) carry no information and are left out
        self.N = torch.where(self.invN > 0, 1.0 / self.invN.clamp_min(1e-300), torch.zeros_like(self.invN))
        self.n_matmul = 0

    # -- communicator helpers
    def _allreduce(self, t):
        c = self.info.comm
        if self.info.dist and c.size > 1:
            c.allreduce_sum_(t)
        return t

    def mpi_dot_product(self, a, b):
        """commander3/src/comm_utils.f90:599-614"""
        s = self.torch.dot(a.reshape(-1), b.reshape(-1)).reshape(1)
        self._allreduce(s)
        return float(s.item())

    # -- operators
    def matmulA(self, x):
        """cr_matmulA, commander3/src/comm_cr_mod.f90:771-1024 for one band / one diffuse component."""
        m = self.buf
        self.torch.mul(x, self.sSbl, out=m.alm)   # sqrtS_x :797-836, then evalDiffuseBand: F_mean = 1, beam :2089
        m.Y()                         # :888-892
        m.map.mul_(self.invN)         # N%invN, :905
        m.Yt()                        # :913-918
        self.n_matmul += 1
        return self.torch.addcmul(x, m.alm, self.sSbl)   # projectDiffuseBand (B^T), sqrtS :957-1008, + x

    def invM(self, r):
        """cr_invM, :1026-1077: 'diagonal' (default) or 'pseudoinv' preconditioner."""
        if self.precond == "pseudoinv":
            return self.invM_pseudoinv(r)
        return r * self.Minv

    def invM_pseudoinv(self, r):
        """applyDiffPrecond_pseudoinv, commander3/src/comm_diffuse_comp_mod.f90:2237-2380, for one band and one
        component.  The system is A = V^T diag(T, 1) V with V = [U; 1], U = alpha b_l sqrt(C_l) per (l, pol) and
        T = Y^T N^-1 Y / alpha^2; its pseudo-inverse preconditioner is V^+ diag(T^+, 1) V^+T with V^+ = [U, 1] / (U^2 + 1)
        (the columns of P_cr%invM_diff, :1313-1557) and T^+ = alpha^2 YtW N WY (:2288-2292: `call invN_x%WY`,
        `call data(k)%N%N(invN_x)`, `call invN_x%YtW`)."""
        m = self.buf
        m.alm.copy_(r)
        m.alm.mul_(self.Uplus)                 # sum over (U^plus)^t, :2270-2285
        m.WY()                                 # :2288
        m.map.mul_(self.N)                     # N%N: noise covariance, :2290
        m.YtW()                                # :2292
        m.alm.mul_(self.alpha2)                # alpha_nu^2, :2293-2295
        z = m.alm * self.Uplus                 # sum over U^plus, :2300-2315
        return z + r * self.Pplus2             # prior terms, :2322-2346

    def computeRHS(self, data, eta_pix=None, eta_alm=None):
        """cr_computeRHS, :542-769: mean-field term, plus the two fluctuation terms when the white
        noise draws are given ('sample' branch)."""
        m = self.buf
        m.map.copy_(data * self.invN)
        if eta_pix is not None:
            m.map.add_(self.siN * eta_pix)          # N^-1/2 eta
        m.Yt()                                       # :615
        m.alm.mul_(self.bl)                          # B^T, :616
        m.alm.mul_(self.sqrtS)                       # :652
        b = m.alm.clone()
        if eta_alm is not None:
            b += eta_alm
        return b

    def x2amp(self, x):
        """cr_x2amp after multiplying with sqrt(S) (comm_cr_mod.f90:350-390): the signal a_lm."""
        return x * self.sqrtS


def solve_cr_eqn_by_CG(sys: cr_cmb_system, b, maxiter=300, cg_tol=1e-8, cg_conv_crit="residual",
                       cg_miniter=5, cg_check_conv_freq=1, x0=None, verbose=False):
    """solve_cr_eqn_by_CG, commander3/src/comm_cr_mod.f90:201-348 (same update order, same
    convergence test).  Returns (x, iterations done, residual history)."""
    torch = sys.torch
    x = torch.zeros_like(b) if x0 is None else x0.clone()
    r = b - sys.matmulA(x)
    d = sys.invM(r)
    if d.data_ptr() == r.data_ptr():
        d = d.clone()                             # an identity preconditioner may hand r back; d is updated in place
    delta_new = sys.mpi_dot_product(r, d)
    delta0 = sys.mpi_dot_product(b, sys.invM(b))
    if cg_conv_crit not in ("residual", "fixed_iter"):
        raise ValueError("Unsupported convergence criterion = " + cg_conv_crit)
    lim_convergence = cg_tol * delta0
    val_convergence = 1e2 * lim_convergence
    hist = [delta_new]
    it = 0
    for i in range(1, maxiter + 1):
        if i % cg_check_conv_freq == 0:
            val_convergence = delta_new
            if (val_convergence < lim_convergence and (i >= cg_miniter or delta_new <= 1e-30 * delta0)
                    and cg_conv_crit != "fixed_iter"):
                break
        q = sys.matmulA(d)
        alpha = delta_new / sys.mpi_dot_product(d, q)
        x.add_(d, alpha=alpha)                    # x = x + alpha d   (in place: x, r, d are this routine's own)
        r.add_(q, alpha=-alpha)                   # r = r - alpha q
        s = sys.invM(r)
        delta_old = delta_new
        delta_new = sys.mpi_dot_product(r, s)
        beta = delta_new / delta_old
        d.mul_(beta).add_(s)                      # d = s + beta d
        hist.append(delta_new)
        it = i
        if verbose:
            print(f"  CG iter. {i:5d} -- res = {delta_new:13.5e}, tol = {lim_convergence:13.5e}")
    return x, it, hist


# =====================================================================================================
# General system: several diffuse components seen through several bands (cr_matmulA as written,
# commander3/src/comm_cr_mod.f90:771-1024, diffuse components only)
# =====================================================================================================

class cr_component:
    """What cr_matmulA needs of a `comm_diffuse_comp`: the amplitude layout x%info (nside, lmax_amp, nmaps), an
    optional diagonal prior C_l (cltype /= 'none'), and per band either F_mean (nmaps scalars, spectral parameters
    constant on the sky) or a per-pixel mixing map F (commander3/src/comm_diffuse_comp_mod.f90:2070-2083)."""

    def __init__(self, x_info: comm_mapinfo, Cl=None, F_mean=None, F=None):
        self.x_info = x_info
        self.lmax_amp = x_info.lmax
        self.nmaps = x_info.nmaps
        self.Cl = None if Cl is None else np.asarray(Cl, dtype=np.float64)
        self.F_mean = np.asarray(F_mean, dtype=np.float64)     # (numband, nmaps); also feeds the preconditioner
        self.F = F                                             # None or a list (numband) of None / (nmaps, np) arrays


class cr_band:
    """One frequency band: data(i)%info, N%invN as siN^2 (x mask) per pixel, beam b_l(0:lmax, nmaps)."""

    def __init__(self, info: comm_mapinfo, invN, b_l):
        self.info, self.invN, self.b_l = info, invN, np.asarray(b_l, dtype=np.float64)


class cr_system:
    """A = P + sqrt(S) sum_nu F^t B^t Y^t N^-1 Y B F sqrt(S) over all diffuse components (P = 1 on components
    with a prior, 0 on the others; sqrt(S) = 1 on the latter).  x is the flat vector of cr_extract_comp /
    cr_insert_comp (:408-540): component after component, each (nmaps, nalm) in memory order."""

    def __init__(self, comps, bands, device, precond: str = "diagonal"):
        import torch
        from .comm_diffuse_comp import diffuse_band
        if precond not in ("diagonal", "pseudoinv"):
            raise ValueError("Preconditioner type not supported: " + precond)
        self.precond = precond
        self.torch, self.dev = torch, device
        self.comps, self.bands = list(comps), list(bands)
        self.off = [0]
        for c in self.comps:
            self.off.append(self.off[-1] + c.nmaps * c.x_info.nalm)
        self.ncr = self.off[-1]
        self.lmax = max(max(c.lmax_amp for c in self.comps), 2)                 # :809
        self.sqrtS = []
        for c in self.comps:
            if c.Cl is None:
                self.sqrtS.append(None)
                continue
            l = c.x_info.lm[0].astype(np.int64)
            sS = np.stack([np.sqrt(np.maximum(c.Cl[l, j], 0.0)) for j in range(c.nmaps)])
            for j in range(1, c.nmaps):
                sS[j, l < 2] = 0.0
            self.sqrtS.append(torch.as_tensor(sS, device=device))
        # (component, band) operators: re-pack + mixing + beam and its transpose
        self.cb = []
        for c in self.comps:
            row = []
            for q, b in enumerate(self.bands):
                nm = min(b.info.nmaps, c.nmaps)
                binfo = b.info if nm == b.info.nmaps else comm_mapinfo(b.info.comm, b.info.nside, b.info.lmax, nm, nm == 3)
                Fq = None if c.F is None else c.F[q]
                if Fq is not None and not hasattr(Fq, "device"):
                    Fq = torch.as_tensor(np.ascontiguousarray(Fq[:nm]), device=device)
                row.append(diffuse_band(c.x_info, binfo, b.b_l[:, :nm], F=Fq,
                                        F_mean=None if Fq is not None else c.F_mean[q, :nm], device=device))
            self.cb.append(row)
        # one buffer pair per band: the band layout, and the synthesis layout at lmax = max lmax_amp (:877-882)
        self.bmap = [comm_map(b.info, device=device) for b in self.bands]
        self.ymap = [comm_map(comm_mapinfo(b.info.comm, b.info.nside, self.lmax, b.info.nmaps, b.info.nmaps == 3), device=device)
                     for b in self.bands]
        self.xbuf = [comm_map(c.x_info, device=device) for c in self.comps]
        self.n_matmul = 0
        self.Minv = None

    # -- vector layout
    def extract_comp(self, i, x):
        """cr_extract_comp: view of component i as (nmaps, nalm)."""
        c = self.comps[i]
        return x[self.off[i]:self.off[i + 1]].view(c.nmaps, c.x_info.nalm)

    def _comm(self):
        return self.bands[0].info.comm

    def _allreduce(self, t):
        c = self._comm()
        if self.bands[0].info.dist and c.size > 1:
            c.allreduce_sum_(t)
        return t

    def mpi_dot_product(self, a, b):
        s = self.torch.dot(a.reshape(-1), b.reshape(-1)).reshape(1)
        self._allreduce(s)
        return float(s.item())

    # -- band passes
    def _to_band(self, q, sx):
        """sum over components of getBand(q, alm_out) (:858-864), then Y at lmax (:877-882); returns the band map."""
        m = self.bmap[q]
        m.alm.zero_()
        for i, c in enumerate(self.comps):
            xb = self.xbuf[i]
            xb.alm.copy_(self.extract_comp(i, sx))
            a = self.cb[i][q].evalDiffuseBand(xb, alm_out=True)
            m.alm[:a.shape[0]] += a
        y = self.ymap[q]
        m.alm_equal(y)
        y.Y()
        return y

    def _from_band(self, q, y, out):
        """Yt at lmax (:913-918), then projectBand(q, alm_in) into every component, accumulated into `out` (:926-934)."""
        m = self.bmap[q]
        y.Yt()
        y.alm_equal(m)
        for i, c in enumerate(self.comps):
            nm = self.cb[i][q].band_info.nmaps
            sub = m if nm == m.info.nmaps else _view_maps(m, self.cb[i][q].band_info, nm)
            self.extract_comp(i, out).add_(self.cb[i][q].projectDiffuseBand(sub, alm_in=True))

    def matmulA(self, x):
        torch = self.torch
        sx = x.clone()
        for i, sS in enumerate(self.sqrtS):
            if sS is not None:
                self.extract_comp(i, sx).mul_(sS)                               # :797-836
        y = torch.zeros_like(x)
        for q, b in enumerate(self.bands):
            ym = self._to_band(q, sx)
            ym.map.mul_(b.invN)                                                 # :905
            self._from_band(q, ym, y)
        for i, sS in enumerate(self.sqrtS):
            if sS is not None:
                yi = self.extract_comp(i, y)
                yi.mul_(sS)                                                     # :957-1008
                yi.add_(self.extract_comp(i, x))
        self.n_matmul += 1
        return y

    def computeRHS(self, data, eta_pix=None, eta_alm=None):
        """cr_computeRHS (:542-769): sum over bands of sqrt(S) F^t B^t Y^t (N^-1 d + N^-1/2 eta_nu), plus the prior
        fluctuation eta_0 on the components that have a prior."""
        torch = self.torch
        rhs = torch.zeros(self.ncr, dtype=torch.float64, device=self.dev)
        for q, b in enumerate(self.bands):
            ym = self.ymap[q]
            ym.map.copy_(data[q] * b.invN)
            if eta_pix is not None:
                ym.map.add_(torch.sqrt(b.invN) * eta_pix[q])
            self._from_band(q, ym, rhs)
        for i, sS in enumerate(self.sqrtS):
            if sS is not None:
                ri = self.extract_comp(i, rhs)
                ri.mul_(sS)
                if eta_alm is not None:
                    ri.add_(self.extract_comp(i, eta_alm))
        return rhs

    # -- preconditioner
    def initDiffPrecond_diagonal(self):
        """initDiffPrecond_diagonal + updateDiffPrecond_diagonal, commander3/src/comm_diffuse_comp_mod.f90:1167-1252,
        1313-1557: per (l, m, pol) the npre x npre matrix sqrt(S) [sum_nu N^-1_lm b_l^2 F_k1 F_k2] sqrt(S) + P on the
        components that reach this l, inverted; N^-1_lm from compute_invN_lm on every band."""
        torch = self.torch
        npre = len(self.comps)
        nmaps_pre = max(c.nmaps for c in self.comps)
        b0 = self.bands[0].info
        pre = comm_mapinfo(b0.comm, b0.nside, self.lmax, nmaps_pre, nmaps_pre == 3)
        self.info_pre = pre
        l, m = pre.lm[0].astype(np.int64), pre.lm[1].astype(np.int64)
        mat = torch.zeros((nmaps_pre, pre.nalm, npre, npre), dtype=torch.float64, device=self.dev)
        for q, b in enumerate(self.bands):
            nd = comm_map(b.info, device=self.dev)
            nd.map.copy_(b.invN)
            compute_invN_lm(nd)                                                  # data(q)%N%invN_diag
            i2 = b.info.lm2i_vec(l, m)
            ok = torch.as_tensor(i2 >= 0, device=self.dev)
            idx = torch.as_tensor(np.maximum(i2, 0), device=self.dev)
            for j in range(min(nmaps_pre, b.info.nmaps)):
                w = torch.where(ok, nd.alm[j, idx], torch.zeros((), dtype=torch.float64, device=self.dev))
                w = w * torch.as_tensor(b.b_l[np.minimum(l, b.info.lmax), j] ** 2, device=self.dev)
                for k1, c1 in enumerate(self.comps):
                    if j >= c1.nmaps:
                        continue
                    r1 = torch.as_tensor((l <= c1.lmax_amp) * c1.F_mean[q, j], device=self.dev)
                    for k2, c2 in enumerate(self.comps):
                        if j >= c2.nmaps:
                            continue
                        r2 = torch.as_tensor((l <= c2.lmax_amp) * c2.F_mean[q, j], device=self.dev)
                        mat[j, :, k1, k2] += w * r1 * r2
        active = torch.diagonal(mat, dim1=2, dim2=3) > 0.0                       # comp2ind /= -1, :1232-1239
        # sqrt(S) on both sides and the unit prior term for components with a C_l (:1350-1470)
        for k, c in enumerate(self.comps):
            if c.Cl is None:
                continue
            sS = np.zeros((nmaps_pre, pre.nalm))
            for j in range(c.nmaps):
                sS[j] = np.sqrt(np.maximum(c.Cl[np.minimum(l, c.lmax_amp), j], 0.0)) * (l <= c.lmax_amp)
                if j > 0:
                    sS[j, l < 2] = 0.0
            sS = torch.as_tensor(sS, device=self.dev)
            mat[:, :, k, :] *= sS[:, :, None]
            mat[:, :, :, k] *= sS[:, :, None]
            unit = torch.as_tensor((l <= c.lmax_amp).astype(np.float64), device=self.dev)[None, :] * active[:, :, k]
            mat[:, :, k, k] += unit
        # invert on the active set: inactive components pass through unchanged (applyDiffPrecond_diagonal, :2186-2235)
        eye = torch.eye(npre, dtype=torch.float64, device=self.dev)
        act2 = active[:, :, :, None] & active[:, :, None, :]
        full = torch.where(act2, mat, torch.zeros_like(mat)) + eye * (~active)[:, :, :, None]
        self.Minv = torch.linalg.inv(full)
        # index maps between every component's layout and info_pre
        self.pre_idx = []
        for c in self.comps:
            k = pre.lm2i_vec(c.x_info.lm[0], c.x_info.lm[1])
            self.pre_idx.append(torch.as_tensor(k, device=self.dev))

    # -- pseudo-inverse preconditioner
    def compute_alpha_nu(self, q):
        """N%alpha_nu of band q for the pseudo-inverse preconditioner (commander3/src/comm_N_rms_mod.f90:218-247):
        tau = Y Yt (siN^2), alpha = sqrt(sum tau^2 / sum tau), T alone and Q,U together."""
        torch = self.torch
        b = self.bands[q]
        m = comm_map(b.info, device=self.dev)
        m.map.copy_(b.invN)
        m.Yt()
        m.Y()
        nm = b.info.nmaps
        groups = [slice(0, 1)] + ([slice(1, 3)] if nm == 3 else [])
        alpha = torch.zeros(nm, dtype=torch.float64, device=self.dev)
        for g in groups:
            t = torch.stack([m.map[g].sum(), (m.map[g] ** 2).sum()])
            self._allreduce(t)
            alpha[g] = torch.sqrt(t[1] / t[0]) if float(t[0]) > 0.0 else 0.0
        return alpha.cpu().numpy()

    def initDiffPrecond_pseudoinv(self):
        """initDiffPrecond_pseudoinv + updateDiffPrecond_pseudoinv, commander3/src/comm_diffuse_comp_mod.f90:1255-1294,
        1560-1658: per (l, pol) the (numband + npre) x npre matrix V = [alpha_nu b_l F sqrt(S); P] and its pseudo-inverse."""
        torch = self.torch
        npre, nb = len(self.comps), len(self.bands)
        nmaps_pre = max(c.nmaps for c in self.comps)
        b0 = self.bands[0].info
        pre = comm_mapinfo(b0.comm, b0.nside, self.lmax, nmaps_pre, nmaps_pre == 3)
        self.info_pre = pre
        self.alpha_nu = [self.compute_alpha_nu(q) for q in range(nb)]
        V = np.zeros((nmaps_pre, self.lmax + 1, nb + npre, npre))
        for j in range(nmaps_pre):
            for q, b in enumerate(self.bands):
                if j >= b.info.nmaps:
                    continue
                lb = min(b.info.lmax, self.lmax)
                for k, c in enumerate(self.comps):
                    if j >= c.nmaps:
                        continue
                    lk = min(lb, c.lmax_amp)
                    v = self.alpha_nu[q][j] * b.b_l[:lk + 1, j] * c.F_mean[q, j]
                    if c.Cl is not None:
                        v = v * np.sqrt(np.maximum(c.Cl[:lk + 1, j], 0.0))
                        if j > 0:
                            v[:2] = 0.0          # sqrt(S) carries no l < 2 polarisation modes (matmulA zeroes them too)
                    V[j, :lk + 1, q, k] = v
            for k, c in enumerate(self.comps):
                if c.Cl is not None and j < c.nmaps:
                    V[j, :c.lmax_amp + 1, nb + k, k] = 1.0
        self.pinvV = torch.linalg.pinv(torch.as_tensor(V, device=self.dev))     # (nmaps_pre, lmax+1, npre, nb + npre)
        self.pre_idx = []
        for c in self.comps:
            self.pre_idx.append(torch.as_tensor(pre.lm2i_vec(c.x_info.lm[0], c.x_info.lm[1]), device=self.dev))
        self.l_pre = torch.as_tensor(pre.lm[0].astype(np.int64), device=self.dev)
        # band layout <-> info_pre layout (:2277-2279: `if (l > info_pre%lmax) cycle; call info_pre%lm2i(l,m,j)`)
        self.band_pre = []
        for b in self.bands:
            j = pre.lm2i_vec(b.info.lm[0], b.info.lm[1])
            ok = (j >= 0) & (b.info.lm[0] <= pre.lmax)
            self.band_pre.append((torch.as_tensor(np.nonzero(ok)[0], device=self.dev), torch.as_tensor(j[ok], device=self.dev),
                                  torch.as_tensor(b.info.lm[0][ok].astype(np.int64), device=self.dev)))
        self.Nmap = [torch.where(b.invN > 0, 1.0 / b.invN.clamp_min(1e-300), torch.zeros_like(b.invN)) for b in self.bands]

    def invM_pseudoinv(self, r):
        """applyDiffPrecond_pseudoinv, commander3/src/comm_diffuse_comp_mod.f90:2237-2380."""
        torch = self.torch
        if getattr(self, "pinvV", None) is None:
            self.initDiffPrecond_pseudoinv()
        npre, nb = len(self.comps), len(self.bands)
        nmaps_pre, nalm_pre = self.info_pre.nmaps, self.info_pre.nalm
        y = torch.zeros((npre, nmaps_pre, nalm_pre), dtype=torch.float64, device=self.dev)           # :2255-2268
        for i, c in enumerate(self.comps):
            y[i, :c.nmaps, self.pre_idx[i]] = self.extract_comp(i, r)
        z = torch.zeros_like(y)
        for q, b in enumerate(self.bands):                                                           # :2271-2318
            m = comm_map(b.info, device=self.dev)
            bi, pj, lb = self.band_pre[q]
            nm = b.info.nmaps
            for p_ in range(min(nm, nmaps_pre)):
                Mq = self.pinvV[p_, lb, :, q]                       # (n, npre): M(qq, k) at this slot's l
                m.alm[p_, bi] = (Mq * y[:, p_, pj].T).sum(dim=1)    # sum over (U^plus)^t
            m.WY()                                                  # :2288
            m.map.mul_(self.Nmap[q])                                # N%N
            m.YtW()                                                 # :2292
            for p_ in range(nm):
                m.alm[p_].mul_(float(self.alpha_nu[q][p_]) ** 2)    # :2293-2295
            for p_ in range(min(nm, nmaps_pre)):
                Mq = self.pinvV[p_, lb, :, q]
                z[:, p_, pj] += (Mq * m.alm[p_, bi][:, None]).T     # sum over U^plus
        Mp = self.pinvV[:, self.l_pre][..., nb:]                     # (nmaps_pre, nalm_pre, npre, npre): prior columns, :2322-2346
        w2 = torch.einsum("jakb,kja->bja", Mp, y)                    # w2(j) = sum_k M(k, numband + j) w(k)
        z += torch.einsum("jakb,bja->kja", Mp, w2)                   # w(j)  = sum_k M(j, numband + k) w2(k)
        out = torch.empty_like(r)
        for i, c in enumerate(self.comps):                           # :2350-2363
            self.extract_comp(i, out).copy_(z[i, :c.nmaps, self.pre_idx[i]])
        return out

    def invM(self, r):
        """cr_invM: applyDiffPrecond_diagonal (:2186-2235) or, with precond = 'pseudoinv', applyDiffPrecond_pseudoinv."""
        torch = self.torch
        if getattr(self, "precond", "diagonal") == "pseudoinv":
            return self.invM_pseudoinv(r)
        if self.Minv is None:
            self.initDiffPrecond_diagonal()
        npre = len(self.comps)
        nmaps_pre, nalm_pre = self.Minv.shape[0], self.Minv.shape[1]
        yv = torch.zeros((nmaps_pre, nalm_pre, npre), dtype=torch.float64, device=self.dev)
        for i, c in enumerate(self.comps):
            yv[:c.nmaps, self.pre_idx[i], i] = self.extract_comp(i, r)
        yv = torch.einsum("jakb,jab->jak", self.Minv, yv)
        out = torch.empty_like(r)
        for i, c in enumerate(self.comps):
            self.extract_comp(i, out).copy_(yv[:c.nmaps, self.pre_idx[i], i])
        return out


def _view_maps(m: comm_map, info: comm_mapinfo, nm: int) -> comm_map:
    """The first nm columns of m's a_lm as a comm_map on `info` (same nside / lmax, fewer maps)."""
    v = comm_map.__new__(comm_map)
    v.info, v.device = info, m.device
    v.alm, v.map = m.alm[:nm], m.map[:nm]
    return v


# =====================================================================================================
# The same CMB system behind the C ABI (cmdr_cr_*, commander_b200/csrc/cr.cu): no torch in the operator, the
# sqrt(S) / beam / N^-1 passes fused into the transform kernels, dot products reduced on the device.
# =====================================================================================================

def _draw_args(seed, draw, pixel, prior):
    """(seed, draw, terms) of cmdr_cr_compute_rhs_draw, after the range checks."""
    from . import sharp
    for name, v in (("seed", seed), ("draw", draw)):
        if not isinstance(v, (int, np.integer)) or not 0 <= int(v) < 2 ** 64:
            raise ValueError(f"{name} must be an integer in [0, 2^64), got {v!r}")
    return int(seed), int(draw), (sharp.CMDR_CR_ETA_PIX if pixel else 0) | (sharp.CMDR_CR_ETA_ALM if prior else 0)


def _cuda_probe(device=None):
    """An empty float64 tensor on `device` (default: the current CUDA device): what output buffers follow when no input
    array says where they live."""
    import torch
    return torch.empty(0, dtype=torch.float64, device=device if device is not None else torch.device("cuda", torch.cuda.current_device()))


def _ptrs(arrs):
    """Array of column pointers over a list of 1-D views (numpy or torch); returns (ctypes array, keep-alive)."""
    import ctypes as C
    p = (C.c_void_p * len(arrs))()
    for i, a in enumerate(arrs):
        if isinstance(a, np.ndarray):
            if a.dtype != np.float64 or not a.flags.c_contiguous:
                raise ValueError("expected contiguous float64 columns")
            p[i] = a.ctypes.data
        else:
            import torch
            if a.dtype != torch.float64 or not a.is_contiguous():
                raise ValueError("expected contiguous float64 columns")
            p[i] = a.data_ptr()
    return p, arrs


class cr_native_system:
    """One signal component with a diagonal prior C_l (or none) seen through `nbands` bands that share `info`:
    handle of cmdr_cr_setup.  invN: list (per band) of (nmaps, np) arrays, numpy or torch; b_l: list (per band) of
    (lmax+1, nmaps) beams (times mb_eff and F_mean); Cl: (lmax+1, nmaps) or None; precond 'diagonal' | 'none'."""

    def __init__(self, info: comm_mapinfo, invN, b_l, Cl=None, precond: str = "diagonal"):
        from . import sharp
        self.info = info
        self.nbands, self.nmaps = len(invN), info.nmaps
        if len(b_l) != self.nbands:
            raise ValueError("one beam per band")
        if precond not in ("diagonal", "none"):
            raise ValueError("Preconditioner type not supported: " + precond)
        nm = self.nmaps
        icols = [invN[b][c] for b in range(self.nbands) for c in range(nm)]
        self._bl = [np.ascontiguousarray(np.asarray(b_l[b], dtype=np.float64)[:, c]) for b in range(self.nbands) for c in range(nm)]
        self._sS = None
        if Cl is not None:
            self._sS = [np.ascontiguousarray(np.sqrt(np.maximum(np.asarray(Cl, dtype=np.float64)[:, c], 0.0))) for c in range(nm)]
        ip, _k1 = _ptrs(icols)
        bp, _k2 = _ptrs(self._bl)
        sp = None
        if self._sS is not None:
            sp, _k3 = _ptrs(self._sS)
        c = info.comm
        comm = c.handle if (info.dist and c.size > 1) else -1
        gp = info.geom_info_P.handle if info.geom_info_P is not None else None
        self.handle = sharp.lib().cmdr_cr_setup(comm, self.nbands, nm, info.geom_info_T.handle, gp, info.alm_info.handle,
                                                ip, bp, sp, 1 if precond == "diagonal" else 0)
        self.L = sharp.lib()

    def __del__(self):
        if getattr(self, "handle", None):
            self.L.cmdr_cr_destroy(self.handle)
            self.handle = None

    def _like(self, v):
        if isinstance(v, np.ndarray):
            return np.empty((self.nmaps, self.info.nalm))
        import torch
        return torch.empty((self.nmaps, self.info.nalm), dtype=torch.float64, device=v.device)

    @property
    def n_matmul(self):
        return int(self.L.cmdr_cr_matmul_count(self.handle))

    def matmulA(self, x):
        """cr_matmulA, commander3/src/comm_cr_mod.f90:771-1024"""
        y = self._like(x)
        xp, _a = _ptrs([x[c] for c in range(self.nmaps)])
        yp, _b = _ptrs([y[c] for c in range(self.nmaps)])
        self.L.cmdr_cr_matmulA(self.handle, xp, yp, None)
        return y

    def invM(self, r):
        """cr_invM, commander3/src/comm_cr_mod.f90:1026-1077 (diagonal)"""
        z = self._like(r)
        rp, _a = _ptrs([r[c] for c in range(self.nmaps)])
        zp, _b = _ptrs([z[c] for c in range(self.nmaps)])
        self.L.cmdr_cr_invM(self.handle, rp, zp, None)
        return z

    def Minv(self):
        out = np.empty((self.nmaps, self.info.nalm))
        op, _a = _ptrs([out[c] for c in range(self.nmaps)])
        self.L.cmdr_cr_get_precond_diag(self.handle, op)
        return out

    def computeRHS(self, data, eta_pix=None, eta_alm=None):
        """cr_computeRHS, commander3/src/comm_cr_mod.f90:542-769; data / eta_pix: lists (per band) of (nmaps, np) arrays."""
        nm = self.nmaps
        b = self._like(data[0])
        dp, _a = _ptrs([data[q][c] for q in range(self.nbands) for c in range(nm)])
        ep = None
        if eta_pix is not None:
            ep, _b = _ptrs([eta_pix[q][c] for q in range(self.nbands) for c in range(nm)])
        ap = None
        if eta_alm is not None:
            ap, _c = _ptrs([eta_alm[c] for c in range(nm)])
        bp, _d = _ptrs([b[c] for c in range(nm)])
        self.L.cmdr_cr_compute_rhs(self.handle, dp, ep, ap, bp, None)
        return b

    def computeRHS_draw(self, data, seed, draw, pixel=True, prior=True):
        """cr_computeRHS with the fluctuation terms drawn on the device (cmdr_cr_compute_rhs_draw, stream of
        commander_b200/csrc/rng.cuh): data as for computeRHS, or None for the fluctuation terms alone (d = 0); seed and
        draw unsigned 64-bit (draw: e.g. the Gibbs sample index); pixel / prior: the N^-1/2 eta_nu and eta_0 terms (eta_0
        only with a prior).  b follows data (numpy or torch on its device); with data None it is a torch tensor on the
        current CUDA device.  Collective."""
        seed, draw, terms = _draw_args(seed, draw, pixel, prior)
        nm = self.nmaps
        b = self._like(data[0] if data is not None else _cuda_probe())
        dp = None
        if data is not None:
            dp, _a = _ptrs([data[q][c] for q in range(self.nbands) for c in range(nm)])
        bp, _d = _ptrs([b[c] for c in range(nm)])
        self.L.cmdr_cr_compute_rhs_draw(self.handle, dp, seed, draw, terms, bp, None)
        return b

    def draw_eta(self, seed, draw, device=None):
        """The draws of computeRHS_draw written out (cmdr_cr_draw_eta): (eta_pix, eta_alm) in computeRHS's layouts, a
        list (per band) of (nmaps, np) and one (nmaps, nalm), zeros without a prior; torch tensors on `device` (default:
        the current CUDA device).  computeRHS(data, *draw_eta(s, d)) equals computeRHS_draw(data, s, d) bit for bit."""
        import torch
        seed, draw, _ = _draw_args(seed, draw, True, True)
        dev = _cuda_probe(device).device
        eta_pix = [torch.empty((self.nmaps, self.info.np), dtype=torch.float64, device=dev) for _ in range(self.nbands)]
        eta_alm = torch.empty((self.nmaps, self.info.nalm), dtype=torch.float64, device=dev)
        ep, _a = _ptrs([e[c] for e in eta_pix for c in range(self.nmaps)])
        ap, _b = _ptrs([eta_alm[c] for c in range(self.nmaps)])
        self.L.cmdr_cr_draw_eta(self.handle, seed, draw, ep, ap, None)
        return eta_pix, eta_alm

    def solve(self, b, x0=None, maxiter=300, cg_tol=1e-8, cg_conv_crit="residual", cg_miniter=5, cg_check_conv_freq=1):
        """solve_cr_eqn_by_CG, commander3/src/comm_cr_mod.f90:201-348.  Returns (x, iterations done, residual history)."""
        import ctypes as C
        if cg_conv_crit not in ("residual", "fixed_iter"):
            raise ValueError("Unsupported convergence criterion = " + cg_conv_crit)
        x = self._like(b)
        if x0 is not None:
            x[...] = x0
        bp, _a = _ptrs([b[c] for c in range(self.nmaps)])
        xp, _b = _ptrs([x[c] for c in range(self.nmaps)])
        hist = (C.c_double * (maxiter + 1))()
        it = self.L.cmdr_cr_solve(self.handle, bp, xp, 1 if x0 is not None else 0, int(maxiter), float(cg_tol),
                                  0 if cg_conv_crit == "residual" else 1, int(cg_miniter), int(cg_check_conv_freq), hist, None)
        return x, int(it), [float(hist[i]) for i in range(it + 1)]


# =====================================================================================================
# The general system behind the C ABI (cmdr_cr_setup_multi, commander_b200/csrc/cr_multi.cu): the components and bands
# of cr_system, F_mean mixing, the block-diagonal preconditioner; vectors in cr_system's flat layout.
# =====================================================================================================

class cr_native_multi_system:
    """Several diffuse components seen through bands of their own nside, lmax, beam and noise: the handle of
    cmdr_cr_setup_multi.  `comps` / `bands` are the cr_component / cr_band objects of cr_system; vectors are flat
    float64 arrays of length ncr in cr_system's layout (component after component, each (nmaps, nalm)), numpy or torch.
    precond: 'diagonal' (the block-diagonal preconditioner of cr_system.initDiffPrecond_diagonal, from F_mean) or 'none'.
    pixel_mixing: install every per-pixel mixing map c.F[q] that is not None (cmdr_cr_set_mixing_map); without it a
    component that carries one is refused.  set_mixing_map replaces or removes one between solves; set_pseudoinv switches
    to the pseudo-inverse preconditioner and back."""

    def __init__(self, comps, bands, precond: str = "diagonal", pixel_mixing: bool = False):
        import ctypes as C
        from . import sharp
        self.comps, self.bands = list(comps), list(bands)
        if not self.comps or not self.bands:
            raise ValueError("at least one component and one band")
        if precond not in ("diagonal", "none"):
            raise ValueError("Preconditioner type not supported: " + str(precond))
        nb, nc = len(self.bands), len(self.comps)
        for b in self.bands:
            if not isinstance(b, cr_band):
                raise ValueError("bands must be cr_band objects")
            nm = b.info.nmaps
            if tuple(b.invN.shape) != (nm, b.info.np):
                raise ValueError(f"band invN has shape {tuple(b.invN.shape)}, expected {(nm, b.info.np)}")
            if b.b_l.ndim != 2 or b.b_l.shape[0] < b.info.lmax + 1 or b.b_l.shape[1] < nm:
                raise ValueError(f"band b_l has shape {b.b_l.shape}, expected at least {(b.info.lmax + 1, nm)}")
        F = np.zeros((nb, nc, 3))
        for k, c in enumerate(self.comps):
            if not isinstance(c, cr_component):
                raise ValueError("comps must be cr_component objects")
            if c.F is not None and any(f is not None for f in c.F):
                if not pixel_mixing:
                    raise ValueError("per-pixel mixing F is not supported by the native system (use cr_system)")
                if len(c.F) != nb:
                    raise ValueError(f"component F has {len(c.F)} entries, expected one per band ({nb})")
            if c.F_mean.ndim != 2 or c.F_mean.shape[0] != nb or c.F_mean.shape[1] < c.nmaps:
                raise ValueError(f"component F_mean has shape {c.F_mean.shape}, expected ({nb}, {c.nmaps})")
            F[:, k, :c.nmaps] = c.F_mean[:, :c.nmaps]
            if c.Cl is not None and (c.Cl.ndim != 2 or c.Cl.shape[0] < c.lmax_amp + 1 or c.Cl.shape[1] < c.nmaps):
                raise ValueError(f"component Cl has shape {c.Cl.shape}, expected at least {(c.lmax_amp + 1, c.nmaps)}")
        self.off = [0]
        for c in self.comps:
            self.off.append(self.off[-1] + c.nmaps * c.x_info.nalm)
        self.ncr = self.off[-1]
        self._F = np.ascontiguousarray(F)
        mixing = []                                           # (q, k, columns), checked before anything is allocated
        if pixel_mixing:
            for k, c in enumerate(self.comps):
                for q, f in enumerate(c.F or []):
                    if f is not None:
                        mixing.append((q, k, self._mixing_cols(q, k, f)))
        # host columns the library reads during setup
        sS = []
        for c in self.comps:
            for j in range(c.nmaps):
                sS.append(None if c.Cl is None else np.ascontiguousarray(np.sqrt(np.maximum(c.Cl[:c.lmax_amp + 1, j], 0.0))))
        bl = [np.ascontiguousarray(b.b_l[:b.info.lmax + 1, j]) for b in self.bands for j in range(b.info.nmaps)]
        icols = [b.invN[j] for b in self.bands for j in range(b.info.nmaps)]
        ip, _k1 = _ptrs(icols)
        bp, _k2 = _ptrs(bl)
        sp = (C.c_void_p * len(sS))(*[None if a is None else a.ctypes.data for a in sS])

        def handles(hs):
            return (C.c_void_p * len(hs))(*[None if h is None else h.handle.value for h in hs])
        comp_alm = handles([c.x_info.alm_info for c in self.comps])
        comp_nm = (C.c_int * nc)(*[c.nmaps for c in self.comps])
        gT = handles([b.info.geom_info_T for b in self.bands])
        gP = handles([b.info.geom_info_P if b.info.nmaps == 3 else None for b in self.bands])
        band_alm = handles([b.info.alm_info for b in self.bands])
        band_nm = (C.c_int * nb)(*[b.info.nmaps for b in self.bands])
        info = self.bands[0].info
        comm = info.comm.handle if (info.dist and info.comm.size > 1) else -1
        self.L = sharp.lib()
        self.handle = self.L.cmdr_cr_setup_multi(comm, nc, comp_alm, comp_nm, sp, nb, gT, gP, band_alm, band_nm, ip, bp,
                                                 self._F.ctypes.data, 1 if precond == "diagonal" else 0)
        for q, k, cols in mixing:
            fp, _keep = _ptrs(cols)
            self.L.cmdr_cr_set_mixing_map(self.handle, q, k, fp, None)

    def set_mixing_map(self, q, k, F):
        """Per-pixel mixing of component k in band q (the Y, x F, YtW branch of evalDiffuseBand / projectDiffuseBand,
        commander3/src/comm_diffuse_comp_mod.f90:2070-2083, 2142-2151): F of shape (>= min(nmaps_q, nmaps_k), np_q),
        this rank's pixels of the band, numpy or torch; None returns the pair to F_mean mixing.  Collective."""
        if F is None:
            self._mixing_cols(q, k, None)
            self.L.cmdr_cr_set_mixing_map(self.handle, q, k, None, None)
            return
        fp, _keep = _ptrs(self._mixing_cols(q, k, F))
        self.L.cmdr_cr_set_mixing_map(self.handle, q, k, fp, None)

    def set_pseudoinv(self, on=True):
        """Selects the pseudo-inverse preconditioner (cr_system's precond = 'pseudoinv': applyDiffPrecond_pseudoinv,
        commander3/src/comm_diffuse_comp_mod.f90:2237-2380) for invM and solve, built on the device the first time; on=False
        returns to the preconditioner chosen at construction.  Collective; invM is collective while it is selected."""
        self.L.cmdr_cr_set_pseudoinv(self.handle, 1 if on else 0, None)

    def _mixing_cols(self, q, k, F):
        """The min(nmaps_q, nmaps_k) float64 columns of a mixing map, after the range and shape checks."""
        nb, nc = len(self.bands), len(self.comps)
        if not 0 <= q < nb:
            raise ValueError(f"band {q} out of range ({nb} bands)")
        if not 0 <= k < nc:
            raise ValueError(f"component {k} out of range ({nc} components)")
        if F is None:
            return None
        if not hasattr(F, "data_ptr"):
            F = np.asarray(F, dtype=np.float64)
        info = self.bands[q].info
        n = min(info.nmaps, self.comps[k].nmaps)
        shape = tuple(F.shape)
        if len(shape) != 2 or shape[0] < n or shape[1] != info.np:
            raise ValueError(f"F of component {k} in band {q} has shape {shape}, expected ({n} or more, {info.np})")
        if isinstance(F, np.ndarray):
            return [np.ascontiguousarray(F[j], dtype=np.float64) for j in range(n)]
        import torch
        return [F[j].to(torch.float64).contiguous() for j in range(n)]

    def __del__(self):
        if getattr(self, "handle", None):
            self.L.cmdr_cr_destroy(self.handle)
            self.handle = None

    @property
    def n_matmul(self):
        return int(self.L.cmdr_cr_matmul_count(self.handle))

    def _cols(self, v):
        """Column pointers of a flat vector of length ncr (component-major, each (nmaps, nalm))."""
        shape = tuple(v.shape)
        if shape != (self.ncr,):
            raise ValueError(f"vector of shape {shape}, expected ({self.ncr},)")
        cols = []
        for k, c in enumerate(self.comps):
            n = c.x_info.nalm
            cols += [v[self.off[k] + j * n:self.off[k] + (j + 1) * n] for j in range(c.nmaps)]
        return _ptrs(cols)

    def _like(self, v):
        if isinstance(v, np.ndarray):
            return np.empty(self.ncr)
        import torch
        return torch.empty(self.ncr, dtype=torch.float64, device=v.device)

    def _band_cols(self, maps, what):
        if len(maps) != len(self.bands):
            raise ValueError(f"{what}: one map array per band")
        cols = []
        for b, m in zip(self.bands, maps):
            if tuple(m.shape) != (b.info.nmaps, b.info.np):
                raise ValueError(f"{what}: shape {tuple(m.shape)}, expected {(b.info.nmaps, b.info.np)}")
            cols += [m[j] for j in range(b.info.nmaps)]
        return _ptrs(cols)

    def matmulA(self, x):
        """cr_matmulA, commander3/src/comm_cr_mod.f90:771-1024"""
        y = self._like(x)
        xp, _a = self._cols(x)
        yp, _b = self._cols(y)
        self.L.cmdr_cr_matmulA(self.handle, xp, yp, None)
        return y

    def invM(self, r):
        """cr_invM with the block-diagonal preconditioner (comm_diffuse_comp_mod.f90:2186-2235), the identity, or the
        pseudo-inverse after set_pseudoinv()"""
        z = self._like(r)
        rp, _a = self._cols(r)
        zp, _b = self._cols(z)
        self.L.cmdr_cr_invM(self.handle, rp, zp, None)
        return z

    def computeRHS(self, data, eta_pix=None, eta_alm=None):
        """cr_computeRHS, commander3/src/comm_cr_mod.f90:542-769; data / eta_pix: lists (per band) of (nmaps, np) arrays,
        eta_alm: a flat vector (used on the components with a prior)."""
        b = self._like(data[0])
        dp, _a = self._band_cols(data, "data")
        ep = ap = None
        if eta_pix is not None:
            ep, _b = self._band_cols(eta_pix, "eta_pix")
        if eta_alm is not None:
            ap, _c = self._cols(eta_alm)
        bp, _d = self._cols(b)
        self.L.cmdr_cr_compute_rhs(self.handle, dp, ep, ap, bp, None)
        return b

    def computeRHS_draw(self, data, seed, draw, pixel=True, prior=True):
        """cr_computeRHS with the fluctuation terms drawn on the device (cmdr_cr_compute_rhs_draw, stream of
        commander_b200/csrc/rng.cuh): data as for computeRHS, or None for the fluctuation terms alone (d = 0); seed and
        draw unsigned 64-bit; pixel / prior: the N^-1/2 eta_nu and eta_0 terms (eta_0 on the components with a prior).
        b follows data (numpy or torch on its device); with data None it is a torch tensor on the current CUDA device.
        Collective."""
        seed, draw, terms = _draw_args(seed, draw, pixel, prior)
        b = self._like(data[0] if data is not None else _cuda_probe())
        dp = None
        if data is not None:
            dp, _a = self._band_cols(data, "data")
        bp, _d = self._cols(b)
        self.L.cmdr_cr_compute_rhs_draw(self.handle, dp, seed, draw, terms, bp, None)
        return b

    def draw_eta(self, seed, draw, device=None):
        """The draws of computeRHS_draw written out (cmdr_cr_draw_eta): (eta_pix, eta_alm) in computeRHS's layouts, a
        list (per band) of (nmaps_q, np_q) and a flat vector of length ncr (zeros on the components without a prior);
        torch tensors on `device` (default: the current CUDA device)."""
        import torch
        seed, draw, _ = _draw_args(seed, draw, True, True)
        dev = _cuda_probe(device).device
        eta_pix = [torch.empty((b.info.nmaps, b.info.np), dtype=torch.float64, device=dev) for b in self.bands]
        eta_alm = torch.empty(self.ncr, dtype=torch.float64, device=dev)
        ep, _a = self._band_cols(eta_pix, "eta_pix")
        ap, _b = self._cols(eta_alm)
        self.L.cmdr_cr_draw_eta(self.handle, seed, draw, ep, ap, None)
        return eta_pix, eta_alm

    def solve(self, b, x0=None, maxiter=300, cg_tol=1e-8, cg_conv_crit="residual", cg_miniter=5, cg_check_conv_freq=1):
        """solve_cr_eqn_by_CG, commander3/src/comm_cr_mod.f90:201-348.  Returns (x, iterations done, residual history)."""
        import ctypes as C
        if cg_conv_crit not in ("residual", "fixed_iter"):
            raise ValueError("Unsupported convergence criterion = " + cg_conv_crit)
        x = self._like(b)
        if x0 is not None:
            x[...] = x0
        bp, _a = self._cols(b)
        xp, _b = self._cols(x)
        hist = (C.c_double * (maxiter + 1))()
        it = self.L.cmdr_cr_solve(self.handle, bp, xp, 1 if x0 is not None else 0, int(maxiter), float(cg_tol),
                                  0 if cg_conv_crit == "residual" else 1, int(cg_miniter), int(cg_check_conv_freq), hist, None)
        return x, int(it), [float(hist[i]) for i in range(it + 1)]
