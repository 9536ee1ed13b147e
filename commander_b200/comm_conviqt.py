"""Host-side mirror of `comm_conviqt_mod` (commander3/src/comm_conviqt_mod.f90): the 4pi beam convolution
cube used for sidelobe corrections of time-ordered data.

    comm_conviqt(...)       constructor,    :60-153   beam table, psi grid, cube, then precompute_sky
    %precompute_sky(map)    :207-292                  bmax+1 spin-j syntheses + a psi FFT per pixel
    %get_alms(m_b, map)     :294-357                  (kept for inspection; the library does it on the device)
    %interp(pix, psi)       :155-205                  psi lookup / linear interpolation (host restatement; on the
                                                      device: make_sampler() -> conviqt_sampler.interp)

In the reference precompute_sky loops `sharp_execute(SHARP_Y, j, 2, ...)` over host arrays and then runs FFTW
c2r per pixel on the host.  Here it is ONE library call (`cmdr_sht_conviqt_cube`): the coefficient products,
the syntheses and the psi transform all run on the device and only the sky a_lm go in and the
single-precision cube comes out (or stays in HBM with device='cuda').

Layout: `c` has shape (psisteps, np) over this rank's pixels `info.pix` -- c%a(pix+1, psi+1) of the
reference, which keeps all ranks' pixels in one MPI shared-memory window (:140-141); `alm_beam` has shape
(ntri, nmaps) complex64 -- alm_beam%a(nmaps, nalm_tot) in memory order, triangular index l(l+1)/2 + m.
"""
from __future__ import annotations

import math

import numpy as np

from . import sharp
from .comm_map import comm_map, comm_mapinfo


class comm_conviqt:
    def __init__(self, nside, lmax, nmaps, bmax, beam: comm_map, map: comm_map, optim=0, device=None,
                 precompute=True):
        """constructor, :60-153 (the shared-memory communicator arguments have no counterpart: every process
        holds the beam table, as every node does in the reference)."""
        self.lmax = lmax
        self.mmax = min(beam.info.lmax, lmax)             # beam%info%mmax = its lmax (comm_map_mod.f90:189)
        self.bmax = bmax
        self.nside = nside
        self.nmaps = nmaps
        self.npix = 12 * nside ** 2
        self.comm = map.info.comm
        self.optim = optim
        self.device = device
        self.psisteps = 2 * bmax                          # :91
        self.psires = np.float32(2.0 * math.pi / self.psisteps)   # real(sp), :39, :92
        l = np.arange(lmax + 1, dtype=np.float64)
        self.lnorm = 0.5 * np.sqrt(4.0 * math.pi / (2.0 * l + 1.0))   # :94-97
        self.info = comm_mapinfo(map.info.comm, nside, lmax, nmaps, nmaps == 3)   # :99
        self.alm_beam = self._beam_table(beam)            # :101-125
        if device is None:
            self.c = np.zeros((self.psisteps, self.info.np), dtype=np.float32)    # :128-129
        else:
            import torch
            self.c = torch.zeros((self.psisteps, self.info.np), dtype=torch.float32, device=device)
            self.alm_beam = torch.as_tensor(self.alm_beam, device=device)
        if precompute:
            self.precompute_sky(map)                      # :131

    def _beam_table(self, beam: comm_map):
        """:101-125: single-precision complex beam coefficients for every (l, m >= 0), all ranks' m's."""
        info = self.info
        ntri = (self.lmax + 1) * (self.lmax + 2) // 2
        tab = np.zeros((ntri, self.nmaps, 2), dtype=np.float32)
        l, m = info.lm[0].astype(np.int64), info.lm[1].astype(np.int64)
        sel = m >= 0
        l, m = l[sel], m[sel]
        k = beam.info.lm2i_vec(l, m)
        ok = k >= 0
        l, m, k = l[ok], m[ok], k[ok]
        j = l * (l + 1) // 2 + m
        balm = beam.alm if isinstance(beam.alm, np.ndarray) else beam.alm.cpu().numpy()
        q = min(self.nmaps, balm.shape[0])
        s2 = np.float32(math.sqrt(np.float32(2.0)))
        z = m == 0
        tab[j[z], :q, 0] = balm[:q, k[z]].T.astype(np.float32)
        nz = ~z
        tab[j[nz], :q, 0] = balm[:q, k[nz]].T.astype(np.float32) / s2
        tab[j[nz], :q, 1] = balm[:q, k[nz] + 1].T.astype(np.float32) / s2
        if info.dist and info.comm.size > 1:
            # sync_shared_2d_spc_alm (:124-125): every rank contributes its own m's
            import torch
            import torch.distributed as dist
            t = torch.from_numpy(tab)
            if dist.get_backend() == "nccl":
                t = t.cuda()
            dist.all_reduce(t)
            tab = t.cpu().numpy()
        return np.ascontiguousarray(tab).view(np.complex64).reshape(ntri, self.nmaps)

    def _comm(self):
        c = self.info.comm
        return c.handle if (self.info.dist and c.size > 1) else None

    def precompute_sky(self, map: comm_map, cube=None):
        """:207-292.  `map` must hold a_lm on the layout of self.info.  Fills self.c (or `cube`, which may be
        float64 to see the values before the reference's real(., sp) rounding)."""
        if map.info.nalm != self.info.nalm or map.info.nmaps < self.nmaps:
            raise ValueError("map must hold a_lm on the conviqt layout (nside, lmax, nmaps of the constructor)")
        out = self.c if cube is None else cube
        sharp.conviqt_cube(map.alm[:self.nmaps], self.alm_beam, self.bmax, self.info.geom_info_T,
                           self.info.alm_info, out, comm=self._comm())
        return out

    def get_alms(self, m_b, map: comm_map):
        """:294-357, vectorised on the host; returns alm (2, nalm).  Inspection/tests only: precompute_sky does
        this step inside the library."""
        info = self.info
        salm = map.alm if isinstance(map.alm, np.ndarray) else map.alm.cpu().numpy()
        beam = self.alm_beam if isinstance(self.alm_beam, np.ndarray) else self.alm_beam.cpu().numpy()
        l, m = info.lm[0].astype(np.int64), info.lm[1].astype(np.int64)
        i = np.nonzero((m >= 0) & (l >= m_b))[0]
        l, m = l[i], m[i]
        ineg = np.where(m > 0, i + 1, i)
        spinsign = -1.0 if m_b else 1.0
        mfac = np.where(m & 1, -1.0, 1.0)
        alm_b = beam[l * (l + 1) // 2 + m_b].astype(np.complex128)             # (n, nmaps)
        s = salm[:self.nmaps]
        alm_s = np.where(m > 0, 1.0 / math.sqrt(2.0) * (s[:, i] + 1j * s[:, ineg]), s[:, i] + 0j).T
        v1 = (alm_s * alm_b).sum(axis=1)
        v2 = (np.conj(alm_s) * alm_b).sum(axis=1) * mfac
        out = np.zeros((2, info.nalm))
        almc = spinsign * self.lnorm[l] * (v1 + np.conj(v2) * mfac)
        f = np.where(m > 0, math.sqrt(2.0), 1.0)
        nz = m > 0
        out[0, i] = almc.real * f
        out[0, ineg[nz]] = almc.imag[nz] * f[nz]
        if m_b > 0:
            almc = -1j * spinsign * self.lnorm[l] * (v1 - np.conj(v2) * mfac)
            out[1, i] = almc.real * f
            out[1, ineg[nz]] = almc.imag[nz] * f[nz]
        return out

    def interp(self, pix, psi):
        """:155-205, vectorised over samples: `pix` global RING pixel numbers owned by this rank, `psi` angles.
        Single-precision arithmetic as in the reference."""
        f = np.float32
        c = self.c if isinstance(self.c, np.ndarray) else self.c.cpu().numpy()
        pix = np.atleast_1d(np.asarray(pix, dtype=np.int64))
        if self.info.np == self.npix:
            loc = pix
        else:
            loc = np.searchsorted(self.info.pix, pix)
            if np.any(loc >= self.info.np) or np.any(self.info.pix[np.minimum(loc, self.info.np - 1)] != pix):
                raise IndexError("pixel not owned by this rank")
        twopi = f(2.0 * math.pi)
        unwrap = np.fmod(-np.atleast_1d(np.asarray(psi)).astype(f), twopi).astype(f)
        unwrap = np.where(unwrap < 0, unwrap + twopi, unwrap).astype(f)         # Fortran modulo
        if self.optim == 2:
            bpsi = np.maximum(np.rint(unwrap / self.psires).astype(np.int64), 0)
            bpsi[bpsi == self.psisteps] = 0
            return c[bpsi, loc]
        psii = (unwrap / self.psires).astype(np.int64)
        psiu = psii + 1
        psiu[psiu >= self.psisteps] = 0
        x0 = (psii.astype(f) * self.psires).astype(f)
        x1 = (psiu.astype(f) * self.psires).astype(f)
        with np.errstate(divide="ignore", invalid="ignore"):
            return ((c[psii, loc] * (x1 - unwrap) + c[psiu, loc] * (unwrap - x0)) / (x1 - x0)).astype(f)

    def make_sampler(self):
        """The cube of ALL ranks on every GPU of the group, ready for interp at any pixel: the device counterpart of the
        reference's node-shared window (:140-141).  Collective on the communicator of self.info; build it after
        precompute_sky (later updates of self.c do not reach it)."""
        return conviqt_sampler(self.c, self.bmax, self.npix, self.optim, self.info.geom_info_T, comm=self._comm())

    def dealloc(self):
        """:360-368"""
        self.c = None
        self.alm_beam = None


class conviqt_sampler:
    """interp (:155-205) on the device (cmdr_sht_conviqt_interp), bit for bit the single-precision arithmetic of the
    reference, for any global RING pixel on any rank."""

    def __init__(self, cube, bmax, npix, optim, geom_T, comm=None):
        import torch
        self.npix, self.optim = npix, optim
        self.device = torch.device("cuda", torch.cuda.current_device()) if isinstance(cube, np.ndarray) else cube.device
        with torch.cuda.device(self.device):
            st = None if isinstance(cube, np.ndarray) else torch.cuda.current_stream().cuda_stream
            self.handle = sharp.conviqt_sampler(cube, bmax, geom_T, stream=st, comm=comm)

    def interp(self, pix, psi, out=None):
        """Samples at global RING pixels `pix` and angles `psi` (broadcast together): numpy in, numpy out; torch in, torch
        out (on the sampler's device, or host tensors).  psi is rounded to float32 first, as the mirror does.  A pixel
        outside 0 .. 12 nside^2 - 1 raises IndexError after the call (its entry of `out` is NaN)."""
        import torch
        if isinstance(pix, torch.Tensor) or isinstance(psi, torch.Tensor):
            p = torch.as_tensor(pix)
            p, q = torch.broadcast_tensors(p, torch.as_tensor(psi, device=p.device))
            if p.is_cuda and p.device != self.device:
                raise ValueError(f"samples on {p.device}, sampler on {self.device}")
            shape = p.shape
            p, q = p.reshape(-1), q.reshape(-1)
            if p.dtype != torch.int32:
                p = torch.where((p < 0) | (p >= self.npix), -1, p).to(torch.int32)
            p, q = p.contiguous(), q.to(torch.float32).contiguous()
            if out is None:
                out = torch.empty(shape, dtype=torch.float32, device=p.device)
            st = torch.cuda.current_stream(self.device).cuda_stream if p.is_cuda else None
        else:
            p, q = np.broadcast_arrays(np.atleast_1d(np.asarray(pix)), np.atleast_1d(np.asarray(psi)))
            shape = p.shape
            p = p.reshape(-1)
            if p.dtype != np.int32:
                p = np.where((p < 0) | (p >= self.npix), -1, p).astype(np.int32)
            p, q = np.ascontiguousarray(p), np.ascontiguousarray(q.reshape(-1), dtype=np.float32)
            if out is None:
                out = np.empty(shape, dtype=np.float32)
            st = None
        if tuple(out.shape) != tuple(shape) or not (out.flags.c_contiguous if isinstance(out, np.ndarray)
                                                    else out.is_contiguous()):
            raise ValueError(f"out must be contiguous with shape {tuple(shape)}")
        with torch.cuda.device(self.device):
            nbad = sharp.conviqt_interp(self.handle, p, q, self.optim, out.reshape(-1), stream=st)
        if nbad:
            raise IndexError(f"{nbad} pixel(s) outside 0..{self.npix - 1}")
        return out

    def close(self):
        if getattr(self, "handle", None):
            sharp.conviqt_sampler_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()
