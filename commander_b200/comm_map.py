"""Host-side mirror of the hot-path part of `comm_map_mod`
(commander3/src/comm_map_mod.f90): the `comm_mapinfo` layout object and the
`comm_map` container with its Y / Yt / YtW / WY operators.  Names, argument meaning
and index conventions follow the Fortran so that tests read like the reference's.

Only what the SHT path needs is mirrored (SURVEY.md 8a rows a1, a5-a11); FITS/HDF IO,
udgrade and the power-spectrum helpers are out of scope.
"""
from __future__ import annotations

import math
import os

import numpy as np

from . import sharp


class SelfComm:
    """Stand-in for an MPI communicator of one rank (comm_chain with -np 1)."""

    rank, size, handle = 0, 1, None


def _in_ring_count(nside: int, ring: int) -> int:
    north = 4 * nside - ring if ring > 2 * nside else ring
    return 4 * north if north < nside else 4 * nside


def _ring_start(nside: int, ring: int) -> int:
    """First RING-scheme pixel index of a ring (what HEALPix `in_ring` lists)."""
    npix = 12 * nside * nside
    north = 4 * nside - ring if ring > 2 * nside else ring
    if north < nside:
        ofs, nph = 2 * north * (north - 1), 4 * north
    else:
        ofs, nph = 2 * nside * (nside - 1) + (north - nside) * 4 * nside, 4 * nside
    return ofs if north == ring else npix - nph - ofs


_repack_cache: dict = {}   # alm_equal index pairs for device-resident maps
_mapinfos: list = []   # the `mapinfos` linked list, commander3/src/comm_map_mod.f90:157-169


def load_ring_weights(nside: int, ncol: int):
    """Ring weights W(2*nside, ncol) = file + 1 (commander3/src/comm_map_mod.f90:266-282).

    The reference reads $HEALPIX/data/weight_ring_nNNNNN.fits through cfitsio.  Neither
    HEALPix nor cfitsio exists in this image, so this mirror accepts the same table as
    $HEALPIX/data/weight_ring_nNNNNN.npy (shape (2*nside, >=ncol), the raw file values) and
    otherwise uses unit weights (file value 0)."""
    hp = os.environ.get("HEALPIX", "")
    path = os.path.join(hp, "data", "weight_ring_n%05d.npy" % nside)
    if hp and os.path.exists(path):
        raw = np.load(path)[:, :ncol]
    else:
        raw = np.zeros((2 * nside, ncol))
    return np.ascontiguousarray(raw.T + 1.0)   # shape (ncol, 2*nside)


class comm_mapinfo:
    """constructor_mapinfo, commander3/src/comm_map_mod.f90:134-305."""

    def __new__(cls, comm, nside, lmax, nmaps, pol, dist=True, weights=None):
        comm = comm if comm is not None else SelfComm()
        if weights is None:
            for p in _mapinfos:
                if (p.nside, p.lmax, p.nmaps, p.pol, p.dist) == (nside, lmax, nmaps, pol, dist) and p.comm is comm \
                        and not p._custom_w:
                    return p
        self = super().__new__(cls)
        self._init(comm, nside, lmax, nmaps, pol, dist, weights)
        if weights is None:
            _mapinfos.append(self)
        return self

    def _init(self, comm, nside, lmax, nmaps, pol, dist, weights):
        self.comm = comm
        if dist:
            self.myid, self.nprocs = comm.rank, comm.size
        else:
            self.myid, self.nprocs = 0, 1
        myid, nprocs = self.myid, self.nprocs
        self.nside, self.nmaps, self.lmax, self.pol, self.dist = nside, nmaps, lmax, pol, dist
        self.nspec = nmaps * (nmaps + 1) // 2
        self.npix = 12 * nside ** 2
        self._custom_w = weights is not None
        # rings and pixels, :193-226
        rings = []
        for i in range(1 + myid, 2 * nside + 1, nprocs):
            rings.append(i)
            if i < 2 * nside:
                rings.append(4 * nside - i)
        rings.sort()
        self.rings = np.array(rings, dtype=np.int32)
        self.nring = len(rings)
        self.pix = np.concatenate([np.arange(_ring_start(nside, r), _ring_start(nside, r) + _in_ring_count(nside, r))
                                   for r in rings]) if rings else np.zeros(0, dtype=np.int64)
        self.np = int(self.pix.size)
        # m's, :228-261
        self.ms = np.arange(myid, lmax + 1, nprocs, dtype=np.int32)
        self.nm = len(self.ms)
        self.mind = np.full(lmax + 1, -1, dtype=np.int32)
        lm = []
        ind = 0
        for m in self.ms:
            self.mind[m] = ind
            ls = np.arange(m, lmax + 1)
            if m == 0:
                lm.append(np.stack([ls, np.zeros_like(ls)]))
                ind += lmax + 1
            else:
                blk = np.empty((2, 2 * ls.size), dtype=np.int64)
                blk[0, 0::2] = ls; blk[0, 1::2] = ls
                blk[1, 0::2] = m;  blk[1, 1::2] = -m
                lm.append(blk)
                ind += 2 * ls.size
        self.nalm = ind
        self.lm = np.concatenate(lm, axis=1).astype(np.int32) if lm else np.zeros((2, 0), dtype=np.int32)
        # ring weights + sharp handles, :263-282
        self.alm_info = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=self.ms)
        ncol = 1 if nmaps == 1 else 2
        self.W = load_ring_weights(nside, ncol) if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        self.geom_info_T = sharp.sharp_make_healpix_geom_info(nside, rings=self.rings, weight=self.W[0])
        self.geom_info_P = None
        if nmaps != 1:
            self.geom_info_P = sharp.sharp_make_healpix_geom_info(nside, rings=self.rings, weight=self.W[1])
        assert self.alm_info.n_local == self.nalm and self.geom_info_T.n_local == self.np

    # commander3/src/comm_map_mod.f90:1213-1245
    def lm2i(self, l, m):
        if l > self.lmax or abs(m) > l:
            return -1
        if self.mind[abs(m)] == -1:
            return -1
        if m == 0:
            return int(self.mind[0]) + l
        i = int(self.mind[abs(m)]) + 2 * (l - abs(m))
        return i + 1 if m < 0 else i

    # commander3/src/comm_map_mod.f90:1247-1262
    def i2lm(self, i):
        if i > self.nalm:
            return -1, -1
        return int(self.lm[0, i]), int(self.lm[1, i])

    def lm2i_vec(self, l, m):
        """Vectorised lm2i over arrays (same semantics, -1 where not local)."""
        l = np.asarray(l); m = np.asarray(m); am = np.abs(m)
        ok = (l <= self.lmax) & (am <= l)
        base = np.where(ok, self.mind[np.minimum(am, self.lmax)], -1)
        i = np.where(m == 0, base + l, base + 2 * (l - am) + (m < 0))
        return np.where(ok & (base >= 0), i, -1)

    # commander3/src/comm_map_mod.f90:419-431
    def dealloc(self):
        sharp.sharp_destroy_alm_info(self.alm_info)
        sharp.sharp_destroy_geom_info(self.geom_info_T)
        if self.geom_info_P is not None:
            sharp.sharp_destroy_geom_info(self.geom_info_P)
        if self in _mapinfos:
            _mapinfos.remove(self)


class comm_map:
    """constructor_map / the Y,Yt,YtW,WY family, commander3/src/comm_map_mod.f90:307-579.

    `map` has shape (nmaps, np) and `alm` (nmaps, nalm): the Fortran (n, nmaps) arrays in
    memory order.  With device='cuda' both live in HBM as torch tensors and no host copy
    happens in the transforms; the default (numpy) reproduces the Fortran host-buffer call."""

    def __init__(self, info: comm_mapinfo, device=None):
        self.info = info
        self.device = device
        if device is None:
            self.map = np.zeros((info.nmaps, info.np))
            self.alm = np.zeros((info.nmaps, info.nalm))
        else:
            import torch
            self.map = torch.zeros((info.nmaps, info.np), dtype=torch.float64, device=device)
            self.alm = torch.zeros((info.nmaps, info.nalm), dtype=torch.float64, device=device)

    def _comm(self):
        c = self.info.comm
        return c.handle if (self.info.dist and c.size > 1) else None

    def _exec(self, job):
        """exec_sharp_Y / WY / Yt / YtW, commander3/src/comm_map_mod.f90:437-475, 511-564."""
        info = self.info
        comm = self._comm()
        if info.pol:
            sharp.sharp_execute(job, 0, 1, self.alm[0:1], info.alm_info, self.map[0:1], info.geom_info_T, comm=comm)
            if info.nmaps == 3:
                sharp.sharp_execute(job, 2, 2, self.alm[1:3], info.alm_info, self.map[1:3], info.geom_info_P, comm=comm)
        else:
            # the reference passes all nmaps columns in one spin-0 call (and libsharp2 transforms
            # the first); each column is an independent scalar transform here
            for i in range(info.nmaps):
                sharp.sharp_execute(job, 0, 1, self.alm[i:i + 1], info.alm_info, self.map[i:i + 1],
                                    info.geom_info_T, comm=comm)

    def Y(self):
        self._exec(sharp.SHARP_Y)

    def WY(self):
        self._exec(sharp.SHARP_WY)

    def Yt(self):
        self._exec(sharp.SHARP_Yt)

    def YtW(self):
        self._exec(sharp.SHARP_YtW)

    def _exec_scalar(self, job):
        """exec_sharp_Y_scalar / Yt_scalar / YtW_scalar, :477-489, 532-544, 567-579."""
        info = self.info
        for i in range(info.nmaps):
            sharp.sharp_execute(job, 0, 1, self.alm[i:i + 1], info.alm_info, self.map[i:i + 1],
                                info.geom_info_T, comm=self._comm())

    def Y_scalar(self):
        self._exec_scalar(sharp.SHARP_Y)

    def Yt_scalar(self):
        self._exec_scalar(sharp.SHARP_Yt)

    def YtW_scalar(self):
        self._exec_scalar(sharp.SHARP_YtW)

    def Y_EB(self):
        """exec_sharp_Y_EB, :491-509: every column as a spin-0 field."""
        self._exec_scalar(sharp.SHARP_Y)

    def alm2map_der1(self, i=0):
        """Gradient maps {dT/dtheta, (1/sin theta) dT/dphi} of a_lm column `i`, shape (2, np), on the T geometry
        (SHARP_ALM2MAP_DERIV1).  On this object's device; collective on the info's communicator when distributed."""
        info = self.info
        if self.device is None:
            grad = np.zeros((2, info.np))
        else:
            import torch
            grad = torch.zeros((2, info.np), dtype=torch.float64, device=self.alm.device)
        sharp.alm2map_der1(self.alm[i:i + 1], info.alm_info, grad, info.geom_info_T, comm=self._comm())
        return grad

    # fused variants (additive; one library call for T and QU)
    def _exec_iqu(self, job):
        info = self.info
        assert info.pol and info.nmaps == 3
        sharp.execute_iqu(job, self.alm, self.map, info.geom_info_T, info.geom_info_P, info.alm_info,
                          comm=self._comm())

    def Y_iqu(self):
        self._exec_iqu(sharp.SHARP_Y)

    def Yt_iqu(self):
        self._exec_iqu(sharp.SHARP_Yt)

    def YtW_iqu(self):
        self._exec_iqu(sharp.SHARP_YtW)

    def WY_iqu(self):
        self._exec_iqu(sharp.SHARP_WY)

    # ---- band batches (extended API): the per-band loops of commander3/src/comm_cr_mod.f90:880-918
    @staticmethod
    def _exec_batch(job, maps):
        info = maps[0].info
        assert info.pol and info.nmaps == 3 and not (info.dist and info.comm is not None and info.comm.size > 1)
        assert all(m.info is info for m in maps), "a batch shares one comm_mapinfo"
        sharp.execute_iqu_batch(job, [m.alm for m in maps], [m.map for m in maps], info.geom_info_T,
                                info.geom_info_P, info.alm_info)

    @staticmethod
    def Y_batch(maps):
        """`call map%Y()` for every band of the list, host<->device copies pipelined band against band."""
        comm_map._exec_batch(sharp.SHARP_Y, maps)

    @staticmethod
    def Yt_batch(maps):
        comm_map._exec_batch(sharp.SHARP_Yt, maps)

    @staticmethod
    def YtW_batch(maps):
        comm_map._exec_batch(sharp.SHARP_YtW, maps)

    @staticmethod
    def WY_batch(maps):
        comm_map._exec_batch(sharp.SHARP_WY, maps)

    # commander3/src/comm_map_mod.f90:1109-1142
    def smooth(self, fwhm, fwhm_pol=None):
        if fwhm <= 0.0 and fwhm_pol is None:
            return
        self.YtW()
        sigma = fwhm * math.pi / 180.0 / 60.0 / math.sqrt(8.0 * math.log(2.0))
        sigma_pol = sigma if fwhm_pol is None else fwhm_pol * math.pi / 180.0 / 60.0 / math.sqrt(8.0 * math.log(2.0))
        fact_pol = math.exp(2.0 * sigma_pol ** 2)
        l = self.info.lm[0].astype(np.float64)
        bl_T = np.exp(-0.5 * l * (l + 1) * sigma ** 2)
        bl_P = np.exp(-0.5 * l * (l + 1) * sigma_pol ** 2) * fact_pol
        for j in range(self.info.nmaps):
            bl = bl_T if j == 0 else bl_P
            if self.device is None:
                self.alm[j] *= bl
            else:
                import torch
                self.alm[j] *= torch.as_tensor(bl, device=self.alm.device)
        self.Y()

    # commander3/src/comm_map_mod.f90:1148-1211
    def alm_equal(self, other: "comm_map"):
        """other%alm = self%alm on the (l,m) both hold, zero elsewhere."""
        q = min(self.info.nmaps, other.info.nmaps)
        other.alm[...] = 0.0
        if self.device is None and other.device is None:
            j = self.info.lm2i_vec(other.info.lm[0], other.info.lm[1])
            ok = j >= 0
            other.alm[:q, ok] = self.alm[:q, j[ok]]
        else:
            # the index pair is a function of the two layouts only: built once per (layout, layout, device)
            # (the reference redoes the lm2i loop on every call, comm_cr_mod.f90:858-861 -- every CG iteration)
            import torch
            key = (id(self.info), id(other.info), str(other.alm.device))
            hit = _repack_cache.get(key)
            if hit is None:
                j = self.info.lm2i_vec(other.info.lm[0], other.info.lm[1])
                ok = j >= 0
                hit = (torch.as_tensor(np.nonzero(ok)[0], device=other.alm.device),
                       torch.as_tensor(j[ok], device=self.alm.device), self.info, other.info)
                _repack_cache[key] = hit
            other.alm[:q, hit[0]] = self.alm[:q, hit[1]]

    # ---- the chain-file order of a_lm: global index l^2 + l + m, all (l, m) of the sphere, single precision on disk
    def alm_to_chain_order(self, dtype=np.float32):
        """This rank's contribution to the `alm` dataset writeFITS puts into the chain file
        (commander3/src/comm_map_mod.f90:712-739): array ((lmax+1)^2, nmaps) with alm(l^2+l+m, :) = self%alm(j, :),
        zero for the (l, m) other ranks own (the reference gathers them on the root with mpi_recv; summing the
        ranks' arrays is the same thing), cast to real(sp) as `real(alm, sp)` does."""
        info = self.info
        l, m = info.lm[0].astype(np.int64), info.lm[1].astype(np.int64)
        out = np.zeros(((info.lmax + 1) ** 2, info.nmaps))
        a = self.alm if isinstance(self.alm, np.ndarray) else self.alm.cpu().numpy()
        out[l * l + l + m, :] = a.T
        return out.astype(dtype)

    def alm_from_chain_order(self, alms):
        """readHDF, commander3/src/comm_map_mod.f90:860-889: self%alm(i, :) = alms(l^2 + l + m, :) for the local (l, m);
        `alms` is the full ((lmax+1)^2, nmaps) dataset every rank receives by mpi_bcast."""
        info = self.info
        l, m = info.lm[0].astype(np.int64), info.lm[1].astype(np.int64)
        loc = np.ascontiguousarray(np.asarray(alms, dtype=np.float64)[l * l + l + m, :].T)
        if isinstance(self.alm, np.ndarray):
            self.alm[...] = loc
        else:
            import torch
            self.alm.copy_(torch.as_tensor(loc))

    def add_alm(self, alm, info: comm_mapinfo):
        j = self.info.lm2i_vec(info.lm[0], info.lm[1])
        q = min(self.info.nmaps, info.nmaps)
        ok = j >= 0
        self.alm[:q, j[ok]] += alm[:q, ok]

    def set_alm(self, alm, info: comm_mapinfo):
        j = self.info.lm2i_vec(info.lm[0], info.lm[1])
        q = min(self.info.nmaps, info.nmaps)
        ok = j >= 0
        self.alm[:q, j[ok]] = alm[:q, ok]
