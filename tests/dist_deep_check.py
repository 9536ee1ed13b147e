"""torchrun worker: the distributed transforms value by value against the single-GPU path on every rank's own GPU.
Launched by tests/test_gpu_dist_deep.py (or by hand:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 3 --master-addr 127.0.0.1 --master-port 29513 \
      tests/dist_deep_check.py).

Why a single-GPU run is an exact reference.  When every ring pair belongs to one rank, the distributed work order is the
single-GPU order (get_plan sorts all ranks' pairs by colatitude, a single-GPU geometry is sorted already), so every warp
gets the same rings and takes the same skip / front-phase / cut-off decisions; the ring-FFT folds sum over m by value,
not by owner; and seeded synthesis is bit-identical to the unseeded kernels the distributed path runs.  So distributed
synthesis must reproduce the single-GPU maps bit for bit, on the union of the ranks' rings and m's, for device, pinned
and pageable arrays, fused or NCCL exchange, pipelined or not.  Analysis may differ only by the order of its
accumulations.  The single-GPU path itself is tied to the mpmath reference by test_gpu_deep_parity.py; with
DIST_DEEP_LARGEST=1 one probe run (slam_ref.run_probes) ties the distributed path to it directly.

Layouts (built on every rank from a seed; see layout()):
  mapinfo   comm_mapinfo's round robin                                                   synthesis bit-identical
  lopsided  rank 0 holds no ring, the last rank no m; the unpaired equator ring on the last rank, the other pairs
            spread unevenly over ranks 1.. (padding slots); rank 0 holds m = 0..lmax/2   synthesis bit-identical
  subset    about a third of the pairs and one band of m left out of the union; each rank's ring list in scrambled
            order                                                                         bit-identical to a run on the union
  blocks    contiguous ring blocks of equal pixel count (most pairs split between two ranks: two work slots at one
            colatitude, other warps) and contiguous m blocks                             per ring / m column <= 2e-11

Environment: DIST_DEEP_LARGEST=1 adds nside 2048 / lmax 4000 (mapinfo and lopsided) and the probe run;
DIST_DEEP_SAVE=<path> writes the SHA-256 of every synthesis result of this rank to <path>.rank<r>.json."""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LAYOUTS = ("mapinfo", "lopsided", "subset", "blocks")
BIT_EXACT = ("mapinfo", "lopsided", "subset")
EPS_ANAL = 1e-13      # analysis, per (component, m) column, relative to the column's largest reference value
EPS_BLOCKS = 2e-11    # blocks layout, per ring and per m column: EPS_SPIN0 of test_gpu_deep_parity.py


# ---------------------------------------------------------------------------------------------------------------------
# Bookkeeping (no GPU; tested by tests/test_dist_layouts_cpu.py)
# ---------------------------------------------------------------------------------------------------------------------
def ring_nph(nside, rings):
    r = np.asarray(rings, dtype=np.int64)
    north = np.where(r > 2 * nside, 4 * nside - r, r)
    return np.where(north < nside, 4 * north, 4 * nside)


def m_count(lmax, ms):
    m = np.asarray(ms, dtype=np.int64)
    return (lmax + 1 - m) * np.where(m == 0, 1, 2)


def pipeline_nside(world):
    """Smallest power-of-two nside that takes the chunked host pipeline at this world size (12 nside^2 >= 2^20 ranks)."""
    n = 1
    while 12 * n * n < (1 << 20) * world:
        n *= 2
    return n


def sizes(world, largest):
    pn = pipeline_nside(world)
    out = [(64, 150), (256, 1100), (pn, 3 * pn // 2)]
    return out + [(2048, 4000)] if largest else out


def pipeline_chunks(nvalid, env=None):
    """Work-slot chunks of the host pipeline (dist.cu get_plan): CMDR_SHT_DIST_CHUNKS, default 8, at most 24."""
    v = os.environ.get("CMDR_SHT_DIST_CHUNKS") if env is None else env
    k = min(24, int(v)) if v and int(v) > 0 else 8
    per = max(128, ((nvalid + k - 1) // k + 127) // 128 * 128)
    return -(-nvalid // per)


def _pair_rings(nside, i):
    return [i, 4 * nside - i] if i < 2 * nside else [i]


def layout(name, nside, lmax, world, seed=0):
    """[(rings, ms)] per rank, int32 arrays, in the order the rank hands them to the library."""
    W = world
    rng = np.random.default_rng([seed, nside, lmax, W, LAYOUTS.index(name)])
    rings = [[] for _ in range(W)]
    ms = [[] for _ in range(W)]
    if name == "mapinfo":
        from oracle import sht_def as D
        rings = [D.mapinfo_rings(nside, r, W) for r in range(W)]
        ms = [D.mapinfo_ms(lmax, r, W) for r in range(W)]
    elif name == "lopsided":
        rings[W - 1].append(2 * nside)                       # the unpaired equator ring
        share = np.arange(1, W, dtype=np.float64)            # rank k of 1..W-1 gets a share ~ k of the other pairs
        owner = 1 + rng.choice(W - 1, size=2 * nside - 1, p=share / share.sum())
        for i in range(1, 2 * nside):
            rings[owner[i - 1]] += _pair_rings(nside, i)
        rings = [sorted(r) for r in rings]
        ms[0] = list(range(lmax // 2 + 1))
        for j, m in enumerate(range(lmax // 2 + 1, lmax + 1)):
            ms[j % (W - 1)].append(m)
        ms = [sorted(m) for m in ms]
    elif name == "subset":
        drop = int(rng.integers(3))                          # every third pair, from a random first one
        owner = rng.integers(W, size=2 * nside)
        for i in range(1, 2 * nside + 1):
            if i % 3 != drop:
                rings[owner[i - 1]] += _pair_rings(nside, i)
        rings = [list(rng.permutation(r)) for r in rings]
        b0 = lmax // 3
        band = range(b0, b0 + max(1, lmax // 8))
        mo = rng.integers(W, size=lmax + 1)
        for m in range(lmax + 1):
            if m not in band:
                ms[mo[m]].append(m)
    elif name == "blocks":
        allr = np.arange(1, 4 * nside)
        nph = ring_nph(nside, allr)
        mid = np.cumsum(nph) - nph / 2.0
        owner = np.minimum(W - 1, (mid * W / nph.sum()).astype(np.int64))
        rings = [list(allr[owner == r]) for r in range(W)]
        allm = np.arange(lmax + 1)
        cnt = m_count(lmax, allm)
        mid = np.cumsum(cnt) - cnt / 2.0
        owner = np.minimum(W - 1, (mid * W / cnt.sum()).astype(np.int64))
        ms = [list(allm[owner == r]) for r in range(W)]
    else:
        raise ValueError(name)
    return [(np.asarray(r, dtype=np.int32), np.asarray(m, dtype=np.int32)) for r, m in zip(rings, ms)]


def union(lay):
    """(rings, ms) of the single-GPU reference: the union of the ranks' lists, sorted."""
    rings = np.sort(np.concatenate([r for r, _ in lay])).astype(np.int32)
    ms = np.sort(np.concatenate([m for _, m in lay])).astype(np.int32)
    return rings, ms


def _ranges(starts, counts):
    if len(counts) == 0:
        return np.zeros(0, dtype=np.int64)
    return np.concatenate([np.arange(s, s + c, dtype=np.int64) for s, c in zip(starts, counts)])


def pix_index(nside, ref_rings, rings):
    """Position in the reference map (ref_rings in storage order) of every local pixel (rings in list order)."""
    nph = ring_nph(nside, ref_rings)
    ofs = dict(zip(ref_rings.tolist(), (np.cumsum(nph) - nph).tolist()))
    return _ranges([ofs[int(r)] for r in rings], ring_nph(nside, rings))


def alm_index(lmax, ref_ms, ms):
    """Position in the reference real-packed m-major a_lm (over ref_ms) of every local coefficient (ms in list order)."""
    cnt = m_count(lmax, ref_ms)
    ofs = dict(zip(np.asarray(ref_ms).tolist(), (np.cumsum(cnt) - cnt).tolist()))
    return _ranges([ofs[int(m)] for m in ms], m_count(lmax, ms))


def segments(counts):
    """Segment id (0..len(counts)-1) of every element of a concatenation of blocks of the given sizes."""
    return np.repeat(np.arange(len(counts), dtype=np.int64), np.asarray(counts, dtype=np.int64))


# ---------------------------------------------------------------------------------------------------------------------
# The GPU run
# ---------------------------------------------------------------------------------------------------------------------
SYNTH_JOBS = ("Y", "WY", "Y+add")
ANAL_JOBS = ("Yt", "YtW", "Yt+add")


class Case:
    """One (layout, size) on this rank: handles, inputs, single-GPU references, the local slices."""

    def __init__(self, sharp, torch, dev, name, nside, lmax, world, rank):
        self.sharp, self.torch, self.dev = sharp, torch, dev
        self.name, self.nside, self.lmax = name, nside, lmax
        lay = layout(name, nside, lmax, world)
        self.lay = lay
        self.rings, self.ms = lay[rank]
        self.ref_rings, self.ref_ms = union(lay)
        self.nvalid = sum(len({min(int(r), 4 * nside - int(r)) for r in rr}) for rr, _ in lay)
        npix, nalm = int(ring_nph(nside, self.ref_rings).sum()), int(m_count(lmax, self.ref_ms).sum())
        g = torch.Generator(device=dev)
        g.manual_seed(1000003 * nside + lmax + 7 * LAYOUTS.index(name))    # the same numbers on every rank

        def rnd(*shape):
            return torch.randn(shape, generator=g, dtype=torch.float64, device=dev)
        self.alm_g, self.map_g = rnd(3, nalm), rnd(3, npix)
        self.base_map, self.base_alm = rnd(3, npix), rnd(3, nalm)
        self.w = (0.5 + torch.rand((2, 2 * nside), generator=g, dtype=torch.float64, device=dev)).cpu().numpy()
        mk_g, mk_a = sharp.sharp_make_healpix_geom_info, sharp.sharp_make_mmajor_real_packed_alm_info
        self.ref_g = [mk_g(nside, rings=self.ref_rings)] + [mk_g(nside, rings=self.ref_rings, weight=self.w[c])
                                                            for c in (0, 1)]
        self.ref_a = mk_a(lmax, ms=self.ref_ms)
        self.loc_g = [mk_g(nside, rings=self.rings)] + [mk_g(nside, rings=self.rings, weight=self.w[c]) for c in (0, 1)]
        self.loc_a = mk_a(lmax, ms=self.ms)
        self.pidx = torch.as_tensor(pix_index(nside, self.ref_rings, self.rings), device=dev)
        self.aidx = torch.as_tensor(alm_index(lmax, self.ref_ms, self.ms), device=dev)
        self.pseg = torch.as_tensor(segments(ring_nph(nside, self.rings)), device=dev)
        self.aseg = torch.as_tensor(segments(m_count(lmax, self.ms)), device=dev)
        self.refs = {}

    def close(self):
        for gi in self.ref_g + self.loc_g:
            self.sharp.sharp_destroy_geom_info(gi)
        self.sharp.sharp_destroy_alm_info(self.ref_a)
        self.sharp.sharp_destroy_alm_info(self.loc_a)

    @staticmethod
    def comps(entry):
        return [0] if entry == "s0" else ([0, 1, 2] if entry == "iqu" else [1, 2])

    def run(self, entry, job, alm, map_, local, add=False, comm=None):
        """One transform through sharp_execute (entry s<spin>) or execute_iqu (entry iqu)."""
        S = self.sharp
        jt = {"Y": S.SHARP_Y, "WY": S.SHARP_WY, "Yt": S.SHARP_Yt, "YtW": S.SHARP_YtW}[job]
        weighted = job in ("WY", "YtW")
        gs, a = (self.loc_g, self.loc_a) if local else (self.ref_g, self.ref_a)
        if entry == "iqu":
            gT, gP = (gs[1], gs[2]) if weighted else (gs[0], gs[0])
            S.execute_iqu(jt, alm, map_, gT, gP, a, add=add, comm=comm)
        else:
            spin = int(entry[1:])
            g = gs[(1 if spin == 0 else 2) if weighted else 0]
            S.sharp_execute(jt, spin, len(self.comps(entry)), alm, a, map_, g, add=add, comm=comm)

    def reference(self, entry, job):
        """Single-GPU result on the union handles, device arrays (cached)."""
        key = (entry, job)
        if key not in self.refs:
            torch = self.torch
            cs = self.comps(entry)
            if job in ("Y", "WY"):
                out = torch.full((len(cs), self.map_g.shape[1]), float("nan"), dtype=torch.float64, device=self.dev)
                self.run(entry, job, self.alm_g[cs].contiguous(), out, local=False)
            else:
                out = torch.full((len(cs), self.alm_g.shape[1]), float("nan"), dtype=torch.float64, device=self.dev)
                self.run(entry, job, out, self.map_g[cs].contiguous(), local=False)
            torch.cuda.synchronize()
            self.refs[key] = out
        return self.refs[key]


def _host(torch, t, kind):
    """A (nc, n) float64 copy of device tensor t as device tensor, pinned numpy or pageable numpy array."""
    if kind == "device":
        return t.clone()
    a = t.cpu().numpy()
    if kind == "pinned" and a.shape[1] > 0:
        p = torch.empty(a.shape, dtype=torch.float64).pin_memory().numpy()
        p[:] = a
        return p
    return np.array(a, order="C")


def _col_check(torch, out, exp, seg, nseg, eps):
    """max over (component, segment) of max|out - exp| / max|exp|; inf where a segment whose reference is all zero is
    not exactly zero, or any value is not finite."""
    if out.numel() == 0:
        return 0.0, True
    if not bool(torch.isfinite(out).all()):
        return float("inf"), False
    d, r = (out - exp).abs(), exp.abs()
    idx = seg.unsqueeze(0).expand_as(d)
    z = torch.zeros((out.shape[0], nseg), dtype=torch.float64, device=out.device)
    dm = z.scatter_reduce(1, idx, d, "amax", include_self=True)
    rm = z.clone().scatter_reduce(1, idx, r, "amax", include_self=True)
    rel = torch.where(rm > 0, dm / torch.where(rm > 0, rm, 1.0), torch.where(dm > 0, float("inf"), 0.0))
    worst = float(rel.max())
    return worst, worst <= eps


def main():
    from datetime import timedelta

    import torch
    import torch.distributed as dist
    from commander_b200 import sharp
    from commander_b200 import dist as cdist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    comm = cdist.init_from_torch(dev)
    side = dist.new_group(backend="gloo", timeout=timedelta(minutes=60))
    largest = os.environ.get("DIST_DEEP_LARGEST", "0") == "1"
    save = os.environ.get("DIST_DEEP_SAVE")
    digests, failures = {}, []
    nlines = 0

    def agree(worst, exact):
        t = torch.tensor([worst, 0.0 if exact else 1.0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), int(t[1]) == 0

    def fail(msg):
        failures.append(f"rank {rank}: {msg}")

    for nside, lmax in sizes(world, largest):
        pipe_size = 12 * nside * nside >= (1 << 20) * world
        huge = nside >= 2048
        for name in LAYOUTS:
            if huge and name not in ("mapinfo", "lopsided"):
                continue
            C = Case(sharp, torch, dev, name, nside, lmax, world, rank)
            K = pipeline_chunks(C.nvalid)
            entries = ["iqu"] if huge else ["s0", "s2", "iqu"] + (["s1", "s3", "s17", "s32"] if nside == 64 else [])
            kinds = ("device", "pageable") if huge else ("device", "pinned", "pageable")
            for exch in (1, 0):
                comm.set_exchange(exch)
                for entry in entries:
                    cs = C.comps(entry)
                    arbitrary = entry not in ("s0", "s2", "iqu")
                    jobs = ("Y", "YtW") if huge else (("Y", "Yt") if arbitrary else SYNTH_JOBS + ANAL_JOBS)
                    for job in jobs:
                        add = job.endswith("+add")
                        base_job = job.replace("+add", "")
                        synth = base_job in ("Y", "WY")
                        ref = C.reference(entry, base_job)
                        if synth:
                            exp = ref[:, C.pidx]
                            base = C.base_map[cs][:, C.pidx].contiguous()
                            src = C.alm_g[cs][:, C.aidx].contiguous()
                        else:
                            exp = ref[:, C.aidx]
                            base = C.base_alm[cs][:, C.aidx].contiguous()
                            src = C.map_g[cs][:, C.pidx].contiguous()
                        if add:
                            exp = base + exp
                        dev_launches = None
                        for kind in kinds:
                            inp = _host(torch, src, kind)
                            out = _host(torch, base if add else torch.full_like(base, float("nan")), kind)
                            torch.cuda.synchronize()
                            n0 = sharp.launch_count()
                            if synth:
                                C.run(entry, base_job, inp, out, local=True, add=add, comm=comm.handle)
                            else:
                                C.run(entry, base_job, out, inp, local=True, add=add, comm=comm.handle)
                            torch.cuda.synchronize()
                            launches = sharp.launch_count() - n0
                            got = out if kind == "device" else torch.from_numpy(out).to(dev)
                            path = f"{kind}/{'fused' if exch else 'nccl'}/{entry}"
                            tag = f"{name} nside {nside} lmax {lmax} {path} {job}"
                            # the chunked host pipeline: K + 1 exchange barriers instead of 2 (and K Legendre / FFT
                            # launches instead of 1), so at least K - 1 launches more than on device arrays
                            if kind == "device":
                                dev_launches = launches
                            elif pipe_size:
                                extra = launches - dev_launches
                                want = (name == "mapinfo" and exch == 1 and entry != "iqu" and not add)
                                if want and not extra >= K - 1:
                                    fail(f"{tag}: the host pipeline did not run ({extra} launches more than on device "
                                         f"arrays, expected >= {K - 1})")
                                if not want and not extra < K - 1:
                                    fail(f"{tag}: {extra} launches more than on device arrays where every rank must "
                                         "fall back to the staged path")
                                if want and rank == 0:
                                    print(f"PIPELINE {tag}: +{extra} launches over device arrays (K = {K})")
                            if synth:
                                if save:
                                    digests[f"{name}/{nside}/{path}/{job}"] = hashlib.sha256(
                                        got.cpu().numpy().tobytes()).hexdigest()
                                if name in BIT_EXACT:
                                    exact = bool(torch.equal(got, exp))
                                    worst = float((got - exp).abs().max()) if got.numel() else 0.0
                                    if not exact:
                                        fail(f"{tag}: not bit-identical to the single-GPU maps (max|delta| {worst:.3e})")
                                else:
                                    worst, ok = _col_check(torch, got, exp, C.pseg, len(C.rings), EPS_BLOCKS)
                                    exact = bool(torch.equal(got, exp))
                                    if not ok:
                                        fail(f"{tag}: per-ring deviation {worst:.3e} > {EPS_BLOCKS:.0e}")
                            else:
                                eps = EPS_ANAL if name in BIT_EXACT else EPS_BLOCKS
                                worst, ok = _col_check(torch, got, exp, C.aseg, len(C.ms), eps)
                                exact = bool(torch.equal(got, exp))
                                if not ok:
                                    fail(f"{tag}: per-(component, m) column deviation {worst:.3e} > {eps:.0e}")
                            gw, gexact = agree(worst, exact)
                            nlines += 1
                            if rank == 0:
                                crit = "bit-identical" if (synth and name in BIT_EXACT) else "rel per column"
                                print(f"DEEP {tag}: worst {gw:.3e} ({crit}), bit-identical on all ranks: {gexact}")
            comm.set_exchange(-1)
            C.close()
            torch.cuda.empty_cache()
    if largest:
        _probe_run(sharp, torch, dist, dev, comm, side, rank, world, fail)
    if save:
        with open(f"{save}.rank{rank}.json", "w") as f:
            json.dump(digests, f)
    nf = torch.tensor([len(failures)], dtype=torch.int64, device=dev)
    dist.all_reduce(nf)
    for msg in failures[:20]:
        print("FAIL " + msg, flush=True)
    dist.barrier()
    if rank == 0 and int(nf) == 0:
        print(f"DIST_DEEP_OK world={world} lines={nlines}")
    cdist.destroy(comm)
    dist.destroy_process_group()
    if int(nf):
        sys.exit(1)


def _probe_run(sharp, torch, dist, dev, comm, side, rank, world, fail, nside=1024, lmax=2048):
    """slam_ref.run_probes through the distributed path (blocks layout, nside 1024 / lmax 2048, spins 0 and 2): rank 0
    drives, every request -- (ring, ms, x) or (m, rings, a) -- is broadcast over a gloo group, every rank runs the
    collective transform on its own handles and sends its piece back to rank 0."""
    import slam_ref as R
    from test_gpu_deep_parity import EPS, EPS_POLAR, EPS_SPIN0
    lay = layout("blocks", nside, lmax, world)
    rings, ms = lay[rank]
    nph = ring_nph(nside, rings)
    rofs = dict(zip(rings.tolist(), (np.cumsum(nph) - nph).tolist()))
    cnt = m_count(lmax, ms)
    mofs = dict(zip(ms.tolist(), zip((np.cumsum(cnt) - cnt).tolist(), cnt.tolist())))
    w = np.random.default_rng(nside + lmax).uniform(0.5, 1.5, 2 * nside)
    gi = sharp.sharp_make_healpix_geom_info(nside, rings=rings)
    gw = sharp.sharp_make_healpix_geom_info(nside, rings=rings, weight=w)
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax, ms=ms)
    npix, nalm = int(nph.sum()), int(cnt.sum())
    for spin in (0, 2):
        nc = 1 if spin == 0 else 2

        def serve(req):
            if req[0] == "A":
                _, r, want, x, weighted = req
                mp = torch.zeros((nc, npix), dtype=torch.float64, device=dev)
                if r in rofs:
                    mp[:, rofs[r]:rofs[r] + x.shape[1]] = torch.from_numpy(x).to(dev)
                alm = torch.full((nc, nalm), float("nan"), dtype=torch.float64, device=dev)
                sharp.sharp_execute(sharp.SHARP_YtW if weighted else sharp.SHARP_Yt, spin, nc, alm, ai, mp,
                                    gw if weighted else gi, comm=comm.handle)
                a = alm.cpu().numpy()
                return {m: a[:, mofs[m][0]:mofs[m][0] + mofs[m][1]] for m in want if m in mofs}
            _, m, want, a = req
            alm = torch.zeros((nc, nalm), dtype=torch.float64, device=dev)
            if m in mofs:
                alm[:, mofs[m][0]:mofs[m][0] + mofs[m][1]] = torch.from_numpy(a).to(dev)
            mp = torch.full((nc, npix), float("nan"), dtype=torch.float64, device=dev)
            sharp.sharp_execute(sharp.SHARP_Y, spin, nc, alm, ai, mp, gi, comm=comm.handle)
            out = mp.cpu().numpy()
            return {r: out[:, rofs[r]:rofs[r] + int(ring_nph(nside, [r])[0])] for r in want if r in rofs}

        def request(req):
            box = [req]
            dist.broadcast_object_list(box, src=0, group=side)
            if box[0] is None:
                return None
            mine = serve(box[0])
            pieces = [None] * world if rank == 0 else None
            dist.gather_object(mine, pieces, dst=0, group=side)
            if rank != 0:
                return True
            merged = {}
            for p in pieces:
                merged.update(p)
            return merged

        if rank != 0:
            while request(None) is not None:
                pass
            continue
        pairs = R.probe_set(nside, lmax, spin, full=True)
        R.prefetch(nside, lmax, spin, pairs)

        def analyse(weighted):
            def f(r, want, x):
                got = request(("A", r, list(want), np.ascontiguousarray(x), weighted))
                return np.concatenate([got[m] for m in want], axis=1)
            return f

        def synthesise(m, want, a):
            return request(("S", m, list(want), np.ascontiguousarray(a)))

        wr = (1, nside, 2 * nside, 4 * nside - 1)
        try:
            recs = R.run_probes(nside, lmax, spin, pairs, analyse(False), synthesise, seed=spin + 7,
                                weighted_rings=wr, analyse_w=analyse(True), weight=w)
        finally:
            dist.broadcast_object_list([None], src=0, group=side)
        print(R.summarize(recs, f"PROBES distributed blocks world {world} nside {nside} lmax {lmax} spin {spin}"))
        bad = []
        for q in recs:
            polar = R.ring_trig(nside, q["ring"])[1] < R.POLAR_STH
            eps = EPS_POLAR if polar else (EPS_SPIN0 if spin == 0 else EPS)
            if not q["zero_ok"] or not (q["excess"] <= eps):
                bad.append(q)
        if bad or not any(q["kind"].startswith("YtW") for q in recs):
            fail(f"probes spin {spin}: {len(bad)} of {len(recs)} readings out of bounds, e.g. " + "; ".join(
                f"{q['kind']} ring {q['ring']} m {q['m']}: {q['excess']:.2e} zero_ok={q['zero_ok']}" for q in bad[:8]))
    for h in (gi, gw):
        sharp.sharp_destroy_geom_info(h)
    sharp.sharp_destroy_alm_info(ai)


if __name__ == "__main__":
    main()
