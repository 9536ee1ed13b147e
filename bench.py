#!/usr/bin/env python
"""bench.py -- SHT pairs/s (alm2map + map2alm, IQU) at nside 2048 / lmax 4000 (BASELINE.json).

One "step" = one pair = comm_map%Y() followed by comm_map%YtW() on an IQU object
(commander3/src/comm_map_mod.f90:437-455, 546-564): four sharp_execute calls.

  value : whole-job pairs/s with alm and map resident in HBM (CUDA events, max over ranks)
  e2e   : the same pair through the reference-facing call with HOST buffers -- pageable arrays as the
          Fortran caller passes them (headline) and caller-pinned arrays (note) -- so the H2D copy of
          the inputs and the D2H copy of the outputs are inside the timed region
  parity / checksums : the transform of this very run against the CPU oracle on an m-subset, and
          N-independent global checksums of its outputs (the SCALE lines must agree)
  roofline     : dominant kernel (spin-2 Legendre) against the FP64-FMA peak measured live
  cpu_baseline : the CPU restatement (oracle/sht_cpu.c, "port": libsharp2 itself is not
                 available) on the box's host cores, on a bounded m-subset of the same workload

N > 1 (torchrun): ONE transform pair distributed over N GPUs exactly as libsharp's MPI mode
shards it (m's and ring pairs round-robin, commander3/src/comm_map_mod.f90:197-261) with an
the m <-> ring exchange of the phases fused into the Legendre kernels over NVLink (NCCL all-to-all as fallback)
-> strong scaling.

--impl reference times the CPU path (all host threads) on the same config/metric.

--dump-outputs DIR (N = 1) writes the map and a_lm of the last timed step as DIR/map.npy and DIR/alm.npy (float64, a
fixed seeded sample of columns at large sizes), so that two builds can be compared output for output.  The inputs are the
same in every run; the outputs agree to rounding, not bit for bit, because the analysis kernels accumulate with atomics
(two runs of the default workload: 1.1e-14 relative L2, B200 at 1000 W).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SHT pairs/sec (alm2map+map2alm, IQU) at nside 2048 lmax 4000"
UNIT = "pairs/s"


def ntriples(nside, lmax):
    return (lmax + 1) * (lmax + 2) / 2 * 2 * nside


def executed_fraction(nside, lmax, spin, ms):
    """Fraction of the nominal (l, m, ring pair) triples the kernels actually visit: rings beyond the
    per-ring m cut-off (same formula as commander_b200/csrc/legendre_core.cuh mlim_for_ring) are
    skipped.  The underflow region (ring not yet accumulating) still runs the recurrence and is
    counted as visited."""
    import numpy as np
    i = np.arange(1, 2 * nside + 1, dtype=np.float64)
    z = np.where(i < nside, 1.0 - i * i / (3.0 * nside * nside), (2.0 * nside - i) * 2.0 / (3.0 * nside))
    sth, cth = np.sqrt(np.maximum(1.0 - z * z, 0.0)), z
    ofs = max(100.0, 0.01 * lmax)
    b = -2.0 * spin * np.abs(cth)
    t1 = lmax * sth + ofs
    c = spin * spin - t1 * t1
    discr = b * b - 4 * c
    mlim = np.where(discr <= 0, lmax, np.minimum((-b + np.sqrt(np.maximum(discr, 0))) / 2.0, lmax) + 0.5).astype(np.int64)
    wpair = np.ones_like(i); wpair[-1] = 0.5          # the equator ring has no mirror
    ms = np.asarray(ms, dtype=np.int64)
    l0 = np.maximum(ms, spin)
    nl = np.maximum(lmax + 1 - l0, 0).astype(np.float64)
    visited = sum(float(nl[k]) * float(wpair[mlim >= ms[k]].sum()) for k in range(len(ms)))
    nominal = float(sum(lmax + 1 - m for m in ms)) * float(wpair.sum())
    return visited / nominal


def workload(args):
    return {"workload": f"comm_map Y+YtW pair, IQU, nside={args.nside} lmax={args.lmax}, synthetic Gaussian alm",
            "nside": args.nside, "lmax": args.lmax, "nmaps": 3,
            "l2_policy": "inputs larger than L2 (alm 0.38 GB, map 1.2 GB, phases 1.6 GB per direction)",
            "parallelism": "m-distributed alm / ring-distributed map; m<->ring exchange fused into the Legendre kernels over NVLink "
                           "(NCCL all-to-all as fallback)",
            "ring_fft": "one shared-memory kernel per ring class, no cuFFT at this size: whole-ring chirp-z (work length <= 8192), "
                        "radix-4 split chirp-z (4 x work length 4096) for the cap rings longer than 4096, whole-ring FFT for the belt"
                        + "".join(f"; {k}={os.environ[k]}" for k in ("CMDR_SHT_FUSED_BLUE", "CMDR_SHT_RING_SPLIT", "CMDR_SHT_BELT_FUSED",
                                                                    "CMDR_SHT_FFT_BLOCKED", "CMDR_SHT_SPLIT_MIN", "CMDR_SHT_PH_LAYOUT",
                                                                    "CMDR_SHT_BELT_HALF")
                                  if k in os.environ),
            "legendre": "FP64 recurrence kernels, one warp per CTA: spin 0 two l per recurrence step (3 DFMA per (l,m,ring pair)), spin 2 "
                        "two coupled recurrences (12 DFMA) with a scalar front phase while all rings of a warp are below the threshold"
                        + "".join(f"; {k}={os.environ[k]}" for k in ("CMDR_SHT_FRONT", "CMDR_SHT_R_S0", "CMDR_SHT_R_S2", "CMDR_SHT_R_A0",
                                                                    "CMDR_SHT_R_A2", "CMDR_SHT_MINB_S0", "CMDR_SHT_MINB_S2",
                                                                    "CMDR_SHT_MINB_A0", "CMDR_SHT_MINB_A2") if k in os.environ)}


# ------------------------------------------------------------------ CPU baseline / reference arm
def cpu_pair_sample(nside, lmax, stride, nthreads=0):
    """Times Y + YtW (spin 0 and spin 2) of the CPU restatement on the m-subset
    m = 0, stride, 2*stride, ... with all rings.  The Legendre stage scales with the m-subset,
    the per-ring FFT stage does not, so the two are timed separately inside the C code and the
    full-workload time is estimated as  t_legendre / work_fraction + t_fft.
    stride == 1 is the complete workload (no extrapolation).
    Returns dict(seconds_full_est, frac, threads, simd, t_leg, t_fft)."""
    import numpy as np
    from oracle import sht_cpu as S
    S.build()
    if nthreads == 0:   # torchrun exports OMP_NUM_THREADS=1; the CPU arm uses every core it may run on
        nthreads = len(os.sched_getaffinity(0))
    # one-off FFT plan tables (not part of a transform; libsharp2 also plans once per geometry)
    tiny = np.array([0], dtype=np.int32)
    S.execute(S.Y, 0, nside, lmax, alm=np.zeros((1, lmax + 1)), ms=tiny, nthreads=nthreads, mlim_skip=True)
    ms = np.arange(0, lmax + 1, stride, dtype=np.int32)
    frac = float(sum(lmax + 1 - m for m in ms)) / ((lmax + 1) * (lmax + 2) / 2)
    nalm = S.alm_count(lmax, ms)
    rng = np.random.default_rng(9)
    almT, almP = rng.standard_normal((1, nalm)), rng.standard_normal((2, nalm))
    t_leg = t_fft = 0.0

    def acc():
        nonlocal t_leg, t_fft
        a, b = S.last_times()
        t_leg += a
        t_fft += b
    t0 = time.perf_counter()
    mT = S.execute(S.Y, 0, nside, lmax, alm=almT, ms=ms, nthreads=nthreads, mlim_skip=True); acc()
    mP = S.execute(S.Y, 2, nside, lmax, alm=almP, ms=ms, nthreads=nthreads, mlim_skip=True); acc()
    S.execute(S.YtW, 0, nside, lmax, map=mT, ms=ms, nthreads=nthreads, mlim_skip=True); acc()
    S.execute(S.YtW, 2, nside, lmax, map=mP, ms=ms, nthreads=nthreads, mlim_skip=True); acc()
    wall = time.perf_counter() - t0
    other = max(wall - t_leg - t_fft, 0.0)   # geometry setup, buffers
    full = t_leg / frac + t_fft + other
    return {"seconds_full_est": full, "frac": frac, "wall": wall, "t_leg": t_leg, "t_fft": t_fft,
            "threads": nthreads, "simd": S.lib().variant}


def cpu_pick_stride(nside, lmax, budget_s=20.0):
    """Chooses the m stride of the CPU sample so that it costs about `budget_s` seconds on this
    box (a 1-core box and a 64-core box differ by two orders of magnitude): a stride-64 probe
    measures the rate first."""
    probe = cpu_pair_sample(nside, lmax, 64)
    est_full = probe["seconds_full_est"]
    stride = 1
    while est_full / stride > budget_s and stride < 64:
        stride *= 2
    return stride


def cpu_sample_text(r, stride):
    if stride == 1:
        return f"the complete workload, one pair, {r['wall']:.1f} s wall (Legendre {r['t_leg']:.1f} s, FFT {r['t_fft']:.1f} s)"
    return (f"m = 0,{stride},{2 * stride},... = {100 * r['frac']:.1f}% of the (l,m) work with all rings, {r['wall']:.1f} s wall; "
            f"full pair estimated as t_legendre/fraction + t_fft = {r['t_leg']:.2f}/{r['frac']:.4f} + {r['t_fft']:.2f} s")


def run_reference(args):
    """The reference arm: the CPU implementation of the path on all host threads.  libsharp2 is not
    available (not under /root/reference, no network), so this is the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    stride = args.cpu_stride if args.cpu_stride > 0 else cpu_pick_stride(args.nside, args.lmax, 12.0)
    ests = []
    r = None
    for i in range(args.warmup + args.steps):
        r = cpu_pair_sample(args.nside, args.lmax, stride)
        if i >= args.warmup:
            ests.append(r["seconds_full_est"])
    mean_t = sum(ests) / len(ests)
    value = 1.0 / mean_t
    cg = None
    if not args.no_cg:
        sec, nth = cpu_cg_sample(CG_NSIDE, CG_LMAX, 2)
        cg = {"metric": "CR CG iters/sec", "value": 1.0 / sec, "unit": "iter/s", "ms_per_iter": 1e3 * sec, "cores": nth,
              "sample": f"2 iterations of solve_cr_eqn_by_CG at nside={CG_NSIDE} lmax={CG_LMAX} IQU (1 band, CMB only, diagonal N^-1, "
                        "10' beam): oracle/sht_cpu.c as SHT engine, numpy vector passes",
              "kind": "port"}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * mean_t, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": r["threads"], "kind": "port",
                             "sample": "each step: " + cpu_sample_text(r, stride), "simd": r["simd"],
                             "note": "oracle/sht_cpu.c (OpenMP restatement of the libsharp2 algorithm); libsharp2 "
                                     "itself is not in /root/reference and cannot be built offline"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "cg": cg}
    print(json.dumps(line))


# ------------------------------------------------------------------ clocks sampling
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thr.join(timeout=2)
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 9 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 9 and r[2].isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}



# ------------------------------------------------------------------ correctness evidence inside the bench records
PARITY_MS = [0, 1, 2, 777, 2048, 3100, 3999, 4000]


def _hash_gauss_np(key, c):
    """Deterministic pseudo-Gaussian from a global index (Box-Muller on sine hashes): the same value whatever the
    number of ranks."""
    import numpy as np
    u1 = np.clip(np.abs(np.modf(np.sin(key * 12.9898 + 78.233 * (c + 1)) * 43758.5453)[0]), 1e-12, 1.0)
    u2 = np.abs(np.modf(np.sin(key * 39.3468 + 11.135 * (c + 1)) * 24634.6345)[0])
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2 * np.pi * u2)


def run_parity(args, info, comm, dev, world, m, alm_in):
    """(i) N-independent global checksums of the map after Y and of the a_lm after YtW of the bench input;
    (ii) the transform through the (distributed) entry point against the CPU oracle on an m-subset x all rings,
    Y and Yt, spin 0 and spin 2, in both exchange modes when N > 1.  Tolerance 1e-10 relative L2 (north_star)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from commander_b200 import comm_map
    from oracle import sht_cpu as S
    nside, lmax = args.nside, args.lmax

    def allsum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return [float(v) for v in t.tolist()]

    pix = torch.as_tensor(info.pix.astype(np.int64), device=dev).double()
    l_t = torch.as_tensor(info.lm[0].astype(np.int64), device=dev)
    m_t = torch.as_tensor(info.lm[1].astype(np.int64), device=dev)
    lmkey = (l_t * (l_t + 1) + m_t).double()
    out = {}
    # ---- (i) checksums of the bench transform itself
    m.alm.copy_(alm_in)
    m.Y()
    cs = {}
    for c, nm in enumerate("TQU"):
        x = m.map[c]
        r = torch.frac(torch.sin(pix * 0.618 + 1.7 * (c + 1)) * 9871.137)
        s1, s2, sa, pr, rr = allsum([float(x.sum()), float((x * x).sum()), float(x.abs().sum()), float((x * r).sum()),
                                     float((r * r).sum())])
        cs["map_" + nm] = {"sum": s1, "sum_sq": s2, "sum_abs": sa, "proj": pr, "proj_scale": (s2 * rr) ** 0.5}
    m.YtW()
    for c, nm in enumerate("TEB"):
        x = m.alm[c]
        r = torch.frac(torch.sin(lmkey * 0.377 + 2.9 * (c + 1)) * 7919.733)
        s1, s2, sa, pr, rr = allsum([float(x.sum()), float((x * x).sum()), float(x.abs().sum()), float((x * r).sum()),
                                     float((r * r).sum())])
        cs["alm_" + nm] = {"sum": s1, "sum_sq": s2, "sum_abs": sa, "proj": pr, "proj_scale": (s2 * rr) ** 0.5}
    out["checksums"] = cs
    out["checksums_note"] = ("global (all-reduced) sums of the map after Y and of the a_lm after YtW(Y(a)) of the bench input; inputs are "
                             "functions of (l, m) / the global pixel index only, so every N must print the same numbers to <= 1e-12 of "
                             "sum_abs (sum, proj: relative to sum_abs / proj_scale, they are sums with cancellation)")
    # ---- (ii) oracle parity on an m-subset x all rings, through the distributed entry point
    ms_sub = np.array([mm for mm in PARITY_MS if mm <= lmax], dtype=np.int32)
    nthreads = max(1, len(os.sched_getaffinity(0)) // world)
    # inputs are generated with numpy on the host for the GPU and the oracle alike (bit-identical; the device's sin()
    # differs from libm's in the last place, which the hash would amplify)
    lk_np = info.lm[0].astype(np.float64) * (info.lm[0].astype(np.float64) + 1.0) + info.lm[1].astype(np.float64)
    in_sub = np.isin(np.abs(info.lm[1]), ms_sub)
    a_np = np.stack([np.where(in_sub, _hash_gauss_np(lk_np, c + 3), 0.0) for c in range(3)])
    a_np[1:3, info.lm[0] < 2] = 0.0
    a_sub = torch.as_tensor(a_np, device=dev)
    # the same a_lm in the oracle's own m-major order over the subset
    blocks = []
    for mm in ms_sub:
        ls = np.arange(mm, lmax + 1, dtype=np.float64)
        if mm == 0:
            blocks.append(np.stack([_hash_gauss_np(ls * (ls + 1), c + 3) for c in range(3)]))
        else:
            b = np.empty((3, 2 * ls.size))
            for c in range(3):
                b[c, 0::2] = _hash_gauss_np(ls * (ls + 1) + mm, c + 3)
                b[c, 1::2] = _hash_gauss_np(ls * (ls + 1) - mm, c + 3)
            blocks.append(b)
    alm_o = np.concatenate(blocks, axis=1)
    lo = np.concatenate([np.repeat(np.arange(mm, lmax + 1), 1 if mm == 0 else 2) for mm in ms_sub])
    alm_o[1:3, lo < 2] = 0.0
    refY = np.concatenate([S.execute(S.Y, 0, nside, lmax, alm=alm_o[0:1], ms=ms_sub, nthreads=nthreads),
                           S.execute(S.Y, 2, nside, lmax, alm=alm_o[1:3], ms=ms_sub, nthreads=nthreads)])
    refY_loc = torch.as_tensor(refY[:, info.pix], device=dev)
    del refY
    # analysis input: a map that is a function of the global pixel index
    gp = np.arange(12 * nside * nside, dtype=np.float64)
    xg = np.stack([_hash_gauss_np(gp, c + 6) for c in range(3)])
    refA = np.concatenate([S.execute(S.Yt, 0, nside, lmax, map=xg[0:1], ms=ms_sub, nthreads=nthreads),
                           S.execute(S.Yt, 2, nside, lmax, map=xg[1:3], ms=ms_sub, nthreads=nthreads)])
    x_loc = torch.as_tensor(xg[:, info.pix], device=dev)
    del xg
    # position of my local (l, m) slots of the subset inside the oracle's subset order
    mstart = {}
    pos = 0
    for mm in ms_sub:
        mstart[int(mm)] = pos
        pos += (lmax + 1 - mm) * (1 if mm == 0 else 2)
    l_np, m_np = info.lm[0].astype(np.int64), info.lm[1].astype(np.int64)
    sel = np.nonzero(np.isin(np.abs(m_np), ms_sub))[0]
    am = np.abs(m_np[sel])
    base = np.array([mstart[int(v)] for v in am], dtype=np.int64)
    oidx = base + np.where(am == 0, l_np[sel], 2 * (l_np[sel] - am) + (m_np[sel] < 0))
    refA_loc = torch.as_tensor(refA[:, oidx], device=dev)
    sel_t = torch.as_tensor(sel, device=dev)
    modes = [("single GPU", None)] if world == 1 else [("fused peer stores over NVLink", 1), ("NCCL all-to-all", 0)]
    par = []
    p = comm_map(info, device=dev)
    for name, mode in modes:
        if mode is not None:
            comm.set_exchange(mode)
        p.alm.copy_(a_sub)
        p.Y()
        errs = {}
        for tag, sl in (("Y_spin0", slice(0, 1)), ("Y_spin2", slice(1, 3))):
            d2, n2 = allsum([float(((p.map[sl] - refY_loc[sl]) ** 2).sum()), float((refY_loc[sl] ** 2).sum())])
            errs[tag] = (d2 / n2) ** 0.5
        p.map.copy_(x_loc)
        p.Yt()
        for tag, sl in (("Yt_spin0", slice(0, 1)), ("Yt_spin2", slice(1, 3))):
            got = p.alm[sl][:, sel_t]
            d2, n2 = allsum([float(((got - refA_loc[sl]) ** 2).sum()), float((refA_loc[sl] ** 2).sum())])
            errs[tag] = (d2 / max(n2, 1e-300)) ** 0.5
        par.append({"mode": name, "rel_l2": max(errs.values()), "per_job": errs})
    if world > 1:
        comm.set_exchange(-1)
    out["parity"] = {"rel_l2": max(q["rel_l2"] for q in par), "tolerance": 1e-10, "mode": [q["mode"] for q in par],
                     "detail": par, "m_subset": [int(v) for v in ms_sub],
                     "what": "comm_map Y and Yt (spin 0 + spin 2) through sharp_execute[_mpi_fortran] on this run's N GPUs vs the CPU "
                             "oracle (oracle/sht_cpu.c) on the m-subset x all rings, global relative L2 over all ranks"}
    out["parity_ok"] = bool(out["parity"]["rel_l2"] <= 1e-10)
    return out


DUMP_COLS = 1_000_000    # per dumped array: 3 x 1e6 float64 = 24 MB, so map + alm stay under 64 MB


def dump_outputs(path, arrays):
    """Writes each (ncomp, n) array as path/<name>.npy in float64.  An array with more than DUMP_COLS columns is
    reduced to a seeded sample of DUMP_COLS columns, the same columns for every component and for every run of the
    same size."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, x in arrays.items():
        n = x.shape[-1]
        if n > DUMP_COLS:
            cols = np.sort(np.random.default_rng(20).choice(n, DUMP_COLS, replace=False))
            x = x[:, torch.as_tensor(cols, device=x.device)]
        np.save(os.path.join(path, name + ".npy"), x.cpu().numpy())

# ------------------------------------------------------------------ GPU arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from commander_b200 import comm_map, comm_mapinfo, sharp
    from commander_b200 import dist as cdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a single-GPU run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        comm = cdist.init_from_torch(dev)
    nside, lmax = args.nside, args.lmax
    info = comm_mapinfo(comm, nside, lmax, 3, True)

    # synthetic Gaussian alm: value depends on (l, m) only, so results are independent of N
    g = torch.Generator(device=dev).manual_seed(9)
    full = None
    m = comm_map(info, device=dev)
    l_t = torch.as_tensor(info.lm[0].astype(np.int64), device=dev)
    m_t = torch.as_tensor(info.lm[1].astype(np.int64), device=dev)
    key = (l_t * (l_t + 1) + m_t).double()
    for c in range(3):
        # cheap deterministic pseudo-Gaussian from a hash of the global index (Box-Muller)
        u1 = torch.frac(torch.sin(key * 12.9898 + 78.233 * (c + 1)) * 43758.5453).abs().clamp_(1e-12, 1.0)
        u2 = torch.frac(torch.sin(key * 39.3468 + 11.135 * (c + 1)) * 24634.6345).abs()
        m.alm[c] = torch.sqrt(-2.0 * torch.log(u1)) * torch.cos(2 * np.pi * u2)
    m.alm[1:3, l_t < 2] = 0.0
    del g, full
    alm_in = m.alm.clone()

    def pair_dev():
        m.Y()
        m.YtW()

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # plan creation (coefficient tables, cuFFT plans, Bluestein filters) happens in the warm-up
    for _ in range(max(args.warmup, 3)):
        m.alm.copy_(alm_in)
        pair_dev()
    sync_all()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    sharp.set_profiling(True)
    sharp.last_legendre_ms()
    n0 = sharp.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    sync_all()
    ev[0].record()
    for _ in range(args.steps):
        pair_dev()
    ev[1].record()
    sync_all()
    launches = sharp.launch_count() - n0
    ms_total = ev[0].elapsed_time(ev[1])
    leg = sharp.last_legendre_ms()
    sharp.set_profiling(False)
    if args.dump_outputs:
        # what the caller of the last timed step receives: the map of Y() and the a_lm of YtW()
        dump_outputs(args.dump_outputs, {"map": m.map, "alm": m.alm})
    tmax = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_per_step = float(tmax.item()) / args.steps
    value = 1e3 / ms_per_step

    # ---- end to end through the reference-facing call with HOST buffers: pageable arrays (what the Fortran
    # caller passes, commander3/src/sharp.f90:219-224: the library stages them through its pinned arena) and, as a
    # note, caller-pinned arrays (copied in place)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def time_host(h):
        def pair_host():
            h.Y()      # H2D alm, kernels, D2H map
            h.YtW()    # H2D map, kernels, D2H alm
        pair_host()
        sync_all()
        t0 = time.perf_counter()
        ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev2[0].record()
        for _ in range(e2e_steps):
            pair_host()
        ev2[1].record()
        sync_all()
        wall = (time.perf_counter() - t0) * 1e3
        # host-side staging runs between the GPU operations, so the wall clock is the honest number; the two agree
        # for pinned buffers
        t = torch.tensor([max(ev2[0].elapsed_time(ev2[1]), 0.0), wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.max().item()) / e2e_steps

    alm_host = alm_in.cpu().numpy()
    h = comm_map(info)               # plain numpy arrays = pageable memory, as the Fortran caller has them
    h.alm[:] = alm_host
    e2e_pageable_ms = time_host(h)
    hp = comm_map(info)
    pin_alm = torch.empty((3, info.nalm), dtype=torch.float64).pin_memory()
    pin_map = torch.empty((3, info.np), dtype=torch.float64).pin_memory()
    hp.alm, hp.map = pin_alm.numpy(), pin_map.numpy()
    hp.alm[:] = alm_host
    e2e_pinned_ms = time_host(hp)
    e2e_same = float(np.abs(h.alm - hp.alm).max()) <= 1e-12 * float(np.abs(hp.alm).max())
    del h, hp, pin_alm, pin_map
    e2e_ms = e2e_pageable_ms if args.e2e_headline == "pageable" else e2e_pinned_ms
    parity = run_parity(args, info, comm, dev, world, m, alm_in) if not args.no_parity else None
    clocks = sampler.stop() if rank == 0 else None
    cg = run_cg_metric(args, comm, dev, world) if not args.no_cg else None
    batch = run_batch_metric(dev) if (world == 1 and not args.no_batch) else None
    conviqt = run_conviqt_metric(dev) if (world == 1 and not args.no_conviqt) else None
    bytes_alm, bytes_map = 3 * info.nalm * 8, 3 * info.np * 8

    # ---- roofline of the dominant kernel (spin-2 Legendre), FP64 pipe
    fp64_peak = sharp.measure_fp64_tflops(4096, 5)
    fp64_3op = sharp.measure_fp64_tflops_3op(4096, 3)
    per, stages = {}, {}
    for spin, direction, msv in leg:
        if spin >= 100:     # 100+spin: ring-FFT stage, 200/201: exchange barriers or all-to-all
            nm = (f"ringfft_spin{int(spin) - 100}" if spin < 200 else ("exchange_pre" if spin == 200 else "exchange_post")) + ("_analysis" if direction else "_synthesis")
            stages.setdefault(nm, []).append(msv)
            continue
        per.setdefault((spin, direction), []).append(msv)
    # per step totals: with the chunked two-stream path one launch per ring-pair chunk is recorded
    avg = {k: sum(v) / args.steps for k, v in per.items()}
    share = sum(sum(v) for v in per.values()) / max(ms_total, 1e-9)
    local_frac = float(sum(lmax + 1 - int(mm) for mm in info.ms)) / ((lmax + 1) * (lmax + 2) / 2)
    flops2 = 28.0 * ntriples(nside, lmax) * local_frac   # nominal flops of one spin-2 launch on this rank
    dom = max(((k, v) for k, v in avg.items() if k[0] == 2), key=lambda kv: kv[1], default=((2, 1), float("nan")))
    achieved = flops2 / (dom[1] * 1e-3) / 1e12
    exe = {0: executed_fraction(nside, lmax, 0, info.ms), 2: executed_fraction(nside, lmax, 2, info.ms)}
    # FP64-pipe instructions the kernel really issues per visited triple: 3 (spin 0, two l per recurrence step) / 12 (spin 2) DFMA
    achieved_exec = 2.0 * 12.0 * ntriples(nside, lmax) * local_frac * exe[2] / (dom[1] * 1e-3) / 1e12
    kern = {f"spin{k[0]}_{'analysis' if k[1] else 'synthesis'}_ms": round(v, 4) for k, v in sorted(avg.items())}
    kern["legendre_share_of_step"] = round(share, 4)
    kern["other_stages_ms"] = {k: round(sum(v) / args.steps, 4) for k, v in sorted(stages.items())}
    for k, v in sorted(avg.items()):
        fl = (8.0 if k[0] == 0 else 28.0) * ntriples(nside, lmax) * local_frac
        kern[f"spin{k[0]}_{'analysis' if k[1] else 'synthesis'}_tflops_nominal"] = round(fl / (v * 1e-3) / 1e12, 3)
        fe = 2.0 * (3.0 if k[0] == 0 else 12.0) * ntriples(nside, lmax) * local_frac * exe[k[0]]
        kern[f"spin{k[0]}_{'analysis' if k[1] else 'synthesis'}_tflops_executed"] = round(fe / (v * 1e-3) / 1e12, 3)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
        prof = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_summary.json")))
        key = next(k for k in prof if k.startswith("anal2_kernel" if dom[0][1] else "synth2_kernel"))
        if world == 1 and nside == 2048 and lmax == 4000:
            traffic = prof[key]["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError, StopIteration):
        pass
    traffic_source = ("dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture "
                      "profiles/r02_ncu_summary.json (not measured by this run)") if traffic is not None else None
    roofline = {"bound": "fp64", "traffic_source": traffic_source, "kernel": f"spin-2 Legendre {'analysis (anal2_kernel)' if dom[0][1] else 'synthesis (synth2_kernel)'}",
                "achieved": round(achieved, 3), "peak": round(fp64_peak, 3), "unit": "TFLOP/s",
                "frac": round(achieved / fp64_peak, 4), "traffic": traffic,
                "peak_source": "measured live: cmdr_sht_measure_fp64_tflops, DFMA probe with two vector-register operands "
                               "(MEASURED_PEAKS.json has no FP64 entry; nominal 148 SM x 64 FMA/clk x 2 x 1.965 GHz = 37.2)",
                "flop_convention": "achieved = nominal 28 flops per (l,m,ring pair) for spin 2 (8 for spin 0; SURVEY 8d), no work "
                                   "subtracted for the m cut-off, divided by the kernel's mean launch time (CUDA events on its stream)",
                "achieved_executed": round(achieved_exec, 3), "frac_executed": round(achieved_exec / fp64_peak, 4),
                "executed_convention": "DFMA instructions really issued: 12 per visited (l,m,ring pair) for spin 2 (3 for spin 0) x 2 flops; "
                                       f"visited = {exe[2]:.3f} of the nominal triples (rings beyond the per-ring m cut-off are skipped); an upper bound since the "
                                       "scalar front phase of the spin-2 kernels issues 1 instead of 4 recurrence DFMAs for the triples it covers",
                "peak_3operand": round(fp64_3op, 3),
                "peak_3operand_note": "DFMA with three distinct vector-register operands (no operand-reuse-cache hit): the register file "
                                      "feeds one 64-bit operand per cycle per scheduler, so such a DFMA issues every 3 cycles instead of 2",
                "kernels": kern}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    if peaks.get("hbm_gbs"):
        hbm_bytes = 2 * (bytes_alm + bytes_map + 2 * 32.0 * 3 * info.nm * 2 * nside)   # per pair, this rank
        roofline["hbm_secondary"] = {"algorithmic_GB_per_pair": round(hbm_bytes / 1e9, 3),
                                     "achieved_GBs": round(hbm_bytes / 1e9 / (ms_per_step * 1e-3), 1),
                                     "peak_GBs_measured": peaks["hbm_gbs"]}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:   # contract: rank 0 at N=1 only
            st = args.cpu_stride if args.cpu_stride > 0 else cpu_pick_stride(nside, lmax, 20.0)
            r = cpu_pair_sample(nside, lmax, st)
            cpu = {"value": 1.0 / r["seconds_full_est"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                   "simd": r["simd"], "sample": cpu_sample_text(r, st)}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload(args), "clocks": clocks, "gpu_launches": int(launches),
                "gpu_launches_note": "kernels launched by rank 0 inside the timed region (cuFFT execs count 1 each)",
                "e2e": {"value": 1e3 / e2e_ms, "unit": UNIT, "ms_per_step": e2e_ms, "steps": e2e_steps,
                        "h2d_bytes_per_step": bytes_alm + bytes_map, "d2h_bytes_per_step": bytes_alm + bytes_map,
                        "host_buffers": args.e2e_headline,
                        "pageable": {"value": 1e3 / e2e_pageable_ms, "ms_per_step": e2e_pageable_ms,
                                     "note": "ordinary (pageable) caller arrays, as commander3/src/sharp.f90:219-224 passes them: staged "
                                             "through the library's pinned arena by its copy threads inside the chunk pipeline"},
                        "pinned": {"value": 1e3 / e2e_pinned_ms, "ms_per_step": e2e_pinned_ms,
                                   "note": "caller-pinned arrays (cudaHostAlloc), copied in place"},
                        "pageable_equals_pinned_result": bool(e2e_same),
                        "timer": "max(CUDA events, wall clock) over ranks",
                        "api": "comm_map.Y(); comm_map.YtW()  (4 sharp_execute calls)"},
                "roofline": roofline, "cpu_baseline": cpu, "cg": cg, "batch": batch, "conviqt": conviqt}
        if parity is not None:
            line.update(parity)
        print(json.dumps(line))
    if world > 1:
        cdist.destroy(comm)
        dist.destroy_process_group()


def run_batch_metric(dev, nbands=30, nside=512, lmax=1500):
    """BASELINE.json configs[4]: 30 frequency maps (nside 512, lmax 1500, IQU) through Y / YtW per Gibbs
    step, pinned host buffers: (i) band by band through the ABI, (ii) through the batched entry point
    that pipelines the bands' PCIe copies against the kernels."""
    import numpy as np
    import torch
    from commander_b200 import comm_map, comm_mapinfo
    info = comm_mapinfo(None, nside, lmax, 3, True)
    maps = []
    rng = np.random.default_rng(100)
    for b in range(nbands):
        m = comm_map(info)
        m.alm = torch.empty((3, info.nalm), dtype=torch.float64).pin_memory().numpy()
        m.map = torch.empty((3, info.np), dtype=torch.float64).pin_memory().numpy()
        m.alm[:] = rng.standard_normal((3, info.nalm))
        maps.append(m)

    def seq():
        for m in maps:
            m.Y()
        for m in maps:
            m.YtW()

    def bat():
        comm_map.Y_batch(maps)
        comm_map.YtW_batch(maps)
    out = {}
    for name, fn in (("sequential", seq), ("batched", bat)):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        out[name] = nbands * reps / (time.perf_counter() - t0)
    nbytes = 2 * 3 * (info.nalm + info.np) * 8
    return {"metric": "SHT pairs/sec over a 30-band batch (nside 512, lmax 1500, IQU), host buffers", "unit": "pairs/s",
            "sequential_abi_calls": round(out["sequential"], 2), "batched_entry_point": round(out["batched"], 2),
            "pcie_bytes_per_pair": nbytes, "bands": nbands, "host_buffers": "pinned",
            "api": "comm_map.Y()/YtW() per band  vs  comm_map.Y_batch()/YtW_batch() (cmdr_sht_execute_iqu_batch)"}


def run_conviqt_metric(dev, nside=512, lmax=1000, bmax=8):
    """SURVEY 8f rank 4: the conviqt convolution cube (comm_conviqt%precompute_sky, commander3/src/comm_conviqt_mod.f90:207-292):
    bmax+1 spin-j syntheses and the psi transform, sky a_lm / beam table / cube device resident."""
    import numpy as np
    import torch
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    info = comm_mapinfo(None, nside, lmax, 3, True)
    rng = np.random.default_rng(200)
    sky = comm_map(info, device=dev)
    sky.alm.copy_(torch.as_tensor(rng.standard_normal((3, info.nalm))))
    beam = comm_map(info)
    beam.alm[...] = rng.standard_normal(beam.alm.shape) / (1.0 + info.lm[0])
    cv = comm_conviqt(nside, lmax, 3, bmax, beam, sky, device=dev)    # first call: plans, tables
    torch.cuda.synchronize()
    reps = 3
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        cv.precompute_sky(sky)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    psi_bytes = info.np * (8 * (2 * bmax + 1) + 4 * 2 * bmax)
    return {"metric": "conviqt cubes/sec (precompute_sky)", "value": round(1e3 / ms, 3), "unit": "cubes/s", "ms_per_cube": round(ms, 3),
            "config": f"nside={nside} lmax={lmax} IQU sky x beam, bmax={bmax} (1 spin-0 + {bmax} spin-j syntheses, {2 * bmax} psi planes, "
                      "float32 cube), device-resident",
            "psi_kernel_algorithmic_bytes": psi_bytes}


CG_NSIDE, CG_LMAX, CG_ITERS = 1024, 2000, 50


def _cg_inputs(nside, lmax):
    import numpy as np
    l = np.arange(lmax + 1, dtype=np.float64)
    Cl = np.stack([1.0 / (l * (l + 1) + 1.0)] * 3, axis=1)
    sigma0 = float(np.sqrt(Cl[min(1000, lmax // 2), 0] * 12 * nside ** 2 / (4 * np.pi)))
    return Cl, sigma0


def run_cg_metric(args, comm, dev, world):
    """Second half of BASELINE.json's metric: CR CG iterations/s on configs[2] (nside 1024, lmax 2000, IQU, diagonal
    N^-1 + Gaussian beam, CMB only), criterion fixed_iter with 50 iterations as shipped
    (parameter_files/param_BP8.1_v1.txt:40-47), through the C ABI (cmdr_cr_solve): vectors device resident, sqrt(S) / beam /
    N^-1 fused into the transform kernels, dot products reduced on the device, no host synchronisation in the loop."""
    import numpy as np
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_cmb_system, cr_native_system, gaussian_beam, solve_cr_eqn_by_CG
    nside, lmax, iters = CG_NSIDE, CG_LMAX, CG_ITERS
    info = comm_mapinfo(comm, nside, lmax, 3, True)
    Cl, sigma0 = _cg_inputs(nside, lmax)
    g = torch.Generator(device=dev).manual_seed(5 + (comm.rank if comm else 0))
    pix = torch.as_tensor(info.pix, device=dev).double()
    z = 1.0 - 2.0 * (pix + 0.5) / (12 * nside ** 2)            # ~cos(theta) of the pixel in ring order
    siN = (1.0 / (sigma0 * (1.0 + 0.5 * (1.0 - z * z)))).expand(3, -1).contiguous()
    bl = gaussian_beam(lmax, 10.0)
    sysn = cr_native_system(info, [siN * siN], [bl], Cl)
    data = torch.empty((3, info.np), dtype=torch.float64, device=dev).normal_(generator=g) / siN
    b = sysn.computeRHS([data])
    sysn.solve(b, maxiter=2, cg_conv_crit="fixed_iter")       # warm-up / plans
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t0 = time.perf_counter()
    ev[0].record()
    x, it, hist = sysn.solve(b, maxiter=iters, cg_conv_crit="fixed_iter")
    ev[1].record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    ms = torch.tensor([max(ev[0].elapsed_time(ev[1]), wall)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    # the round-1 torch mirror of the same system (eager element-wise passes, two host syncs per iteration), for comparison
    sysm = cr_cmb_system(info, siN, bl, Cl)
    bm = sysm.computeRHS(data)
    solve_cr_eqn_by_CG(sysm, bm, maxiter=2, cg_conv_crit="fixed_iter")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    xm, itm, histm = solve_cr_eqn_by_CG(sysm, bm, maxiter=10, cg_conv_crit="fixed_iter")
    torch.cuda.synchronize()
    ms_m = torch.tensor([(time.perf_counter() - t0) * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_m, op=dist.ReduceOp.MAX)
    agree = float(abs(hist[10] - histm[10]) / abs(histm[10]))
    return {"metric": "CR CG iters/sec", "value": it / (ms * 1e-3), "unit": "iter/s",
            "config": f"nside={nside} lmax={lmax} IQU, 1 band, CMB only, diagonal N^-1, 10' Gaussian beam, diagonal preconditioner "
                      f"(full N_lm), fixed_iter x{iters} (x0 = 0: one A application per iteration), cmdr_cr_solve through the C ABI",
            "ms_per_iter": ms / it, "iterations": it, "residual_drop": hist[-1] / hist[0],
            "torch_mirror_iters_per_s": 11.0 / (float(ms_m.item()) * 1e-3),
            "native_vs_mirror_residual_after_10_iterations_rel": agree}


def cpu_cg_sample(nside, lmax, iters, nthreads=0):
    """The reference's CG iteration on the host cores: cr_matmulA (commander3/src/comm_cr_mod.f90:771-1024) with the CPU
    restatement as SHT engine and numpy for the vector passes, `iters` iterations of solve_cr_eqn_by_CG (:201-348).
    Returns seconds per iteration (what the reference prints at :326-335)."""
    import numpy as np
    from oracle import sht_cpu as S
    S.build()
    if nthreads == 0:
        nthreads = len(os.sched_getaffinity(0))
    Cl, sigma0 = _cg_inputs(nside, lmax)
    npix = 12 * nside * nside
    z = 1.0 - 2.0 * (np.arange(npix) + 0.5) / npix
    invN = np.stack([(1.0 / (sigma0 * (1.0 + 0.5 * (1.0 - z * z)))) ** 2] * 3)
    sigma = 10.0 * np.pi / 180.0 / 60.0 / np.sqrt(8.0 * np.log(2.0))
    lo = np.concatenate([np.repeat(np.arange(m, lmax + 1), 1 if m == 0 else 2) for m in range(lmax + 1)])
    blT = np.exp(-0.5 * lo * (lo + 1.0) * sigma ** 2)
    f = np.stack([blT, blT * np.exp(2 * sigma ** 2), blT * np.exp(2 * sigma ** 2)]) * np.sqrt(1.0 / (lo * (lo + 1.0) + 1.0))
    f[1:, lo < 2] = 0.0

    def A(v):
        w = f * v
        mp = np.concatenate([S.execute(S.Y, 0, nside, lmax, alm=w[0:1], nthreads=nthreads, mlim_skip=True),
                             S.execute(S.Y, 2, nside, lmax, alm=w[1:3], nthreads=nthreads, mlim_skip=True)])
        mp *= invN
        a = np.concatenate([S.execute(S.Yt, 0, nside, lmax, map=mp[0:1], nthreads=nthreads, mlim_skip=True),
                            S.execute(S.Yt, 2, nside, lmax, map=mp[1:3], nthreads=nthreads, mlim_skip=True)])
        return v + f * a
    rng = np.random.default_rng(5)
    b = rng.standard_normal(f.shape)
    Minv = 1.0 / (1.0 + f * f * float(invN.mean()) * npix / (4 * np.pi))
    A(b)                                                      # warm-up: FFT plans, page faults
    x = np.zeros_like(b); r = b.copy(); d = Minv * r
    dn = float(np.sum(r * d))
    t0 = time.perf_counter()
    for _ in range(iters):
        q = A(d); alpha = dn / float(np.sum(d * q)); x += alpha * d; r -= alpha * q
        s = Minv * r; do = dn; dn = float(np.sum(r * s)); d = s + dn / do * d
    return (time.perf_counter() - t0) / iters, nthreads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nside", type=int, default=2048)
    ap.add_argument("--lmax", type=int, default=4000)
    ap.add_argument("--cpu-stride", type=int, default=0,
                    help="CPU sample: every stride-th m (0: chosen so that the sample costs ~10-20 s of CPU time on this box)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the checksum / oracle-parity block")
    ap.add_argument("--e2e-headline", default="pageable", choices=["pageable", "pinned"],
                    help="which host-buffer kind e2e.value reports (both are always measured)")
    ap.add_argument("--no-cg", action="store_true", help="skip the secondary CG iters/s measurement")
    ap.add_argument("--no-batch", action="store_true", help="skip the 30-band batch measurement (config 5)")
    ap.add_argument("--no-conviqt", action="store_true", help="skip the conviqt cube measurement (SURVEY 8f rank 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the map and a_lm of the last timed step as DIR/map.npy and DIR/alm.npy (float64; a fixed "
                         f"seeded sample of {DUMP_COLS} columns when larger)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
