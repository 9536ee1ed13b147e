"""Times SHARP_ALM2MAP_DERIV1 against the two syntheses it sits between, device-resident, in one process:

  deriv1   the gradient job (prep_d1_kernel + synth_d1_kernel, 4 accumulate FMAs per l and ring pair)
  spin1    the general spin-1 SHARP_Y fed with E = -sqrt(l(l+1)) a, B = 0 (same maps; synth2_kernel, 8 FMAs)
  spin0    SHARP_Y of the same a_lm (one map)

Whole calls are timed with CUDA events, the three alternating over --reps rounds after --warmup rounds; the Legendre
kernel times come from cmdr_sht_set_profiling / cmdr_sht_last_legendre_ms in a separate pass.  Prints the card name
and power limit read in the same run, and one JSON line.

  python tools/deriv_bench.py [--nside 2048] [--lmax 4000] [--reps 20] [--warmup 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unknown ({e})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nside", type=int, default=2048)
    ap.add_argument("--lmax", type=int, default=4000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("deriv_bench needs a CUDA device")
    from commander_b200 import sharp
    nside, lmax = args.nside, args.lmax
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    rng = np.random.default_rng(0)
    a = rng.standard_normal((1, ai.n_local))
    l = np.concatenate([np.repeat(np.arange(m, lmax + 1), 1 if m == 0 else 2) for m in range(lmax + 1)]).astype(np.float64)
    alm = torch.from_numpy(a).cuda()
    eb = torch.zeros((2, ai.n_local), dtype=torch.float64, device="cuda")
    eb[0] = torch.from_numpy(-np.sqrt(l * (l + 1)) * a[0]).cuda()
    m2 = torch.empty((2, gi.n_local), dtype=torch.float64, device="cuda")
    m2b = torch.empty_like(m2)
    m1 = torch.empty((1, gi.n_local), dtype=torch.float64, device="cuda")
    jobs = {
        "deriv1": lambda: sharp.alm2map_der1(alm, ai, m2, gi),
        "spin1": lambda: sharp.sharp_execute(sharp.SHARP_Y, 1, 2, eb, ai, m2b, gi),
        "spin0": lambda: sharp.sharp_execute(sharp.SHARP_Y, 0, 1, alm, ai, m1, gi),
    }
    for _ in range(args.warmup):
        for f in jobs.values():
            f()
    torch.cuda.synchronize()
    rel = float(torch.linalg.norm(m2 - m2b) / torch.linalg.norm(m2b))
    ms = {k: [] for k in jobs}
    for _ in range(args.reps):
        for k, f in jobs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    # Legendre kernel times: profiling pass of its own (events around the Legendre launch of every call)
    leg = {k: [] for k in jobs}
    sharp.set_profiling(True)
    sharp.last_legendre_ms()
    for _ in range(max(3, args.reps // 4)):
        for k, f in jobs.items():
            f()
            torch.cuda.synchronize()
            leg[k] += [t for s, d, t in sharp.last_legendre_ms() if s < 100 and d == 0]
    sharp.set_profiling(False)
    res = {"nside": nside, "lmax": lmax, "reps": args.reps, "card": card(), "deriv1_vs_spin1_rel_l2": rel}
    for k in jobs:
        res[f"{k}_call_ms_median"] = statistics.median(ms[k])
        res[f"{k}_call_ms_min"] = min(ms[k])
        res[f"{k}_legendre_ms_median"] = statistics.median(leg[k]) if leg[k] else None
    print(f"card: {res['card']}")
    for k in jobs:
        print(f"{k:7s} call {res[f'{k}_call_ms_median']:8.3f} ms (min {res[f'{k}_call_ms_min']:.3f})   "
              f"Legendre {res[f'{k}_legendre_ms_median']:.3f} ms")
    print(json.dumps(res))
    sharp.sharp_destroy_alm_info(ai)
    sharp.sharp_destroy_geom_info(gi)


if __name__ == "__main__":
    main()
