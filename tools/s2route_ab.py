#!/usr/bin/env python
"""s2route_ab.py -- what running spin 2 as scalar sums (cmdr_sht_set_spin2_scalar) saves, per Legendre stage.

Times synth0, anal0, synth2 and anal2 (the Legendre stage of SHARP_Y / SHARP_YtW at spin 0 and 2, device-resident data,
cmdr_sht_set_profiling events around each Legendre stage; with the route on, "synth2" / "anal2" are the whole spin-2
stage: prep, both scalar launches, the polar spin-2 launch and, for analysis, the post kernel) with the route off and
on, alternating in the same process, and reports medians over --rounds rounds.  The same calls give the largest
difference between the two routes' spin-2 maps and a_lm relative to the largest value and as relative L2.  Prints the
card name, power limit and SM clock read in the same run, and one JSON line (also written to --out when given).

  python tools/s2route_ab.py [--nside 2048] [--lmax 4000] [--rounds 12] [--warmup 2] [--out FILE]
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

KERNELS = {(0, 0): "synth0", (0, 1): "anal0", (2, 0): "synth2", (2, 1): "anal2"}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unknown ({e})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nside", type=int, default=2048)
    ap.add_argument("--lmax", type=int, default=4000)
    ap.add_argument("--rounds", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("s2route_ab needs a CUDA device")
    from commander_b200 import sharp
    nside, lmax = args.nside, args.lmax
    ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
    gi = sharp.sharp_make_healpix_geom_info(nside)
    rng = np.random.default_rng(0)
    alm = {s: torch.from_numpy(rng.standard_normal((1 if s == 0 else 2, ai.n_local))).cuda() for s in (0, 2)}
    maps = {s: torch.empty((1 if s == 0 else 2, gi.n_local), dtype=torch.float64, device="cuda") for s in (0, 2)}
    back = {s: torch.empty_like(alm[s]) for s in (0, 2)}

    def run(route):
        """One Y + YtW per spin; returns the Legendre ms per kernel and the outputs."""
        sharp.set_spin2_scalar(route)
        out, ms = {}, {}
        for s in (0, 2):
            sharp.sharp_execute(sharp.SHARP_Y, s, maps[s].shape[0], alm[s], ai, maps[s], gi)
            sharp.sharp_execute(sharp.SHARP_YtW, s, maps[s].shape[0], back[s], ai, maps[s], gi)
            torch.cuda.synchronize()
            for sp, d, t in sharp.last_legendre_ms():
                if (sp, d) in KERNELS:
                    ms[KERNELS[(sp, d)]] = t
            out[s] = (maps[s].clone(), back[s].clone())
        return ms, out

    sharp.set_profiling(True)
    sharp.last_legendre_ms()
    for _ in range(args.warmup):
        run(False)
        run(True)
    times = {False: {k: [] for k in KERNELS.values()}, True: {k: [] for k in KERNELS.values()}}
    diff = {"map_max": 0.0, "map_rel_l2": 0.0, "alm_max": 0.0, "alm_rel_l2": 0.0}
    for _ in range(args.rounds):
        ref = None
        for route in (False, True):
            ms, out = run(route)
            for k, t in ms.items():
                times[route][k].append(t)
            if not route:
                ref = out
            else:
                for i, what in ((0, "map"), (1, "alm")):
                    for c in range(2):
                        a, b = out[2][i][c], ref[2][i][c]
                        diff[f"{what}_max"] = max(diff[f"{what}_max"], float((a - b).abs().max() / b.abs().max()))
                        diff[f"{what}_rel_l2"] = max(diff[f"{what}_rel_l2"], float(torch.linalg.norm(a - b) / torch.linalg.norm(b)))
    sharp.set_profiling(False)
    sharp.set_spin2_scalar(True)
    res = {"nside": nside, "lmax": lmax, "rounds": args.rounds, "card": card(),
           "seed_table_bytes": sharp.legendre_seed_bytes(), **{f"spin2_{k}": v for k, v in diff.items()}}
    tot = {False: 0.0, True: 0.0}
    for k in KERNELS.values():
        for route, name in ((False, "spin2"), (True, "scalar")):
            med = statistics.median(times[route][k])
            res[f"{k}_{name}_ms"] = round(med, 4)
            res[f"{k}_{name}_spread_ms"] = round(max(times[route][k]) - min(times[route][k]), 4)
            tot[route] += med
        res[f"{k}_saved_pct"] = round(100.0 * (1.0 - res[f"{k}_scalar_ms"] / res[f"{k}_spin2_ms"]), 2)
    res["pair_spin2_route_ms"] = round(tot[False], 4)
    res["pair_scalar_route_ms"] = round(tot[True], 4)
    print(f"card: {res['card']}")
    for k in KERNELS.values():
        print(f"{k:7s} route off {res[f'{k}_spin2_ms']:8.3f} ms   on {res[f'{k}_scalar_ms']:8.3f} ms   "
              f"saved {res[f'{k}_saved_pct']:5.2f} %")
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    sharp.sharp_destroy_alm_info(ai)
    sharp.sharp_destroy_geom_info(gi)


if __name__ == "__main__":
    main()
