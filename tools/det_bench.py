"""det_bench.py -- what the deterministic mode (cmdr_sht_set_deterministic) costs, default and deterministic runs
alternated in one process and timed with CUDA events:
  - device-resident IQU YtW and Yt (cmdr_sht_execute_iqu) at nside 2048 / lmax 4000;
  - the pinned end-to-end pair (Y then YtW from pinned host arrays, sharp_execute per spin);
  - CG iterations per second of bench.py's `cg` configuration (cmdr_cr_solve, nside 1024 / lmax 2000, IQU, one band,
    diagonal preconditioner, 50 fixed_iter iterations per timed call);
  - the partials bytes of the analysis launches at that size (computed from det.h's layout).
Writes profiles/<round>_det_bench.json with the card name and power limit.
Usage: python tools/det_bench.py --round r10 [--reps 5] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
        name, pl = [s.strip() for s in q.split(",")]
        return name, pl
    except Exception as e:   # noqa: BLE001
        return f"unknown ({e})", "unknown"


def partial_bytes(nside, lmax):
    npairs = 2 * nside
    nm = lmax + 1
    s0 = -(-npairs // 256) * nm * 2 * (lmax + 1) * 8                 # anal0_kernel, one component
    s2s = -(-npairs // 256) * nm * 2 * (lmax + 3) * 8 * 2            # spin 2 as scalar sums, two components
    s2 = -(-npairs // 128) * nm * 2 * (lmax + 1) * 8 * 2             # anal2_kernel, E and B
    return dict(spin0=s0, spin2_scalar_route=s2s, spin2_kernels=s2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r10")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--nside", type=int, default=2048)
    ap.add_argument("--lmax", type=int, default=4000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "det_bench.py measures on a GPU"
    from commander_b200 import comm_mapinfo, sharp
    info = comm_mapinfo(None, a.nside, a.lmax, 3, True)
    gT, gP, ai = info.geom_info_T, info.geom_info_P, info.alm_info
    rng = np.random.default_rng(0)
    mp = torch.from_numpy(rng.standard_normal((3, gT.n_local))).cuda()
    alm = torch.from_numpy(rng.standard_normal((3, ai.n_local))).cuda()
    out_a = torch.empty_like(alm)
    mp_pin = mp.cpu().pin_memory()
    alm_pin = alm.cpu().pin_memory()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(fn):
        torch.cuda.synchronize()
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1])

    # bench.py's `cg` configuration (run_cg_metric): CMB-only system, N^-1 varying with latitude, 10' beam
    from commander_b200.comm_cr import cr_native_system, gaussian_beam
    cg_nside, cg_lmax, cg_iters = 1024, 2000, 50
    cinfo = comm_mapinfo(None, cg_nside, cg_lmax, 3, True)
    l = np.arange(cg_lmax + 1, dtype=np.float64)
    Cl = np.stack([1.0 / (l * (l + 1) + 1.0)] * 3, axis=1)
    sigma0 = float(np.sqrt(Cl[min(1000, cg_lmax // 2), 0] * 12 * cg_nside ** 2 / (4 * np.pi)))
    pix = torch.as_tensor(cinfo.pix, device="cuda").double()
    z = 1.0 - 2.0 * (pix + 0.5) / (12 * cg_nside ** 2)
    siN = (1.0 / (sigma0 * (1.0 + 0.5 * (1.0 - z * z)))).expand(3, -1).contiguous()
    cg_sys = cr_native_system(cinfo, [siN * siN], [gaussian_beam(cg_lmax, 10.0)], Cl)
    g = torch.Generator(device="cuda").manual_seed(5)
    cg_b = cg_sys.computeRHS([torch.empty((3, cinfo.np), dtype=torch.float64, device="cuda").normal_(generator=g) / siN])
    cases = {
        "iqu_YtW_device_ms": lambda: sharp.execute_iqu(sharp.SHARP_YtW, out_a, mp, gT, gP, ai),
        "iqu_Yt_device_ms": lambda: sharp.execute_iqu(sharp.SHARP_Yt, out_a, mp, gT, gP, ai),
        "pinned_pair_ms": lambda: (sharp.sharp_execute(sharp.SHARP_Y, 0, 1, alm_pin[0:1], ai, mp_pin[0:1], gT),
                                   sharp.sharp_execute(sharp.SHARP_Y, 2, 2, alm_pin[1:3], ai, mp_pin[1:3], gP),
                                   sharp.sharp_execute(sharp.SHARP_YtW, 0, 1, alm_pin[0:1], ai, mp_pin[0:1], gT),
                                   sharp.sharp_execute(sharp.SHARP_YtW, 2, 2, alm_pin[1:3], ai, mp_pin[1:3], gP)),
        "cg_50_iters_ms": lambda: cg_sys.solve(cg_b, maxiter=cg_iters, cg_conv_crit="fixed_iter"),
    }
    res = {k: {"default": [], "deterministic": []} for k in cases}
    try:
        for mode in (False, True):             # warm-up of both modes (plans, seed tables, partials buffer)
            sharp.set_deterministic(mode)
            for fn in cases.values():
                timed(fn)
        for _ in range(a.reps):
            for mode in (False, True):
                sharp.set_deterministic(mode)
                for k, fn in cases.items():
                    res[k]["deterministic" if mode else "default"].append(timed(fn))
    finally:
        sharp.set_deterministic(False)
    name, pl = card()
    summary = {}
    for k, v in res.items():
        d, t = np.median(v["default"]), np.median(v["deterministic"])
        summary[k] = dict(default_median=d, deterministic_median=t, overhead_pct=100.0 * (t - d) / d,
                          default_runs=v["default"], deterministic_runs=v["deterministic"])
    cg = summary["cg_50_iters_ms"]
    summary["cg_iters_per_s"] = dict(default=1e3 * cg_iters / cg["default_median"],
                                     deterministic=1e3 * cg_iters / cg["deterministic_median"],
                                     change_pct=100.0 * (cg["default_median"] / cg["deterministic_median"] - 1.0))
    doc = dict(card=name, power_limit=pl, nside=a.nside, lmax=a.lmax, reps=a.reps, timing="CUDA events around each call",
               results=summary, partials_bytes=partial_bytes(a.nside, a.lmax))
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, f"{a.round}_det_bench.json")
    with open(path, "w") as f:
        json.dump(doc, f, indent=1)
    for k, s in summary.items():
        if "overhead_pct" not in s:
            print(k, {a: round(b, 3) for a, b in s.items()})
            continue
        print(f"{k}: default {s['default_median']:.2f} ms, deterministic {s['deterministic_median']:.2f} ms "
              f"({s['overhead_pct']:+.1f} %)")
    print("card", name, "power limit", pl, "->", path)


if __name__ == "__main__":
    main()
