"""Time the right-hand side of a constrained realisation with its fluctuation terms from the host (numpy draws passed to
computeRHS, pageable and pinned) against the same terms drawn on the device (computeRHS_draw,
commander_b200/csrc/cr_draw.cu), on two configurations:
  (a) the CG configuration: nside 1024 / lmax 2000 IQU, one band, cr_native_system (cmdr_cr_setup);
  (b) config 5: 30 IQU bands at nside 512 / lmax 1500, one CMB component, cr_native_multi_system (cmdr_cr_setup_multi).
`data` is device resident in every arm, so the arms differ only in where eta comes from.

  python tools/cr_rhs_draw_bench.py --out DIR [--reps 3] [--only a|b]

Per configuration: the host draw time of numpy default_rng().standard_normal for the same arrays (host clock), each
computeRHS arm (host clock around calls that end in a device synchronise; median of --reps after a warm-up call), and the
draw kernels' time from a torch.profiler run of its own, with their share of the HBM bound (bytes / 7.7 TB/s), of the
FP64 bound (FP64 instructions over the FP64 rate measured in the same run by cmdr_sht_measure_fp64_tflops) and of the
instruction-issue bound (SASS instructions per draw over 4 warp instructions per SM and clock at the maximum SM clock),
and the same kernel writing the draws alone (draw_eta: no reads).  Writes
DIR/r09_cr_rhs_draw_bench.json with the card name, power limit and maximum SM clock read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBS = 7.7                 # HGX B200 data sheet, one GPU
ISSUE_RATE = float("nan")     # set in main() from the SM count and the maximum SM clock
# Per drawn pixel on the loop path of k_rhs_map_draw that computeRHS_draw runs (N^-1 and d given), counted in its SASS
# (cuobjdump -sass of the sm_100a build, the branches taken for ordinary values): 287 instructions, 67 of them FP64
# (DFMA / DMUL / DADD / DSETP: log, sqrt, cospi, the product and the fma), 59 IMAD (Philox's 32-bit products and the
# index arithmetic).  Static counts of one path, not counters of executed instructions.
SASS_INSTR_PER_DRAW = 287
FP64_INSTR_PER_DRAW = 67
ISSUE_PER_SM_CLK = 4 * 32     # four schedulers per SM, one warp instruction each per clock


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def median_ms(fn, reps):
    import torch
    fn()                                                   # warm-up: every shape of the timed window
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), ts


PROFILED_CALLS = 3


def kernel_us(fn, names):
    """Device time (us) per call of the kernels whose names contain one of `names`, from PROFILED_CALLS calls of fn in one
    profiler run after a warm-up call (the profiler can miss the first kernel record of a run: one call alone may then lack
    a launch), and the launches matched over all calls"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(PROFILED_CALLS):
            fn()
        torch.cuda.synchronize()
    per = {n: 0.0 for n in names}
    count = {n: 0 for n in names}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        for n in names:
            if n in ev.name:
                per[n] += t / PROFILED_CALLS
                count[n] += 1
    return per, count


def draw_eta_into(sysn, out_pix, out_alm):
    """cmdr_cr_draw_eta into preallocated device buffers (the Python draw_eta allocates its outputs)"""
    from commander_b200.comm_cr import _ptrs
    cols = [m[j] for m in out_pix for j in range(m.shape[0])]
    if out_alm.dim() == 2:
        acols = [out_alm[j] for j in range(out_alm.shape[0])]
    else:
        acols = sysn._cols(out_alm)[1]
    ep, _a = _ptrs(cols)
    ap, _b = _ptrs(acols)
    sysn.L.cmdr_cr_draw_eta(sysn.handle, 42, 7, ep, ap, None)


def setup_a(dev, rng):
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_native_system, gaussian_beam
    nside, lmax = 1024, 2000
    info = comm_mapinfo(None, nside, lmax, 3, True)
    l = np.arange(lmax + 1, dtype=np.float64)
    Cl = np.stack([1.0 / (l * (l + 1) + 1.0)] * 3, axis=1)
    invN = torch.as_tensor((1.0 / (0.5 + rng.uniform(size=(3, info.np)))) ** 2, device=dev)
    sysn = cr_native_system(info, [invN], [gaussian_beam(lmax, 10.0)], Cl, precond="none")
    data = [torch.as_tensor(rng.standard_normal((3, info.np)), device=dev)]
    return sysn, data, [(3, info.np)], (3, info.nalm), [invN]


def setup_b(dev, rng):
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, gaussian_beam
    nside, lmax, nb = 512, 1500, 30
    info = comm_mapinfo(None, nside, lmax, 3, True)
    l = np.arange(lmax + 1, dtype=np.float64)
    Cl = np.stack([1.0 / (l * (l + 1) + 1.0)] * 3, axis=1)
    bands = [cr_band(info, torch.as_tensor((1.0 / (0.5 + rng.uniform(size=(3, info.np)))) ** 2, device=dev),
                     gaussian_beam(lmax, 14.0 + q)) for q in range(nb)]
    comp = cr_component(info, Cl=Cl, F_mean=np.ones((nb, 3)))
    nat = cr_native_multi_system([comp], bands, precond="none")
    data = [torch.as_tensor(rng.standard_normal((3, info.np)), device=dev) for _ in range(nb)]
    return nat, data, [(3, info.np)] * nb, (nat.ncr,), [b.invN for b in bands]


def run_config(name, build, dev, reps, fp64_tflops):
    import torch
    rng = np.random.default_rng(9)
    sysn, data, pix_shapes, alm_shape, invN = build(dev, rng)
    npix_tot = int(sum(a * b for a, b in pix_shapes))
    nalm_tot = int(np.prod(alm_shape))
    res = {"config": name, "draws_pixel": npix_tot, "draws_prior": nalm_tot,
           "host_eta_bytes": 8 * (npix_tot + nalm_tot)}
    # host draws: numpy's generator for the same arrays
    hrng = np.random.default_rng(123)
    t0 = time.perf_counter()
    eta_pix = [hrng.standard_normal(s) for s in pix_shapes]
    eta_alm = hrng.standard_normal(alm_shape)
    res["host_draw_ms"] = 1e3 * (time.perf_counter() - t0)
    pin_pix = [torch.from_numpy(e).pin_memory() for e in eta_pix]
    pin_alm = torch.from_numpy(eta_alm).pin_memory()
    dev_pix = [e.to(dev) for e in pin_pix]
    dev_alm = pin_alm.to(dev)
    arms = {
        "computeRHS_pageable_eta": lambda: sysn.computeRHS(data, eta_pix, eta_alm),
        "computeRHS_pinned_eta": lambda: sysn.computeRHS(data, pin_pix, pin_alm),
        "computeRHS_device_eta": lambda: sysn.computeRHS(data, dev_pix, dev_alm),
        "computeRHS_draw": lambda: sysn.computeRHS_draw(data, 42, 7),
        "computeRHS_no_eta": lambda: sysn.computeRHS(data),
    }
    for k, fn in arms.items():
        ms, ts = median_ms(fn, reps)
        res[k + "_ms"] = ms
        res[k + "_all_ms"] = ts
    res["host_draw_plus_pageable_ms"] = res["host_draw_ms"] + res["computeRHS_pageable_eta_ms"]
    # the draw kernels alone (profiled run of its own) and the mean-field map kernel they replace
    per, cnt = kernel_us(lambda: sysn.computeRHS_draw(data, 42, 7), ["k_rhs_map_draw", "k_eta_alm_draw"])
    base, _ = kernel_us(lambda: sysn.computeRHS(data), ["k_rhs_map"])
    # the draws alone (draw_eta into device buffers): the same kernel writing eta only (8 B per pixel, nothing read).  If it
    # takes about as long as the 24-byte RHS pass, memory traffic is not what limits the pass.
    out_pix = [torch.empty(s, dtype=torch.float64, device=dev) for s in pix_shapes]
    out_alm = torch.empty(alm_shape, dtype=torch.float64, device=dev)
    raw, raw_cnt = kernel_us(lambda: draw_eta_into(sysn, out_pix, out_alm), ["k_rhs_map_draw", "k_eta_alm_draw"])
    ev_ms, _ = median_ms(lambda: draw_eta_into(sysn, out_pix, out_alm), reps)
    t_draw = per["k_rhs_map_draw"] * 1e-6
    bytes_draw = 24 * npix_tot                             # N^-1 and d read, m written
    hbm_s = bytes_draw / (HBM_TBS * 1e12)
    fp64_s = FP64_INSTR_PER_DRAW * npix_tot / (fp64_tflops * 1e12 / 2)   # the probe counts an FMA as 2 flops
    res["kernels"] = {
        "k_rhs_map_draw_ms": t_draw * 1e3,
        "k_rhs_map_draw_launches": cnt["k_rhs_map_draw"],
        "k_eta_alm_draw_ms": per["k_eta_alm_draw"] * 1e-3,
        "k_eta_alm_draw_launches": cnt["k_eta_alm_draw"],
        "draw_only_k_rhs_map_draw_ms (writes eta, 8 B per pixel)": raw["k_rhs_map_draw"] * 1e-3,
        "draw_only_k_eta_alm_draw_ms": raw["k_eta_alm_draw"] * 1e-3,
        "draw_only_launches": raw_cnt,
        "draw_eta_call_ms (host clock, device outputs)": ev_ms,
        "k_rhs_map_ms (mean-field pass of computeRHS without eta)": base["k_rhs_map"] * 1e-3,
        "k_rhs_map_draw_bytes": bytes_draw,
        "k_rhs_map_draw_GB_per_s": bytes_draw / t_draw / 1e9 if t_draw > 0 else None,
        "hbm_bound_ms": hbm_s * 1e3,
        "hbm_share": hbm_s / t_draw if t_draw > 0 else None,
        "fp64_instr_per_draw_estimate": FP64_INSTR_PER_DRAW,
        "fp64_bound_ms": fp64_s * 1e3,
        "fp64_share": fp64_s / t_draw if t_draw > 0 else None,
        "sass_instr_per_draw": SASS_INSTR_PER_DRAW,
        "issue_bound_ms": SASS_INSTR_PER_DRAW * npix_tot / ISSUE_RATE * 1e3,
        "issue_share": SASS_INSTR_PER_DRAW * npix_tot / ISSUE_RATE / t_draw if t_draw > 0 else None,
        "bound": max((("HBM", hbm_s), ("FP64", fp64_s), ("instruction issue", SASS_INSTR_PER_DRAW * npix_tot / ISSUE_RATE)),
                     key=lambda kv: kv[1])[0],
    }
    del sysn, data, invN, dev_pix, dev_alm, out_pix, out_alm
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", choices=("a", "b"), default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("cr_rhs_draw_bench: needs a CUDA device")
    from commander_b200 import sharp
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    fp64 = float(sharp.lib().cmdr_sht_measure_fp64_tflops(4096, 5))
    cd = card()
    try:
        mhz = float(cd.split(",")[-1].split()[0])
    except ValueError:
        mhz = float("nan")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    global ISSUE_RATE
    ISSUE_RATE = sms * ISSUE_PER_SM_CLK * mhz * 1e6          # thread instructions per second at the maximum SM clock
    res = {"card": cd, "fp64_tflops_measured": fp64, "hbm_TB_per_s_datasheet": HBM_TBS, "sms": sms,
           "issue_thread_instr_per_s_at_max_clock": ISSUE_RATE, "configs": []}
    if args.only in (None, "a"):
        res["configs"].append(run_config("a: nside 1024 / lmax 2000 IQU, one band (cmdr_cr_setup)", setup_a, dev, args.reps, fp64))
    if args.only in (None, "b"):
        res["configs"].append(run_config("b: 30 IQU bands, nside 512 / lmax 1500, one CMB component (cmdr_cr_setup_multi)",
                                         setup_b, dev, args.reps, fp64))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r09_cr_rhs_draw_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
