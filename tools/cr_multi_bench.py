"""Time the native multi-component constrained-realisation solve (cmdr_cr_setup_multi) against the torch mirror
comm_cr.cr_system on the sampling group of tests/test_gpu_cr_multi_native.py::real_size_problem: bands (nside / lmax)
512 / 1500, 1024 / 2000, 1024 / 2000; components CMB (3 maps, lmax 2000, prior), dust (3, 1500, prior) and a 1-map
low-l component without prior.  With --pixel-F the dust component is mixed per pixel in every band
(cmdr_cr_set_mixing_map; the mirror gets the same maps) and the result goes to cr_mix_bench[_nN].json.  With
--precond pseudoinv both solvers use the pseudo-inverse preconditioner (cmdr_cr_set_pseudoinv on the native handle,
precond = 'pseudoinv' on the mirror), the switch's setup time is recorded, and the result goes to
cr_pinv_bench[_nN].json.  Either preconditioner also records the iterations (and time) to cg_tol = 1e-8 in 'residual'
mode, which with the per-iteration rate settles what a preconditioner buys on this group.

  python tools/cr_multi_bench.py --out DIR [--pixel-F] [--precond {diagonal,pseudoinv}]     (one GPU)
  python -m torch.distributed.run --nproc-per-node N tools/cr_multi_bench.py --out DIR

Each solve runs `fixed_iter` iterations after a warm-up solve and is timed with CUDA events around work that ends in a
synchronise.  A separate torch.profiler run gives the kernel time of the gathers and of the block-preconditioner apply,
and their GB/s from the bytes the shapes imply.  Writes DIR/cr_multi_bench[_nN].json with the card name, power limit
and maximum SM clock read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def nalm(lmax, ms):
    return int(sum((lmax + 1 - m) * (1 if m == 0 else 2) for m in ms if m <= lmax))


def kernel_bytes(comps, bands, ms, mixed=()):
    """Bytes each new kernel moves per CG iteration (one matmulA + one preconditioner apply), from the shapes.  `mixed`:
    the (band, component) pairs mixed per pixel, whose band-gather input is their buffer at the band's L_q."""
    lmax_pre = max(c["lmax"] for c in comps)
    L = [min(b["lmax"], lmax_pre) for b in bands]
    bnm = [b.get("nmaps", 3) for b in bands]
    band = sum(8 * (bnm[q] * nalm(L[q], ms) + sum(min(c["nmaps"], bnm[q]) * nalm(L[q] if (q, k) in mixed else min(c["lmax"], L[q]), ms)
                                                  for k, c in enumerate(comps)))
               for q in range(len(bands)))
    comp = sum(8 * (c["nmaps"] * nalm(c["lmax"], ms) * (2 if c["Cl"] is not None else 1)
                    + sum(min(c["nmaps"], bnm[q]) * nalm(min(c["lmax"], L[q]), ms) for q in range(len(bands))))
               for c in comps)
    npre, nmaps_pre = len(comps), max(c["nmaps"] for c in comps)
    pre = 8 * (npre * (npre + 1) // 2 * nmaps_pre * nalm(lmax_pre, ms) + 2 * sum(c["nmaps"] * nalm(c["lmax"], ms) for c in comps))
    return {"k_cr_band_gather": band, "k_cr_comp_gather": comp, "k_cr_pre_apply": pre}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--mirror-iters", type=int, default=10)
    ap.add_argument("--pixel-F", action="store_true", help="mix the dust component per pixel in every band")
    ap.add_argument("--precond", choices=("diagonal", "pseudoinv"), default="diagonal",
                    help="block-diagonal (default) or pseudo-inverse preconditioner")
    ap.add_argument("--residual-maxiter", type=int, default=2000,
                    help="iteration cap of the 'residual' solve to cg_tol = 1e-8 (0: skip it)")
    args = ap.parse_args()
    import torch
    from commander_b200 import comm_mapinfo
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, cr_system, solve_cr_eqn_by_CG
    from test_gpu_cr_multi_native import real_size_problem
    if not torch.cuda.is_available():
        sys.exit("cr_multi_bench: needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    comm = None
    rank = 0
    if world > 1:
        import torch.distributed as dist
        from commander_b200 import dist as cdist
        dist.init_process_group("nccl", device_id=dev)
        rank = dist.get_rank()
        comm = cdist.init_from_torch(dev)
    bands, comps = real_size_problem(np.random.default_rng(15))
    binfo = [comm_mapinfo(comm, b["nside"], b["lmax"], 3, True) for b in bands]
    cb = [cr_band(i, torch.as_tensor(np.ascontiguousarray(b["invN"][:, i.pix]), device=dev), b["b_l"]) for i, b in zip(binfo, bands)]
    mixed = ()
    if args.pixel_F:                                            # dust, F_mean times a smooth-ish per-pixel factor
        frng = np.random.default_rng(17)
        comps[1]["F"] = [torch.as_tensor(np.ascontiguousarray((f[0] * (1.0 + 0.3 * frng.uniform(size=(3, 12 * b["nside"] ** 2))))[:, i.pix]),
                                         device=dev) for f, b, i in zip(comps[1]["F_mean"], bands, binfo)]
        mixed = tuple((q, 1) for q in range(len(bands)))
    cc = [cr_component(comm_mapinfo(comm, c["nside"], c["lmax"], c["nmaps"], c["nmaps"] == 3), Cl=c["Cl"], F_mean=c["F_mean"],
                       F=c.get("F")) for c in comps]
    nat = cr_native_multi_system(cc, cb, pixel_mixing=args.pixel_F)
    rng = np.random.default_rng(16)
    data = [torch.as_tensor(rng.standard_normal((3, i.np)), device=dev) for i in binfo]
    b = nat.computeRHS(data)
    setup_ms = None
    if args.precond == "pseudoinv":                             # the call synchronises: a host clock is exact here
        import time
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        nat.set_pseudoinv(True)
        setup_ms = 1e3 * (time.perf_counter() - t0)

    def timed(fn, n):
        fn(2)                                                   # warm-up: every shape of the timed window
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(n)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    ms_nat = timed(lambda n: nat.solve(b, maxiter=n, cg_conv_crit="fixed_iter"), args.iters)
    res = {"world": world, "card": card(), "precond": args.precond, "iters_native": args.iters,
           "native_ms_per_iter": ms_nat / args.iters, "native_iter_per_s": 1e3 * args.iters / ms_nat}
    if setup_ms is not None:
        res["pseudoinv_setup_ms"] = setup_ms
    if args.residual_maxiter > 0:
        # a data-like right-hand side: noise-weighted white data, so the residual solve sees the signal-to-noise of a
        # real run rather than the unit-variance maps of the timing loop
        dres = [torch.as_tensor(rng.standard_normal((3, i.np)), device=dev) / torch.sqrt(c.invN) for i, c in zip(binfo, cb)]
        bres = nat.computeRHS(dres)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _, it_res, _ = nat.solve(bres, maxiter=args.residual_maxiter, cg_tol=1e-8, cg_conv_crit="residual")
        e1.record()
        torch.cuda.synchronize()
        res.update(residual_cg_tol=1e-8, residual_iters=it_res, residual_ms=e0.elapsed_time(e1),
                   residual_maxiter=args.residual_maxiter)
    if args.mirror_iters > 0:
        mir = cr_system(cc, cb, dev, precond=args.precond)
        ms_mir = timed(lambda n: solve_cr_eqn_by_CG(mir, b.clone(), maxiter=n, cg_conv_crit="fixed_iter"), args.mirror_iters)
        res.update(iters_mirror=args.mirror_iters, mirror_ms_per_iter=ms_mir / args.mirror_iters,
                   mirror_iter_per_s=1e3 * args.mirror_iters / ms_mir)
        del mir
    # kernel share, profiler on, separate run
    from torch.profiler import ProfilerActivity, profile
    nat.solve(b, maxiter=2, cg_conv_crit="fixed_iter")
    torch.cuda.synchronize()
    nprof = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        nat.solve(b, maxiter=nprof, cg_conv_crit="fixed_iter")
        torch.cuda.synchronize()
    tot, per = 0.0, {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        tot += t
        for k in ("k_cr_band_gather", "k_cr_comp_gather", "k_cr_pre_apply", "k_cr_mix_pack", "k_cr_pinv_prior"):
            if k in ev.name:
                per[k] = per.get(k, 0.0) + t
    ms_local = cc[0].x_info.ms                                  # the largest lmax: every local m
    nbytes = kernel_bytes(comps, bands, ms_local, mixed)
    iters = nprof + 1                                           # the solve's matmulA / precond count: one extra at the start
    kern = {}
    for k, us in per.items():
        kern[k] = {"ms_per_iter": us / 1e3 / iters}
        if k in nbytes and args.precond == "diagonal":       # the byte model counts one gather pass per iteration
            kern[k].update(GB_per_iter=nbytes[k] / 1e9, GB_per_s=nbytes[k] / (us / 1e6 / iters) / 1e9 if us > 0 else None)
    res["kernels"] = kern
    res["pixel_F"] = [f"dust in band {q}" for q, _ in mixed]
    res["profiled_gpu_ms_per_iter"] = tot / 1e3 / iters
    res["new_kernel_share"] = sum(per.values()) / tot if tot > 0 else None
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        name = "cr_mix_bench" if args.pixel_F else ("cr_pinv_bench" if args.precond == "pseudoinv" else "cr_multi_bench")
        path = os.path.join(args.out, f"{name}.json" if world == 1 else f"{name}_n{world}.json")
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))
    if world > 1:
        import torch.distributed as dist
        from commander_b200 import dist as cdist
        cdist.destroy(comm)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
