"""Throughput of the conviqt sampler (cmdr_sht_conviqt_interp) at nside 1024 / bmax 8, and the time to build it.

  python tools/conviqt_interp_bench.py --out DIR                                     (one GPU: samples/s and build time)
  python -m torch.distributed.run --nproc-per-node N tools/conviqt_interp_bench.py --out DIR        (build time on N)

Two sample streams of --n samples (default 1e8), both in device memory: scan-ordered (consecutive pixels along the
rings, slowly varying psi: what one detector scan looks like) and uniformly random pixels and angles.  Each rate is
CUDA events around --calls calls after two warm-up calls; every call ends in its stream synchronise, as in use.  The
table (805 MB) is larger than L2.  Beside each rate: the algorithmic bytes per sample (4 pix + 4 psi + 4 out + 4 per
table read: 2 reads for linear interpolation, 1 for the nearest bin) over the time, and that as a share of the B200's
7.7 TB/s HBM data-sheet bandwidth.  The numpy mirror (comm_conviqt.interp on a host cube) gives the CPU reference rate
on 1e6 samples of each stream.  The build time is a host clock around make_sampler (which ends in a synchronise), from a
device cube and from a host cube, after one warm-up build; on N GPUs the slowest rank's time.  Writes
DIR/conviqt_interp_bench[_nN].json with the card name and power limit read in the same run."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12     # B/s, one B200 (data sheet)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def make_conviqt(comm, nside, lmax, bmax, device, seed):
    from commander_b200 import comm_map, comm_mapinfo
    from commander_b200.comm_conviqt import comm_conviqt
    info = comm_mapinfo(comm, nside, lmax, 1, False)
    rng = np.random.default_rng(seed)
    sky, beam = comm_map(info), comm_map(info)
    sky.alm[...] = rng.standard_normal(sky.alm.shape)
    beam.alm[...] = rng.standard_normal(beam.alm.shape) / (1.0 + info.lm[0])
    return comm_conviqt(nside, lmax, 1, bmax, beam, sky, device=device)


def build_seconds(cv, reps, barrier=None):
    import torch
    cv.make_sampler().close()                               # warm-up
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        if barrier:
            barrier()
        t0 = time.perf_counter()
        s = cv.make_sampler()
        ts.append(time.perf_counter() - t0)
        s.close()
    return ts


def streams(n, npix, dev, seed):
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    i = torch.arange(n, device=dev, dtype=torch.int64)
    scan = ((i + 12345) % npix).to(torch.int32), (0.3 + 2e-6 * i.to(torch.float64)).to(torch.float32)
    rand = (torch.randint(0, npix, (n,), device=dev, generator=g, dtype=torch.int32),
            (-2 * math.pi * torch.rand(n, device=dev, generator=g, dtype=torch.float64)).to(torch.float32))
    return {"scan": scan, "random": rand}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--nside", type=int, default=1024)
    ap.add_argument("--bmax", type=int, default=8)
    ap.add_argument("--lmax", type=int, default=256, help="of the sky and beam (the cube's values do not change the rates)")
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--mirror-n", type=int, default=1_000_000)
    args = ap.parse_args()
    import torch
    from commander_b200 import sharp
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.makedirs(args.out, exist_ok=True)
    res = {"card": card(), "nside": args.nside, "bmax": args.bmax, "world": world,
           "table_bytes": 4 * 2 * args.bmax * 12 * args.nside ** 2}

    if world > 1:
        import torch.distributed as dist
        from commander_b200 import dist as cdist
        dist.init_process_group("nccl", device_id=dev)
        comm = cdist.init_from_torch(dev)
        cv = make_conviqt(comm, args.nside, args.lmax, args.bmax, dev, 7)
        ts = build_seconds(cv, 3, barrier=dist.barrier)
        t = torch.tensor(ts, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["build_s_device_cube"] = t.tolist()
        if dist.get_rank() == 0:
            path = os.path.join(args.out, f"conviqt_interp_bench_n{world}.json")
            with open(path, "w") as f:
                json.dump(res, f, indent=1)
            print(json.dumps(res))
        cdist.destroy(comm)
        dist.destroy_process_group()
        return

    cv = make_conviqt(None, args.nside, args.lmax, args.bmax, dev, 7)
    cvh = make_conviqt(None, args.nside, args.lmax, args.bmax, None, 7)
    res["build_s_device_cube"] = build_seconds(cv, 5)
    res["build_s_host_cube"] = build_seconds(cvh, 3)
    s = cv.make_sampler()
    st = torch.cuda.current_stream()
    npix = cv.npix
    out = torch.empty(args.n, dtype=torch.float32, device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res["rates"] = {}
    for name, (pix, psi) in streams(args.n, npix, dev, 11).items():
        for optim in (0, 2):
            for _ in range(2):
                assert sharp.conviqt_interp(s.handle, pix, psi, optim, out, stream=st.cuda_stream) == 0
            ev0.record(st)
            for _ in range(args.calls):
                sharp.conviqt_interp(s.handle, pix, psi, optim, out, stream=st.cuda_stream)
            ev1.record(st)
            ev1.synchronize()
            sec = ev0.elapsed_time(ev1) / 1e3 / args.calls
            nbytes = args.n * (12 + 4 * (1 if optim == 2 else 2))
            # the mirror on the host, on the first mirror_n samples of the same stream
            cvh.optim = optim
            p_h, q_h = pix[:args.mirror_n].cpu().numpy(), psi[:args.mirror_n].cpu().numpy()
            cvh.interp(p_h[:1000], q_h[:1000])
            t0 = time.perf_counter()
            ref = cvh.interp(p_h, q_h)
            th = time.perf_counter() - t0
            assert np.array_equal(ref.view(np.uint32), out[:args.mirror_n].cpu().numpy().view(np.uint32))
            res["rates"][f"{name}_optim{optim}"] = {
                "ms_per_call": sec * 1e3, "samples_per_s": args.n / sec, "algorithmic_bytes_per_s": nbytes / sec,
                "share_of_hbm_datasheet": nbytes / sec / HBM_PEAK, "mirror_host_samples_per_s": args.mirror_n / th}
    s.close()
    path = os.path.join(args.out, "conviqt_interp_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
