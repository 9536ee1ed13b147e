"""torchrun worker: the deterministic mode (cmdr_sht_set_deterministic) on N GPUs.  Checks bit for bit:
  - cmdr_sht_allreduce_sum: every rank gets the sum of the ranks' values in rank order;
  - repeated YtW / Yt of spin 0 and spin 2 on a comm_mapinfo layout, in both exchange modes, and the two modes against
    each other;
  - device arrays against pinned and pageable ones at a size where the chunked distributed pipeline runs (its Legendre
    launches cut on warp blocks, one ordered reduce per m range before the download);
  - two draw-and-solve runs of a multi-component system (pseudo-inverse preconditioner, so that its alpha sums go through
    the all-reduce too): x on every rank, and the residual history, which must also be the same on every rank.
Launched by tests/test_gpu_det_dist.py (or by hand:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29521 tests/det_dist_check.py)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    from commander_b200 import comm_map, comm_mapinfo, sharp
    from commander_b200 import dist as cdist
    from commander_b200.comm_cr import cr_band, cr_component, cr_native_multi_system, gaussian_beam
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    sharp.set_deterministic(True)
    comm = cdist.init_from_torch(dev)

    def gather(t):
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t.contiguous())
        return [o.cpu() for o in out]

    def same_on_every_rank(t, what):
        g = gather(t)
        assert all(torch.equal(g[0], x) for x in g[1:]), f"{what} differs between ranks"

    # 1. the all-reduce of the CG scalars: gather + sum in rank order
    r = np.random.default_rng(100 + rank)
    v = torch.as_tensor(r.standard_normal(1001) * 10.0 ** r.uniform(-8, 8, 1001), device=dev)
    parts = gather(v)
    want = parts[0].clone()
    for p in parts[1:]:
        want = want + p
    got = comm.allreduce_sum_(v.clone())
    torch.cuda.synchronize()
    assert torch.equal(got.cpu(), want), "allreduce_sum is not the rank-order sum"
    same_on_every_rank(got, "allreduce_sum")

    # 2. transforms: repeated, both exchange modes, device against pinned / pageable arrays (pipelined at this size)
    nside, lmax = 1024, 1500
    info = comm_mapinfo(comm, nside, lmax, 3, True)
    rng = np.random.default_rng(7)                      # identical global map on every rank
    mloc = np.ascontiguousarray(rng.standard_normal((3, 12 * nside ** 2))[:, info.pix])
    res = {}
    for mode in (1, 0):                                 # fused NVLink peer stores, NCCL all-to-all
        comm.set_exchange(mode)
        for job in ("YtW", "Yt"):
            runs = []
            for _ in range(2):
                m = comm_map(info, device=dev)
                m.map.copy_(torch.as_tensor(mloc, device=dev))
                getattr(m, job)()
                torch.cuda.synchronize()
                runs.append(m.alm.cpu())
            assert torch.equal(runs[0], runs[1]), f"{job} exchange {mode}: not repeatable"
            res[(mode, job)] = runs[0]
    for job in ("YtW", "Yt"):
        assert torch.equal(res[(1, job)], res[(0, job)]), f"{job}: the exchange modes differ"
    comm.set_exchange(1)                                # the chunked pipeline rides on the fused exchange
    for kind in ("pinned", "pageable"):
        m = comm_map(info)
        if kind == "pinned":
            m.alm = torch.empty((3, info.nalm), dtype=torch.float64).pin_memory().numpy()
            m.map = torch.empty((3, info.np), dtype=torch.float64).pin_memory().numpy()
        for job in ("YtW", "Yt"):
            m.map[:] = mloc
            getattr(m, job)()
            assert torch.equal(torch.from_numpy(np.array(m.alm)), res[(1, job)]), f"{job} {kind}: differs from device arrays"
    info.dealloc()

    # 3. two draw-and-solve runs of a multi-component system
    def put(a):
        return torch.as_tensor(np.ascontiguousarray(a), device=dev)

    rng = np.random.default_rng(31)
    bspec = [(16, 24, 500.0, 1.0), (32, 40, 300.0, 0.7)]
    binvN = [(1.0 / (s * (1.0 + 0.5 * rng.uniform(size=(3, 12 * ns ** 2))))) ** 2 for ns, _, _, s in bspec]
    datm = [rng.standard_normal((3, 12 * ns ** 2)) for ns, _, _, _ in bspec]
    lc = np.arange(33, dtype=np.float64)
    Clc = np.stack([10.0 / (lc * (lc + 1) + 1.0)] * 3, axis=1)
    binfo = [comm_mapinfo(comm, ns, lm, 3, True) for ns, lm, _, _ in bspec]
    bands = [cr_band(i, put(v[:, i.pix]), gaussian_beam(lm, fw, 3)) for i, v, (_, lm, fw, _) in zip(binfo, binvN, bspec)]
    cinfo = [comm_mapinfo(comm, 32, 32, 3, True), comm_mapinfo(comm, 32, 8, 1, False)]
    comps = [cr_component(cinfo[0], Cl=Clc, F_mean=np.ones((2, 3))),
             cr_component(cinfo[1], Cl=None, F_mean=np.array([[1.5], [0.6]]))]
    data = [put(d[:, i.pix]) for d, i in zip(datm, binfo)]
    sols = []
    for _ in range(2):
        nat = cr_native_multi_system(comps, bands, precond="diagonal")
        nat.set_pseudoinv(True)
        b = nat.computeRHS_draw(data, 0xC0FFEE, 5)
        x, it, hist = nat.solve(b, maxiter=30, cg_conv_crit="fixed_iter")
        torch.cuda.synchronize()
        assert it == 30
        sols.append((x.cpu(), torch.tensor(hist, dtype=torch.float64)))
        del nat
    assert torch.equal(sols[0][0], sols[1][0]), "x differs between two draw-and-solve runs"
    assert torch.equal(sols[0][1], sols[1][1]), "hist differs between two draw-and-solve runs"
    same_on_every_rank(sols[0][1].to(dev), "hist")
    comm.set_exchange(-1)
    if rank == 0:
        print(f"DET_DIST_CHECK_OK world={world}")
    cdist.destroy(comm)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
