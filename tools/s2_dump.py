#!/usr/bin/env python
"""s2_dump.py -- spin-2 outputs of one source tree, for comparing two builds output for output.

  python tools/s2_dump.py dump TREE OUTDIR   SHARP_Y maps (route on, second call so that the seed tables are in use) and
                                             SHARP_YtW a_lm of seeded standard-normal inputs, built in TREE, at nside 2048 /
                                             lmax 4000, 256 / 37 and 512 / 700, as OUTDIR/{Y,YtW}_<nside>.npy
  python tools/s2_dump.py cmp DIR_A DIR_B    whether each pair is bit-identical, and its relative L2 difference

The synthesis of two builds whose accumulation chains are the same fma sequences must agree bit for bit; the analysis
adds with atomics and agrees to rounding only."""
import os
import sys

import numpy as np

SIZES = ((2048, 4000), (256, 37), (512, 700))


def dump(root, out):
    sys.path.insert(0, os.path.abspath(root))
    import torch
    from commander_b200 import sharp
    if not os.path.abspath(sharp.__file__).startswith(os.path.abspath(root)):
        raise SystemExit(f"imported {sharp.__file__}, not the tree {root}")
    os.makedirs(out, exist_ok=True)
    for nside, lmax in SIZES:
        ai = sharp.sharp_make_mmajor_real_packed_alm_info(lmax)
        gi = sharp.sharp_make_healpix_geom_info(nside)
        rng = np.random.default_rng(1234 + nside)
        alm = torch.from_numpy(rng.standard_normal((2, ai.n_local))).cuda()
        mp = torch.empty((2, gi.n_local), dtype=torch.float64, device="cuda")
        sharp.sharp_execute(sharp.SHARP_Y, 2, 2, alm, ai, mp, gi)
        sharp.sharp_execute(sharp.SHARP_Y, 2, 2, alm, ai, mp, gi)
        back = torch.empty_like(alm)
        sharp.sharp_execute(sharp.SHARP_YtW, 2, 2, back, ai, mp, gi)
        torch.cuda.synchronize()
        np.save(os.path.join(out, f"Y_{nside}.npy"), mp.cpu().numpy())
        np.save(os.path.join(out, f"YtW_{nside}.npy"), back.cpu().numpy())
        sharp.sharp_destroy_alm_info(ai)
        sharp.sharp_destroy_geom_info(gi)


def cmp(a, b):
    for nside, _ in SIZES:
        for k in ("Y", "YtW"):
            x, y = np.load(os.path.join(a, f"{k}_{nside}.npy")), np.load(os.path.join(b, f"{k}_{nside}.npy"))
            same = bool(np.array_equal(x.view(np.int64), y.view(np.int64)))
            print(f"{k} nside {nside}: bit-identical {same} rel_l2 {np.linalg.norm(x - y) / np.linalg.norm(x):.3e}")


if __name__ == "__main__":
    if len(sys.argv) != 4 or sys.argv[1] not in ("dump", "cmp"):
        raise SystemExit(__doc__)
    (dump if sys.argv[1] == "dump" else cmp)(sys.argv[2], sys.argv[3])
