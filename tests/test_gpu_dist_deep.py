"""The distributed transforms value by value against the single-GPU path (tests/dist_deep_check.py under torchrun) on
2, 3 and 8 GPUs (each skipped when fewer are visible): four rank layouts (comm_mapinfo's round robin, ranks without
rings or m's, a scrambled subset of the sphere, pairs split between ranks), device / pinned / pageable arrays, fused and
NCCL exchange, sharp_execute (spins 0, 2 and 1, 3, 17, 32) and execute_iqu, Y / WY / Yt / YtW and the add forms, up
to the size that takes the chunked host pipeline.  Synthesis must be bit-identical to the single-GPU maps wherever
every ring pair belongs to one rank.  At the largest world the box can run, nside 2048 / lmax 4000 and a probe run
against the mpmath reference (slam_ref) are added, and a second launch with the NCCL stream barrier and 3 pipeline
chunks (both switches are read once per process) must reproduce the first launch's maps bit for bit.
Run with -s to see one line per (layout, size, path, job)."""
import json
import os
import signal
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORLDS = [2, 3, 8]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _launch(world, env, timeout):
    """torchrun in its own process group: on timeout the whole group is killed, so that no rank is left behind."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "dist_deep_check.py")]
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, cwd=ROOT,
                         env=dict(os.environ, **env), start_new_session=True)
    try:
        out, _ = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)
        out, _ = p.communicate()
        pytest.fail(f"world {world} timed out after {timeout} s:\n" + out[-6000:])
    print(out)
    assert p.returncode == 0, out[-6000:]
    assert f"DIST_DEEP_OK world={world}" in out, out[-6000:]
    return out


def _digests(prefix, world):
    d = []
    for r in range(world):
        with open(f"{prefix}.rank{r}.json") as f:
            d.append(json.load(f))
    return d


@pytest.mark.parametrize("world", WORLDS)
def test_distributed_deep(shtlib, world, tmp_path):
    import torch
    n = torch.cuda.device_count()
    if n < world:
        pytest.skip(f"needs >= {world} GPUs")
    largest = world == max(w for w in WORLDS if w <= n)
    first = str(tmp_path / "default")
    _launch(world, {"DIST_DEEP_LARGEST": "1" if largest else "0", "DIST_DEEP_SAVE": first},
            3000 if largest else 1500)
    if not largest:
        return
    second = str(tmp_path / "nccl_barrier_3_chunks")
    _launch(world, {"DIST_DEEP_LARGEST": "0", "DIST_DEEP_SAVE": second, "CMDR_SHT_FLAG_BARRIER": "0",
                    "CMDR_SHT_DIST_CHUNKS": "3"}, 1500)
    a, b = _digests(first, world), _digests(second, world)
    for r in range(world):
        assert b[r], f"rank {r} saved no maps"
        diff = [k for k in b[r] if a[r].get(k) != b[r][k]]
        assert not diff, f"rank {r}: {len(diff)} synthesis results differ between the launches, e.g. {diff[:5]}"
