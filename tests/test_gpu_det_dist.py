"""The deterministic mode on 2, 4 and 8 GPUs (skipped with fewer): tests/det_dist_check.py under torchrun.  Bit for bit:
the rank-order all-reduce, repeated analyses in both exchange modes, device against pinned / pageable arrays through the
chunked distributed pipeline, and two draw-and-solve runs of a multi-component system (x and hist, hist on every rank)."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("world", [2, 4, 8])
def test_deterministic_distributed(shtlib, world):
    import torch
    n = torch.cuda.device_count()
    if n < world:
        pytest.skip(f"needs >= {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "det_dist_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "DET_DIST_CHECK_OK" in out.stdout
