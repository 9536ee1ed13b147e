"""SHARP_ALM2MAP_DERIV1 on 2, 4 and 8 GPUs (skipped with fewer than 2): tests/deriv_dist_check.py under torchrun, both
exchange modes, device / pinned / pageable arrays, against the single-GPU maps and the CPU oracle."""
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
def test_deriv1_distributed(shtlib, cpu_oracle, world):
    import torch
    n = torch.cuda.device_count()
    if n < world:
        pytest.skip(f"needs >= {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "deriv_dist_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "DERIV_DIST_CHECK_OK" in out.stdout
