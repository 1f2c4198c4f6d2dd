"""-m gpu, needs >= 2 GPUs on the box (skipped otherwise): the multi-candidate mode compressed across 2 or 4
ranks with distributed.compress_dynamic_sharded (every rank walks its own input range, entry tables folded over
NCCL, fragments assembled on rank 0) gives engine.compress_dynamic_device's body, and
distributed.decompress_sharded decodes that body back to the input."""
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_dynamic_compress_of_one_input(world):
    if _gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_dyn_shard_worker.py")]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    sys.stdout.write(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "DYN SHARD OK" in r.stdout
