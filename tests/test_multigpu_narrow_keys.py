"""Narrow keys through lsb_sort_device_typed on 2/4/8 GPUs: one process per GPU under torchrun, each rank passes its
shard and checks its slice of the global stable sort (tests/mgpu_narrow_keys_worker.py).  Skipped below the number of
GPUs a case needs."""
import os
import subprocess
import sys

import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multigpu_narrow_keys(world):
    if _ngpus() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29660 + world),
           os.path.join(ROOT, "tests", "mgpu_narrow_keys_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("multi-GPU narrow-key sort ok") == world
