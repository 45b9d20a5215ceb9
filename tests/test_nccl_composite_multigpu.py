"""Composite keys across real NCCL ranks: torchrun with 2 ranks (one per GPU), where only rank 1's shard has null keys,
so the ranks' own key layouts differ and the step has to agree on one.  The gathered result of the C-ABI communicator
and of distributed.py's sharded step is compared with the oracle on the whole data set (tests/nccl_composite_worker.py).
Needs 2 GPUs; skipped on a single-GPU box."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2])
def test_nccl_composite_ranks_match_oracle(world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29551", os.path.join(ROOT, "tests", "nccl_composite_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0 and "NCCL COMPOSITE PARITY OK" in r.stdout
