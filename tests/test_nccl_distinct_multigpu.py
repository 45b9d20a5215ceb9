"""count_distinct / all / any across real NCCL ranks: torchrun with 2 ranks (one per GPU); the gathered result of the
C-ABI communicator and of distributed.py's sharded step is compared with the oracle on the whole data set
(tests/nccl_distinct_worker.py).  Needs 2 GPUs; skipped on a single-GPU box."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2])
def test_nccl_distinct_ranks_match_oracle(world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tests", "nccl_distinct_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0 and "NCCL DISTINCT PARITY OK" in r.stdout
