"""utf8 keys across real NCCL ranks: torchrun with 2 ranks (one per GPU), through the C-ABI communicator and through
distributed.py, compared with the oracle on the whole column (tests/nccl_strkeys_worker.py); and the collision hook
across two real ranks, where both ranks retry with seed 1.  Needs 2 GPUs; skipped on a single-GPU box."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("hook", [False, True])
def test_nccl_strkeys_ranks_match_oracle(hook):
    import torch
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29553" if hook else "29552", os.path.join(ROOT, "tests", "nccl_strkeys_worker.py")] + (["--hook"] if hook else [])
    env = dict(os.environ, **({"PA_TEST_STR_HASH_BITS": "0"} if hook else {}))
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    print(r.stdout[-4000:], r.stderr[-4000:])
    assert r.returncode == 0 and "NCCL STRKEYS PARITY OK" in r.stdout
