"""Cost of composite keys in the sharded step: config 3's key (int32 of 1000 values x dictionary<int32 -> utf8> of 64
symbols, 1 % null keys in each column) over a nullable fp64 value (10 % nulls), a pa_comm of world size 1 on one GPU.
The columns are generated on the device (pab.synth) and handed over as host Arrow arrays (the library copies them to
the device once, when the handle is made).  For sum / mean / count / min / max it reports, per step: the step time
(host clock around the synchronous step), pa_comm_last_phases, the key-layout gather (pa_comm_last_key_layout), and the
single-GPU aggregate of the same handle, alternating step by step.  It also times the one-time repack a rank pays when
its shard of k1 has no nulls and the agreed layout gives k1 a null bit (host clock around set_key_layout on a second
handle, synchronised).  With one rank the gather is an all-gather of one 64-byte layout and nothing is repacked by the
step itself.  Prints JSON lines with the card's name and power limit read in the same run.
python scripts/prof_sharded_composite.py [rows] [steps] [warmup] [out.json]"""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pyarrow as pa
import torch
import torch.distributed as dist

import pandasarrow_b200 as pab
from pandasarrow_b200 import distributed as D

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000_000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
warmup = int(sys.argv[3]) if len(sys.argv) > 3 else 2
out_path = sys.argv[4] if len(sys.argv) > 4 else None
AGGS = ["sum", "mean", "count", "min", "max"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def host_int32(t, bits=None):
    """A device int32 tensor (and optional validity bitmap) as a zero-copy host Arrow array."""
    data = pa.py_buffer(t.cpu().numpy())
    valid = pa.py_buffer(bits.cpu().numpy()) if bits is not None else None
    return pa.Array.from_buffers(pa.int32(), t.numel(), [valid, data], null_count=-1 if bits is not None else 0)


torch.cuda.set_device(0)
dist.init_process_group("gloo", store=dist.FileStore(os.path.join(tempfile.mkdtemp(), "s"), 1), rank=0, world_size=1)
comm = D.Comm(device=0)
gpu = card()
t64 = torch.empty(n, dtype=torch.int64, device="cuda")
pab.synth.keys(t64, 1000, 0)
k1 = t64.to(torch.int32)
pab.synth.keys(t64, 64, 12345)
k2 = t64.to(torch.int32)
del t64
nb = (n + 7) // 8
b1, b2, bv = (torch.empty(nb, dtype=torch.uint8, device="cuda") for _ in range(3))
pab.synth.validity(b1, n, 0, seed=7, null_every=100)
pab.synth.validity(b2, n, 0, seed=8, null_every=100)
pab.synth.validity(bv, n, 0, seed=9, null_every=10)
v = torch.empty(n, dtype=torch.float64, device="cuda")
pab.synth.vals(v, 0)
torch.cuda.synchronize()
dictionary = pa.array([f"sym{i:02d}" for i in range(64)])
a1 = host_int32(k1, b1)
a2 = pa.DictionaryArray.from_arrays(host_int32(k2, b2), dictionary)
dv = pab.DeviceColumn.from_torch(v, valid=bv, null_count=-1)
t0 = time.perf_counter()
gb = pab.GroupBy(["k1", "k2"], {"k1": a1, "k2": a2}, expected_groups=65 * 1001)
torch.cuda.synchronize()
create_ms = (time.perf_counter() - t0) * 1e3
layout = gb.key_layout()
times = {"comm_step": [], "single_gpu_aggregate": []}
phases, agree = [], []
for it in range(warmup + steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m = comm.sharded_aggregate(gb, dv, AGGS)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) * 1e3
    if it >= warmup:
        times["comm_step"].append(dt)
        phases.append(comm.phases())
        agree.append(comm.key_layout_info())
    groups = m.groupSize()
    m.close()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gb.aggregate(dv, AGGS, fetch=False)
    torch.cuda.synchronize()
    if it >= warmup:
        times["single_gpu_aggregate"].append((time.perf_counter() - t0) * 1e3)
single_groups = gb.groupSize()
gb.close()
line = {"rows": n, "groups": groups, "single_gpu_groups": single_groups, "aggs": ",".join(AGGS), "steps": steps,
        "layout": {"bits": list(layout.bits[:2]), "nullable": list(layout.nullable[:2])},
        "step_ms_median": float(np.median(times["comm_step"])), "step_ms_min": float(np.min(times["comm_step"])),
        "single_gpu_aggregate_ms_median": float(np.median(times["single_gpu_aggregate"])),
        "phases_ms_median": {k: float(np.median([p[k] for p in phases])) for k in phases[0]},
        "agree_ms_median": float(np.median([a["agree_ms"] for a in agree])),
        "step_repack_ms": max(a["repack_ms"] for a in agree), "create_ms": create_ms, "gpu": gpu}
print(json.dumps(line), flush=True)
lines = [line]
# the one-time repack of a rank whose k1 shard has no nulls: own layout k1 without a null bit, agreed with one
a1c = host_int32(k1)
repack = []
for it in range(3):
    g2 = pab.GroupBy(["k1", "k2"], {"k1": a1c, "k2": a2})
    wider = g2.key_layout()
    wider.nullable[0] = 1
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    g2.set_key_layout(wider)
    g2.sync()
    torch.cuda.synchronize()
    repack.append((time.perf_counter() - t0) * 1e3)
    g2.close()
line = {"rows": n, "what": "one-time repack (k1 gains its null bit)", "repack_ms": repack, "gpu": gpu}
print(json.dumps(line), flush=True)
lines.append(line)
comm.close()
dist.destroy_process_group()
if out_path:
    with open(out_path, "w") as f:
        json.dump(lines, f, indent=1)
