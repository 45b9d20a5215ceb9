"""Cost of count_distinct in the sharded step: a pa_comm of world size 1 on one GPU, synthetic device columns
(pab.synth), for two value distributions — (a) int64 values floor(v * 1000), about 1000 distinct per group, and (b) the
synthetic fp64 values themselves, where every value is distinct and the distinct pairs D are about the rows.  For each:
per-step time (host clock around the synchronous step), pa_comm_last_phases, the pairs sent / received and the set's
slots (pa_comm_last_distinct), and the single-GPU count_distinct (pa_groupby_aggregate) on the same data, alternating
step by step.  Prints one JSON line per distribution with the card's name and power limit read in the same run, and
writes the list to out.json when a path is given.
python scripts/prof_sharded_distinct.py [rows] [groups] [steps] [warmup] [out.json]"""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import pandasarrow_b200 as pab
from pandasarrow_b200 import distributed as D

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000_000
G = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
warmup = int(sys.argv[4]) if len(sys.argv) > 4 else 1
out_path = sys.argv[5] if len(sys.argv) > 5 else None


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t0) * 1e3


torch.cuda.set_device(0)
dist.init_process_group("gloo", store=dist.FileStore(os.path.join(tempfile.mkdtemp(), "s"), 1), rank=0, world_size=1)
comm = D.Comm(device=0)
gpu = card()
lines = []
k = torch.empty(n, dtype=torch.int64, device="cuda")
pab.synth.keys(k, G, 0)
dk = pab.DeviceColumn.from_torch(k)
gb = pab.GroupBy("k", {"k": dk}, expected_groups=G)
for dist_name in ("a: int64, ~1000 distinct per group", "b: fp64, all distinct"):
    v = torch.empty(n, dtype=torch.float64, device="cuda")
    pab.synth.vals(v, 0)
    if dist_name.startswith("a"):
        v = torch.floor(v * 1000).to(torch.int64)
    torch.cuda.synchronize()
    dv = pab.DeviceColumn.from_torch(v)
    step_ms, single_ms, phases = [], [], []
    info = {}
    for it in range(warmup + steps):
        m, dt = timed(lambda: comm.sharded_aggregate(gb, dv, ["count_distinct"]))
        ph, info = comm.phases(), comm.distinct_info()
        m.close()
        _, ds = timed(lambda: gb.aggregate(dv, ["count_distinct"], fetch=False))
        if it >= warmup:
            step_ms.append(dt); phases.append(ph); single_ms.append(ds)
    line = {"rows": n, "groups": G, "values": dist_name, "step_ms_median": float(np.median(step_ms)),
            "step_ms_min": float(np.min(step_ms)),
            "phases_ms_median": {key: float(np.median([p[key] for p in phases])) for key in phases[0]},
            "single_gpu_count_distinct_ms_median": float(np.median(single_ms)), **info, "steps": steps, "gpu": gpu}
    print(json.dumps(line), flush=True)
    lines.append(line)
    del v, dv
    torch.cuda.empty_cache()
gb.close()
comm.close()
dist.destroy_process_group()
if out_path:
    with open(out_path, "w") as f:
        json.dump(lines, f, indent=1)
