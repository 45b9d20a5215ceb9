"""Cost of product / variance / stddev in the sharded step: a pa_comm of world size 1 on one GPU, synthetic device
columns (pab.synth), per-step time (host clock around the synchronous step) and pa_comm_last_phases for
["sum", "mean", "count"] (compact records) against ["mean", "variance", "stddev"] and ["product"] (stage-2 records), at
each group count.  The aggregate sets alternate step by step so that all see the same machine state.  Prints one JSON
line per (groups, aggregates) with the card's name and power limit read in the same run, and writes the list to
out.json when a path is given.
python scripts/prof_sharded_stage2.py [rows] [groups,groups,...] [steps] [warmup] [out.json]"""
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
groups = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1000,1000000").split(",")]
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
warmup = int(sys.argv[4]) if len(sys.argv) > 4 else 2
out_path = sys.argv[5] if len(sys.argv) > 5 else None
SETS = {"sum,mean,count": ["sum", "mean", "count"], "mean,variance,stddev": ["mean", "variance", "stddev"], "product": ["product"]}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


torch.cuda.set_device(0)
dist.init_process_group("gloo", store=dist.FileStore(os.path.join(tempfile.mkdtemp(), "s"), 1), rank=0, world_size=1)
comm = D.Comm(device=0)
gpu = card()
lines = []
for G in groups:
    k = torch.empty(n, dtype=torch.int64, device="cuda")
    v = torch.empty(n, dtype=torch.float64, device="cuda")
    pab.synth.keys(k, G, 0); pab.synth.vals(v, 0)
    v += 0.5                                     # [0.5, 1.5): products of a group stay away from 0
    torch.cuda.synchronize()
    dk, dv = pab.DeviceColumn.from_torch(k), pab.DeviceColumn.from_torch(v)
    gb = pab.GroupBy("k", {"k": dk, "v": dv}, expected_groups=G)
    times = {name: [] for name in SETS}
    phases = {name: [] for name in SETS}
    info = {}
    for it in range(warmup + steps):
        for name, aggs in SETS.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = comm.sharded_aggregate(gb, dv, aggs)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            if it >= warmup:
                times[name].append(dt)
                phases[name].append(comm.phases())
            info[name] = comm.exchange_info()
            m.close()
    for name in SETS:
        ph = {key: float(np.median([p[key] for p in phases[name]])) for key in phases[name][0]}
        line = {"rows": n, "groups": G, "aggs": name, "step_ms_median": float(np.median(times[name])),
                "step_ms_min": float(np.min(times[name])), "steps": steps, "phases_ms_median": ph,
                "record_bytes": info[name]["record_bytes"], "gpu": gpu}
        print(json.dumps(line), flush=True)
        lines.append(line)
    gb.close()
    del k, v, dk, dv
    torch.cuda.empty_cache()
comm.close()
dist.destroy_process_group()
if out_path:
    with open(out_path, "w") as f:
        json.dump(lines, f, indent=1)
