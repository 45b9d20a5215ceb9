"""Cost of a hashed composite key (csrc/rowkeys.cuh): two int64 key columns whose tuple needs 128 bits — k1 from
pa_synth_keys_i64, k2 = k1 * (odd constant) + 2^40 — and an fp64 value, all generated on the device, at 1000 groups
over 1 B rows and 1 M groups over 500 M rows.  It reports create (the row hash, host clock to a device synchronise),
the first aggregate (the pass plus the row check against each group's first row), and the steady-state
sum / mean / count per step over K steps (the handle's own CUDA event timing, pa_groupby_last_timing, and the host
clock around the synchronous call), alternated with the same steps on the single int64 key k1 — the same group
structure, the scattered-key baseline.  Writes one JSON line, with the card's name and power limit read in the same
run, to <out_dir>/prof_hashed_keys.json.  python scripts/prof_hashed_keys.py [out_dir] [steps] [warmup]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pandasarrow_b200 as pab

out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
warmup = int(sys.argv[3]) if len(sys.argv) > 3 else 2
AGGS = ["sum", "mean", "count"]
ODD = 0x2545F4914F6CDD1D   # odd: k2 is one value per k1 (int64 wraps)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


torch.cuda.set_device(0)
result = {"gpu": card(), "aggs": ",".join(AGGS), "steps": steps, "warmup": warmup, "cases": []}
for G, n in ((1000, 1_000_000_000), (1_000_000, 500_000_000)):
    k1 = torch.empty(n, dtype=torch.int64, device="cuda")
    pab.synth.keys(k1, G, 0)
    k2 = k1 * ODD + (1 << 40)
    v = torch.empty(n, dtype=torch.float64, device="cuda")
    pab.synth.vals(v, 0)
    dv = pab.DeviceColumn.from_torch(v)
    create_ms, gb = host_ms(lambda: pab.GroupBy(["k1", "k2"], {"k1": pab.DeviceColumn.from_torch(k1), "k2": pab.DeviceColumn.from_torch(k2)}))
    first_ms, _ = host_ms(lambda: gb.aggregate(dv, AGGS, fetch=False))
    assert gb.groupSize() == G and gb.key_hash_seed() == 0
    base = pab.GroupBy("k1", {"k1": pab.DeviceColumn.from_torch(k1)})
    t = {"hashed_event": [], "hashed_host": [], "int64_event": [], "int64_host": []}
    for it in range(warmup + steps):
        for name, h in (("hashed", gb), ("int64", base)):
            dt, _ = host_ms(lambda: h.aggregate(dv, AGGS, fetch=False))
            if it >= warmup:
                t[name + "_host"].append(dt)
                t[name + "_event"].append(h.timing()["total_ms"])
    same = all(gb.fetch(a).equals(base.fetch(a)) for a in ("count",))
    case = {"groups": G, "rows": n, "create_ms": create_ms, "first_aggregate_ms": first_ms, "counts_equal_int64": same,
            **{k + "_ms_median": float(np.median(x)) for k, x in t.items()},
            **{k + "_ms_min": float(np.min(x)) for k, x in t.items()},
            "path": gb.timing()["path"], "mode": gb.timing()["mode"], "int64_mode": base.timing()["mode"]}
    case["hashed_over_int64"] = case["hashed_event_ms_median"] / case["int64_event_ms_median"]
    print(json.dumps(case), flush=True)
    result["cases"].append(case)
    gb.close(); base.close()
    del k1, k2, v, dv
    torch.cuda.empty_cache()
os.makedirs(out_dir, exist_ok=True)
with open(os.path.join(out_dir, "prof_hashed_keys.json"), "w") as f:
    f.write(json.dumps(result) + "\n")
print(json.dumps(result))
