"""Cost of a utf8 key in the sharded step: a large_utf8 key column on the device over 1 B rows, words of a fixed width L
(8 or 24 bytes), so that the column is one device gather (offsets = L * i) with no per-byte index, at 1000 and 1 M
distinct words; an fp64 value without nulls; a pa_comm of world size 1 on one GPU.  For sum / mean / count and
mean / variance / stddev it reports, per step: the step time (host clock around the synchronous step),
pa_comm_last_phases, the key bytes sent and received and the attempts (pa_comm_last_key_strings), the single-GPU
aggregate of the same handle alternated with the step, and the same step on an int64 key of the same cardinality — the
difference is what carrying the strings costs.  Prints JSON lines with the card's name and power limit read in the
same run.  python scripts/prof_sharded_strkeys.py [rows] [steps] [warmup] [out.json]"""
import ctypes as C
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
from pandasarrow_b200 import _lib
from pandasarrow_b200 import distributed as D
from pandasarrow_b200.groupby import _check, _options

n = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000_000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
warmup = int(sys.argv[3]) if len(sys.argv) > 3 else 2
out_path = sys.argv[4] if len(sys.argv) > 4 else None
AGG_SETS = [["sum", "mean", "count"], ["mean", "variance", "stddev"]]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def device_string_handle(offsets, data, n_rows):
    """pa_groupby_create on a large_utf8 column whose offsets and bytes are device tensors (borrowed)."""
    L = _lib.load()
    dev, sc = _lib.ArrowDeviceArray(), _lib.ArrowSchema()
    bufs = (C.c_void_p * 3)(None, offsets.data_ptr(), data.data_ptr())
    fmt = C.c_char_p(b"U")
    a = dev.array
    a.length, a.null_count, a.offset, a.n_buffers, a.n_children = n_rows, 0, 0, 3, 0
    a.buffers = C.cast(bufs, C.POINTER(C.c_void_p))
    dev.device_id, dev.device_type = 0, _lib.ARROW_DEVICE_CUDA
    sc.format, sc.name, sc.flags = fmt, b"", 2
    h = C.c_void_p()
    opt = _options(0, "auto", 0, None)
    _check(L.pa_groupby_create(C.byref(dev), C.byref(sc), 1, C.byref(opt), C.byref(h)))
    gb = pab.GroupBy(None, _handle=h)
    gb._keep = (bufs, fmt, offsets, data)
    return gb


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


torch.cuda.set_device(0)
dist.init_process_group("gloo", store=dist.FileStore(os.path.join(tempfile.mkdtemp(), "s"), 1), rank=0, world_size=1)
comm = D.Comm(device=0)
gpu = card()
v = torch.empty(n, dtype=torch.float64, device="cuda")
pab.synth.vals(v, 0)
dv = pab.DeviceColumn.from_torch(v)
lines = []
for G in (1000, 1_000_000):
    ik = torch.empty(n, dtype=torch.int64, device="cuda")
    pab.synth.keys(ik, G, 0)
    for width in (8, 24):
        table = torch.tensor(np.frombuffer(b"".join(f"w{i:0{width - 1}d}".encode() for i in range(G)), dtype=np.uint8).reshape(G, width),
                             device="cuda")
        data = table.index_select(0, ik).reshape(-1)             # one gather: row i's bytes at [L i, L (i + 1))
        offsets = torch.arange(n + 1, dtype=torch.int64, device="cuda") * width
        gb = device_string_handle(offsets, data, n)
        gi = pab.GroupBy("k", {"k": pab.DeviceColumn.from_torch(ik)})
        for aggs in AGG_SETS:
            t = {"str_step": [], "single_gpu_aggregate": [], "int64_step": []}
            phases, ks = [], []
            for it in range(warmup + steps):
                dt, m = timed(lambda: comm.sharded_aggregate(gb, dv, aggs))
                groups = m.groupSize()
                m.close()
                if it >= warmup:
                    t["str_step"].append(dt)
                    phases.append(comm.phases())
                    ks.append({**comm.key_strings_info(), "unordered": comm.exchange_info()["unordered_export"]})
                dt, _ = timed(lambda: gb.aggregate(dv, aggs, fetch=False))
                if it >= warmup:
                    t["single_gpu_aggregate"].append(dt)
                dt, m = timed(lambda: comm.sharded_aggregate(gi, dv, aggs))
                m.close()
                if it >= warmup:
                    t["int64_step"].append(dt)
            line = {"rows": n, "groups": groups, "word_bytes": width, "aggs": ",".join(aggs), "steps": steps,
                    **{k + "_ms_median": float(np.median(x)) for k, x in t.items()},
                    "str_step_ms_min": float(np.min(t["str_step"])),
                    "phases_ms_median": {k: float(np.median([p[k] for p in phases])) for k in phases[0]},
                    "key_bytes_sent": ks[-1]["bytes_sent"], "key_bytes_received": ks[-1]["bytes_received"],
                    "attempts": max(k["attempts"] for k in ks), "seed": ks[-1]["seed"],
                    "unordered_export": ks[-1]["unordered"], "gpu": gpu}
            print(json.dumps(line), flush=True)
            lines.append(line)
        gb.close()
        gi.close()
        del data, offsets, table
        torch.cuda.empty_cache()
    del ik
comm.close()
dist.destroy_process_group()
if out_path:
    with open(out_path, "w") as f:
        json.dump(lines, f, indent=1)
