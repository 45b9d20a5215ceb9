"""Full dense pass against the sum-only pass of a handle whose groups are known (csrc/lowcard_known.cuh), on the bench's
headline workload: int64 keys over 1000 dense groups and fp64 values from pa_synth_*, sum / mean / count, one handle.
Rounds alternate the two (PA_LC_NO_KNOWN=1 forces the full pass); each round queues `passes` deferred passes like
bench.py's steps and times them with CUDA events around the stream, then reads the last pass's scan time
(pa_groupby_last_timing).  Also times the handle's first pass (the one that records the facts) on a fresh handle, and
checks that both kinds of pass give the same bits.  Writes one JSON line, with the card's name and power limit read in
the same run, to <out_dir>/prof_lowcard_known.json.
python scripts/prof_lowcard_known.py [out_dir] [rows] [rounds] [passes]"""
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pandasarrow_b200 as pab

out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
rows = int(sys.argv[2]) if len(sys.argv) > 2 else 1_000_000_000
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 7
passes = int(sys.argv[4]) if len(sys.argv) > 4 else 10
GROUPS = 1000
AGGS = ["sum", "mean", "count"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip()


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def outputs(gb):
    return {a: np.asarray(gb.fetch(a).to_numpy(zero_copy_only=False)).tobytes() for a in AGGS}


def main():
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    keys = torch.empty(rows, dtype=torch.int64, device=dev)
    vals = torch.empty(rows, dtype=torch.float64, device=dev)
    pab.synth.keys(keys, GROUPS, 0)
    pab.synth.vals(vals, 0)
    torch.cuda.synchronize()
    dk, dv = pab.DeviceColumn.from_torch(keys), pab.DeviceColumn.from_torch(vals)

    def first_pass():
        with pab.GroupBy("k", {"k": dk}, stream=stream.cuda_stream) as h:
            h.aggregate(dv, AGGS, fetch=False)
            return h.timing()

    first_pass()                                            # (module load, allocator)
    firsts = [first_pass() for _ in range(3)]

    gb = pab.GroupBy("k", {"k": dk}, stream=stream.cuda_stream)
    gb.aggregate(dv, AGGS, fetch=False)                     # records the facts
    step = {"full": [], "known": []}
    scan = {"full": [], "known": []}
    modes = {}
    bits = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for r in range(rounds):
        for kind in (("full", "known") if r % 2 == 0 else ("known", "full")):
            if kind == "full":
                os.environ["PA_LC_NO_KNOWN"] = "1"
            else:
                os.environ.pop("PA_LC_NO_KNOWN", None)
            gb.aggregate(dv, AGGS, fetch=False, wait=False)   # warm this kind
            gb.sync()
            torch.cuda.synchronize()
            e0.record(stream)
            for _ in range(passes):
                gb.aggregate(dv, AGGS, fetch=False, wait=False)
            e1.record(stream)
            t = gb.timing()
            torch.cuda.synchronize()
            step[kind].append(e0.elapsed_time(e1) / passes)
            scan[kind].append(t["scan_ms"])
            modes[kind] = t["mode"]
            bits.setdefault(kind, outputs(gb))
    os.environ.pop("PA_LC_NO_KNOWN", None)
    gb.close()
    line = {
        "card": card(), "rows": rows, "groups": GROUPS, "aggs": AGGS, "rounds": rounds, "passes_per_round": passes,
        "modes": modes, "same_bits": bits["full"] == bits["known"],
        "step_ms": {k: spread(v) for k, v in step.items()},
        "scan_ms": {k: spread(v) for k, v in scan.items()},
        "first_pass": {"total_ms": spread([t["total_ms"] for t in firsts]), "scan_ms": spread([t["scan_ms"] for t in firsts]),
                       "mode": firsts[0]["mode"]},
        "step_gain": 1.0 - statistics.median(step["known"]) / statistics.median(step["full"]),
        "scan_gain": 1.0 - statistics.median(scan["known"]) / statistics.median(scan["full"]),
    }
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "prof_lowcard_known.json"), "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
