#!/usr/bin/env python
"""bench.py — group-by aggregation throughput on B200 (BASELINE.json metric).

One "step" = one fused pass of the hot path (stages 1-3 + merge + emit) over one batch of synthetic
rows: int64 key, fp64 value, sum + mean + count, N rows per GPU, G groups.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--rows R] [--groups G] [--sweep] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for how every field is derived.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AGGS = ["sum", "mean", "count"]
SWEEP_AGGS = ["sum", "min", "max", "count"]
SWEEP_G = [16, 256, 4096, 65536, 1 << 20, 1 << 24, 100_000_000]
METRIC = "groupby_agg_rows_per_s"
UNIT = "rows/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU")
    ap.add_argument("--groups", type=int, default=1000)
    ap.add_argument("--sweep", action="store_true", help="(default at N=1) config-2 cardinality sweep, device resident")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--config5-groups", type=int, default=100_000_000, help="N>1: groups of the config-5 extra (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--sm-reserve", type=int, default=-1, help="SMs the scan leaves free (pa_options.sm_reserve; default 0: measured slower at N=2 — 3.57 / 3.59 / 3.61 / 3.65 ms per step with 0 / 1 / 2 / 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-rows", type=int, default=100_000_000, help="rows of the bounded CPU-baseline sample")
    ap.add_argument("--extras", action="store_true", help="(default at N=1) config 3 (multi-key, nullable), config 4 (resample OHLC), scattered keys, ...")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (group keys and one array "
                    "per aggregate) to DIR/<name>.npy as float64; a fixed seeded sample of the groups beyond 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must be at least 0")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def _source_sha(rel: str) -> str:
    import hashlib
    return hashlib.sha256(open(os.path.join(ROOT, rel), "rb").read()).hexdigest()[:16]


def measured_traffic(kernel: str, n_rows: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the committed
    `ncu --set full` capture (profiles/r2_traffic.json); scaled linearly when the capture used another row count.
    The capture is stamped with the hash of the kernel's source file: a stale capture reads as null."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))[kernel]
        if t.get("source_sha") != _source_sha(t["source"]):
            return None
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) * (n_rows / t["rows"])
    except Exception:
        return None


def algorithmic_bytes(n_rows: int, n_groups: int, n_aggs: int) -> float:
    # SURVEY §8d: 16 B/row in (int64 key + fp64 value) + G x (8 B key + 8 B per aggregate) out
    return 16.0 * n_rows + n_groups * (8.0 + 8.0 * n_aggs)


DUMP_BYTES = 64_000_000      # --dump-outputs: bytes on disk over all files (and all ranks)
NPY_HEADER_BYTES = 4096      # allowance per file for the .npy header (128 bytes for a 1-D float64 array)


def step_outputs(h, limit_bytes: int) -> dict:
    """What a caller of the timed path receives from handle `h`: the group keys in result order and one array per
    aggregate, as float64 (the benchmark's keys are group ids below 2^53: exact).  When their .npy files would take
    more than `limit_bytes`, every array keeps the same fixed seeded sample of group positions, which is stored as
    `group_index`."""
    import numpy as np
    out = {"keys": h.unique().to_numpy(zero_copy_only=False).astype(np.float64)}
    for a in AGGS:
        out[a] = h.fetch(a).to_numpy(zero_copy_only=False).astype(np.float64)
    n = len(out["keys"])
    if len(out) * (NPY_HEADER_BYTES + 8 * n) > limit_bytes:
        files = len(out) + 1
        cap = max(0, (limit_bytes - files * NPY_HEADER_BYTES) // (8 * files))
        pos = np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
        out = {k: v[pos] for k, v in out.items()}
        out["group_index"] = pos.astype(np.float64)
    return out


def dump_outputs(h, outdir: str, rank: int = 0, world: int = 1):
    """--dump-outputs: step_outputs(h) as outdir/<name>.npy; with several ranks each writes the groups it owns as
    <name>_rank<r>.npy within its share of the byte limit."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    tag = f"_rank{rank}" if world > 1 else ""
    for name, a in step_outputs(h, DUMP_BYTES // world).items():
        np.save(os.path.join(outdir, f"{name}{tag}.npy"), a)


def _hostgen():
    """hostgen.py (numpy data generator) loaded by path: importing the package would load libpa_b200.so,
    which must not appear in the reference arm's process."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("pa_hostgen", os.path.join(ROOT, "pandasarrow_b200", "hostgen.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_reference(rows: int, groups: int, repeats: int = 1) -> dict:
    """The reference's CPU path (oracle port of its Arrow call sequence) on this box's host cores:
    GroupBy ctor (hash + groupings + gathers of index and every column + per-group map inserts:
    single-threaded, as in the reference) followed by sum/mean/count with the over-groups loop on all
    cores (OpenMP standing in for TBB)."""
    import pyarrow as pa
    from oracle import oracle as orc
    hg = _hostgen()
    threads = os.cpu_count() or 1
    rb = pa.record_batch({"k": pa.array(hg.keys(rows, groups)), "v": pa.array(hg.vals(rows))})
    index = pa.array(range(rows), pa.int64())
    best = None
    detail = {}
    for _ in range(repeats):
        t0 = time.perf_counter()
        g = orc.OracleGroupBy(rb, "k", index=index, materialize=True)
        t1 = time.perf_counter()
        for a in AGGS:
            g.agg(a, "v", nthreads=threads)
        t2 = time.perf_counter()
        tm = g.timing_ms()
        g.close()
        if best is None or (t2 - t0) < best:
            best = t2 - t0
            detail = {"ctor_s": t1 - t0, "aggs_s": t2 - t1, "consume_ms": tm["consume"], "groupings_ms": tm["groupings"],
                      "gather_ms": tm["gather"]}
    return {"value": rows / best, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{rows} rows x {groups} groups, int64 key + fp64 value, GroupBy ctor (1 thread, as the reference) "
                      f"+ sum/mean/count ({threads} threads); ctor {detail['ctor_s']:.3f}s aggs {detail['aggs_s']:.3f}s",
            "seconds": best}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    rows = min(args.cpu_rows, args.rows)
    for _ in range(min(warm, 1)):
        cpu_reference(min(rows, 1_000_000), args.groups)
    t0 = time.perf_counter()
    vals = [cpu_reference(rows, args.groups) for _ in range(steps)]
    dt = time.perf_counter() - t0
    secs = sorted(v["seconds"] for v in vals)
    med = secs[len(secs) // 2]
    value = rows / med
    base = vals[0]
    base["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"group_by(int64 key, {args.groups} groups).sum/mean/count, fp64 value; CPU sample of "
                                   f"{rows} rows (the reference path needs ~4x input RAM and int32 row ids)",
                       "rows_per_step": rows, "groups": args.groups},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": dt}
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import pyarrow as pa
    import pandasarrow_b200 as pab

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    n, G = args.rows, args.groups
    first_row = rank * n                        # row-range shard of a world*n-row data set (weak scaling)
    stream = torch.cuda.Stream(device=dev)

    keys = torch.empty(n, dtype=torch.int64, device=dev)
    vals = torch.empty(n, dtype=torch.float64, device=dev)
    pab.synth.keys(keys, G, first_row)
    pab.synth.vals(vals, first_row)
    torch.cuda.synchronize()
    dk, dv = pab.DeviceColumn.from_torch(keys), pab.DeviceColumn.from_torch(vals)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput (`value`) ----------------
    # N = 1: one fused pass (stages 1-3 + merge + emit).  N > 1: the same on this rank's row shard, then
    # partial records -> NCCL all-to-all -> owner-side merge (pandasarrow_b200/distributed.py).
    from pandasarrow_b200 import distributed as D
    sm_reserve = max(args.sm_reserve, 0)
    gb = pab.GroupBy("k", {"k": dk, "v": dv}, stream=stream.cuda_stream, device=local, row_base=first_row, sm_reserve=sm_reserve)
    scan_ms, launches, merged_groups = [], 0, 0

    # N > 1: the serial tail of a step (all-to-all of ~1000 partial records -> single-CTA merge: ~0.15 ms of launch and
    # NCCL latency on a handful of CTAs) runs on a second stream behind an event, so that the next step's scan starts
    # as soon as this step's records are exported.  Scans never overlap each other (they stay on one stream).
    tail_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    handles = []          # multi-GPU: merged handles of the steps in flight

    def step():
        # Every step queues its whole pipeline (local pass -> export -> all-to-all -> merge -> result formatting)
        # without a host round trip; results are read after the timed region.  Steps therefore overlap their
        # launch latency with the previous step's kernels, exactly like a streaming consumer would.
        nonlocal launches, merged_groups
        if world == 1:
            gb.aggregate(dv, AGGS, fetch=False, wait=False)
        else:
            with torch.cuda.stream(stream):
                # (more groups than a padded block holds: counted exchange, which reads the counts back)
                big = args.groups > D.PADDED_BLOCK_RECORDS
                m = D.sharded_aggregate(gb, dv, AGGS, "g", "l", stream=stream.cuda_stream, wait=big, padded=False if big else None,
                                        tail_stream=None if big else tail_stream)
            handles.append(m)
            if len(handles) > 2:
                handles.pop(0).close()      # (recycled by the library without synchronising)

    def finish_steps(dump_dir=None):
        nonlocal launches, merged_groups
        t = gb.timing()                     # completes the last local pass (reads its status words)
        scan_ms.append(t["scan_ms"])
        launches += t["launches"] * args.steps
        if world > 1:
            m = handles[-1]
            merged_groups = m.groupSize()   # completes the last merge
            launches += (2 + m.timing()["launches"]) * args.steps
            if dump_dir:
                dump_outputs(m, dump_dir, rank, world)
            while handles:
                handles.pop().close()
        elif dump_dir:
            dump_outputs(gb, dump_dir)

    for _ in range(args.warmup):
        step()
    if args.warmup:
        finish_steps()
    scan_ms.clear(); launches = 0
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    if tail_stream is not None:
        stream.wait_stream(tail_stream)     # the region ends when the last step's merge has finished
    e1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    finish_steps(args.dump_outputs)
    ms = e0.elapsed_time(e1)
    tms = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_per_step = tms.item() / args.steps
    path = gb.timing()["path"]
    n_groups_found = gb.groupSize()
    if dist is not None:
        tg = torch.tensor([merged_groups], device=dev, dtype=torch.int64)
        dist.all_reduce(tg)
        total_groups = int(tg.item())
    else:
        total_groups = n_groups_found
    value = world * n / (ms_per_step * 1e-3)
    scan = sorted(scan_ms)[len(scan_ms) // 2]
    peak, peak_src = peaks()
    alg = algorithmic_bytes(n, n_groups_found, len(AGGS))
    achieved = alg / (scan * 1e-3) / 1e9
    kernel = "k_lowcard_scan" if path == "lowcard" else "k_gtable_scan"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": measured_traffic(kernel, n), "kernel": kernel,
                "kernel_ms": scan, "algorithmic_bytes": alg, "peak_source": peak_src,
                "frac_of_step": scan / ms_per_step}

    # ---------------- optional cardinality sweep (config 2), device resident ----------------
    sweep = None
    do_sweep = (args.sweep or world == 1) and not args.no_sweep and world == 1
    do_extras = (args.extras or world == 1) and not args.no_extras and world == 1
    if do_sweep and rank == 0:
        sweep = []
        for g_ in SWEEP_G:
            if g_ > n:
                continue
            pab.synth.keys(keys, g_, first_row)
            torch.cuda.synchronize()
            h = pab.GroupBy("k", {"k": dk, "v": dv}, stream=stream.cuda_stream, device=local, expected_groups=g_)
            for _ in range(3):
                h.aggregate(dv, SWEEP_AGGS, fetch=False)
            ts = []
            for _ in range(3):
                h.aggregate(dv, SWEEP_AGGS, fetch=False)
                ts.append(h.timing())
            ts.sort(key=lambda t: t["total_ms"])
            t = ts[len(ts) // 2]
            ab = algorithmic_bytes(n, h.groupSize(), len(SWEEP_AGGS))
            sweep.append({"groups": g_, "found": h.groupSize(), "path": t["path"], "mode": t["mode"], "total_ms": t["total_ms"],
                          "scan_ms": t["scan_ms"], "rows_per_s": n / (t["total_ms"] * 1e-3),
                          "scan_GBps": ab / (t["scan_ms"] * 1e-3) / 1e9, "frac": ab / (t["scan_ms"] * 1e-3) / 1e9 / peak})
            h.close()
        pab.synth.keys(keys, G, first_row)
        torch.cuda.synchronize()

    # ---------------- optional: configs 3 and 4, device resident ----------------
    extras = None
    if do_extras and rank == 0:
        extras = {}
        try:
            # the headline workload with SCATTERED 64-bit keys (an odd multiplier + offset over the same group
            # ids: the key set is no dense window, so the shared-memory kernel runs in hash mode)
            for g_, tag in ((G, "scattered_keys"), (4096, "scattered_keys_4096")):
                pab.synth.keys(keys, g_, first_row)
                keys.mul_(0x2545F4914F6CDD1D).add_(0x1234567)
                torch.cuda.synchronize()
                h = pab.GroupBy("k", {"k": dk, "v": dv}, stream=stream.cuda_stream, device=local)
                tl = []
                for _ in range(3):
                    h.aggregate(dv, AGGS, fetch=False)
                for _ in range(5):
                    h.aggregate(dv, AGGS, fetch=False)
                    tl.append(h.timing())
                tl.sort(key=lambda t: t["total_ms"])
                t = tl[len(tl) // 2]
                ab = algorithmic_bytes(n, h.groupSize(), len(AGGS))
                extras[tag] = {"rows": n, "groups": h.groupSize(), "path": t["path"], "mode": t["mode"], "total_ms": t["total_ms"],
                               "scan_ms": t["scan_ms"], "rows_per_s": n / (t["total_ms"] * 1e-3),
                               "scan_GBps": ab / (t["scan_ms"] * 1e-3) / 1e9, "frac": ab / (t["scan_ms"] * 1e-3) / 1e9 / peak}
                h.close()
            pab.synth.keys(keys, G, first_row)
            torch.cuda.synchronize()
            # config 4: sorted timestamp[ns] index, 1-minute buckets (~1000 ticks each), OHLC + sum
            ts = torch.empty(n, dtype=torch.int64, device=dev)
            pab.synth.timestamps(ts)
            torch.cuda.synchronize()
            dts = pab.DeviceColumn.from_torch(ts, fmt="tsn:")
            r = pab.resample({"v": dv}, dts, 60 * 10**9, stream=stream.cuda_stream, device=local)
            tl = []
            for _ in range(4):                                     # warm-up: stream-ordered pool growth
                r.aggregate(dv, ["first", "max", "min", "last", "sum"], fetch=False)
            for _ in range(5):
                r.aggregate(dv, ["first", "max", "min", "last", "sum"], fetch=False)
                tl.append(r.timing())
            tl.sort(key=lambda t: t["total_ms"])
            t = tl[len(tl) // 2]
            extras["resample_ohlc_sum"] = {"rows": n, "buckets": r.groupSize(), "total_ms": t["total_ms"], "scan_ms": t["scan_ms"],
                                           "rows_per_s": n / (t["total_ms"] * 1e-3), "scan_GBps": 16.0 * n / (t["scan_ms"] * 1e-3) / 1e9,
                                           "frac": 16.0 * n / (t["scan_ms"] * 1e-3) / 1e9 / peak}
            r.close(); del ts, dts
            # config 3: int32 key (1 K values) x int32 dictionary indices (64 symbols) packed into one 64-bit key,
            # nullable fp64 value (10 % nulls)
            m = min(n, 500_000_000)
            k1 = torch.empty(m, dtype=torch.int64, device=dev); pab.synth.keys(k1, 1000, 0)
            k2 = torch.empty(m, dtype=torch.int64, device=dev); pab.synth.keys(k2, 64, 12345)
            k1i, k2i = k1.to(torch.int32), k2.to(torch.int32)
            del k1, k2
            bits = torch.empty((m + 7) // 8, dtype=torch.uint8, device=dev)
            pab.synth.validity(bits, m)
            torch.cuda.synchronize()
            c1 = pab.DeviceColumn.from_torch(k1i)
            c2 = pab.DeviceColumn.from_torch(k2i)          # (the int32 indices of a dictionary column are what the kernels see)
            cv = pab.DeviceColumn.from_torch(vals[:m], valid=bits, null_count=-1)
            h = pab.GroupBy(["k1", "k2"], {"k1": c1, "k2": c2, "v": cv}, stream=stream.cuda_stream, device=local, expected_groups=64000)
            tl = []
            for _ in range(3):
                h.aggregate(cv, ["sum", "mean", "count", "min", "max"], fetch=False)
            for _ in range(4):
                h.aggregate(cv, ["sum", "mean", "count", "min", "max"], fetch=False)
                tl.append(h.timing())
            tl.sort(key=lambda t: t["total_ms"])
            t = tl[len(tl) // 2]
            extras["multikey_nullable"] = {"rows": m, "groups": h.groupSize(), "path": t["path"], "total_ms": t["total_ms"],
                                           "pack_ms": t["pack_ms"], "scan_ms": t["scan_ms"], "rows_per_s": m / (t["total_ms"] * 1e-3)}
            h.close()
            # second-stage aggregates (SURVEY §8f-1) on the headline workload: variance + stddev + product, which is
            # the ordinary pass (sum / mean / count) plus one more pass over keys and values
            h = pab.GroupBy("k", {"k": dk, "v": dv}, stream=stream.cuda_stream, device=local)
            tl = []
            for _ in range(3):
                h.aggregate(dv, ["variance", "stddev", "product"], fetch=False)
            for _ in range(4):
                h.aggregate(dv, ["variance", "stddev", "product"], fetch=False)
                tl.append(h.timing())
            tl.sort(key=lambda t: t["total_ms"])
            t = tl[len(tl) // 2]
            extras["variance_stddev_product"] = {"rows": n, "groups": h.groupSize(), "total_ms": t["total_ms"], "first_pass_ms": t["scan_ms"],
                                                 "second_pass_ms": t["emit_ms"], "rows_per_s": n / (t["total_ms"] * 1e-3)}
            h.close()
            # group materialisation (SURVEY §8f-2): MakeGroupings + ApplyGroupings of one fp64 column on the device
            # (int32 offsets like the reference: < 2^31 rows); device times only, the host copies are not in them
            m = min(n, 200_000_000)
            ck, cv2 = pab.DeviceColumn.from_torch(keys[:m]), pab.DeviceColumn.from_torch(vals[:m])
            for _ in range(2):                                       # first round: stream-ordered pool growth
                h = pab.GroupBy("k", {"k": ck, "v": cv2}, stream=stream.cuda_stream, device=local)
                h.groupSize()
                h.groupings(rows=False)
                h.take_grouped(cv2)
                t = h.groupings_timing()
                if _ == 0:
                    h.close()
            extras["materialise_groups"] = {"rows": m, "groups": h.groupSize(), "groupings_build_ms": t["build_ms"], "take_column_ms": t["take_ms"],
                                            "rows_per_s_build": m / (t["build_ms"] * 1e-3), "rows_per_s_take": m / (t["take_ms"] * 1e-3)}
            h.close()
        except Exception as ex:  # noqa: BLE001
            extras["error"] = repr(ex)[:300]
        # the same roofline figure for the general (hash-table) mode of the headline kernel and for config 4's scan,
        # next to the dense-key headline: 16 B/row of the same workload / that scan's duration / the same peak
        if "scattered_keys" in extras:
            sk = extras["scattered_keys"]
            roofline["scattered_keys"] = {"kernel": "k_lowcard_scan (hash mode)", "kernel_ms": sk["scan_ms"],
                                          "achieved": sk["scan_GBps"], "frac": sk["frac"]}
        if "resample_ohlc_sum" in extras:
            rk = extras["resample_ohlc_sum"]
            roofline["resample_ohlc_sum"] = {"kernel": "k_resample_scan", "kernel_ms": rk["scan_ms"],
                                             "achieved": rk["scan_GBps"], "frac": rk["frac"]}

    # ---------------- N > 1: config 5 (BASELINE configs[4]): 1 B rows per GPU, 100 M groups, counted exchange ----------------
    if world > 1 and args.config5_groups > 0 and not args.no_extras:
        extras = extras or {}
        try:
            g5 = args.config5_groups
            pab.synth.keys(keys, g5, first_row)
            torch.cuda.synchronize()
            h5 = pab.GroupBy("k", {"k": dk, "v": dv}, stream=stream.cuda_stream, device=local, row_base=first_row, expected_groups=g5)
            local_ms = []
            for _ in range(3):                                   # local pass alone (what one GPU does for its shard)
                h5.aggregate(dv, AGGS, fetch=False)
                local_ms.append(h5.timing()["total_ms"])
            # the whole sharded step is ONE C call on the library's own NCCL communicator (pa_groupby_sharded_aggregate)
            comm = D.Comm(device=local)
            def step5():
                return comm.sharded_aggregate(h5, dv, AGGS)
            m5 = step5()                                         # warm-up (allocations, NCCL channels)
            m5.close()
            barrier()
            k5 = 3
            t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
            t0.record(stream)
            found = 0
            phases = []
            for _ in range(k5):
                m5 = step5()
                phases.append(comm.phases())
                found = m5.groupSize()
                m5.close()
            t1.record(stream)
            barrier()
            t5 = torch.tensor([t0.elapsed_time(t1) / k5, min(local_ms)], device=dev, dtype=torch.float64)
            dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            tg5 = torch.tensor([found], device=dev, dtype=torch.int64)
            dist.all_reduce(tg5)
            ph = {k: sorted(p_[k] for p_ in phases)[len(phases) // 2] for k in phases[0]}
            xi = comm.exchange_info()
            extras["config5"] = {"rows_per_gpu": n, "groups": g5, "groups_found_global": int(tg5.item()), "aggs": AGGS,
                                 "exchange": "pa_comm (C ABI): ncclAllGather of counts + grouped ncclSend/ncclRecv of records",
                                 "record_bytes": xi["record_bytes"], "unordered_export": xi["unordered_export"],
                                 "merge_table_slots": xi["merge_table_slots"],
                                 "steps": k5, "ms_per_step": t5[0].item(),
                                 "local_pass_ms": t5[1].item(), "rows_per_s": world * n / (t5[0].item() * 1e-3),
                                 "efficiency_vs_local_pass": t5[1].item() / t5[0].item(), "phases_rank0_ms": ph}
            comm.close()
            h5.close()
        except Exception as ex:  # noqa: BLE001
            extras["config5"] = {"error": repr(ex)[:300]}
        pab.synth.keys(keys, G, first_row)
        torch.cuda.synchronize()

    # ---------------- end to end through the C ABI with HOST buffers (`e2e`) ----------------
    e2e = None
    if not args.no_e2e:
        try:
            # one process per GPU, each on the NUMA node of its GPU while it allocates (first-touches) the pinned host
            # columns: with 4-8 ranks the host -> device copies otherwise share one node's DRAM and the socket link
            from pandasarrow_b200.numa import bind_to_device_numa
            with bind_to_device_numa(local) as numa_bind:
                hk = torch.empty(n, dtype=torch.int64, pin_memory=True)
                hv = torch.empty(n, dtype=torch.float64, pin_memory=True)
                hk.copy_(keys); hv.copy_(vals)
                torch.cuda.synchronize()
            ak = pa.Array.from_buffers(pa.int64(), n, [None, pa.py_buffer(hk.numpy())])
            av = pa.Array.from_buffers(pa.float64(), n, [None, pa.py_buffer(hv.numpy())])

            def e2e_step():
                with pab.GroupBy("k", {"k": ak, "v": av}, device=local) as h:
                    r = h.aggregate(av, AGGS)                      # H2D of keys + values, kernels, D2H of results
                    return sum(len(x) * 8 for x in r.values())

            e2e_steps = max(2, min(args.steps, 3))
            d2h = e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_step()
            barrier()
            dt = (time.perf_counter() - t0) / e2e_steps
            tt = torch.tensor([dt], device=dev, dtype=torch.float64)
            if dist is not None:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e = {"value": world * n / tt.item(), "unit": UNIT, "h2d_bytes_per_step": 16 * n,
                   "d2h_bytes_per_step": d2h, "ms_per_step": tt.item() * 1e3, "steps": e2e_steps,
                   "note": "pinned host Arrow buffers -> pa_groupby_create/aggregate/fetch; wall clock around synchronous calls",
                   "host_numa": numa_bind.info}
            # the same call with ORDINARY (pageable) host memory — what an Arrow heap buffer / an IPC blob is: the library
            # stages it through its own pinned double buffer with a few copy threads (h2d_copy in capi.cu)
            if world == 1:
                try:
                    import numpy as np
                    pk, pv = np.array(hk.numpy()), np.array(hv.numpy())
                    del ak, av
                    bk = pa.Array.from_buffers(pa.int64(), n, [None, pa.py_buffer(pk)])
                    bv = pa.Array.from_buffers(pa.float64(), n, [None, pa.py_buffer(pv)])

                    def e2e_step_pageable():
                        with pab.GroupBy("k", {"k": bk, "v": bv}, device=local) as h:
                            h.aggregate(bv, AGGS)

                    e2e_step_pageable()
                    t0 = time.perf_counter()
                    for _ in range(2):
                        e2e_step_pageable()
                    torch.cuda.synchronize()
                    dtp = (time.perf_counter() - t0) / 2
                    e2e["pageable"] = {"value": n / dtp, "unit": UNIT, "ms_per_step": dtp * 1e3, "h2d_GBps": 16.0 * n / dtp / 1e9,
                                       "note": "ordinary (pageable) numpy / Arrow heap buffers through the same calls: pinned staging inside the library"}
                    del pk, pv, bk, bv
                except Exception as ex:  # noqa: BLE001
                    e2e["pageable"] = {"error": repr(ex)[:200]}
            del hk, hv
        except Exception as ex:  # noqa: BLE001
            e2e = {"value": None, "unit": UNIT, "error": repr(ex)[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_reference(min(args.cpu_rows, n), G)
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "error": repr(ex)[:300]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"group_by(int64 key, {G} groups).sum/mean/count over {n} rows per GPU, fp64 value "
                                       f"(BASELINE configs[1] row count at configs[0] cardinality)",
                           "rows_per_gpu": n, "groups": G, "groups_found_global": total_groups, "aggs": AGGS, "path": path,
                           "parallelism": "1 GPU" if world == 1 else f"row-range shards x{world}, hash-partitioned partials, NCCL all-to-all, owner merge; "
                                                                             f"exchange + merge of step k on a second stream while step k+1 scans",
                           "l2": "inputs (16 B/row x rows) far exceed the 126 MB L2; no explicit flush",
                           "hbm_GBps_whole_step": alg / (ms_per_step * 1e-3) / 1e9},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks}
        if sweep is not None:
            line["sweep"] = sweep
        if extras is not None:
            line["extras"] = extras
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
