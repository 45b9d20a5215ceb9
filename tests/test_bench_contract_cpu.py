"""The committed bench lines (profiles/r2_bench_line*.json: what `python bench.py` printed on the GPU box for the
final build of the round) carry every key of the bench contract, and their roofline arithmetic follows from their
own numbers.  CPU only: nothing is measured here."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"]


def _line(name):
    return json.load(open(os.path.join(ROOT, "profiles", name)))


@pytest.mark.parametrize("name,n", [("r2_bench_line.json", 1), ("r2_bench_line_n2.json", 2), ("r2_bench_line_n8.json", 8)])
def test_line_has_the_contract_keys(name, n):
    d = _line(name)
    for k in BASE_KEYS:
        assert k in d, f"{name}: {k} missing"
    assert d["n_gpus"] == n and d["metric"] == "groupby_agg_rows_per_s" and d["unit"] == "rows/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["steps"] >= 1 and d["warmup"] >= 3 and d["gpu_launches"] > 0
    rows = d["config"]["rows_per_gpu"]
    # value = rows all ranks processed / the step time
    assert d["value"] == pytest.approx(n * rows / (d["ms_per_step"] * 1e-3), rel=1e-9)
    c = d["clocks"]
    assert not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert c["sm_mhz"] >= 0.9 * c["sm_max_mhz"]


def test_roofline_follows_from_the_line():
    d = _line("r2_bench_line.json")
    r = d["roofline"]
    rows, groups = d["config"]["rows_per_gpu"], d["config"]["groups_found_global"]
    alg = 16.0 * rows + groups * (8.0 + 8.0 * len(d["config"]["aggs"]))      # SURVEY §8d
    assert r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert r["algorithmic_bytes"] == pytest.approx(alg, rel=1e-12)
    assert r["achieved"] == pytest.approx(alg / (r["kernel_ms"] * 1e-3) / 1e9, rel=1e-9)
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-12)
    assert r["kernel_ms"] <= d["ms_per_step"] and r["frac"] < 1.0
    # measured DRAM traffic of the capture the line cites: within 1 % of the algorithmic bytes, never below them
    assert r["traffic"] is not None and alg <= r["traffic"] <= 1.01 * alg
    for sub in ("scattered_keys", "resample_ohlc_sum"):
        s = r[sub]
        assert s["achieved"] == pytest.approx(16.0 * rows / (s["kernel_ms"] * 1e-3) / 1e9, rel=1e-4)
        assert s["frac"] == pytest.approx(s["achieved"] / r["peak"], rel=1e-9)


def test_e2e_and_cpu_baseline_are_declared():
    d = _line("r2_bench_line.json")
    e, c = d["e2e"], d["cpu_baseline"]
    rows = d["config"]["rows_per_gpu"]
    assert e["unit"] == "rows/s" and e["h2d_bytes_per_step"] == 16 * rows and e["d2h_bytes_per_step"] > 0
    assert e["value"] == pytest.approx(rows / (e["ms_per_step"] * 1e-3), rel=1e-6)
    assert e["value"] < d["value"]                     # end to end includes PCIe: it cannot repeat the device number
    assert c["kind"] == "port" and c["cores"] >= 1 and c["unit"] == "rows/s" and "rows" in c["sample"]
    assert {s["groups"] for s in d["sweep"]} >= {16, 4096, 65536, 1048576, 100000000}
    for k in ("scattered_keys", "resample_ohlc_sum", "multikey_nullable"):
        assert k in d["extras"]


def test_traffic_stamp_matches_the_kernel_source():
    """`roofline.traffic` comes from a committed ncu capture stamped with the hash of lowcard.cuh: a kernel edit without a
    new capture must read as null, never as a stale number."""
    import hashlib
    t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["k_lowcard_scan"]
    sha = hashlib.sha256(open(os.path.join(ROOT, t["source"]), "rb").read()).hexdigest()[:16]
    assert t["source_sha"] == sha, "lowcard.cuh changed after the traffic capture: re-capture (scripts/r2_run50.sh) and restamp"


@pytest.mark.parametrize("flags", [["--steps", "0"], ["--warmup", "-1"]])
def test_bench_refuses_step_counts_it_cannot_time(flags):
    """--steps is the number of timed steps: zero of them has no time per step, so the run stops before any work."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "must be at least" in r.stderr, r.stderr[-2000:]
