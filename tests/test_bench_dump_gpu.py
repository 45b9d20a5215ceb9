"""bench.py --dump-outputs: the files hold what the timed path returned in its last step (group keys in first-appearance
order, sum / mean / count per group, float64), checked against numpy on the generator's host twin; beyond 64 MB of files
every array keeps the same seeded sample of group positions.  Needs a GPU: -m gpu."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,groups", [(2_000_000, 1000), (8_000_000, 4_000_000)])      # the second is sampled
def test_dump_outputs_match_numpy(tmp_path, rows, groups):
    from pandasarrow_b200 import hostgen as hg
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--rows", str(rows),
                        "--groups", str(groups), "--no-sweep", "--no-extras", "--no-e2e", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    got = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64_000_000

    k, v = hg.keys(rows, groups), hg.vals(rows)
    _, first = np.unique(k, return_index=True)
    keys = k[np.sort(first)]                                      # first-appearance order
    cnt = np.bincount(k, minlength=groups)[keys]
    s = np.bincount(k, weights=v, minlength=groups)[keys]
    assert line["steps"] == 2 and line["config"]["groups_found_global"] == len(keys)
    assert ("group_index" in got) == (len(keys) > 2_000_000)        # 4 x 8 B per group do not fit 64 MB beyond 2 M groups
    if "group_index" in got:
        assert set(got) == {"keys", "sum", "mean", "count", "group_index"}
        pos = got["group_index"].astype(np.int64)
        assert 0 < len(pos) < len(keys) and (np.diff(pos) > 0).all() and pos[-1] < len(keys)
    else:
        assert set(got) == {"keys", "sum", "mean", "count"}
        pos = np.arange(len(keys))
    assert np.array_equal(got["keys"], keys[pos].astype(np.float64))
    assert np.array_equal(got["count"], cnt[pos].astype(np.float64))
    assert np.max(np.abs(got["sum"] - s[pos]) / s[pos]) <= 1e-12
    mean = s[pos] / cnt[pos]
    assert np.max(np.abs(got["mean"] - mean) / mean) <= 1e-12
