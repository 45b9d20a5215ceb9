"""Worker of tests/test_nccl_strkeys_multigpu.py: one process per GPU (torchrun), real NCCL.  A utf8 key column (nulls, the
empty string, non-ASCII bytes) is sharded by row range; every step runs through the C-ABI communicator and through
distributed.py's counted exchange, and rank 0 compares the gathered owners' groups, in global first-appearance order,
with the ORACLE on the whole column.  With --hook (run under PA_TEST_STR_HASH_BITS=0) rank 0 holds only "a" and rank 1
only "b": both hash alike under seed 0, the owner sees it, and every rank retries with seed 1.  Exits non-zero on any
mismatch."""
import os
import sys

import numpy as np
import pyarrow as pa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gathered(m, aggs, dist, world):
    part = (m.unique().to_pylist(), {a: m.fetch(a).to_pylist() for a in aggs}, m.first_rows().to_numpy())
    parts = [None] * world
    dist.all_gather_object(parts, part)
    fr = np.concatenate([p[2] for p in parts])
    order = np.argsort(fr, kind="stable")
    keys = [k for p in parts for k in p[0]]
    return [keys[i] for i in order], {a: [v for p in parts for v in p[1][a]] for a in aggs}, order


def main():
    import torch
    import torch.distributed as dist
    import pandasarrow_b200 as pab
    from pandasarrow_b200 import distributed as D
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    comm = D.Comm(device=local)
    stream = torch.cuda.current_stream(dev).cuda_stream
    failures = []
    aggs = ["sum", "count", "min", "max"]
    if "--hook" in sys.argv:
        keys = pa.array(["a"] * 4 + ["b"] * 3)
        vals = pa.array(np.arange(7, dtype=np.float64))
        b, e = (0, 4) if rank == 0 else (4, 7)
        want_keys, want_sum = ["a", "b"], [6.0, 15.0]
    else:
        n = 400_003 * world
        rng = np.random.default_rng(3)
        pool = pa.array(["", "ü", "日本語", "x" * 45] + [f"key{i}" for i in range(5000)])
        idx = rng.integers(0, len(pool), n).astype(np.int32)
        keys = pa.DictionaryArray.from_arrays(pa.array(idx, mask=rng.random(n) < 0.01), pool).cast(pa.large_string())
        vals = pa.array(rng.random(n))
        b, e = D.shard_rows(n, world, rank)
    for run in ("c-abi", "distributed.py"):
        gb = pab.GroupBy("k", {"k": keys.slice(b, e - b)}, device=local, stream=stream, row_base=b)
        v = vals.slice(b, e - b)
        if run == "c-abi":
            m = comm.sharded_aggregate(gb, v, aggs)
            info = comm.key_strings_info()
            if "--hook" in sys.argv and (info["seed"], info["attempts"]) != (1, 2):
                failures.append(f"rank {rank}: key_strings_info {info}")
        else:
            m = D.sharded_aggregate(gb, v, aggs, "g", None, stream=stream)
            if "--hook" in sys.argv and gb.key_hash_seed() != 1:
                failures.append(f"rank {rank}: distributed.py seed {gb.key_hash_seed()}")
        got_keys, got, _ = gathered(m, aggs, dist, world)
        if rank == 0:
            if "--hook" in sys.argv:
                if got_keys != want_keys or got["sum"] != want_sum:
                    failures.append(f"{run}: {got_keys} {got['sum']}")
            else:
                from oracle import oracle as orc
                from util import first_appearance_order
                if m.unique().type != pa.large_string():
                    failures.append(f"{run}: unique() type {m.unique().type}")
                if [(k,) for k in got_keys] != first_appearance_order([keys]):
                    failures.append(f"{run}: global first-appearance order")
                else:
                    ora = orc.OracleGroupBy(pa.record_batch({"k": keys, "v": vals}), "k")
                    pos = {k: i for i, k in enumerate(got_keys)}
                    perm = [pos[k] for k in ora.unique().to_pylist()]
                    for a in aggs:
                        want = ora.agg(a, "v", nthreads=8).to_numpy(zero_copy_only=False)
                        g_ = np.asarray(got[a], dtype=want.dtype)[perm]
                        ok = np.allclose(g_, want, rtol=1e-12, atol=0) if a == "sum" else np.array_equal(g_, want)
                        if not ok:
                            failures.append(f"{run}: {a}")
                    ora.close()
        m.close()
        gb.close()
    comm.close()
    out = [None] * world
    dist.all_gather_object(out, failures)
    dist.destroy_process_group()
    if rank == 0:
        allf = [f for fs in out for f in fs]
        if allf:
            print("FAILURES:", allf)
            sys.exit(1)
        print("NCCL STRKEYS PARITY OK")


if __name__ == "__main__":
    main()
