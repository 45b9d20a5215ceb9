"""Worker of tests/test_nccl_composite_multigpu.py: one process per GPU (torchrun), real NCCL.  Config 3's composite key
(int32 x dictionary<int32 -> utf8>, encoded once over the whole column) is sharded by row range; only the last rank's
shard has null keys.  Each step runs through the C-ABI communicator and through distributed.py (padded and counted
exchange); rank 0 gathers the owners' groups, restores global first-appearance order and compares with the ORACLE run
on the whole data set.  Exits non-zero on any mismatch."""
import os
import sys

import numpy as np
import pyarrow as pa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import faulthandler
    faulthandler.enable()
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
    n = 1_000_003 * world
    for n1 in (30, 1000):
        rng = np.random.default_rng(n1)
        k1 = rng.integers(0, n1, n).astype(np.int32)
        words = pa.array([f"sym{i:02d}" for i in range(64)])
        k2 = rng.integers(0, 64, n).astype(np.int32)
        m1, m2 = rng.random(n) < 0.01, rng.random(n) < 0.01
        b, e = D.shard_rows(n, world, rank)
        last = D.shard_rows(n, world, world - 1)[0]
        m1[:last] = False; m2[:last] = False              # null keys on the last rank only
        v = rng.random(n)
        vm = rng.random(n) < 0.1
        fa = pa.array(v, mask=vm)
        c1 = pa.array(k1[b:e], mask=m1[b:e] if rank == world - 1 else None)
        c2 = pa.DictionaryArray.from_arrays(pa.array(k2[b:e], mask=m2[b:e] if rank == world - 1 else None), words)
        gb = pab.GroupBy(["k1", "k2"], {"k1": c1, "k2": c2}, device=local, stream=stream, row_base=b)
        own = list(gb.key_layout().nullable[:2])
        if own != ([1, 1] if rank == world - 1 else [0, 0]):
            failures.append(f"n1={n1}: own layout {own}")
        vals = fa.slice(b, e - b)
        aggs = ["sum", "mean", "count", "min", "max"]
        runs = [("c-abi", None), ("distributed.py padded", True), ("distributed.py counted", False)]
        if rank == 0:
            from oracle import oracle as orc
            rb = pa.record_batch({"k1": pa.array(k1, mask=m1), "k2": pa.DictionaryArray.from_arrays(pa.array(k2, mask=m2), words), "v": fa})
            ora = orc.OracleGroupBy(rb, ["k1", "k2"])
            theirs = list(zip(ora.unique(0).to_pylist(), ora.unique(1).to_pylist()))
            want = {a: ora.agg(a, "v", nthreads=8).to_pylist() for a in ("count", "min", "max")}
            wsum = ora.agg("sum", "v", nthreads=8).to_numpy(zero_copy_only=False)
            from util import first_appearance_order
            fao = first_appearance_order([rb.column("k1"), rb.column("k2")])
        for name, padded in runs:
            if padded is None:
                m = comm.sharded_aggregate(gb, vals, aggs)
                info = comm.key_layout_info()
                if info["agree_ms"] <= 0 or (rank < world - 1 and n1 == 30 and info["repack_ms"] <= 0):
                    failures.append(f"{name} n1={n1}: agreement / repack not seen ({info})")
            else:
                m = D.sharded_aggregate(gb, vals, aggs, "g", None, stream=stream, padded=padded)
            if list(gb.key_layout().nullable[:2]) != [1, 1]:
                failures.append(f"{name} n1={n1}: rank {rank} did not repack")
            u2 = m.unique(1)
            if not isinstance(u2, pa.DictionaryArray):
                failures.append(f"{name} n1={n1}: unique(1) is {u2.type}")
            owned = {"k1": m.unique(0).fill_null(-1).to_numpy(), "k1null": np.asarray(m.unique(0).is_null()),
                     "k2": np.asarray(u2.cast(pa.string()).fill_null("<null>").to_pylist(), dtype=object),
                     **{a: m.fetch(a).to_numpy(zero_copy_only=False) for a in aggs}}
            fr = m.first_rows().to_numpy()
            m.close()
            res = D.gather_result(owned, fr)
            if rank == 0:
                tag = f"{name} n1={n1}"
                ours = [(None if nl else int(x), None if s == "<null>" else s) for x, nl, s in zip(res["k1"], res["k1null"], res["k2"])]
                if ours != fao:
                    failures.append(f"{tag}: keys / global first-appearance order differ")
                    continue
                pos = {t: i for i, t in enumerate(ours)}
                perm = np.array([pos[t] for t in theirs])
                for a in ("count", "min", "max"):
                    if res[a][perm].tolist() != want[a]:
                        failures.append(f"{tag} {a} differs")
                got = res["sum"][perm]
                if not np.allclose(got, wsum, rtol=1e-12, atol=0):
                    failures.append(f"{tag} sum differs")
        gb.close()
        if rank == 0:
            ora.close()
    if rank == 0:
        print("phases of the last c-abi step:", comm.phases(), comm.key_layout_info())
    bad = torch.tensor([len(failures)], device=dev)
    dist.all_reduce(bad)
    for f in failures:
        print(f"[rank {rank}] FAIL {f}")
    comm.close()
    dist.destroy_process_group()
    if bad.item():
        sys.exit(1)
    if rank == 0:
        print("NCCL COMPOSITE PARITY OK")


if __name__ == "__main__":
    main()
