"""Worker of tests/test_nccl_distinct_multigpu.py: one process per GPU (torchrun), real NCCL.  Every rank aggregates its
row-range shard with count_distinct / all / any; the partial records and the distinct pairs travel over NCCL by the C-ABI
communicator and by distributed.py's counted exchange; rank 0 gathers the owners' groups, restores global
first-appearance order and compares with the ORACLE run on the whole data set.  Exits non-zero on any mismatch."""
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
    from pandasarrow_b200 import hostgen as hg
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    comm = D.Comm(device=local)
    n = 2_000_003                                   # rows per rank
    stream = torch.cuda.current_stream(dev).cuda_stream
    failures = []
    for G in (1000, 60_000):
        first = rank * n
        k = torch.empty(n, dtype=torch.int64, device=dev); pab.synth.keys(k, G, first)
        v = torch.empty(n, dtype=torch.float64, device=dev); pab.synth.vals(v, first)
        q = torch.floor(v * 500).to(torch.int64)    # ~500 distinct values per group, repeated across the ranks
        b = (v < 0.999).to(torch.uint8)
        torch.cuda.synchronize()
        dk, dq = pab.DeviceColumn.from_torch(k), pab.DeviceColumn.from_torch(q)
        bh = pa.array(b.cpu().numpy().astype(bool))
        gb = pab.GroupBy("k", {"k": dk}, device=local, stream=stream, row_base=first)
        runs = [("c-abi", dq, "l", ["count_distinct", "count"]), ("c-abi", bh, "b", ["all", "any", "count_distinct"]),
                ("distributed.py", dq, "l", ["count_distinct", "count"]), ("distributed.py", bh, "b", ["all", "any", "count_distinct"])]
        if rank == 0:
            from oracle import oracle as orc
            import pandas as pd
            kh = hg.keys(world * n, G)
            vh = hg.vals(world * n)
            rb = pa.record_batch({"k": pa.array(kh), "q": pa.array(np.floor(vh * 500).astype(np.int64)), "b": pa.array(vh < 0.999)})
            ora = orc.OracleGroupBy(rb, "k")
            st = np.argsort(ora.unique().to_numpy(), kind="stable")
            want = {("q", a): ora.agg(a, "q", nthreads=8).to_numpy()[st] for a in ("count_distinct", "count")}
            want.update({("b", a): ora.agg(a, "b", nthreads=8).to_numpy(zero_copy_only=False)[st] for a in ("all", "any", "count_distinct")})
            fa = pd.unique(kh)
        for name, col, vfmt, aggs in runs:
            if name == "c-abi":
                m = comm.sharded_aggregate(gb, col, aggs)
                info = comm.distinct_info()
                if info["pairs_received"] <= 0:
                    failures.append(f"{name} G={G}: no pairs received ({info})")
            else:
                m = D.sharded_aggregate(gb, col, aggs, vfmt, "l", stream=stream, padded=None)
            owned = {a: m.fetch(a).to_numpy(zero_copy_only=False) for a in aggs}
            owned["key"] = m.unique().to_numpy()
            fr = m.first_rows().to_numpy()
            if not (D.owner_of(owned["key"], world) == rank).all():
                failures.append(f"{name} G={G}: rank {rank} merged a key it does not own")
            m.close()
            res = D.gather_result(owned, fr)
            if rank == 0:
                tag = f"{name} G={G} {vfmt}"
                if not np.array_equal(res["key"], fa):
                    failures.append(f"{tag}: keys / global first-appearance order differ")
                    continue
                so = np.argsort(res["key"], kind="stable")
                for a in aggs:
                    g_, w_ = res[a][so], want[("q" if vfmt == "l" else "b", a)]
                    if not np.array_equal(g_, w_):
                        failures.append(f"{tag} {a}: {(g_ != w_).sum()} groups differ")
        gb.close()
        if rank == 0:
            ora.close()
    if rank == 0:
        print("phases of the last c-abi step:", comm.phases(), comm.distinct_info())
    bad = torch.tensor([len(failures)], device=dev)
    dist.all_reduce(bad)
    for f in failures:
        print(f"[rank {rank}] FAIL {f}")
    comm.close()
    dist.destroy_process_group()
    if bad.item():
        sys.exit(1)
    if rank == 0:
        print("NCCL DISTINCT PARITY OK")


if __name__ == "__main__":
    main()
