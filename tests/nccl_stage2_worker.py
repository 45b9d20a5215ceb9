"""Worker of tests/test_nccl_stage2_multigpu.py: one process per GPU (torchrun), real NCCL.  Every rank aggregates its
row-range shard with product / variance / stddev; the stage-2 records travel over NCCL by the C-ABI communicator and
by distributed.py's counted exchange (which a stage-2 mask must choose even when the padded one would apply); rank 0
gathers the owners' groups, restores global first-appearance order and compares with the ORACLE run on the whole data
set.  Exits non-zero on any mismatch."""
import os
import sys

import numpy as np
import pyarrow as pa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

AGGS = ["mean", "count", "variance", "stddev", "product"]


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
    n = 2_000_003                                   # rows per rank (odd: partial row groups)
    stream = torch.cuda.current_stream(dev).cuda_stream
    failures = []
    for G in (1000, 60_000):
        first = rank * n
        k = torch.empty(n, dtype=torch.int64, device=dev); pab.synth.keys(k, G, first)
        v = torch.empty(n, dtype=torch.float64, device=dev); pab.synth.vals(v, first)
        v += 0.5                                    # values in [0.5, 1.5): products stay normal numbers
        torch.cuda.synchronize()
        dk, dv = pab.DeviceColumn.from_torch(k), pab.DeviceColumn.from_torch(v)
        gb = pab.GroupBy("k", {"k": dk, "v": dv}, device=local, stream=stream, row_base=first)
        transports = [("c-abi", lambda: comm.sharded_aggregate(gb, dv, AGGS)),
                      ("distributed.py", lambda: D.sharded_aggregate(gb, dv, AGGS, "g", "l", stream=stream, padded=None))]
        if rank == 0:
            from oracle import oracle as orc
            import pandas as pd
            kh = hg.keys(world * n, G)
            vh = hg.vals(world * n) + 0.5
            rb = pa.record_batch({"k": pa.array(kh), "v": pa.array(vh), "sq": pa.array(vh * vh)})
            ora = orc.OracleGroupBy(rb, "k")
            st = np.argsort(ora.unique().to_numpy(), kind="stable")
            want = {a: ora.agg(a, "v", nthreads=8).to_numpy()[st] for a in AGGS}
            m2 = ora.agg("mean", "sq", nthreads=8).to_numpy()[st]                  # mean(x^2): the variance bar's scale
            fa = pd.unique(kh)
        for name, run in transports:
            m = run()
            if name == "c-abi" and comm.exchange_info()["record_bytes"] != 104:
                failures.append(f"{name} G={G}: {comm.exchange_info()['record_bytes']}-byte records, want 104")
            owned = {a: m.fetch(a).to_numpy(zero_copy_only=False) for a in AGGS}
            owned["key"] = m.unique().to_numpy()
            fr = m.first_rows().to_numpy()
            if not (D.owner_of(owned["key"], world) == rank).all():
                failures.append(f"{name} G={G}: rank {rank} merged a key it does not own")
            m.close()
            res = D.gather_result(owned, fr)
            if rank == 0:
                tag = f"{name} G={G}"
                if not np.array_equal(res["key"], fa):
                    failures.append(f"{tag}: keys / global first-appearance order differ")
                    continue
                so = np.argsort(res["key"], kind="stable")
                for a in AGGS:
                    g_, w_ = res[a][so], want[a]
                    if a == "count":
                        if not np.array_equal(g_, w_):
                            failures.append(f"{tag} {a}: {(g_ != w_).sum()} groups differ")
                        continue
                    scale = {"variance": m2, "stddev": np.sqrt(m2)}.get(a, np.abs(w_))
                    rel = np.abs(g_ - w_) / np.maximum(np.abs(w_), scale)
                    if not rel.max() <= 1e-12:
                        failures.append(f"{tag} {a}: rel err {rel.max():.3e}")
        gb.close()
        if rank == 0:
            ora.close()
    if rank == 0:
        print("phases of the last c-abi step:", comm.phases())
    bad = torch.tensor([len(failures)], device=dev)
    dist.all_reduce(bad)
    for f in failures:
        print(f"[rank {rank}] FAIL {f}")
    comm.close()
    dist.destroy_process_group()
    if bad.item():
        sys.exit(1)
    if rank == 0:
        print("NCCL STAGE2 PARITY OK")


if __name__ == "__main__":
    main()
