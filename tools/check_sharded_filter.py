#!/usr/bin/env python
"""Multi-GPU parity check of label filters on the sharded search (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29512 \
        tools/check_sharded_filter.py [N] [D] [nq] [K]

Every rank owns a row shard of the same seeded catalog and sets the same seeded GLOBAL label words through
ShardedFlatIPIndex.set_labels.  For each filter - random label bits at selectivity 0.1 and 0.01, a "clustered" filter
whose allowed rows all lie in the last shard, and the 0.1 filter with each query's own best allowed rows excluded - the
merged top-K of search_device and of search_host_sliced_async (each rank submits its share of the batch and its masks)
must equal, ids and scores bit for bit, the filtered top-K of one unsharded index on rank 0's GPU.
"""
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
import two_tower_model_v2_b200 as pkg  # noqa: E402


def global_labels(n_total, world):
    """Bit 1: s = 0.1, bit 2: s = 0.01, bit 3: 1 % of the catalog, all in the last shard; bits 8-31 noise."""
    g = torch.Generator(device="cuda").manual_seed(808)
    lab = torch.randint(0, 1 << 24, (n_total,), device="cuda", generator=g) << 8
    lab |= (torch.rand(n_total, device="cuda", generator=g) < 0.1).to(torch.int64) << 1
    lab |= (torch.rand(n_total, device="cuda", generator=g) < 0.01).to(torch.int64) << 2
    lo, hi = pkg.shard_bounds(n_total, world, world - 1)
    last = torch.zeros(n_total, device="cuda", dtype=torch.bool)
    last[lo:hi] = torch.rand(hi - lo, device="cuda", generator=g) < 0.01 * n_total / (hi - lo)
    return lab | (last.to(torch.int64) << 3)


def main():
    n_total = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
    d = int(sys.argv[2]) if len(sys.argv) > 2 else 384
    nq = int(sys.argv[3]) if len(sys.argv) > 3 else 256
    k = int(sys.argv[4]) if len(sys.argv) > 4 else 50
    world, rank, local = bench.dist_setup(0)
    torch.cuda.set_device(local)
    index, lo, hi = bench.make_shard(n_total, d, world, rank)
    sharded = pkg.ShardedFlatIPIndex(index, n_total)
    labels = global_labels(n_total, world)
    sharded.set_labels(labels)
    q = torch.randn((nq, d), device="cuda", generator=torch.Generator(device="cuda").manual_seed(4326))
    full = None
    if rank == 0:
        full, _, _ = bench.make_shard(n_total, d, 1, 0)
        full.set_labels(labels)
    nl = nq // world
    ok = True
    for name, bit, excl in (("s=0.1", 1, False), ("s=0.01", 2, False), ("clustered", 3, False),
                            ("s=0.1+exclude", 1, True)):
        req = np.array([1 << bit, 0])
        kw = {}
        if excl:       # each query's own 20 best allowed rows (rank 0 finds them; every rank gets the same list)
            ex = torch.empty((nq, 20), device="cuda", dtype=torch.int64)
            if rank == 0:
                ex.copy_(full.search_checked_device(q, 20, require=req)[1])
            if world > 1:
                dist.broadcast(ex, 0)
            kw["exclude"] = ex
        s, i, n_bad = sharded.search_device(q, k, require=req, **kw)
        if not excl:    # the sliced call takes masks but no exclusion list
            hs, hi_, _ = sharded.search_host_sliced_async(q[rank * nl:(rank + 1) * nl].cpu().numpy(), k,
                                                          require=req).result()
        torch.cuda.synchronize()
        if rank == 0:
            fs, fi, fbad = full.search_checked_device(q, k, require=req, **kw)
            same = torch.equal(i, fi) and torch.equal(s, fs)
            sliced = excl or (np.array_equal(hi_, fi[:nl].cpu().numpy()) and np.array_equal(hs, fs[:nl].cpu().numpy()))
            allowed = bool(((labels[i[i >= 0]] >> bit) & 1).all())
            print(f"world {world} N {n_total} D {d} nq {nq} K {k} {name}: sharded == single {same}, sliced {sliced}, "
                  f"only allowed rows {allowed}, re-run sharded {n_bad} single {fbad}, exchange {sharded.exchange_used}",
                  flush=True)
            ok &= same and sliced and allowed
    flag = torch.tensor([1 if ok else 0], device="cuda")
    sharded.close()
    if world > 1:
        dist.broadcast(flag, 0)
        dist.destroy_process_group()
    if rank == 0:
        print("OK" if ok else "FAIL", flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == "__main__":
    main()
