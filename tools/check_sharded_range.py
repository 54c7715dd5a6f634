#!/usr/bin/env python
"""Multi-GPU parity check of range search on the sharded catalog (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port 29513 \
        tools/check_sharded_range.py [N] [D] [nq]

Every rank owns a row shard of the same seeded catalog (rank 0 also builds the whole catalog on its GPU).  With L = 1000
and radii at about 10, 1000 and 20 000 qualifying rows per query (the last: counts above L), a label filter plus
exclusion lists of global ids, and a per-query radius array, ShardedFlatIPIndex.range_search_device must give rank 0
the counts, ids and scores of FlatIPIndex.range_search_async on the whole catalog.
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


def main():
    n_total = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
    d = int(sys.argv[2]) if len(sys.argv) > 2 else 384
    nq = int(sys.argv[3]) if len(sys.argv) > 3 else 256
    L = 1000
    world, rank, local = bench.dist_setup(0)
    torch.cuda.set_device(local)
    index, lo, hi = bench.make_shard(n_total, d, world, rank)
    sharded = pkg.ShardedFlatIPIndex(index, n_total)
    g = torch.Generator(device="cuda").manual_seed(909)
    labels = torch.randint(0, 1 << 24, (n_total,), device="cuda", generator=g) << 8
    labels |= (torch.rand(n_total, device="cuda", generator=g) < 0.3).to(torch.int64) << 1
    sharded.set_labels(labels)
    q = torch.randn((nq, d), device="cuda", generator=torch.Generator(device="cuda").manual_seed(4327))
    full = None
    if rank == 0:
        full, _, _ = bench.make_shard(n_total, d, 1, 0)
        full.set_labels(labels)
    # radii from the whole catalog's scores on rank 0 (the rank-r score of each query), sent to every rank
    rad = torch.empty((3, nq), device="cuda")
    if rank == 0:
        ts, _ = bench.torch_flat_topk(full.xn, q, 20_001)
        for j, r in enumerate((10, 1000, 20_000)):
            rad[j] = 0.5 * (ts[:, r - 1] + ts[:, r])
    ex = torch.empty((nq, 20), device="cuda", dtype=torch.int64)
    if rank == 0:
        ex.copy_(full.search_checked_device(q, 20, require=np.array([2, 0]))[1])
    if world > 1:
        dist.broadcast(rad, 0)
        dist.broadcast(ex, 0)
    per_query = torch.stack([rad[j % 3, j] for j in range(nq)])
    ok = True
    for name, radius, kw in (("~10 rows", rad[0], {}), ("~1000 rows", rad[1], {}), ("~20000 rows (> L)", rad[2], {}),
                             ("~1000 rows, filter + exclusions", rad[1], {"require": np.array([2, 0]), "exclude": ex}),
                             ("per-query radii", per_query, {})):
        c, s, i, n_bad = sharded.range_search_device(q, radius, L, **kw)
        torch.cuda.synchronize()
        if rank == 0:
            fc, fs, fi, n_t, n_x = full.range_search_async(q, radius, L, **kw).result()
            same_c = torch.equal(c, fc)
            same_l = torch.equal(i, fi) and torch.equal(s, fs)
            print(f"world {world} N {n_total} D {d} nq {nq} L {L} {name}: counts {int(c.min())}..{int(c.max())}, "
                  f"counts equal {same_c}, ids/scores equal {same_l}, re-run sharded {n_bad} single {n_t}+{n_x}",
                  flush=True)
            ok &= same_c and same_l
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
