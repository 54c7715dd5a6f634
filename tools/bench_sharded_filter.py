"""Per-shard cost of label filters on the global-threshold sharded search, G shards emulated on one GPU.

    python tools/bench_sharded_filter.py --out profiles/bench_sharded_filter_n1.json

Every emulated shard is the same 10M x 384 rows (views of one catalog, id_offset r * 10M) with its own label words, so a
catalog of G * 10M rows is searched the way G ranks would search it: the per-rank calls (shard_sample, the gathered
top-r lists, shard_search_into) run in sequence on one device, then tt_shard_merge.  G = 4 and 8, K 100, nq 1024 and
4096.  Arms, alternated with warm-ups first: no filter | random label bits at selectivity 0.5, 0.1, 1e-2, 1e-3 |
"clustered" (1 % of the catalog allowed, every allowed row in the last shard).  Per arm and shard: the main-scan kernel
time (tt_profile_scan_*) and the records that overflowed their candidate segments; per arm, the queries the merged
certificate rejects (not re-run: a query is certified once for the whole catalog, not per shard).  Because every shard
holds the same rows, each catalog row appears G times: the per-shard scan time is that of a real 10M-row shard, but the
sampled threshold and the uncertified counts are those of this duplicated catalog.  The device name and power limit are
read in the same run.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import bench  # noqa: E402
import two_tower_model_v2_b200 as pkg  # noqa: E402
from bench_exclude import device_info  # noqa: E402
from two_tower_model_v2_b200 import _native, ops  # noqa: E402
from two_tower_model_v2_b200.sharded import record_layout, record_views  # noqa: E402

N_SHARD, D, K = 10_000_000, 384, 100
SELECTIVITY_BITS = {0.5: 1, 0.1: 2, 1e-2: 3, 1e-3: 4}      # label bit b is set with probability s
CLUSTERED_BIT = 5


def make_shards(base, G):
    gen = torch.Generator(device="cuda").manual_seed(17 + G)
    shards = []
    for r in range(G):
        idx = pkg.FlatIPIndex(base.d, base.device)
        idx.xn = idx._xn_store = base.xn
        idx.xh = idx._xh_store = base.xh
        idx.stats = base.stats
        idx.id_offset = r * N_SHARD
        lab = torch.zeros(N_SHARD, device="cuda", dtype=torch.int64)
        for s, b in SELECTIVITY_BITS.items():
            lab |= (torch.rand(N_SHARD, device="cuda", generator=gen) < s).to(torch.int64) << b
        if r == G - 1:          # 1 % of the whole catalog, all of it here
            lab |= (torch.rand(N_SHARD, device="cuda", generator=gen) < 0.01 * G).to(torch.int64) << CLUSTERED_BIT
        idx.set_labels(lab)
        shards.append(idx)
    return shards


def step(shards, q, req, bufs):
    """One sharded search of q: every shard's sample, the gathered lists, every shard's main scan + finalize, merge.
    -> (uncertified queries after the merge, per-shard count of records that overflowed their candidate segments)."""
    G, nq, n_total = len(shards), q.shape[0], len(shards) * N_SHARD
    topr_g, lay, gathered = bufs
    kw = {} if req is None else {"require": req}
    for r, idx in enumerate(shards):
        idx.shard_sample(q, K, n_total, topr_g[r], **kw)
    for r, idx in enumerate(shards):
        s, i, b, f = record_views(gathered[r], lay, nq, K)
        idx.shard_search_into(nq, K, n_total, topr_g, s, i, b, f, **kw)
    _, _, _, nunc = ops.shard_merge(gathered, lay.off_scores, lay.off_ids, lay.off_bound, lay.off_flags, nq, K)
    f = record_views(gathered, lay, nq, K)[3]
    return nunc, ((f <= 0) & (((-f) & 1) == 1)).sum(1)


def time_arm(shards, qs, req, steps, bufs):
    lib = _native.load()
    G = len(shards)
    lib.tt_profile_scan_arm(G * steps)
    torch.cuda.synchronize()
    out = [step(shards, qs[j % len(qs)], req, bufs) for j in range(steps)]
    torch.cuda.synchronize()
    sm = torch.empty(G * steps, dtype=torch.float32)
    n = lib.tt_profile_scan_read(sm.data_ptr(), G * steps)
    assert n == G * steps, n
    return (sm.view(steps, G).mean(0).tolist(), int(sum(int(u.item()) for u, _ in out)),
            torch.stack([o for _, o in out]).sum(0).tolist())


def case(shards, nq, steps, rounds):
    G = len(shards)
    assert shards[0].shard_plan_ok(G * N_SHARD, nq, K, N_SHARD)
    g = torch.Generator(device="cuda").manual_seed(4325 + nq)
    qs = [torch.randn((nq, D), device="cuda", generator=g) for _ in range(3)]
    lay = record_layout(nq, K)
    bufs = (torch.empty((G, nq, _native.TT_SHARD_TOPR), device="cuda"), lay,
            torch.zeros((G, lay.nbytes), dtype=torch.uint8, device="cuda"))
    arms = {"no_filter": None}
    arms.update({f"s={s:g}": np.array([1 << b, 0]) for s, b in SELECTIVITY_BITS.items()})
    arms["clustered_s=0.01"] = np.array([1 << CLUSTERED_BIT, 0])
    for req in arms.values():
        time_arm(shards, qs, req, 1, bufs)
    acc = {a: [] for a in arms}
    for _ in range(rounds):
        for a, req in arms.items():
            acc[a].append(time_arm(shards, qs, req, steps, bufs))
    rows = []
    for a in arms:
        per_shard = np.array([r[0] for r in acc[a]])          # [rounds, G]
        rows.append({"G": G, "rows_per_shard": N_SHARD, "d": D, "nq": nq, "k": K, "arm": a,
                     "scan_ms_per_shard": per_shard.mean(0).round(4).tolist(),
                     "scan_ms_mean": float(per_shard.mean()), "scan_ms_rounds": per_shard.mean(1).round(4).tolist(),
                     "uncertified": int(sum(r[1] for r in acc[a])),
                     "overflow_records_per_shard": np.sum([r[2] for r in acc[a]], 0).tolist(),
                     "queries": nq * steps * rounds})
        print(json.dumps(rows[-1]), flush=True)
    for r in rows:
        r["scan_vs_no_filter"] = r["scan_ms_mean"] / rows[0]["scan_ms_mean"]
        r["scan_vs_no_filter_per_shard"] = (np.array(r["scan_ms_per_shard"]) /
                                            np.array(rows[0]["scan_ms_per_shard"])).round(3).tolist()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=4)
    args = ap.parse_args()
    out = {"info": device_info(), "note": "G shards emulated on one GPU (each the same 10M x 384 rows with its own "
           "labels; 15.4 GB fp32 + 7.7 GB bf16, far above L2); per-rank calls in sequence; alternating arms, warm-ups "
           "first; scan_ms = main scan kernel per shard (CUDA events); uncertified = queries the merged certificate "
           "rejects (a real search re-runs them exactly)", "rows": []}
    print(json.dumps(out["info"]), flush=True)
    base, _, _ = bench.make_shard(N_SHARD, D, 1, 0)
    for G in (4, 8):
        shards = make_shards(base, G)
        for nq in (1024, 4096):
            out["rows"] += case(shards, nq, args.steps, args.rounds)
        del shards
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
