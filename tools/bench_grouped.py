"""Cost of the per-group cap on one GPU (tt_flat_search_grouped, RetrievalPipeline(max_per_group=...)).

    python tools/bench_grouped.py --out profiles/bench_grouped_n1.json

Catalog 10M x 384 (bench.make_shard), K 100, nq 1, 128 and 4096, two group layouts over 10 000 groups:
  * random: every row's group drawn uniformly (seeded);
  * clustered: every row's group is the nearest of 10 000 seeded random unit directions (fp32 on the device, in
    chunks), so similar rows share a group and a query's best rows crowd into few groups: the hard case.
Arms, alternated with warm-ups in the same process: plain search_async | grouped search_async with m = 1 | m = 3.
Per arm: mean step time (CUDA events; a step includes the exact re-run of uncertified queries), the finalize kernel's
time (torch.profiler, in a run of its own), how many queries were re-run, and the exact path's time per re-run query
(CUDA events around tt_flat_search_exact_grouped over batches of 8 queries).  /retrieve: batch 1 and 1024, 50-event
histories, with and without max_per_group=2 (random layout).  The device name, power limit and max SM clock are read
in the same run.  Every input is seeded, so a rerun gives the same re-run counts.
"""
import argparse
import json
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import bench  # noqa: E402
import two_tower_model_v2_b200 as pkg  # noqa: E402
from bench_exclude import device_info  # noqa: E402

N_GROUPS = 10_000


def random_groups(n):
    g = torch.Generator(device="cuda").manual_seed(77)
    return torch.randint(0, N_GROUPS, (n,), device="cuda", generator=g)


def clustered_groups(xn, chunk=1 << 18):
    g = torch.Generator(device="cuda").manual_seed(78)
    dirs = torch.randn((N_GROUPS, xn.shape[1]), device="cuda", generator=g)
    dirs /= dirs.norm(dim=1, keepdim=True)
    out = torch.empty(xn.shape[0], device="cuda", dtype=torch.int64)
    for lo in range(0, xn.shape[0], chunk):
        out[lo:lo + chunk] = torch.argmax(xn[lo:lo + chunk] @ dirs.t(), dim=1)
    return out


def time_arm(index, qs, k, m, steps):
    kw = {} if m is None else {"max_per_group": m}
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    n_rerun = 0
    e0.record()
    for j in range(steps):
        n_rerun += index.search_async(qs[j % len(qs)], k, **kw).result()[2]
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, n_rerun


def finalize_ms(index, q, k, m, steps=3):
    """Mean device time per step of the finalize kernel (flat_finalize_kernel / flat_group_finalize_kernel)."""
    kw = {} if m is None else {"max_per_group": m}
    index.search_device(q, k, **kw)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            index.search_device(q, k, **kw)
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "finalize_kernel" in e.key)
    return us / steps / 1e3


def exact_ms_per_query(index, q, k, m, reps=3):
    kw = {} if m is None else {"max_per_group": m}
    qs = q[:8]
    s = torch.empty((qs.shape[0], k), device="cuda")
    i = torch.empty((qs.shape[0], k), device="cuda", dtype=torch.int64)
    index.search_exact_device(qs, k, s, i, **kw)
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        index.search_exact_device(qs, k, s, i, **kw)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps / qs.shape[0]


def search_case(index, layout, nq, k, steps, rounds, nbatch=4):
    g = torch.Generator(device="cuda").manual_seed(4321 + nq)
    qs = [torch.randn((nq, index.d), device="cuda", generator=g) for _ in range(nbatch)]
    arms = {"plain": None, "m=1": 1, "m=3": 3}
    for m in arms.values():
        time_arm(index, qs, k, m, 2)
    acc = {a: [] for a in arms}
    for _ in range(rounds):
        for a, m in arms.items():
            acc[a].append(time_arm(index, qs, k, m, steps))
    rows = []
    for a, m in arms.items():
        ms = [r[0] for r in acc[a]]
        rows.append({"case": "10Mx384", "layout": layout, "nq": nq, "k": k, "arm": a, "ms_per_step": sum(ms) / len(ms),
                     "ms_per_step_rounds": ms, "queries": nq * steps * rounds,
                     "rerun_queries": int(sum(r[1] for r in acc[a])),
                     "finalize_ms": finalize_ms(index, qs[0], k, m),
                     "exact_ms_per_rerun_query": exact_ms_per_query(index, qs[0], k, m)})
        rows[-1]["rerun_rate"] = rows[-1]["rerun_queries"] / rows[-1]["queries"]
        print(json.dumps(rows[-1]), flush=True)
    for r in rows:
        r["step_vs_plain"] = r["ms_per_step"] / rows[0]["ms_per_step"]
    return rows


def retrieve_case(index, k, batch, steps, rounds):
    db = pkg.VectorDatabase(index.d)
    db.index = index
    torch.manual_seed(0)
    pipe = pkg.RetrievalPipeline(pkg.BuyerTower(index.d, "weighted_avg").cuda(), db)
    g = torch.Generator(device="cuda").manual_seed(99 + batch)
    reqs = [(torch.randint(0, index.ntotal, (batch, 50), device="cuda", generator=g),
             torch.rand((batch, 50), device="cuda", generator=g) * 9 + 1) for _ in range(8)]
    arms = {"plain": {}, "max_per_group=2": {"max_per_group": 2}}

    def run(kw, n):
        times, n_unc = [], 0
        for j in range(n):
            idx, w = reqs[j % len(reqs)]
            t0 = time.perf_counter()
            _, _, nb = pipe.retrieve_device_async(idx, w, k, **kw).result()
            times.append((time.perf_counter() - t0) * 1e3)
            n_unc += nb
        return times, n_unc
    for kw in arms.values():
        run(kw, 3)
    acc = {a: ([], 0) for a in arms}
    for _ in range(rounds):
        for a, kw in arms.items():
            t, n = run(kw, steps)
            acc[a] = (acc[a][0] + t, acc[a][1] + n)
    rows = []
    for a in arms:
        t = sorted(acc[a][0])
        rows.append({"case": "retrieve_10Mx384", "layout": "random", "batch": batch, "k": k, "arm": a,
                     "ms_mean": sum(t) / len(t), "ms_p50": t[len(t) // 2],
                     "ms_p99": t[min(len(t) - 1, int(len(t) * 0.99))], "rerun_queries": acc[a][1], "requests": len(t)})
        print(json.dumps(rows[-1]), flush=True)
    for r in rows:
        r["vs_plain"] = r["ms_mean"] / rows[0]["ms_mean"]
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    out = {"info": device_info(), "note": "alternating arms, warm-ups first; step = search_async + exact re-run of "
           "uncertified queries; finalize_ms from torch.profiler in separate runs; catalog 10M x 384 is 15.4 GB fp32 + "
           "7.7 GB bf16, far above L2", "rows": []}
    print(json.dumps(out["info"]), flush=True)
    index, _, _ = bench.make_shard(10_000_000, 384, 1, 0)
    for layout in ("random", "clustered"):
        index.set_groups(random_groups(index.ntotal) if layout == "random" else clustered_groups(index.xn))
        # clustered batches re-run many queries on the exact path (~1 ms per query at 10M rows): fewer steps
        sched = ((1, 100), (128, 30), (4096, 10)) if layout == "random" else ((1, 30), (128, 5), (4096, 2))
        for nq, steps in sched:
            out["rows"] += search_case(index, layout, nq, 100, steps=steps, rounds=args.rounds)
        if layout == "random":
            for batch in (1, 1024):
                out["rows"] += retrieve_case(index, 100, batch, steps=100 if batch == 1 else 10, rounds=args.rounds)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
