"""Cost of exclusion lists on one GPU (tt_flat_search_excl, RetrievalPipeline(exclude_history=True)).

    python tools/bench_exclude.py --out profiles/exclude.json

Cases, each as alternating arms with warm-ups in the same process (device-resident timing, CUDA events):
  * 10M x 384, nq 4096, K 100: no list | 50 random rows per query | each query's own top-50 (the adversarial list)
  * 1M x 384, K 10, nq 1 and 128: no list | each query's own top-100
  * /retrieve on the 10M x 384 catalog, K 100, 50-event histories, batch 1 and 1024: without / with exclude_history
Per arm: mean step time, mean main-scan kernel time (tt_profile_scan_*), uncertified queries (re-run through the
exact path inside the timed step).  The device name and power limit are read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
import two_tower_model_v2_b200 as pkg  # noqa: E402
from two_tower_model_v2_b200 import _native  # noqa: E402


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:          # the numbers stay valid; say that the limit could not be read
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e!r})"
    return info


def own_top(index, q, e):
    """Each query's own top-e rows (fp32 torch checker): the list that costs the search most."""
    return bench.torch_flat_topk(index.xn, q, e)[1].contiguous()


def time_search(index, qs, k, lists, steps):
    """`steps` checked searches (uncertified queries re-run exactly inside the step) -> (ms/step, scan ms, n_unc)."""
    lib = _native.load()
    lib.tt_profile_scan_arm(steps)
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    n_unc = 0
    e0.record()
    for j in range(steps):
        kw = {} if lists is None else {"exclude": lists[j % len(lists)]}
        _, _, n = index.search_checked_device(qs[j % len(qs)], k, **kw)
        n_unc += n
    e1.record()
    torch.cuda.synchronize()
    sm = torch.empty(steps, dtype=torch.float32)
    n = lib.tt_profile_scan_read(sm.data_ptr(), steps)
    return e0.elapsed_time(e1) / steps, float(sm[:n].mean()) if n > 0 else None, n_unc


def search_case(index, name, nq, k, arms, steps, rounds, nbatch):
    """arms: {label: None | function(q) -> list}; alternated `rounds` times after one warm-up pass each."""
    d = index.d
    g = torch.Generator(device="cuda").manual_seed(4321 + nq)
    qs = [torch.randn((nq, d), device="cuda", generator=g) for _ in range(nbatch)]
    lists = {a: (None if f is None else [f(q) for q in qs]) for a, f in arms.items()}
    for a in arms:
        time_search(index, qs, k, lists[a], 2)
    acc = {a: [] for a in arms}
    for _ in range(rounds):
        for a in arms:
            acc[a].append(time_search(index, qs, k, lists[a], steps))
    rows = []
    for a in arms:
        ms = [r[0] for r in acc[a]]
        scan = [r[1] for r in acc[a] if r[1] is not None]
        rows.append({"case": name, "nq": nq, "k": k, "arm": a, "E": 0 if lists[a] is None else int(lists[a][0].shape[1]),
                     "ms_per_step": sum(ms) / len(ms), "ms_per_step_rounds": ms,
                     "scan_ms": sum(scan) / len(scan) if scan else None,
                     "uncertified": int(sum(r[2] for r in acc[a])), "queries": nq * steps * rounds})
        print(json.dumps(rows[-1]), flush=True)
    base = rows[0]["ms_per_step"]
    for r in rows:
        r["vs_no_list"] = r["ms_per_step"] / base
    return rows


def retrieve_case(index, k, batch, steps, rounds):
    """One-GPU /retrieve: 50-event histories -> fused gather + pool -> exact top-k, with and without the history
    as the exclusion list.  Host clock around each request (it ends in the certificate's synchronisation)."""
    db = pkg.VectorDatabase(index.d)
    db.index = index
    torch.manual_seed(0)
    pipe = pkg.RetrievalPipeline(pkg.BuyerTower(index.d, "weighted_avg").cuda(), db)
    g = torch.Generator(device="cuda").manual_seed(99 + batch)
    reqs = [(torch.randint(0, index.ntotal, (batch, 50), device="cuda", generator=g),
             torch.rand((batch, 50), device="cuda", generator=g) * 9 + 1) for _ in range(8)]
    arms = {"no_list": False, "exclude_history": True}

    def run(flag, n):
        times, n_unc = [], 0
        for j in range(n):
            idx, w = reqs[j % len(reqs)]
            t0 = time.perf_counter()
            p = pipe.retrieve_device_async(idx, w, k, exclude_history=True) if flag else pipe.retrieve_device_async(idx, w, k)
            _, _, nb = p.result()
            times.append((time.perf_counter() - t0) * 1e3)
            n_unc += nb
        return times, n_unc
    for f in arms.values():
        run(f, 3)
    acc = {a: ([], 0) for a in arms}
    for _ in range(rounds):
        for a, f in arms.items():
            t, n = run(f, steps)
            acc[a] = (acc[a][0] + t, acc[a][1] + n)
    rows = []
    for a in arms:
        t = sorted(acc[a][0])
        rows.append({"case": "retrieve_10Mx384", "batch": batch, "k": k, "arm": a, "ms_mean": sum(t) / len(t),
                     "ms_p50": t[len(t) // 2], "ms_p99": t[min(len(t) - 1, int(len(t) * 0.99))],
                     "uncertified": acc[a][1], "requests": len(t)})
        print(json.dumps(rows[-1]), flush=True)
    rows[1]["vs_no_list"] = rows[1]["ms_mean"] / rows[0]["ms_mean"]
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    out = {"info": device_info(), "note": "alternating arms, warm-ups first; step = search + exact re-run of "
           "uncertified queries; scan_ms = main scan kernel (CUDA events); catalog 10M x 384 is 15.4 GB fp32 + "
           "7.7 GB bf16, far above L2", "rows": []}
    print(json.dumps(out["info"]), flush=True)
    index, _, _ = bench.make_shard(10_000_000, 384, 1, 0)
    gen = torch.Generator(device="cuda").manual_seed(7)
    out["rows"] += search_case(index, "10Mx384", 4096, 100, {
        "no_list": None,
        "random_50": lambda q: torch.randint(0, index.ntotal, (q.shape[0], 50), device="cuda", generator=gen),
        "own_top_50": lambda q: own_top(index, q, 50)}, steps=10, rounds=args.rounds, nbatch=4)
    for batch in (1, 1024):
        out["rows"] += retrieve_case(index, 100, batch, steps=100 if batch == 1 else 10, rounds=args.rounds)
    del index
    torch.cuda.empty_cache()
    index, _, _ = bench.make_shard(1_000_000, 384, 1, 0)
    for nq in (1, 128):
        out["rows"] += search_case(index, "1Mx384", nq, 10, {"no_list": None, "own_top_100": lambda q: own_top(index, q, 100)},
                                   steps=200 if nq == 1 else 50, rounds=args.rounds, nbatch=8)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
