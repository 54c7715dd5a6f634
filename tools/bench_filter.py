"""Cost of label filters on one GPU (tt_flat_search_filtered, RetrievalPipeline(require_any=...)).

    python tools/bench_filter.py --out profiles/bench_filter_n1.json

Cases, each as alternating arms with warm-ups in the same process (device-resident timing, CUDA events):
  * 10M x 384, K 100, nq 1, 128 and 4096: no filter (tt_flat_search) | the trivial filter (0, 0) through the filtered
    kernels (the cost of the mask alone) | filters of selectivity 0.5, 0.1, 1e-2, 1e-3 (one label bit each)
  * /retrieve on the same catalog, K 100, 50-event histories, batch 1 and 1024: plain | exclude_history | a two-category
    filter (require_any, ~1/4 of the catalog) | both
Per search arm: mean step time, mean main-scan kernel time (tt_profile_scan_*), candidates per query
(tt_flat_debug_read: rows the main scan kept, summed over slices) and uncertified queries (re-run through the exact path
inside the timed step).  The device name and power limit are read in the same run.
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
from two_tower_model_v2_b200 import _native, ops  # noqa: E402

SELECTIVITY_BITS = {0.5: 1, 0.1: 2, 1e-2: 3, 1e-3: 4}      # label bit b is set with probability s
CATEGORY_BIT0, N_CATEGORIES = 8, 8                          # bits 8..15: one category per item


def make_labels(n, gen):
    lab = torch.zeros(n, device="cuda", dtype=torch.int64)
    for s, b in SELECTIVITY_BITS.items():
        lab |= (torch.rand(n, device="cuda", generator=gen) < s).to(torch.int64) << b
    lab |= 1 << (CATEGORY_BIT0 + torch.randint(0, N_CATEGORIES, (n,), device="cuda", generator=gen))
    return lab


def search(index, q, k, req):
    """One checked search; req None = tt_flat_search, else tt_flat_search_filtered with the int32 [nq, 2] masks (also
    when they are all zero).  Uncertified queries are re-run exactly.  -> (workspace, n_uncertified)"""
    lib = _native.load()
    nq = q.shape[0]
    s = torch.empty((nq, k), device="cuda")
    i = torch.empty((nq, k), device="cuda", dtype=torch.int64)
    flags = torch.empty(nq, device="cuda", dtype=torch.int32)
    nunc = torch.empty(1, device="cuda", dtype=torch.int32)
    ws = index._workspace(nq, k)
    args = (q.data_ptr(), nq, index.xn.data_ptr(), index.xh.data_ptr(), index.stats.data_ptr(), index.ntotal, index.d, k,
            0, s.data_ptr(), i.data_ptr(), flags.data_ptr(), nunc.data_ptr())
    if req is None:
        _native.check(lib.tt_flat_search(*args, ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_search")
    else:
        _native.check(lib.tt_flat_search_filtered(*args, index.labels.data_ptr(), req.data_ptr(), None, 0, ws.data_ptr(),
                                                  ws.numel(), ops._stream()), "tt_flat_search_filtered")
    n_bad = int(nunc.item())
    if n_bad:
        qsel = torch.nonzero(flags != 1).flatten().to(torch.int32)
        index.search_exact_device(q, k, s, i, qsel, **({} if req is None else {"require": req}))
    return ws, n_bad


def candidates(index, q, k, req):
    ws, _ = search(index, q, k, req)
    nq = q.shape[0]
    thr = torch.empty(nq, device="cuda")
    cnt = torch.empty(nq, device="cuda", dtype=torch.int32)
    _native.check(_native.load().tt_flat_debug_read(ws.data_ptr(), index.ntotal, index.d, nq, k, thr.data_ptr(),
                                                    cnt.data_ptr(), ops._stream()), "tt_flat_debug_read")
    c = cnt.double()
    return {"cand_mean": float(c.mean()), "cand_min": int(cnt.min()), "cand_max": int(cnt.max()),
            "queries_with_thr_neg_inf": int(torch.isneginf(thr).sum())}


def time_arm(index, qs, k, req, steps):
    lib = _native.load()
    lib.tt_profile_scan_arm(steps)
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    torch.cuda.synchronize()
    n_unc = 0
    e0.record()
    for j in range(steps):
        n_unc += search(index, qs[j % len(qs)], k, req)[1]
    e1.record()
    torch.cuda.synchronize()
    sm = torch.empty(steps, dtype=torch.float32)
    n = lib.tt_profile_scan_read(sm.data_ptr(), steps)
    return e0.elapsed_time(e1) / steps, float(sm[:n].mean()) if n > 0 else None, n_unc


def search_case(index, nq, k, steps, rounds, nbatch):
    g = torch.Generator(device="cuda").manual_seed(4321 + nq)
    qs = [torch.randn((nq, index.d), device="cuda", generator=g) for _ in range(nbatch)]

    def masks(all_bits):
        return torch.tensor([[all_bits, 0]] * nq, device="cuda", dtype=torch.int32)
    arms = {"no_filter": None, "trivial_filter": masks(0)}
    arms.update({f"s={s:g}": masks(1 << b) for s, b in SELECTIVITY_BITS.items()})
    for req in arms.values():
        time_arm(index, qs, k, req, 2)
    acc = {a: [] for a in arms}
    for _ in range(rounds):
        for a, req in arms.items():
            acc[a].append(time_arm(index, qs, k, req, steps))
    rows = []
    for a, req in arms.items():
        ms = [r[0] for r in acc[a]]
        scan = [r[1] for r in acc[a] if r[1] is not None]
        rows.append({"case": "10Mx384", "nq": nq, "k": k, "arm": a, "ms_per_step": sum(ms) / len(ms),
                     "ms_per_step_rounds": ms, "scan_ms": sum(scan) / len(scan) if scan else None,
                     "scan_ms_rounds": scan, "uncertified": int(sum(r[2] for r in acc[a])),
                     "queries": nq * steps * rounds, **candidates(index, qs[0], k, req)})
        print(json.dumps(rows[-1]), flush=True)
    base = rows[0]
    for r in rows:
        r["step_vs_no_filter"] = r["ms_per_step"] / base["ms_per_step"]
        if r["scan_ms"] and base["scan_ms"]:
            r["scan_vs_no_filter"] = r["scan_ms"] / base["scan_ms"]
    return rows


def retrieve_case(index, k, batch, steps, rounds):
    """One-GPU /retrieve: 50-event histories -> fused gather + pool -> exact top-k; host clock around each request (it
    ends in the certificate's synchronisation)."""
    db = pkg.VectorDatabase(index.d)
    db.index = index
    torch.manual_seed(0)
    pipe = pkg.RetrievalPipeline(pkg.BuyerTower(index.d, "weighted_avg").cuda(), db)
    g = torch.Generator(device="cuda").manual_seed(99 + batch)
    reqs = [(torch.randint(0, index.ntotal, (batch, 50), device="cuda", generator=g),
             torch.rand((batch, 50), device="cuda", generator=g) * 9 + 1) for _ in range(8)]
    cat = (1 << CATEGORY_BIT0) | (1 << (CATEGORY_BIT0 + 3))          # two of the eight categories
    arms = {"plain": {}, "exclude_history": {"exclude_history": True}, "category": {"require_any": cat},
            "category_exclude_history": {"require_any": cat, "exclude_history": True}}

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
        rows.append({"case": "retrieve_10Mx384", "batch": batch, "k": k, "arm": a, "ms_mean": sum(t) / len(t),
                     "ms_p50": t[len(t) // 2], "ms_p99": t[min(len(t) - 1, int(len(t) * 0.99))],
                     "uncertified": acc[a][1], "requests": len(t)})
        print(json.dumps(rows[-1]), flush=True)
    for r in rows:
        r["vs_plain"] = r["ms_mean"] / rows[0]["ms_mean"]
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    out = {"info": device_info(), "note": "alternating arms, warm-ups first; step = search + exact re-run of "
           "uncertified queries; scan_ms = main scan kernel (CUDA events); candidates from one extra search per arm; "
           "catalog 10M x 384 is 15.4 GB fp32 + 7.7 GB bf16 + 40 MB of label words, far above L2", "rows": []}
    print(json.dumps(out["info"]), flush=True)
    index, _, _ = bench.make_shard(10_000_000, 384, 1, 0)
    index.set_labels(make_labels(index.ntotal, torch.Generator(device="cuda").manual_seed(5)))
    for nq, steps in ((1, 100), (128, 30), (4096, 10)):
        out["rows"] += search_case(index, nq, 100, steps=steps, rounds=args.rounds, nbatch=4)
    for batch in (1, 1024):
        out["rows"] += retrieve_case(index, 100, batch, steps=100 if batch == 1 else 10, rounds=args.rounds)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
