"""Cost of range search on one GPU (tt_flat_range_search) against the workaround it replaces.

    python tools/bench_range.py --out profiles/bench_range_n1.json

10M x 384 catalog (bench.make_shard), nq 1, 128 and 4096.  Each query's radius lies between its target-th and
(target+1)-th exact fp32 scores, for targets of 10, 100, 1000 and 10000 rows.  Two arms, alternated with warm-ups in the
same process, both ending with the results on the host:
  * topk : search_device with K = min(target, 2048) (uncertified queries re-run exactly), then a host-side cut at the radius
  * range: range_search_async with L = that K (overflowed and uncertified queries re-run inside the step)
Per arm: mean step time, mean main-scan kernel time (tt_profile_scan_*), re-runs (tensor path / exact path) and, for
candidates per query (tt_flat_debug_read for the top-K arm, tt_flat_range_debug_read for the range arm: rows the main
scan kept, summed over slices).
One extra case: 1M x 384, nq 128, a radius at the median score (half the catalog qualifies).  The device name and
power limit are read in the same run.
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
from bench_exclude import device_info  # noqa: E402
from two_tower_model_v2_b200 import _native, ops  # noqa: E402


def radius_at(index, q, target):
    ts, _ = bench.torch_flat_topk(index.xn, q, target + 1)
    return 0.5 * (ts[:, target - 1] + ts[:, target])


def topk_step(index, q, rad, k):
    s, i, n_bad = index.search_checked_device(q, k)
    s, i, r = s.cpu(), i.cpu(), rad.cpu()
    keep = s > r[:, None]                       # the host-side cut
    return int(n_bad), int(keep.sum())


def range_step(index, q, rad, L):
    c, s, i, n_t, n_x = index.range_search_async(q, rad, L).result()
    c, s, i = c.cpu(), s.cpu(), i.cpu()
    return n_t, n_x, int(c.sum())


def time_arm(fn, steps):
    lib = _native.load()
    lib.tt_profile_scan_arm(steps)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = [fn() for _ in range(steps)]
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    scan = torch.empty(steps)
    n = lib.tt_profile_scan_read(scan.data_ptr(), steps)
    return ms, (float(scan[:n].mean()) if n > 0 else None), outs[-1]


def topk_candidates(index, q, k):
    nq = q.shape[0]
    index.search_device(q, k)
    ws = index._workspace(nq, k)
    thr = torch.empty(nq, device="cuda")
    cnt = torch.empty(nq, device="cuda", dtype=torch.int32)
    _native.check(_native.load().tt_flat_debug_read(ws.data_ptr(), index.ntotal, index.d, nq, k, thr.data_ptr(),
                                                    cnt.data_ptr(), ops._stream()), "tt_flat_debug_read")
    return float(cnt.double().mean())


def range_candidates(index, q, L):
    """Rows the range scan kept per query (its segment counters, summed), read from the workspace of the last call."""
    nq = q.shape[0]
    ws = index._range_workspace(nq, index._range_budget(nq, L))
    cnt = torch.empty(nq, device="cuda", dtype=torch.int32)
    _native.check(_native.load().tt_flat_range_debug_read(ws.data_ptr(), index.ntotal, index.d, nq, cnt.data_ptr(),
                                                          ops._stream()), "tt_flat_range_debug_read")
    return float(cnt.double().mean())


def run_case(index, q, rad, k, steps, warmup, rounds=2):
    rec = {"topk": [], "range": []}
    for _ in range(warmup):
        topk_step(index, q, rad, k)
        range_step(index, q, rad, k)
    for _ in range(rounds):                     # alternated: topk, range, topk, range
        ms, scan, (n_bad, kept) = time_arm(lambda: topk_step(index, q, rad, k), steps)
        rec["topk"].append({"step_ms": ms, "scan_ms": scan, "rerun_exact": n_bad, "rows_kept_per_query": kept / q.shape[0]})
        ms, scan, (n_t, n_x, total) = time_arm(lambda: range_step(index, q, rad, k), steps)
        rec["range"].append({"step_ms": ms, "scan_ms": scan, "rerun_tensor": n_t, "rerun_exact": n_x,
                             "rows_above_radius_per_query": total / q.shape[0]})
    rec["topk_candidates_per_query"] = topk_candidates(index, q, k)
    _, _, _, _, need, _ = index.range_search_device(q, rad, k)
    rec["range_largest_segment_count_mean"] = float(need.double().mean())
    rec["range_candidates_per_query"] = range_candidates(index, q, k)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--n", type=int, default=10_000_000)
    args = ap.parse_args()
    out = {"device": device_info(), "catalog": [args.n, 384], "cases": []}
    index, _, _ = bench.make_shard(args.n, 384, 1, 0)
    for nq in (1, 128, 4096):
        for target in (10, 100, 1000, 10000):
            q = torch.randn((nq, 384), device="cuda", generator=torch.Generator(device="cuda").manual_seed(7 + nq + target))
            rad = radius_at(index, q, target)
            k = min(target, _native.TT_FLAT_MAX_K)
            r = run_case(index, q, rad, k, args.steps, args.warmup)
            out["cases"].append({"N": args.n, "nq": nq, "target": target, "k": k, **r})
            print(json.dumps(out["cases"][-1]), flush=True)
    del index
    torch.cuda.empty_cache()
    index, _, _ = bench.make_shard(1_000_000, 384, 1, 0)
    q = torch.randn((128, 384), device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    rad = radius_at(index, q, 500_000)
    for _ in range(args.warmup):
        range_step(index, q, rad, 2048)
    ms, scan, (n_t, n_x, total) = time_arm(lambda: range_step(index, q, rad, 2048), args.steps)
    out["huge_band"] = {"N": 1_000_000, "nq": 128, "L": 2048, "radius": "median score", "step_ms": ms, "scan_ms": scan,
                        "rerun_tensor": n_t, "rerun_exact": n_x, "rows_above_radius_per_query": total / 128}
    print(json.dumps(out["huge_band"]), flush=True)
    out["device_after"] = device_info()
    Path(args.out).write_text(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
