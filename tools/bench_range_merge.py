#!/usr/bin/env python
"""Cost of merging per-rank range-search records (tt_range_merge) next to the local range step, on one GPU:

    python tools/bench_range_merge.py [--out FILE]

For G in {2, 4, 8}, nq in {1, 128, 4096} and L in {100, 1000, 16384}: the merge of G records whose runs are all full
(count > L, so the kernel selects the best L of G*L keys: its costly case), timed with CUDA events after warm-up; the
bytes one rank sends and the bytes the all-gather delivers; and the local first pass of the sharded range search
(FlatIPIndex.range_shard_into, tt_flat_range_search) over one 10M/G x 384 shard at the same nq and L, radius 0.19
(about 1000 rows per query over the whole 10M catalog, 1000/G per shard).  Card name and power limit are read in the
same run.  One JSON record goes to stdout and to --out.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from two_tower_model_v2_b200 import ops  # noqa: E402
from two_tower_model_v2_b200.sharded import range_record_layout, range_record_views  # noqa: E402

N_TOTAL, D, RADIUS = 10_000_000, 384, 0.19


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the measurement still stands; the record says what could not be read
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unread ({e!r})"}


def time_ms(fn, warmup=3, iters=10):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def records(G, nq, L, gen):
    """G full sorted runs per query (random scores, ids unique per query), counts beyond L."""
    lay = range_record_layout(nq, L)
    buf = torch.empty((G, lay.nbytes), dtype=torch.uint8, device="cuda")
    c, s, i, f = range_record_views(buf, lay, nq, L)
    ids = torch.randperm(G * L, device="cuda", generator=gen).view(G, 1, L)
    for g in range(G):
        sc, order = torch.rand((nq, L), device="cuda", generator=gen).sort(dim=1, descending=True)
        s[g].copy_(sc)
        i[g].copy_(ids[g].expand(nq, L).gather(1, order))
    c.fill_(L + 7)
    f.fill_(1)
    return buf, lay


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gen = torch.Generator(device="cuda").manual_seed(11)
    rec = {"tool": "bench_range_merge", "card": card(), "kernel": "tt::range_merge_kernel", "merge": [], "local": []}
    for G in (2, 4, 8):
        for nq in (1, 128, 4096):
            for L in (100, 1000, 16384):
                buf, lay = records(G, nq, L, gen)
                nunc = torch.zeros(1, dtype=torch.int32, device="cuda")
                ms = time_ms(lambda: ops.range_merge(buf, lay, nq, L, nunc), iters=10 if nq * L > 1 << 24 else 50)
                rec["merge"].append({"G": G, "nq": nq, "L": L, "merge_ms": round(ms, 4),
                                     "bytes_per_rank": lay.nbytes, "bytes_gathered": G * lay.nbytes})
                print(json.dumps(rec["merge"][-1]), flush=True)
                del buf
        torch.cuda.empty_cache()
        index, _, _ = bench.make_shard(N_TOTAL, D, G, 0)
        for nq in (1, 128, 4096):
            q = torch.randn((nq, D), device="cuda", generator=gen)
            rad = torch.full((nq,), RADIUS, device="cuda")
            for L in (100, 1000, 16384):
                lay = range_record_layout(nq, L)
                rbuf = torch.empty(lay.nbytes, dtype=torch.uint8, device="cuda")
                views = range_record_views(rbuf, lay, nq, L)
                ms = time_ms(lambda: index.range_shard_into(q, rad, L, *views), iters=5 if nq >= 4096 else 20)
                cnt = views[0]
                rec["local"].append({"G": G, "shard_rows": index.ntotal, "nq": nq, "L": L, "local_ms": round(ms, 4),
                                     "mean_count": float(cnt.double().mean()), "uncertified": int((views[3] != 1).sum())})
                print(json.dumps(rec["local"][-1]), flush=True)
                del rbuf, views
        del index
        torch.cuda.empty_cache()
    loc = {(r["G"], r["nq"], r["L"]): r["local_ms"] for r in rec["local"]}
    for r in rec["merge"]:
        r["merge_over_local"] = round(r["merge_ms"] / loc[(r["G"], r["nq"], r["L"])], 4)
    text = json.dumps(rec, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
