#!/usr/bin/env python
"""Benchmark of the serving hot path (BASELINE.json): exact top-100 inner-product retrieval over a sharded
catalog, buyer-tower pooling, and the device-resident /retrieve path.

    python bench.py --gpus N --steps K --warmup W                     # headline: 10M x 384, nq 4096, top-100
    python bench.py --workload c3|c4|c5 ...                           # the other BASELINE configs (see WORKLOADS)
    python bench.py --impl reference --gpus N --steps K --warmup W    # the reference's CPU path (rank 0 only)
    python bench.py ... --dump-outputs DIR                            # + the last timed step's results as DIR/*.npy

A "step" is one search of a batch of `--nq` queries (c5: one /retrieve batch).  Prints ONE JSON line (rank 0).
Catalogs (>= 768 MB of bf16 per pass) are larger than L2, so no flush is needed between iterations.  Inputs
are synthetic (seeded N(0,1)), generated on the device per shard.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

# BASELINE.json configs; explicit --catalog-rows/--dim/--nq/--topk override the table.
WORKLOADS = {
    "headline": {"catalog_rows": 10_000_000, "dim": 384, "nq": 4096, "topk": 100},   # the `metric` line
    "c3": {"catalog_rows": 1_000_000, "dim": 384, "nq": 4096, "topk": 100},          # configs[2]
    "c4": {"catalog_rows": 10_000_000, "dim": 768, "nq": 4096, "topk": 100},         # configs[3]
    "c5": {"catalog_rows": 100_000_000, "dim": 384, "nq": 1024, "topk": 100},        # configs[4]: /retrieve path
}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "sm_mhz_sustained": (d.get("clocks_under_load") or {}).get("sm_mhz_median"),
                "sm_max_mhz": d.get("sm_max_mhz"), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_mhz_sustained": 1300.0,
            "sm_max_mhz": 1965.0, "source": "fallback"}


def host_threads() -> int:
    """Host cores this process may use (cgroup/affinity aware)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines, self.t0, self.t1 = gpu_index, None, [], 0.0, float("inf")

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln))

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
            # nvidia-smi needs a few hundred ms to start: a short timed region would end before its first sample
            deadline = time.perf_counter() + 3.0
            while not self.lines and time.perf_counter() < deadline:
                time.sleep(0.01)
        except Exception:
            self.proc = None
        self.t0 = time.perf_counter()
        return self

    def __exit__(self, *a):
        self.t1 = time.perf_counter()
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for ts, ln in self.lines if self.t0 <= ts <= self.t1 + 0.06]      # samples of the timed region
        if not inside:                                                                 # (region shorter than one period)
            inside = [ln for ts, ln in self.lines if ts >= self.t0][:2]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus: int):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return world, rank, local


def max_over_ranks(ms: float, world: int) -> float:
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world: int):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def make_shard(n_total: int, d: int, world: int, rank: int):
    """Catalog rows [lo,hi): i.i.d. N(0,1), seeded per 1M-row block so the catalog is the same for any N."""
    import two_tower_model_v2_b200 as pkg
    lo, hi = pkg.shard_bounds(n_total, world, rank)
    xn = torch.empty((hi - lo, d), device="cuda", dtype=torch.float32)
    blk = 1 << 20
    g = torch.Generator(device="cuda")
    r = lo
    while r < hi:
        b = r // blk
        g.manual_seed(1234 + b)
        block = torch.randn((min(blk, n_total - b * blk), d), device="cuda", generator=g)
        s, e = r - b * blk, min(hi, (b + 1) * blk) - b * blk
        xn[r - lo:r - lo + (e - s)].copy_(block[s:e])
        r += e - s
        del block
    idx = pkg.FlatIPIndex.adopt(xn)
    idx.id_offset = lo
    return idx, lo, hi


# ---------------------------------------------------------------------------------------------------------
# Parity checkers used AFTER the timed region (and by tests/): an independent fp32 implementation of
# IndexFlatIP.search in library torch ops (cuBLAS sgemm with TF32 off + torch.topk), and a tie-tolerant
# comparison implementing the north-star acceptance (scores within 1e-5, ids identical except inside score
# ties of 1e-6).  Never on the product path.
def torch_flat_topk(xn: torch.Tensor, q: torch.Tensor, k: int, id_offset: int = 0, chunk_rows: int = 1 << 17):
    """xn f32 [N,D] stored rows, q f32 [nq,D] un-normalised -> (scores [nq,k'], ids [nq,k']) with k' = min(k, N)."""
    assert not torch.backends.cuda.matmul.allow_tf32, "the checker must run true fp32 sgemm"
    qn = q / (q.norm(dim=1, keepdim=True) + 1e-8)              # vector_db.py:152-153
    n = xn.shape[0]
    best_s = torch.empty((q.shape[0], 0), device=q.device)
    best_i = torch.empty((q.shape[0], 0), device=q.device, dtype=torch.int64)
    for lo in range(0, n, chunk_rows):
        hi = min(n, lo + chunk_rows)
        s = qn @ xn[lo:hi].t()
        ts, ti = torch.topk(s, min(k, hi - lo), dim=1)
        cs = torch.cat([best_s, ts], 1)
        ci = torch.cat([best_i, ti + (lo + id_offset)], 1)
        best_s, sel = torch.topk(cs, min(k, cs.shape[1]), dim=1)
        best_i = torch.gather(ci, 1, sel)
        del s
    return best_s, best_i


def compare_topk_device(s, i, rs, ri, score_tol=1e-5, tie_tol=1e-6, noise=4e-7):
    """(s,i) = ours, (rs,ri) = checker; both sorted descending.  Returns a dict; `ok` implements: every score
    within score_tol of the checker's score at the same rank; wherever the ids differ the two rows are tied
    (checker scores within tie_tol, plus fp32 summation noise), or - for an id the checker's list does not
    hold at all - its score ties with the checker's K-th score."""
    K = s.shape[1]
    ds = (s.double() - rs.double()).abs()
    eq = i[:, :, None] == ri[:, None, :]
    present = eq.any(2)
    pos = eq.float().argmax(2)
    mism = i != ri
    tol = tie_tol + noise
    gap_swapped = (torch.gather(rs, 1, pos) - rs).abs()               # same id, different rank: must be a tie
    gap_absent = (s - rs[:, K - 1:K]).abs()                           # id not in the checker's list: boundary tie
    gap = torch.where(present, gap_swapped, gap_absent)
    outside = mism & (gap > tol)
    sorted_ok = bool((s[:, 1:] <= s[:, :-1]).all())
    out = {"queries": int(s.shape[0]), "k": int(K), "score_max_abs_err": float(ds.max()) if ds.numel() else 0.0,
           "queries_with_id_differences": int(mism.any(1).sum()), "id_differences_outside_ties": int(outside.sum()),
           "sorted": sorted_ok}
    out["ok"] = bool(out["score_max_abs_err"] <= score_tol and out["id_differences_outside_ties"] == 0 and sorted_ok)
    return out


def parity_block(searcher, sharded, index, q, s, i, k, world, n_exact=64, n_torch=256):
    """After the timed region, on every rank: a sample of the LAST timed batch against (a) the always-exact fp32
    path of this library and (b) the independent torch fp32 checker (per-shard top-k all-gathered with NCCL and
    merged with torch.topk when the catalog is sharded).  Returns the block of the JSON line."""
    nq = q.shape[0]
    ne, nt = min(n_exact, nq), min(n_torch, nq)
    sel_e = torch.linspace(0, nq - 1, ne, device=q.device).long()
    sel_t = torch.linspace(0, nq - 1, nt, device=q.device).long()
    if sharded is not None:
        es, ei = sharded.search_exact_device(q[sel_e].contiguous(), k)
    else:
        es, ei = index.search_exact_device(q[sel_e].contiguous(), k)
    a = compare_topk_device(s[sel_e], i[sel_e], es, ei)
    ts, ti = torch_flat_topk(index.xn, q[sel_t].contiguous(), k, index.id_offset)
    if world > 1:
        import torch.distributed as dist
        kk = ts.shape[1]
        gs = torch.empty((world, nt, kk), device=q.device)
        gi = torch.empty((world, nt, kk), device=q.device, dtype=torch.int64)
        dist.all_gather_into_tensor(gs.view(-1), ts.contiguous().view(-1))
        dist.all_gather_into_tensor(gi.view(-1), ti.contiguous().view(-1))
        cs, ci = gs.permute(1, 0, 2).reshape(nt, -1), gi.permute(1, 0, 2).reshape(nt, -1)
        ts, sel = torch.topk(cs, k, dim=1)
        ti = torch.gather(ci, 1, sel)
    b = compare_topk_device(s[sel_t], i[sel_t], ts, ti)
    ok = torch.tensor([1 if (a["ok"] and b["ok"]) else 0], device=q.device)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return {"ok_all_ranks": bool(int(ok.item())), "batch": "last timed batch",
            "vs_exact_fp32_path": a, "vs_torch_fp32_sgemm_topk": b,
            "tolerance": "scores 1e-5; ids identical except score ties within 1e-6"}


# ---------------------------------------------------------------------------------------------------------
def bench_pooling(peaks, iters=20):
    """Secondary metric: buyer encodes/s at BASELINE C2 (4096 buyers x 50 events x 384), both modes."""
    import two_tower_model_v2_b200 as pkg
    B, S, D = 4096, 50, 384
    g = torch.Generator(device="cuda").manual_seed(99)
    x = torch.randn((B, S, D), device="cuda", generator=g)
    w = torch.tensor([1.0, 5.0, 10.0], device="cuda")[torch.multinomial(torch.tensor([0.75, 0.18, 0.07], device="cuda"), B * S, True, generator=g)].view(B, S)
    out = {}
    alg_bytes = B * S * D * 4 + B * S * 4 + B * D * 4
    for method in ("weighted_avg", "attention"):
        torch.manual_seed(0)
        m = pkg.BuyerTower(D, method).cuda()
        with torch.no_grad():
            for _ in range(3):
                m(x, w)
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        torch.cuda.synchronize()
        e0.record()
        with torch.no_grad():
            for _ in range(iters):
                m(x, w)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        rec = {"buyer_encodes_per_s": B / (ms * 1e-3), "ms_per_batch": ms,
               "hbm_gbs": alg_bytes / (ms * 1e-3) / 1e9, "hbm_frac": alg_bytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
        if method == "attention":
            flop = B * S * (2 * D * 128 + 2 * 128)
            # algorithmic flops (2*D*H + 2*H per row) per second; the hidden layer runs as two-piece fp16 (3 MMAs per K step) on the tensor cores
            rec["algorithmic_tflops"] = flop / (ms * 1e-3) / 1e12
            rec["mlp_kernel"] = "one fused kernel: tcgen05 kind::f16 on two-piece fp16 operands (fp32-accurate) + softmax + weighted sum + L2 norm"
        out[method] = rec
    out["config"] = "4096 buyers x 50 events x 384 f32 (x 322 MB > L2)"
    return out


def batch_sweep(index, lib, peaks, n_total, d, k, nqs, steps=10):
    """Same search at other query-batch sizes: nq <= ~250 is the HBM-bound regime (catalog streamed once
    per batch), larger batches are tensor-bound.  Device-resident timing, scan kernel timed by events."""
    from two_tower_model_v2_b200 import _native
    dp = int(lib.tt_flat_pitch(d))
    out = []
    for nq in nqs:
        g = torch.Generator(device="cuda").manual_seed(4321 + nq)
        qs = torch.randn((steps + 3, nq, d), device="cuda", generator=g)
        for i in range(3):
            index.search_device(qs[i], k)
        _native.check(lib.tt_profile_scan_arm(steps), "arm")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        nunc = [index.search_device(qs[i], k)[3] for i in range(3, 3 + steps)]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        sm = torch.empty(steps, dtype=torch.float32)
        n = lib.tt_profile_scan_read(sm.data_ptr(), steps)
        scan = float(sm[:n].mean())
        gbs = n_total * dp * 2 / scan / 1e6
        tfl = 2.0 * nq * n_total * d / scan / 1e9
        floor_ms = max(n_total * dp * 2 / (peaks["hbm_gbs"] * 1e6), 2.0 * nq * n_total * d / (peaks["bf16_tflops_sustained"] * 1e9))
        out.append({"catalog": f"{n_total}x{d}", "nq": nq, "queries_per_s": nq / ms * 1e3, "ms_per_step": ms, "scan_ms": scan,
                    "roofline_floor_ms": floor_ms, "step_frac_of_floor": floor_ms / ms,
                    "scan_hbm_gbs": gbs, "hbm_frac": gbs / peaks["hbm_gbs"], "scan_bf16_tflops": tfl,
                    "tensor_frac_sustained": tfl / peaks["bf16_tflops_sustained"],
                    "uncertified": int(torch.stack(nunc).sum().item())})
    return out


def bench_retrieve_path(index, d, k, requests=200, batch=1024):
    """Secondary (BASELINE config C5 shape on one GPU): the /retrieve path = history rows -> fused gather+pool ->
    exact top-K, host to host.  Batch-1 latency percentiles and batch-1024 throughput, 50-event histories."""
    import two_tower_model_v2_b200 as pkg
    db = pkg.VectorDatabase(d)
    db.index, db.product_ids, db.id_to_index, db.index_to_id = index, [], {}, {}
    out = {}
    for method in ("weighted_avg", "attention"):
        torch.manual_seed(0)
        tower = pkg.BuyerTower(d, method).cuda()
        pipe = pkg.RetrievalPipeline(tower, db)
        S, n = 50, index.ntotal
        g = torch.Generator().manual_seed(99)
        w_choices = torch.tensor([1.0, 5.0, 10.0])

        def make(B):
            idx = torch.randint(0, n, (B, S), generator=g, dtype=torch.int64).pin_memory()
            w = w_choices[torch.multinomial(torch.tensor([0.75, 0.18, 0.07]), B * S, True, generator=g)].view(B, S).pin_memory()
            return idx, w

        def request(idx, w):
            s, i, _ = pipe.retrieve_device_async(idx.cuda(non_blocking=True), w.cuda(non_blocking=True), k).result()
            return s.cpu(), i.cpu()
        reqs = [make(1) for _ in range(requests + 10)]
        for r in reqs[:10]:
            request(*r)
        lat = []
        for r in reqs[10:]:
            t = time.perf_counter()
            request(*r)
            lat.append((time.perf_counter() - t) * 1e3)
        lat = np.sort(np.array(lat))
        big = [make(batch) for _ in range(8)]
        request(*big[0]); request(*big[1])
        torch.cuda.synchronize()
        t = time.perf_counter()
        for r in big[2:]:
            request(*r)
        thr = batch * 6 / (time.perf_counter() - t)
        out[method] = {"batch1_latency_ms": {"p50": float(lat[len(lat) // 2]), "p99": float(lat[int(len(lat) * 0.99) - 1]),
                                             "mean": float(lat.mean())},
                       f"batch{batch}_requests_per_s": thr}
        if method == "weighted_avg":
            # 64 single-request clients (threads) sharing catalog passes through the micro-batcher; results come
            # back as array rows (ids i64[k], scores f32[k]) - no per-request Python lists
            def batch_fn(payloads, kk):
                idx = torch.from_numpy(np.stack([p[0] for p in payloads])).pin_memory().cuda(non_blocking=True)
                w = torch.from_numpy(np.stack([p[1] for p in payloads])).pin_memory().cuda(non_blocking=True)
                s, i, _ = pipe.retrieve_device_async(idx, w, kk).result()
                return pkg.ArrayRows(i.cpu().numpy(), s.cpu().numpy())
            clients, per_client = 64, 30
            payloads = [[(reqs[(c * per_client + j) % len(reqs)][0][0].numpy(), reqs[(c * per_client + j) % len(reqs)][1][0].numpy())
                         for j in range(per_client)] for c in range(clients)]
            lat_mb = []
            with pkg.MicroBatcher(batch_fn, max_batch=128, max_wait_ms=0.3) as mb:
                mb(payloads[0][0], k)

                def client(c):
                    for pl in payloads[c]:
                        t0 = time.perf_counter()
                        mb(pl, k)
                        lat_mb.append((time.perf_counter() - t0) * 1e3)
                ths = [threading.Thread(target=client, args=(c,)) for c in range(clients)]
                t = time.perf_counter()
                [th.start() for th in ths]
                [th.join() for th in ths]
                el = time.perf_counter() - t
                lat_mb = np.sort(np.array(lat_mb))
                out["micro_batched_64_clients"] = {"requests_per_s": clients * per_client / el,
                                                   "mean_batch": (mb.requests - 1) / max(mb.batches - 1, 1),
                                                   "latency_ms": {"p50": float(lat_mb[len(lat_mb) // 2]),
                                                                  "p99": float(lat_mb[int(len(lat_mb) * 0.99) - 1])}}
    out["config"] = f"history 50 events, top-{k}, {index.ntotal}x{d} catalog, host round trip per request, 1 GPU"
    return out


# ---------------------------------------------------------------------------------------------------------
# The reference's own CPU path.  faiss-cpu (requirements.txt:26) is not installable in this image, so the
# IndexFlatIP arithmetic is the oracle's torch sgemm+topk port (what faiss does for nq >= 20); when the
# unmodified reference modules are staged in baseline/_ref/ (by __graft_entry__.build() in the authoring
# container) the step drives the reference's own VectorDatabase.build_index / retrieve_batch over
# oracle/faiss_shim, wrapper overhead included, and the pooling baseline runs the reference's own BuyerTower.
def _reference_modules():
    """(VectorDatabase, BuyerTower) of the unmodified reference from baseline/_ref, or (None, None)."""
    ref = ROOT / "baseline" / "_ref"
    if not (ref / "src" / "inference" / "vector_db.py").exists():
        return None, None
    for p in (str(ROOT / "oracle" / "faiss_shim"), str(ref)):
        if p not in sys.path:
            sys.path.insert(0, p)
    try:
        import faiss  # the shim (or a real faiss, should the image ever gain one)
        if hasattr(faiss, "SEARCH_IMPL"):
            faiss.SEARCH_IMPL = "torch"
        from src.inference.vector_db import VectorDatabase
        from src.models.buyer_tower import BuyerTower
        return VectorDatabase, BuyerTower
    except Exception:
        return None, None


class CpuSearchArm:
    """One bounded sample step of the reference CPU search: `nq` queries x top-k over `sample_rows` of the
    `n_total` catalog rows; the step time is scaled by n_total/sample_rows (an inner-product scan is linear in
    the number of rows) - the line says so wherever the number appears."""

    def __init__(self, n_total, d, nq, k, budget_s, steps_total):
        import contextlib
        import io
        from oracle import flat_ip_oracle as fo
        torch.set_num_threads(host_threads())       # torchrun exports OMP_NUM_THREADS=1
        self.fo, self.n_total, self.d, self.nq, self.k = fo, n_total, d, nq, k
        self.cores = torch.get_num_threads()
        VectorDatabase, _ = _reference_modules()
        # calibrate the sgemm rate on a small block, then size the sample to the time budget
        xc = torch.randn((min(65536, n_total), d))
        qc = torch.randn((min(nq, 256), d))
        fo.torch_search(xc, qc, min(k, xc.shape[0]), block=65536)
        t = time.perf_counter()
        fo.torch_search(xc, qc, min(k, xc.shape[0]), block=65536)
        per_pair = (time.perf_counter() - t) / (xc.shape[0] * qc.shape[0])
        rows = int(budget_s / max(steps_total, 1) / (per_pair * nq))
        rows = max(min(rows, n_total, 1 << 20), min(n_total, 16384))
        if rows < n_total:
            rows = max(16384, rows // 16384 * 16384)
        self.sample_rows = rows
        g = torch.Generator().manual_seed(1234)
        x = torch.randn((rows, d), generator=g)
        self.wrapper = None
        if VectorDatabase is not None:
            db = VectorDatabase(embedding_dim=d)
            with contextlib.redirect_stdout(io.StringIO()):
                db.build_index(x.numpy(), [f"p{i}" for i in range(rows)])      # reference normalisation + id maps
            self.db = db
            self.wrapper = "unmodified reference VectorDatabase (baseline/_ref) over oracle/faiss_shim"
        else:
            self.xn = x / (x.norm(dim=1, keepdim=True) + 1e-8)
        self.scale = n_total / rows

    def step(self, q: torch.Tensor):
        if self.wrapper:
            return self.db.retrieve_batch(q.numpy(), self.k)
        return self.fo.torch_search(self.xn, q / (q.norm(dim=1, keepdim=True) + 1e-8), self.k, block=65536)

    def describe(self):
        s = (f"each step: {self.nq} queries x top-{self.k} over {self.sample_rows} of {self.n_total} rows x {self.d} f32; "
             f"IndexFlatIP arithmetic = torch-CPU sgemm+topk port (faiss-cpu not installable here)")
        if self.wrapper:
            s += f"; driven through the {self.wrapper}, Python result lists included"
        if self.scale != 1:
            s += f"; step time EXTRAPOLATED x{self.scale:g} to the full catalog (scan cost is linear in rows)"
        return s


def cpu_baseline_search(n_total, d, nq, k, budget_s=20.0, reps=2):
    arm = CpuSearchArm(n_total, d, nq, k, budget_s, reps + 1)
    q = torch.randn((nq, d), generator=torch.Generator().manual_seed(4321))
    arm.step(q)
    best = float("inf")
    for _ in range(reps):
        t = time.perf_counter()
        arm.step(q)
        best = min(best, time.perf_counter() - t)
    return {"value": nq / (best * arm.scale), "unit": "queries/s", "cores": arm.cores,
            "kind": "port", "sample": arm.describe(), "extrapolated": arm.scale != 1,
            "seconds_per_sample_step": best, "host_cpus": os.cpu_count()}


def cpu_baseline_pooling(buyers=1024, S=50, D=384, H=128, reps=3):
    """Reported baseline for the second half of the metric (buyer encodes/s): the reference BuyerTower on torch-CPU
    (the unmodified module from baseline/_ref when staged, else the oracle's port of the same eager ops) on a
    bounded sample of C2, all host threads."""
    from oracle import buyer_tower_oracle as bo
    torch.set_num_threads(host_threads())
    g = torch.Generator().manual_seed(99)
    x = torch.randn((buyers, S, D), generator=g)
    w = torch.tensor([1.0, 5.0, 10.0])[torch.multinomial(torch.tensor([0.75, 0.18, 0.07]), buyers * S, True, generator=g)].view(buyers, S)
    _, RefTower = _reference_modules()
    out = {"cores": torch.get_num_threads(), "kind": "reference" if RefTower is not None else "port",
           "sample": f"{buyers} of 4096 buyers x {S} events x {D} f32, torch-CPU, " +
                     ("unmodified reference BuyerTower (baseline/_ref)" if RefTower is not None else
                      "eager ops of the reference module (oracle port)")}
    with torch.no_grad():
        for method in ("weighted_avg", "attention"):
            torch.manual_seed(0)
            if RefTower is not None:
                m = RefTower(D, method, H).eval()
                fn = lambda: m(x, w)
            else:
                l1, l2 = torch.nn.Linear(D, H), torch.nn.Linear(H, 1)
                params = (l1.weight.detach(), l1.bias.detach(), l2.weight.detach(), l2.bias.detach())
                fn = lambda: bo.torch_forward(x, w, method, params)
            fn()
            best = float("inf")
            for _ in range(reps):
                t = time.perf_counter()
                fn()
                best = min(best, time.perf_counter() - t)
            out[method] = {"buyer_encodes_per_s": buyers / best, "seconds_per_sample": best}
    return out


def workload_name(args):
    return f"flat_ip_top{args.topk}_{args.catalog_rows}x{args.dim}_nq{args.nq}"


def metric_name(args):
    rows = args.catalog_rows
    pretty = f"{rows // 1_000_000}M" if rows % 1_000_000 == 0 else str(rows)
    return f"exact top-{args.topk} queries/s, {pretty}x{args.dim} catalog"


def run_reference(args):
    """`--impl reference`: rank 0 alone times the reference's CPU path with every host thread it can use; the
    other ranks exit 0 without work.  The whole run is bounded (~60 s of steps) at any --gpus."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_total, d, nq, k = args.catalog_rows, args.dim, args.nq, args.topk
    if args.workload == "c5":
        nq = args.nq
    arm = CpuSearchArm(n_total, d, nq, k, budget_s=float(os.environ.get("TT_BENCH_REF_BUDGET_S", "60")),
                       steps_total=args.warmup + args.steps)
    qs = torch.randn((args.warmup + args.steps, nq, d), generator=torch.Generator().manual_seed(4321))
    for i in range(args.warmup):
        arm.step(qs[i])
    t = time.perf_counter()
    for i in range(args.warmup, args.warmup + args.steps):
        arm.step(qs[i])
    el = time.perf_counter() - t
    sample_ms = el / args.steps * 1e3
    ms_step = sample_ms * arm.scale
    value = nq / (ms_step * 1e-3)
    sample = arm.describe()
    line = {"impl": "reference", "metric": metric_name(args), "value": value,
            "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (CPU" + (f"; catalog-row sample, step time extrapolated x{arm.scale:g}" if arm.scale != 1 else "") + ")",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "catalog_rows": n_total, "dim": d,
                       "topk": k, "query_batch": nq},
            "extrapolated": {"is_extrapolated": arm.scale != 1, "sample_rows": arm.sample_rows, "scale": arm.scale,
                             "measured_ms_per_sample_step": sample_ms, "measured_timed_region_s": el},
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": arm.cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def make_roofline(peaks, clocks, scan_avg_ms, ms_step, n_local, dp, d, nq, world, n_total):
    """Roofline of the dominant kernel (main scan): algorithmic bytes / flops of ONE launch over this rank's shard
    divided by the kernel's own CUDA-event time.  Tensor-bound launches are reported against both measured cuBLAS
    peaks; `frac` uses the sustained one unless the SM clock sampled during the timed region was nearer the burst
    clock (a short or lightly loaded run is not power-capped)."""
    if not scan_avg_ms:
        return None
    alg_bytes = n_local * dp * 2 + nq * dp * 2           # bf16 catalog streamed once + the query block(s)
    alg_flops = 2.0 * nq * n_local * d
    crossover = peaks["bf16_tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)     # flops per byte = nq* (2D per 2D bytes)
    gbs = alg_bytes / (scan_avg_ms * 1e-3) / 1e9
    tfl = alg_flops / (scan_avg_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    tp = ROOT / "profiles" / "scan_traffic.json"      # dram bytes/launch of committed ncu captures (1 GPU only)
    if world == 1 and tp.exists():
        try:
            traffic = json.loads(tp.read_text()).get(f"{n_total}x{d}_nq{nq}")
            traffic_src = "profiles/scan_traffic.json (ncu --set full capture of this workload, not this run)" if traffic else None
        except Exception:
            traffic = None
    if nq < crossover:
        r = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"]}
    else:
        sus, burst = peaks["bf16_tflops_sustained"], peaks["bf16_tflops"]
        mhz = (clocks or {}).get("sm_mhz")
        lo, hi = peaks.get("sm_mhz_sustained") or 1350.0, peaks.get("sm_max_mhz") or 1965.0
        use_burst = mhz is not None and mhz > 0.5 * (lo + hi)
        peak = burst if use_burst else sus
        r = {"bound": "tensor", "achieved": tfl, "peak": peak, "unit": "TFLOP/s", "frac": tfl / peak,
             "peak_basis": ("burst" if use_burst else "sustained") + f" cuBLAS bf16 (SM clock during the timed region {mhz} MHz; "
                           f"sustained peak measured at {lo:.0f} MHz, max {hi:.0f})",
             "frac_sustained": tfl / sus, "frac_burst": tfl / burst}
    r.update({"traffic": traffic, "traffic_source": traffic_src, "kernel": "flat_scan_kernel<main>", "kernel_ms": scan_avg_ms,
              "kernel_share_of_step": scan_avg_ms / ms_step, "algorithmic_bytes": alg_bytes,
              "algorithmic_flops": alg_flops, "hbm_gbs": gbs, "bf16_tflops": tfl, "peaks": peaks["source"],
              "crossover_nq": crossover})
    return r


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, scores, ids):
    """Writes what a caller of the timed path receives for one batch: scores.npy (float32 [rows, k]) and ids.npy
    (float64, exact for any row id below 2**53).  Above DUMP_MAX_BYTES a fixed, seeded sample of query rows is
    kept and rows.npy (float64) lists which; the inputs are seeded too, so two builds can be compared file by file."""
    scores = scores.cpu().numpy().astype(np.float32)
    ids = ids.cpu().numpy().astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    nq, k = scores.shape
    keep = max(1, (DUMP_MAX_BYTES - 4096) // (k * 12 + 8))      # 4096: room for the three .npy headers
    if nq > keep:
        rows = np.sort(np.random.default_rng(0).choice(nq, keep, replace=False))
        scores, ids = scores[rows], ids[rows]
        np.save(out / "rows.npy", rows.astype(np.float64))
    np.save(out / "scores.npy", scores)
    np.save(out / "ids.npy", ids)


def run_pipelined(submit, first, last, depth=2):
    """Steps first..last-1 with `depth` batches in flight: step i+depth-1 is enqueued before step i's certificate is
    looked at, so the device never idles on the host (the sharded search runs a 3-stage pipeline and wants depth 3).
    Every step is checked (uncertified queries re-run through the exact path) inside the timed region.
    Returns (re-run queries, result of the last step)."""
    from collections import deque
    bad, pending, out = 0, deque(), None
    for i in range(first, last):
        pending.append(submit(i))
        if len(pending) >= depth:
            out = pending.popleft().result()
            bad += out[2]
    while pending:
        out = pending.popleft().result()
        bad += out[2]
    return bad, out


def run_search(args):
    world, rank, local = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200 import _native
    lib = _native.load()
    peaks = load_peaks()
    n_total, d, nq, k = args.catalog_rows, args.dim, args.nq, args.topk

    index, lo, hi = make_shard(n_total, d, world, rank)
    n_local = hi - lo
    sharded = pkg.ShardedFlatIPIndex(index, n_total) if world > 1 else None
    total = args.warmup + args.steps
    gq = torch.Generator(device="cuda").manual_seed(4321)
    queries = torch.randn((total, nq, d), device="cuda", generator=gq)
    queries_host = queries.cpu().numpy()
    searcher = sharded if world > 1 else index

    # ---- device-resident timing ---------------------------------------------------------------
    depth = 3 if world > 1 else 2
    run_pipelined(lambda i: searcher.search_async(queries[i], k), 0, args.warmup, depth)
    launches0 = lib.tt_kernel_launch_count()
    _native.check(lib.tt_profile_scan_arm(args.steps), "tt_profile_scan_arm")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    host_s = [0.0]

    def submit_timed(i):        # host time spent enqueueing (ctypes + Python), to tell a host-bound step from a device-bound one
        t = time.perf_counter()
        r = searcher.search_async(queries[i], k)
        host_s[0] += time.perf_counter() - t
        return r
    with ClockSampler(local) as clk:
        barrier(world)          # the sampler's start-up time differs between ranks: line them up again before the clock starts
        e0.record()
        uncertified, last = run_pipelined(submit_timed, args.warmup, total, depth)
        e1.record()
        barrier(world)
    ms_total = max_over_ranks(e0.elapsed_time(e1), world)
    host_enqueue_ms = max_over_ranks(host_s[0] * 1e3, world) / args.steps
    launches = lib.tt_kernel_launch_count() - launches0
    scan_ms = (torch.empty(args.steps, dtype=torch.float32))
    n_rec = lib.tt_profile_scan_read(scan_ms.data_ptr(), args.steps)
    ms_step = ms_total / args.steps
    value = nq / (ms_step * 1e-3)
    clocks = clk.summary()

    dp = int(lib.tt_flat_pitch(d))
    scan_avg_ms = float(scan_ms[:n_rec].mean()) if n_rec > 0 else None
    roofline = make_roofline(peaks, clocks, scan_avg_ms, ms_step, n_local, dp, d, nq, world, n_total)

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0], last[1])

    # ---- parity of the last timed batch (outside the timed region, every rank) -------------------
    parity = parity_block(searcher, sharded, index, queries[total - 1], last[0], last[1], k, world)

    # ---- end to end through the host-facing API (numpy in, numpy out) ----------------------------
    if world > 1 and nq % world == 0:
        # every rank fronts 1/G of the batch: its share goes host -> device, the shares are all-gathered over
        # NVLink, and each rank reads back the results of its own rows (whole job: nq*D*4 in, nq*k*12 out)
        nl = nq // world
        host_submit = lambda i: sharded.search_host_sliced_async(queries_host[i][rank * nl:(rank + 1) * nl], k)
        e2e_api = "ShardedFlatIPIndex.search_host_sliced_async(np.ndarray share) -> numpy share, 2 batches in flight"
    else:
        host_submit = lambda i: searcher.search_host_async(queries_host[i], k)
        e2e_api = ("FlatIPIndex" if world == 1 else "ShardedFlatIPIndex") + ".search_host_async(np.ndarray) -> numpy, 2 batches in flight"
    run_pipelined(host_submit, 0, min(3, args.warmup), depth)
    barrier(world)
    t0 = time.perf_counter()
    run_pipelined(host_submit, args.warmup, total, depth)
    barrier(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world) / args.steps
    e2e = {"value": nq / (e2e_ms * 1e-3), "unit": "queries/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * 12 + 4,
           "api": e2e_api.replace("2 batches in flight", f"{depth} batches in flight")}

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            sharded.close()
            dist.destroy_process_group()
        return

    line = {"metric": metric_name(args), "value": value, "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16 scan + f32 rescoring",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "catalog_rows": n_total, "dim": d, "topk": k,
                       "query_batch": nq, "sharding": (f"catalog rows over {world} GPUs, one catalog-wide threshold, all-gather ({sharded.exchange_used}) + certified merge"
                                    if world > 1 else "none"),
                       "l2": f"inputs ({n_local * dp * 2 / 1e9:.2f} GB bf16 per pass per GPU) exceed L2; no flush"},
            "e2e": e2e, "gpu_launches": int(launches), "uncertified_queries": uncertified,
            "host_enqueue_ms_per_step": host_enqueue_ms,
            "roofline": roofline, "parity": parity, "clocks": clocks}
    if world == 1 and not args.no_secondary:
        sec = {"pooling": bench_pooling(peaks),
               "query_batch_sweep": batch_sweep(index, lib, peaks, n_total, d, k, [1, 128, 1024])}
        sec["retrieve_path"] = bench_retrieve_path(index, d, k)
        if n_total != 1_000_000:
            # BASELINE config C3 (1M x 384) in the HBM-bound regime: the whole step against the scan floor
            del index, searcher
            torch.cuda.empty_cache()
            small, _, _ = make_shard(1_000_000, 384, 1, 0)
            sec["query_batch_sweep_1Mx384"] = batch_sweep(small, lib, peaks, 1_000_000, 384, k, [1, 128], steps=30)
            del small
        line["secondary"] = sec
        line["cpu_baseline"] = cpu_baseline_search(n_total, d, nq, k)
        try:
            sec["pooling"]["cpu_baseline"] = cpu_baseline_pooling()
        except Exception as e:                       # a reported extra must never cost the headline line
            sec["pooling"]["cpu_baseline"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        sharded.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("TT_BENCH_WORKLOAD", "headline"), choices=sorted(WORKLOADS))
    ap.add_argument("--nq", type=int, default=None, help="queries per step")
    ap.add_argument("--catalog-rows", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--topk", type=int, default=None)
    ap.add_argument("--no-secondary", action="store_true", help="skip pooling / cpu baseline extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's results (scores, ids) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    wl = WORKLOADS[args.workload]
    if args.nq is None:
        args.nq = int(os.environ.get("TT_BENCH_NQ", wl["nq"]))
    args.catalog_rows = wl["catalog_rows"] if args.catalog_rows is None else args.catalog_rows
    args.dim = wl["dim"] if args.dim is None else args.dim
    args.topk = wl["topk"] if args.topk is None else args.topk
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    if args.workload == "c5":
        run_c5(args)
    else:
        run_search(args)


def run_c5(args):
    """BASELINE configs[4]: the end-to-end /retrieve path (buyer encode + search) over a 100M x 384 catalog on 8 B200
    (bf16 scan copy 9.6 GB + fp32 rows 19.2 GB per GPU): p50/p99 latency at batch 1, throughput at batch 1024.
    Weak scaling: 12.5M rows per GPU, so N GPUs hold N/8 of the 100M rows.  A request = a 50-event history (global
    catalog row ids + event weights) -> owner-computes pooling over the sharded item table -> exact top-100."""
    world, rank, local = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200 import _native
    lib = _native.load()
    peaks = load_peaks()
    d, k, batch, S = args.dim, args.topk, args.nq, 50
    n_total = args.catalog_rows * world // 8 if args.catalog_rows == WORKLOADS["c5"]["catalog_rows"] else args.catalog_rows
    index, lo, hi = make_shard(n_total, d, world, rank)
    n_local = hi - lo
    sharded = pkg.ShardedFlatIPIndex(index, n_total)
    method = os.environ.get("TT_BENCH_C5_METHOD", "attention")          # configs/config.yaml:12-13 default
    torch.manual_seed(0)
    tower = pkg.BuyerTower(d, method).cuda()
    pipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    g = torch.Generator().manual_seed(99)
    wc = torch.tensor([1.0, 5.0, 10.0])

    def make(B):
        idx = torch.randint(0, n_total, (B, S), generator=g, dtype=torch.int64).pin_memory()
        w = wc[torch.multinomial(torch.tensor([0.75, 0.18, 0.07]), B * S, True, generator=g)].view(B, S).pin_memory()
        return idx, w
    total = args.warmup + args.steps
    big = [make(batch) for _ in range(total)]
    big_dev = [(i.cuda(), w.cuda()) for i, w in big]

    # ---- batch-1024 throughput, device-resident inputs ----------------------------------------------
    run_pipelined(lambda i: pipe.retrieve_device_async(*big_dev[i], k), 0, args.warmup)
    launches0 = lib.tt_kernel_launch_count()
    _native.check(lib.tt_profile_scan_arm(args.steps), "tt_profile_scan_arm")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    with ClockSampler(local) as clk:
        barrier(world)          # (the sampler's start-up time differs between ranks)
        e0.record()
        uncertified, last = run_pipelined(lambda i: pipe.retrieve_device_async(*big_dev[i], k), args.warmup, total)
        e1.record()
        barrier(world)
    ms_step = max_over_ranks(e0.elapsed_time(e1), world) / args.steps
    launches = lib.tt_kernel_launch_count() - launches0
    scan_ms = torch.empty(args.steps, dtype=torch.float32)
    n_rec = lib.tt_profile_scan_read(scan_ms.data_ptr(), args.steps)
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0], last[1])
    dp = int(lib.tt_flat_pitch(d))
    roofline = make_roofline(peaks, clocks, float(scan_ms[:n_rec].mean()) if n_rec > 0 else None, ms_step, n_local, dp, d,
                             batch, world, n_total)
    # parity of the last batch: pooled queries re-derived, then the search checked as in the search workloads
    q_last = pipe.encode_device(*big_dev[total - 1], k)
    parity = parity_block(sharded, sharded, index, q_last, last[0], last[1], k, world)

    # ---- batch-1024 end to end: pinned host histories in, this rank's share of the results out ----------
    share = slice(rank * batch // world, (rank + 1) * batch // world)

    def host_step(i):
        pend = pipe.retrieve_device_async(big[i][0].cuda(non_blocking=True), big[i][1].cuda(non_blocking=True), k)

        class _P:
            def result(self_inner):
                sc, ids, bad = pend.result()
                return sc[share].cpu(), ids[share].cpu(), bad
        return _P()
    run_pipelined(host_step, 0, min(2, args.warmup))
    barrier(world)
    t0 = time.perf_counter()
    run_pipelined(host_step, args.warmup, total)
    barrier(world)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world) / args.steps

    # ---- batch-1 latency, host to host, every rank fronts the same request ------------------------------
    reqs = [make(1) for _ in range(210)]

    def one(r):
        sc, ids, _ = pipe.retrieve_device_async(r[0].cuda(non_blocking=True), r[1].cuda(non_blocking=True), k).result()
        return sc.cpu(), ids.cpu()
    for r in reqs[:10]:
        one(r)
    barrier(world)
    lat = []
    _native.check(lib.tt_profile_scan_arm(200), "tt_profile_scan_arm")
    for r in reqs[10:]:
        t = time.perf_counter()
        one(r)
        lat.append((time.perf_counter() - t) * 1e3)
    sm1 = torch.empty(200, dtype=torch.float32)
    n1 = lib.tt_profile_scan_read(sm1.data_ptr(), 200)
    lat = np.sort(np.array(lat))
    p50 = max_over_ranks(float(lat[len(lat) // 2]), world)
    p99 = max_over_ranks(float(lat[int(len(lat) * 0.99) - 1]), world)
    scan1 = float(sm1[:n1].mean()) if n1 > 0 else None
    floor1 = n_local * dp * 2 / (peaks["hbm_gbs"] * 1e6)
    if rank == 0:
        pretty = f"{n_total // 1_000_000}M"
        line = {"metric": f"/retrieve requests/s at batch {batch} (buyer encode + exact top-{k}), {pretty}x{d} catalog", "value": batch / (ms_step * 1e-3),
                "unit": "requests/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 pooling, bf16 scan + f32 rescoring", "data": "synthetic",
                "config": {"workload": f"c5_retrieve_{n_total}x{d}_hist{S}_top{k}_batch{batch}", "catalog_rows": n_total,
                           "rows_per_gpu": n_local, "dim": d, "topk": k, "batch": batch, "history_events": S,
                           "aggregation_method": method,
                           "sharding": f"catalog rows over {world} GPUs; owner-computes pooling partials + one catalog-wide threshold; exchanges: {sharded.exchange_used}",
                           "hbm_per_gpu_gb": {"bf16_scan_copy": n_local * dp * 2 / 1e9, "fp32_rows": n_local * d * 4 / 1e9},
                           "l2": "inputs exceed L2; no flush"},
                "latency_batch1_ms": {"p50": p50, "p99": p99, "timing": "host perf_counter around history H2D -> pool -> search -> D2H, max over ranks",
                                      "scan_kernel_ms": scan1, "hbm_floor_ms": floor1,
                                      "scan_hbm_frac": (floor1 / scan1) if scan1 else None},
                "e2e": {"value": batch / (e2e_ms * 1e-3), "unit": "requests/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": world * batch * S * 12, "d2h_bytes_per_step": batch * k * 12,
                        "api": "ShardedRetrievalPipeline.retrieve_device_async(pinned history rows + weights) -> this rank's share of (scores, ids) on the host, 2 batches in flight"},
                "gpu_launches": int(launches), "uncertified_queries": uncertified, "roofline": roofline, "parity": parity,
                "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        barrier(world)
        sharded.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
