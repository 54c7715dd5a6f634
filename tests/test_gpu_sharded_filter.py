"""GPU: label filters on the sharded search (tt_flat_search_shard_filtered, tt_flat_shard_sample_filtered,
tt_flat_shard_search_filtered) with shards emulated on one device, the public sharded API at world size 1, and a
2-GPU sharded /retrieve."""
import ctypes

import numpy as np
import pytest
import torch

from filter_oracle import search_filtered, torch_topk_filtered
from oracle import flat_ip_oracle as fo

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def plan(N, D, nq, K):
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    assert _native.load().tt_flat_plan_describe(N, D, nq, K, out) == 0
    return {"route_exact": out[7]}


def shard_views(full, G):
    """G FlatIPIndex shards that view the rows of `full` (no copy; the whole catalog's error statistics bound every
    subset), each with its slice of the labels."""
    import two_tower_model_v2_b200 as pkg
    out = []
    for r in range(G):
        lo, hi = pkg.shard_bounds(full.ntotal, G, r)
        idx = pkg.FlatIPIndex(full.d, full.device)
        idx.xn = idx._xn_store = full.xn[lo:hi]
        idx.xh = idx._xh_store = full.xh[lo:hi]
        idx.stats = full.stats
        idx.id_offset = lo
        idx.set_labels(full.labels[lo:hi])
        out.append(idx)
    return out


def labels_for(kind, N, G, rng):
    """Bit 0 = allowed.  "s<x>": random rows at selectivity x; "clustered": 1 % of the catalog, every row in the last
    shard; the other bits are noise."""
    import two_tower_model_v2_b200 as pkg
    lab = rng.integers(0, 1 << 32, N, dtype=np.uint64) & ~np.uint64(1)
    if kind == "clustered":
        lo, hi = pkg.shard_bounds(N, G, G - 1)
        allowed = np.zeros(N, bool)
        allowed[lo + rng.choice(hi - lo, max(N // 100, 1), replace=False)] = True
    else:
        allowed = rng.random(N) < float(kind[1:])
    return lab | allowed.astype(np.uint64)


def merge(gathered, lay, nq, k):
    from two_tower_model_v2_b200 import ops
    return ops.shard_merge(gathered, lay.off_scores, lay.off_ids, lay.off_bound, lay.off_flags, nq, k)


# ---- per-shard thresholds -----------------------------------------------------------------------------------
KINDS = ["s1", "s0.1", "s0.01", "s0", "clustered", "s0.1+excl"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("G", [2, 3, 4])
def test_shard_records_merge_to_filtered_oracle(G, kind):
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200.sharded import record_layout, record_views
    N, D, nq, k = 40_000, 64, 33, 10
    rng = np.random.default_rng(G * 100 + KINDS.index(kind))
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = labels_for(kind.split("+")[0], N, G, rng)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    ex = None
    if kind.endswith("+excl"):                                   # each query's own best allowed rows, random rows
        top = search_filtered(xn, qn, 20, labels, [1, 0])[1]
        ex = np.concatenate([top, rng.integers(0, N, (nq, 20)), np.full((nq, 2), -1)], 1).astype(np.int64)
    full = pkg.FlatIPIndex(D)
    full.add(x)
    full.set_labels(labels)
    lay = record_layout(nq, k)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    qd = torch.from_numpy(q).to(dev())
    kw = {} if ex is None else {"exclude": torch.from_numpy(ex).to(dev())}
    for g, idx in enumerate(shard_views(full, G)):
        s, i, b, f = record_views(gathered[g], lay, nq, k)
        idx.search_shard_into(qd, k, s, i, b, f, require=np.array([1, 0]), **kw)
    s, i, flags, nunc = merge(gathered, lay, nq, k)
    s, i, flags = s.cpu().numpy(), i.cpu().numpy(), flags.cpu().numpy()
    rs, ri = search_filtered(xn, qn, k, labels, [1, 0], ex)
    short = (ri < 0).any(1)                                      # fewer than k allowed rows: flag -2, padded exactly
    assert np.array_equal(flags[short], np.full(int(short.sum()), -2, np.int32))
    assert np.array_equal(i[short], ri[short]) and np.array_equal(np.isneginf(s[short]), np.isneginf(rs[short]))
    ok = ~short & (flags == 1)
    assert ok.sum() == (~short).sum(), f"{(~short).sum() - ok.sum()} queries uncertified"
    okc, msg = fo.compare_topk(s[ok], i[ok], rs[ok], ri[ok], xn, qn[ok])
    assert okc, msg
    got = i[i >= 0]
    assert (labels[got] & 1).all()
    if ex is not None:
        for r in range(nq):
            assert not np.isin(i[r][i[r] >= 0], ex[r]).any()
    if kind == "s0":
        assert (i == -1).all() and short.all()


def test_route_exact_shard_with_filter_has_unbounded_record():
    """A shard too small for a sampled threshold (K is a large fraction of its rows) is served by the filtered exact
    path: bound -inf, flags 1, the exact filtered top-K of its rows."""
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200.sharded import record_layout, record_views
    N, D, nq, k, G = 60_000, 64, 8, 1000, 2
    assert plan(N // G, D, nq, k)["route_exact"] == 1
    rng = np.random.default_rng(17)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = labels_for("s0.5", N, G, rng)
    full = pkg.FlatIPIndex(D)
    full.add(x)
    full.set_labels(labels)
    lay = record_layout(nq, k)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    for g, idx in enumerate(shard_views(full, G)):
        s, i, b, f = record_views(gathered[g], lay, nq, k)
        idx.search_shard_into(torch.from_numpy(q).to(dev()), k, s, i, b, f, require=np.array([1, 0]))
        assert bool(torch.isneginf(b).all()) and bool((f == 1).all())
    s, i, flags, nunc = merge(gathered, lay, nq, k)
    rs, ri = search_filtered(fo.normalize_rows(x), fo.normalize_rows(q), k, labels, [1, 0])
    assert int(nunc.item()) == 0
    okc, msg = fo.compare_topk(s.cpu().numpy(), i.cpu().numpy(), rs, ri, fo.normalize_rows(x), fo.normalize_rows(q))
    assert okc, msg


# ---- one global threshold ------------------------------------------------------------------------------------
def run_global_threshold(full, q, k, G, req):
    """shard_sample(require=) on every shard, the gathered lists, shard_search_into(require=), merge -> (s, i, flags,
    per-shard flags [G, nq])."""
    from two_tower_model_v2_b200 import _native
    from two_tower_model_v2_b200.sharded import record_layout, record_views
    shards = shard_views(full, G)
    nq, N = q.shape[0], full.ntotal
    assert shards[0].shard_plan_ok(N, nq, k, min(s.ntotal for s in shards))
    topr_g = torch.empty((G, nq, _native.TT_SHARD_TOPR), device=dev())
    for r, idx in enumerate(shards):
        idx.shard_sample(q, k, N, topr_g[r], require=req)
    lay = record_layout(nq, k)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    for r, idx in enumerate(shards):
        s, i, b, f = record_views(gathered[r], lay, nq, k)
        idx.shard_search_into(nq, k, N, topr_g, s, i, b, f, require=req)
    s, i, flags, _ = merge(gathered, lay, nq, k)
    return s, i, flags, record_views(gathered, lay, nq, k)[3], topr_g


def check_against_single(full, q, k, G, allowed, tag):
    """Certified by both: bit-identical to the single index; re-run queries: tie-tolerant against the fp32 checker."""
    import bench
    req = np.array([1, 0])
    s, i, flags, shard_flags, topr_g = run_global_threshold(full, q, k, G, req)
    fs, fi, fflags, _ = full.search_device(q, k, require=req)
    both = (flags == 1) & (fflags == 1)
    assert torch.equal(i[both], fi[both]) and torch.equal(s[both], fs[both])
    bad = torch.nonzero(flags != 1).flatten()
    if bad.numel():
        rs, ri = full.search_exact_device(q[bad].contiguous(), k, require=req)
        s[bad], i[bad] = rs, ri
    ts, ti = torch_topk_filtered(full.xn, q, k, allowed)
    rep = bench.compare_topk_device(s, i, ts, ti)
    assert rep["ok"], rep
    overflow = ((shard_flags <= 0) & ((-shard_flags) & 1 == 1)).sum(1)
    print(f"{tag}: uncertified sharded {int((flags != 1).sum())}, single {int((fflags != 1).sum())}, "
          f"certified by both {int(both.sum())}/{q.shape[0]}, candidate overflows per shard {overflow.tolist()}")
    return shard_flags, topr_g


@pytest.mark.parametrize("kind", ["s0.1", "s0.01", "clustered"])
def test_global_threshold_path_3m_4_shards(kind):
    import two_tower_model_v2_b200 as pkg
    N, D, nq, k, G = 3_000_000, 64, 200, 100, 4
    g = torch.Generator(device="cuda").manual_seed(79)
    full = pkg.FlatIPIndex.adopt(torch.randn((N, D), device=dev(), generator=g))
    q = torch.randn((nq, D), device=dev(), generator=g)
    labels = torch.from_numpy(labels_for(kind, N, G, np.random.default_rng(5)).astype(np.int64)).to(dev())
    full.set_labels(labels)
    shard_flags, topr_g = check_against_single(full, q, k, G, (labels & 1) == 1, f"3M x {D}, {G} shards, {kind}")
    if kind == "clustered":
        # every shard but the last holds no allowed row: all -inf lists, and the last shard takes the whole candidate
        # target without overflowing its segments (make_shard_plan sizes seg_cap for that)
        assert bool(torch.isneginf(topr_g[:G - 1]).all()) and bool(torch.isfinite(topr_g[G - 1, :, 0]).all())
        assert not bool(((shard_flags <= 0) & ((-shard_flags) & 1 == 1)).any())


# ---- public API at world size 1 ------------------------------------------------------------------------------
def test_sharded_api_world1_equals_single_index_and_trivial_filter_is_bit_identical():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(61)
    N, D, nq, k = 50_000, 384, 40, 10
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = torch.from_numpy(rng.standard_normal((nq, D)).astype(np.float32)).to(dev())
    local = pkg.FlatIPIndex(D)
    local.add(x)
    sharded = pkg.ShardedFlatIPIndex(local, N)
    labels = labels_for("s0.1", N, 1, rng)
    rows = np.flatnonzero(labels & 1)
    sharded.set_labels(np.ones(rows.size, np.int64), rows=rows)         # by global row id: bit 0 only
    assert np.array_equal(local.labels.cpu().numpy() & 1, (labels & 1).astype(np.int32))
    req = np.stack([np.ones(nq, np.int64), np.zeros(nq, np.int64)], 1)
    req[3] = [0, 0]
    s, i, _ = sharded.search_device(q, k, require=req)
    fs, fi, _ = local.search_checked_device(q, k, require=req)
    assert torch.equal(i, fi) and torch.equal(s, fs)
    hs, hi, _ = sharded.search_host_async(q.cpu().numpy(), k, require=req).result()
    assert np.array_equal(hi, fi.cpu().numpy())
    ls, li, _ = sharded.search_host_sliced_async(q.cpu().numpy(), k, require=req).result()
    assert np.array_equal(li, fi.cpu().numpy())
    # (0, 0) masks, as numpy or CUDA, run exactly the unfiltered search
    s0, i0, _ = sharded.search_device(q, k)
    for triv in (np.zeros(2, np.int64), torch.zeros((nq, 2), device=dev(), dtype=torch.int32)):
        s1, i1, _ = sharded.search_device(q, k, require=triv)
        assert torch.equal(s0, s1) and torch.equal(i0, i1)
    s2, i2, _ = sharded.search_host_sliced_async(q.cpu().numpy(), k, require=np.zeros(2, np.int64)).result()
    assert np.array_equal(i2, i0.cpu().numpy())


@pytest.mark.parametrize("method", ["weighted_avg", "attention"])
def test_sharded_retrieval_pipeline_world1_require_any_with_exclude_history(method):
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(24)
    N, D, B, S, k = 30000, 384, 16, 50, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    db = pkg.VectorDatabase(D)
    db.build_index(cat, [f"p{i}" for i in range(N)])
    torch.manual_seed(3)
    tower = pkg.BuyerTower(D, method).to(dev())
    pipe = pkg.RetrievalPipeline(tower, db)
    sharded = pkg.ShardedFlatIPIndex(db.index, N)
    labels = (1 << rng.integers(0, 8, N)).astype(np.int64)
    sharded.set_labels(labels)
    spipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    idx = torch.from_numpy(rng.integers(0, N, (B, S))).to(dev())
    idx[:, S // 2:] = -1
    w = torch.from_numpy(rng.random((B, S)).astype(np.float32)).to(dev())
    want_any = np.array([(1 << int(rng.integers(0, 8))) | (1 << int(rng.integers(0, 8))) for _ in range(B)], np.int64)
    ps, pi, _ = pipe.retrieve_device_async(idx, w, k, exclude_history=True, require_any=want_any).result()
    ss, si, _ = spipe.retrieve_device_async(idx, w, k, exclude_history=True, require_any=want_any).result()
    assert torch.equal(si, pi) and torch.allclose(ss, ps, atol=1e-6)
    assert all(labels[r] & want_any[b] for b in range(B) for r in si[b].tolist())
    assert not bool((si[:, :, None] == idx[:, None, :]).any())
    hs, hi, _ = spipe.retrieve_host_async(idx.cpu().pin_memory(), w.cpu().pin_memory(), k, exclude_history=True,
                                          require_any=want_any).result()
    assert np.array_equal(hi, pi.cpu().numpy())


# ---- full size -----------------------------------------------------------------------------------------------
def test_full_size_10m_8_shards_nq4096_k100_s001():
    """The benched shape split into 8 emulated shards, one filter at selectivity 0.01: the merged global-threshold
    result against the single index's filtered result, query by query."""
    import bench
    torch.cuda.empty_cache()
    N, D, nq, k, G = 10_000_000, 384, 4096, 100, 8
    index, _, _ = bench.make_shard(N, D, 1, 0)
    try:
        g = torch.Generator(device="cuda").manual_seed(4324)
        allowed = torch.rand(N, device="cuda", generator=g) < 0.01
        index.set_labels(allowed.to(torch.int32))
        q = torch.randn((nq, D), device="cuda", generator=g)
        check_against_single(index, q, k, G, allowed, f"10M x {D}, {G} shards, nq {nq}, K {k}, s 0.01")
    finally:
        del index
        torch.cuda.empty_cache()


# ---- two GPUs ------------------------------------------------------------------------------------------------
def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_retrieve_worker(rank, world, port, out_dir):
    import os
    import torch.distributed as dist
    import two_tower_model_v2_b200 as pkg
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    N, D, B, S, k = 2_000_000, 384, 64, 40, 10        # K_plan = k + S = 50: the one-threshold plan, pipelined
    g = torch.Generator(device="cuda").manual_seed(92)
    x = torch.randn((N, D), device="cuda", generator=g)
    idx_h = torch.randint(0, N, (B, S), device="cuda", generator=g)
    w_h = torch.rand((B, S), device="cuda", generator=g)
    labels = 1 << torch.randint(0, 8, (N,), device="cuda", generator=g)
    want_any = (1 << torch.randint(0, 8, (B,), generator=torch.Generator().manual_seed(3))).numpy()
    lo, hi = pkg.shard_bounds(N, world, rank)
    local = pkg.FlatIPIndex.adopt(x[lo:hi].clone())
    local.id_offset = lo
    torch.manual_seed(5)
    tower = pkg.BuyerTower(D, "weighted_avg").cuda()
    sharded = pkg.ShardedFlatIPIndex(local, N, exchange="p2p")
    sharded.set_labels(labels)
    spipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    pend = [spipe.retrieve_device_async(idx_h, w_h, k, exclude_history=True, require_any=want_any) for _ in range(3)]
    outs = [p.result() for p in pend]
    if rank == 0:
        full = pkg.FlatIPIndex.adopt(x)
        full.set_labels(labels)
        emb = tower.forward_gather(full.xn, idx_h, w_h, None)
        req = np.stack([np.zeros(B, np.int64), want_any.astype(np.int64)], 1)
        fs, fi, _ = full.search_checked_device(emb, k, exclude=idx_h, require=req)
        np.savez(os.path.join(out_dir, "r0.npz"), s=np.stack([o[0].cpu().numpy() for o in outs]),
                 i=np.stack([o[1].cpu().numpy() for o in outs]), fs=fs.cpu().numpy(), fi=fi.cpu().numpy(),
                 hist=idx_h.cpu().numpy(), labels=labels.cpu().numpy(), want_any=want_any,
                 exchange=np.array(sharded.exchange_used))
    sharded.close()
    dist.destroy_process_group()


def test_sharded_retrieve_require_any_exclude_history_on_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    mp.spawn(_sharded_retrieve_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r = np.load(tmp_path / "r0.npz")
    assert str(r["exchange"]) == "p2p"
    for j in range(r["i"].shape[0]):
        assert np.array_equal(r["i"][j], r["fi"]) and np.allclose(r["s"][j], r["fs"], atol=1e-6)
    for b in range(r["fi"].shape[0]):
        assert not np.isin(r["i"][0][b], r["hist"][b]).any()
        assert (r["labels"][r["i"][0][b]] & r["want_any"][b]).all()
