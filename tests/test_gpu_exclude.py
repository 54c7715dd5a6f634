"""GPU: exclusion lists (tt_flat_search_excl, tt_flat_search_shard_excl, tt_flat_shard_search_excl,
tt_flat_search_exact_excl) against the masked oracle on every route of the planner, the adversarial case of a
query excluding its own best rows, and the Python surfaces built on them."""
import ctypes

import numpy as np
import pytest
import torch

from exclusion_oracle import search_excluding, torch_topk_excluding
from oracle import flat_ip_oracle as fo

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def build(x):
    import two_tower_model_v2_b200 as pkg
    idx = pkg.FlatIPIndex(x.shape[1])
    idx.add(x)
    return idx


def plan(N, D, nq, K):
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    assert _native.load().tt_flat_plan_describe(N, D, nq, K, out) == 0
    return {"supported": out[0], "block": out[1], "use_threshold": out[6], "route_exact": out[7]}


def lists(rng, N, nq, E, top=None):
    """[nq, E] lists: some of each query's best rows, random rows, -1 padding, ids outside the catalog, duplicates."""
    ex = rng.integers(0, N, (nq, E)).astype(np.int64)
    if top is not None:
        h = min(E // 2, top.shape[1])
        ex[:, :h] = top[:, :h]
    if E >= 4:
        ex[:, -1] = -1
        ex[:, -2] = N + 7
        ex[:, -3] = ex[:, 0]
    return ex


def check(idx, x, q, k, ex, expect_certified=True):
    s, i, n_bad = idx.search_checked_device(torch.from_numpy(q).to(dev()), k,
                                            exclude=torch.from_numpy(ex).to(dev()))
    s, i = s.cpu().numpy(), i.cpu().numpy()
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rs, ri = search_excluding(xn, qn, k, ex)
    ok, msg = fo.compare_topk(s, i, rs, ri, xn, qn)
    assert ok, msg
    for r in range(q.shape[0]):
        assert not np.isin(i[r][i[r] >= 0], ex[r]).any(), f"query {r} returned an excluded row"
    if expect_certified:
        assert n_bad == 0, f"{n_bad}/{q.shape[0]} queries were not certified"
    return n_bad


ROUTES = [  # name, N, D, nq, k
    ("every_row_a_candidate", 2_000, 64, 20, 10),
    ("threshold_single_tiling", 200_000, 384, 64, 10),
    ("threshold_pair_tiling", 200_000, 384, 200, 100),
    ("threshold_d768", 100_000, 768, 33, 10),
    ("route_exact", 30_000, 64, 8, 1000),
    ("wide_d1100", 3_000, 1100, 5, 10),            # D > 1024 that the scan still serves (64-query blocks)
    ("unsupported_d1536", 3_000, 1536, 5, 10),     # too wide for the resident-query scan: the exact path
]


@pytest.mark.parametrize("E", [1, 50, 1000])
@pytest.mark.parametrize("name,N,D,nq,k", ROUTES, ids=[r[0] for r in ROUTES])
def test_routes_match_masked_oracle(name, N, D, nq, k, E):
    from two_tower_model_v2_b200 import _native
    p = plan(N, D, nq, _native.plan_k(k, E, N))
    if name == "every_row_a_candidate":
        assert p["use_threshold"] == 0 and p["route_exact"] == 0
    elif name == "route_exact":
        assert p["route_exact"] == 1
    elif name == "unsupported_d1536":
        assert p["supported"] == 0
    elif name == "wide_d1100":
        assert p["supported"] == 1 and p["block"] == 64
    else:     # D = 768 runs 64-query blocks
        assert p["use_threshold"] == 1 and p["block"] == (64 if D == 768 else 256 if nq > 128 else 128)
    rng = np.random.default_rng(N + E)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    top = fo.search(fo.normalize_rows(x), fo.normalize_rows(q), min(E, 64))[1]
    check(build(x), x, q, k, lists(rng, N, nq, E, top), expect_certified=E <= 100 and not p["route_exact"])


@pytest.mark.parametrize("E,k", [(50, 10), (50, 100), (100, 10), (100, 100), (1000, 10)])
def test_excluding_each_querys_true_top_e(E, k):
    """1M x 384: a query excluding its own top-E gets exactly ranks E+1..E+k of the unfiltered search."""
    import bench
    import two_tower_model_v2_b200 as pkg
    g = torch.Generator(device="cuda").manual_seed(500 + E)
    N, D, nq = 1_000_000, 384, 128
    x = torch.randn((N, D), device=dev(), generator=g)
    q = torch.randn((nq, D), device=dev(), generator=g)
    idx = pkg.FlatIPIndex.adopt(x)
    ts, ti = bench.torch_flat_topk(idx.xn, q, E + k)
    ex = ti[:, :E].contiguous()
    s, i, flags, nunc = idx.search_device(q, k, exclude=ex)
    n_unc = int(nunc.item())
    if n_unc:
        idx.search_exact_device(q, k, s, i, torch.nonzero(flags != 1).flatten().to(torch.int32), exclude=ex)
    rep = bench.compare_topk_device(s, i, ts[:, E:].contiguous(), ti[:, E:].contiguous())
    assert rep["ok"], rep
    assert not bool((i[:, :, None] == ex[:, None, :]).any())
    print(f"exclude own top-{E}, k={k}, nq={nq}: {n_unc} uncertified queries (re-run exactly)")
    if E <= 100:
        assert n_unc == 0


def test_fewer_allowed_rows_than_k_pad_and_never_leak():
    rng = np.random.default_rng(3)
    for N, D, nq, k in [(1000, 64, 4, 20), (30_000, 64, 3, 1000)]:
        x = rng.standard_normal((N, D)).astype(np.float32)
        q = rng.standard_normal((nq, D)).astype(np.float32)
        E = 1000 if N == 1000 else 1024
        ex = np.full((nq, E), -1, np.int64)
        if N == 1000:
            ex[0, :995] = np.arange(5, 1000)            # 5 allowed rows
            ex[1, :] = rng.permutation(N)               # nothing allowed
        else:
            ex[0, :] = rng.choice(N, E, replace=False)  # k allowed rows remain plenty; exact route
        ex[2, :10] = np.arange(10)
        idx = build(x)
        check(idx, x, q, k, ex, expect_certified=False)
        s, i, _ = idx.search_checked_device(torch.from_numpy(q).to(dev()), k, exclude=torch.from_numpy(ex).to(dev()))
        s, i = s.cpu().numpy(), i.cpu().numpy()
        if N == 1000:
            assert sorted(i[0, :5].tolist()) == [0, 1, 2, 3, 4] and (i[0, 5:] == -1).all() and np.isneginf(s[0, 5:]).all()
            assert (i[1] == -1).all() and np.isneginf(s[1]).all()
        # the always-exact path alone, with a row selection: the list row is the QUERY row
        es, ei = idx.search_exact_device(torch.from_numpy(q).to(dev()), k, exclude=torch.from_numpy(ex).to(dev()))
        assert np.array_equal(ei.cpu().numpy(), i)
        sel = torch.tensor([2, 0], device=dev(), dtype=torch.int32)
        ss = torch.zeros((nq, k), device=dev())
        si = torch.zeros((nq, k), device=dev(), dtype=torch.int64)
        idx.search_exact_device(torch.from_numpy(q).to(dev()), k, ss, si, sel, exclude=torch.from_numpy(ex).to(dev()))
        assert np.array_equal(si.cpu().numpy()[[2, 0]], i[[2, 0]])


@pytest.mark.parametrize("N,D,nq,k", [(200_000, 384, 64, 10), (10_000, 64, 300, 10), (1_000_000, 384, 1, 10)])
def test_no_list_empty_list_and_foreign_ids_are_bit_identical(N, D, nq, k):
    g = torch.Generator(device="cuda").manual_seed(N + nq)
    x = torch.randn((N, D), device=dev(), generator=g)
    q = torch.randn((nq, D), device=dev(), generator=g)
    import two_tower_model_v2_b200 as pkg
    idx = pkg.FlatIPIndex.adopt(x)
    s0, i0, _ = idx.search_checked_device(q, k)
    s1, i1, _ = idx.search_checked_device(q, k, exclude=torch.empty((nq, 0), device=dev(), dtype=torch.int64))
    foreign = torch.full((nq, 50), -1, device=dev(), dtype=torch.int64)
    foreign[:, ::2] = N + torch.arange(25, device=dev())
    s2, i2, _ = idx.search_checked_device(q, k, exclude=foreign)
    assert torch.equal(i0, i1) and torch.equal(s0, s1)
    assert torch.equal(i0, i2) and torch.equal(s0, s2)


def test_argument_errors():
    x = np.random.default_rng(0).standard_normal((500, 32)).astype(np.float32)
    idx = build(x)
    q = torch.randn((3, 32), device=dev())
    with pytest.raises(ValueError):
        idx.search_device(q, 5, exclude=torch.zeros((3, 1025), device=dev(), dtype=torch.int64))
    with pytest.raises(ValueError):
        idx.search_device(q, 5, exclude=torch.zeros((2, 4), device=dev(), dtype=torch.int64))
    with pytest.raises(ValueError):
        idx.search_device(q, 5, exclude=torch.zeros((3, 4), device=dev(), dtype=torch.int32))


# ---- shard paths on one device -------------------------------------------------------------------------
@pytest.mark.parametrize("N,D,nq,k,G,E", [(40_000, 64, 33, 100, 4, 60), (70_000, 384, 130, 10, 8, 1000),
                                          (900, 32, 5, 300, 3, 500)])
def test_shard_records_with_exclusions_merge_to_masked_oracle(N, D, nq, k, G, E):
    import two_tower_model_v2_b200 as pkg
    from test_sharded_gloo import _merge_oracle
    from two_tower_model_v2_b200 import ops
    from two_tower_model_v2_b200.sharded import record_layout, record_views
    rng = np.random.default_rng(N)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    top = fo.search(fo.normalize_rows(x), fo.normalize_rows(q), min(E, 200))[1]
    ex = lists(rng, N, nq, E, top)
    if N == 900:
        ex[0, :] = -1
        lo1, hi1 = pkg.shard_bounds(N, G, 1)
        ex[0, :hi1 - lo1 - 3] = np.arange(lo1 + 3, hi1)     # shard 1 keeps 3 rows < k: padded record, bound -inf
    lay = record_layout(nq, k)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    qd, exd = torch.from_numpy(q).to(dev()), torch.from_numpy(ex).to(dev())
    for g in range(G):
        lo, hi = pkg.shard_bounds(N, G, g)
        idx = build(x[lo:hi])
        idx.id_offset = lo
        s, i, b, f = record_views(gathered[g], lay, nq, k)
        kl = min(k, hi - lo)
        if kl < k:
            s.fill_(float("-inf")); i.fill_(-1)
        idx.search_shard_into(qd, kl, s, i, b, f, exclude=exd)
    s, i, flags, nunc = ops.shard_merge(gathered, lay.off_scores, lay.off_ids, lay.off_bound, lay.off_flags, nq, k)
    ns, ni, nf, nn = _merge_oracle(gathered.cpu(), lay, nq, k)
    assert torch.equal(s.cpu(), ns) and torch.equal(i.cpu(), ni) and torch.equal(flags.cpu(), nf)
    if N == 900:
        sg, ig, bg, fg = record_views(gathered, lay, nq, k)
        assert int((ig[1, 0] >= 0).sum()) == 3 and float(bg[1, 0]) == float("-inf") and int(flags[0]) == 1
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rs, ri = search_excluding(xn, qn, k, ex)
    ok = np.ones(nq, bool) if E <= 100 else (flags.cpu().numpy() == 1)
    assert int(nunc.item()) == 0 or E > 100
    okc, msg = fo.compare_topk(s.cpu().numpy()[ok], i.cpu().numpy()[ok], rs[ok], ri[ok], xn, qn[ok])
    assert okc, msg


def test_shard_global_threshold_path_with_exclusions():
    """3M rows, 4 shards: tt_flat_shard_sample with K_plan, tt_flat_shard_search_excl, merge == single index."""
    import bench
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200 import _native, ops
    from two_tower_model_v2_b200.sharded import record_layout, record_views
    N, D, nq, k, G, E = 3_000_000, 64, 200, 100, 4, 20     # K_plan = 120 (at 150 this shape has no global plan)
    g = torch.Generator(device="cuda").manual_seed(78)
    x = torch.randn((N, D), device=dev(), generator=g)
    q = torch.randn((nq, D), device=dev(), generator=g)
    full = pkg.FlatIPIndex.adopt(x.clone())
    _, ti = bench.torch_flat_topk(full.xn, q, E // 2)
    ex = torch.cat([ti, torch.randint(0, N, (nq, E - E // 2), device=dev(), generator=g)], 1).contiguous()
    fs, fi, fbad = full.search_checked_device(q, k, exclude=ex)
    assert fbad == 0
    shards = []
    for r in range(G):
        lo, hi = pkg.shard_bounds(N, G, r)
        idx = pkg.FlatIPIndex.adopt(x[lo:hi].clone())
        idx.id_offset = lo
        shards.append(idx)
    n_min = min(s.ntotal for s in shards)
    assert shards[0].shard_plan_ok(N, nq, _native.plan_k(k, E, N), n_min)
    topr_g = torch.empty((G, nq, _native.TT_SHARD_TOPR), device=dev())
    for r, idx in enumerate(shards):
        idx.shard_sample(q, k, N, topr_g[r], exclude=ex)
    lay = record_layout(nq, k)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    for r, idx in enumerate(shards):
        s, i, b, f = record_views(gathered[r], lay, nq, k)
        idx.shard_search_into(nq, k, N, topr_g, s, i, b, f, exclude=ex)
    s, i, flags, nunc = ops.shard_merge(gathered, lay.off_scores, lay.off_ids, lay.off_bound, lay.off_flags, nq, k)
    assert int(nunc.item()) == 0
    assert torch.equal(i, fi) and torch.equal(s, fs)
    ts, tix = torch_topk_excluding(full.xn, q, k, ex)
    rep = bench.compare_topk_device(s, i, ts, tix)
    assert rep["ok"], rep


# ---- Python surfaces --------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["weighted_avg", "attention"])
def test_retrieval_pipeline_exclude_history(method):
    import two_tower_model_v2_b200 as pkg
    from oracle import buyer_tower_oracle as bo
    rng = np.random.default_rng(22)
    N, D, B, S, k = 30000, 384, 16, 50, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    ids = [f"p{i}" for i in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, ids)
    torch.manual_seed(3)
    tower = pkg.BuyerTower(D, method).to(dev())
    pipe = pkg.RetrievalPipeline(tower, db)
    events = ["view", "add_to_cart", "purchase"]
    rows = rng.integers(0, N, (B, S))
    ev = rng.integers(0, 3, (B, S))
    lens = rng.integers(1, S + 1, B)
    batch = [[{"product_id": ids[rows[b, s]], "event_type": events[ev[b, s]]} for s in range(lens[b])] for b in range(B)]
    got = pipe.retrieve_batch(batch, k, exclude_history=True)
    plain = pipe.retrieve_batch(batch, k)
    xn = fo.normalize_rows(cat)
    wts = np.array([1.0, 5.0, 10.0], np.float32)
    n_hist_in_plain = 0
    for b in range(B):
        hist = {ids[r] for r in rows[b, :lens[b]]}
        assert not hist & {p for p, _ in got[b]}, f"buyer {b}: a history item was returned"
        n_hist_in_plain += len(hist & {p for p, _ in plain[b]})
        x = xn[rows[b, :lens[b]]][None]
        w = wts[ev[b, :lens[b]]][None]
        if method == "weighted_avg":
            emb = bo.weighted_average(x, w)
        else:
            emb = bo.attention_aggregation(x, w, *[p.detach().cpu().numpy() for p in tower.attention.parameters()])
        rs, ri = search_excluding(xn, fo.normalize_rows(emb), k, rows[b:b + 1, :lens[b]])
        assert [p for p, _ in got[b]] == [ids[i] for i in ri[0]], f"buyer {b}"
        assert np.allclose([s for _, s in got[b]], rs[0], atol=1e-5)
    assert n_hist_in_plain > 0          # without the filter the history does come back
    one = pipe.retrieve(batch[0], k, exclude_history=True)
    assert [p for p, _ in one] == [p for p, _ in got[0]]


def test_vector_database_exclude_by_product_id():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(9)
    N, D, nq, k = 5000, 96, 6, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    pids = [f"item-{i}" for i in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, pids)
    plain = db.retrieve_batch(q, k)
    exclude = [[p for p, _ in plain[r][:3]] + ["no-such-item"] for r in range(nq)]
    exclude[1] = []
    exclude[2] = [plain[2][0][0]] * 3
    got = db.retrieve_batch(q, k, exclude=exclude)
    rows = np.full((nq, 4), -1, np.int64)
    for r, lst in enumerate(exclude):
        known = [db.id_to_index[p] for p in lst if p in db.id_to_index]
        rows[r, :len(known)] = known
    rs, ri = search_excluding(fo.normalize_rows(cat), fo.normalize_rows(q), k, rows)
    for r in range(nq):
        assert [p for p, _ in got[r]] == [pids[i] for i in ri[r]]
        assert not set(exclude[r]) & {p for p, _ in got[r]}
    assert got[1] == plain[1]
    one = db.retrieve(q[0], k, exclude=exclude[0])
    assert [p for p, _ in one] == [p for p, _ in got[0]]
    s, i = db.search_batch(q, k, exclude_rows=rows)
    assert np.array_equal(i, ri)


# ---- two GPUs ----------------------------------------------------------------------------------------------
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
    N, D, B, S, k = 2_000_000, 384, 64, 50, 100
    g = torch.Generator(device="cuda").manual_seed(91)
    x = torch.randn((N, D), device="cuda", generator=g)
    idx_h = torch.randint(0, N, (B, S), device="cuda", generator=g)
    w_h = torch.rand((B, S), device="cuda", generator=g)
    lo, hi = pkg.shard_bounds(N, world, rank)
    local = pkg.FlatIPIndex.adopt(x[lo:hi].clone())
    local.id_offset = lo
    torch.manual_seed(5)
    tower = pkg.BuyerTower(D, "weighted_avg").cuda()
    sharded = pkg.ShardedFlatIPIndex(local, N)
    spipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    s, i, _ = spipe.retrieve_device_async(idx_h, w_h, k, exclude_history=True).result()
    if rank == 0:
        full = pkg.FlatIPIndex.adopt(x)
        emb = tower.forward_gather(full.xn, idx_h, w_h, None)
        fs, fi, _ = full.search_checked_device(emb, k, exclude=idx_h)
        np.savez(os.path.join(out_dir, "r0.npz"), s=s.cpu().numpy(), i=i.cpu().numpy(), fs=fs.cpu().numpy(),
                 fi=fi.cpu().numpy(), hist=idx_h.cpu().numpy())
    sharded.close()
    dist.destroy_process_group()


def test_sharded_retrieve_exclude_history_on_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    mp.spawn(_sharded_retrieve_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r = np.load(tmp_path / "r0.npz")
    assert np.array_equal(r["i"], r["fi"]) and np.allclose(r["s"], r["fs"], atol=1e-6)
    for b in range(r["i"].shape[0]):
        assert not np.isin(r["i"][b], r["hist"][b]).any()


# ---- full size ---------------------------------------------------------------------------------------------
def test_full_size_10m_nq4096_k100_e50_every_query():
    """The benched shape with 50 exclusions per query (25 of the query's own best rows, 25 random): every query
    against the chunked fp32 torch checker with the listed rows masked."""
    import bench
    torch.cuda.empty_cache()
    N, D, nq, k, E = 10_000_000, 384, 4096, 100, 50
    index, _, _ = bench.make_shard(N, D, 1, 0)
    try:
        g = torch.Generator(device="cuda").manual_seed(4322)
        q = torch.randn((nq, D), device="cuda", generator=g)
        _, ti = bench.torch_flat_topk(index.xn, q, E // 2)
        ex = torch.cat([ti, torch.randint(0, N, (nq, E - E // 2), device="cuda", generator=g)], 1).contiguous()
        s, i, flags, nunc = index.search_device(q, k, exclude=ex)
        n_bad = int(nunc.item())
        if n_bad:
            index.search_exact_device(q, k, s, i, torch.nonzero(flags != 1).flatten().to(torch.int32), exclude=ex)
        print(f"10M x 384, nq {nq}, K {k}, E {E}: {n_bad} uncertified queries")
        assert n_bad <= max(1, nq // 1000)
        assert not bool((i[:, :, None] == ex[:, None, :]).any()) and int(i.min()) >= 0
        ts, tix = torch_topk_excluding(index.xn, q, k, ex)
        rep = bench.compare_topk_device(s, i, ts, tix)
        assert rep["ok"], rep
    finally:
        del index
        torch.cuda.empty_cache()
