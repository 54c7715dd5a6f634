"""GPU: label filters (tt_flat_search_filtered, tt_flat_search_exact_filtered) against the masked oracle on every route
of the planner, over a range of selectivities, with adversarial labels, composed with exclusion lists, and through the
Python surfaces built on them."""
import ctypes

import numpy as np
import pytest
import torch

from filter_oracle import allows, search_filtered, torch_topk_filtered
from oracle import flat_ip_oracle as fo

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def build(x, labels=None):
    import two_tower_model_v2_b200 as pkg
    idx = pkg.FlatIPIndex(x.shape[1])
    idx.add(x)
    if labels is not None:
        idx.set_labels(labels)
    return idx


def plan(N, D, nq, K):
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    assert _native.load().tt_flat_plan_describe(N, D, nq, K, out) == 0
    return {"supported": out[0], "block": out[1], "use_threshold": out[6], "route_exact": out[7]}


def check(idx, x, q, k, labels, req, ex=None, expect_certified=True):
    kw = {} if ex is None else {"exclude": torch.from_numpy(ex).to(dev())}
    s, i, n_bad = idx.search_checked_device(torch.from_numpy(q).to(dev()), k, require=req, **kw)
    s, i = s.cpu().numpy(), i.cpu().numpy()
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rs, ri = search_filtered(xn, qn, k, labels, req, ex)
    ok, msg = fo.compare_topk(s, i, rs, ri, xn, qn)
    assert ok, msg
    r2 = np.broadcast_to(np.asarray(req, np.int64), (q.shape[0], 2))
    for r in range(q.shape[0]):
        got = i[r][i[r] >= 0]
        assert allows(labels[got], r2[r, 0], r2[r, 1]).all(), f"query {r} returned a disallowed row"
        if ex is not None:
            assert not np.isin(got, ex[r]).any(), f"query {r} returned an excluded row"
    if expect_certified:
        assert n_bad == 0, f"{n_bad}/{q.shape[0]} queries were not certified"
    return n_bad


def bit0_labels(rng, N, s):
    """Bit 0 set with probability s, the other bits random."""
    lab = rng.integers(0, 1 << 32, N, dtype=np.uint64) & ~np.uint64(1)
    return lab | (rng.random(N) < s).astype(np.uint64)


ROUTES = [  # name, N, D, nq, k  (200_000 rows end in a partial 64-row tile)
    ("every_row_a_candidate", 2_000, 64, 20, 10),
    ("threshold_single_tiling", 200_000, 384, 64, 10),
    ("threshold_single_nq1", 200_000, 384, 1, 10),          # threshold selected inside the main scan
    ("threshold_pair_tiling", 200_000, 384, 200, 100),
    ("threshold_m64_d768", 100_000, 768, 33, 10),
    ("route_exact", 30_000, 64, 8, 1000),
    ("unsupported_d1536", 3_000, 1536, 5, 10),
]


@pytest.mark.parametrize("s", [1.0, 0.1, 0.01])
@pytest.mark.parametrize("name,N,D,nq,k", ROUTES, ids=[r[0] for r in ROUTES])
def test_routes_match_masked_oracle(name, N, D, nq, k, s):
    p = plan(N, D, nq, k)
    if name == "every_row_a_candidate":
        assert p["use_threshold"] == 0 and p["route_exact"] == 0
    elif name == "route_exact":
        assert p["route_exact"] == 1
    elif name == "unsupported_d1536":
        assert p["supported"] == 0
    else:
        assert p["use_threshold"] == 1 and p["block"] == (64 if D == 768 else 256 if nq > 128 else 128)
    rng = np.random.default_rng(N + nq + int(s * 1000))
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = bit0_labels(rng, N, s)
    check(build(x, labels), x, q, k, labels, [1, 0], expect_certified=not p["route_exact"] and N * s >= k)


@pytest.mark.parametrize("s", [1.0, 0.5, 0.1, 1e-2, 1e-3, 1e-4, 0.0])
def test_selectivity_1m(s):
    """1M x 384, nq 128 and 1, K 10, one filter at selectivity s (0 = a filter nothing matches) against the fp32 torch
    checker over the allowed rows."""
    import bench
    import two_tower_model_v2_b200 as pkg
    g = torch.Generator(device="cuda").manual_seed(77)
    N, D, k = 1_000_000, 384, 10
    x = torch.randn((N, D), device=dev(), generator=g)
    idx = pkg.FlatIPIndex.adopt(x)
    allowed = torch.rand(N, device=dev(), generator=g) < s
    idx.set_labels(allowed.to(torch.int32) | 6)
    for nq in (128, 1):
        q = torch.randn((nq, D), device=dev(), generator=g)
        s_, i_, flags, nunc = idx.search_device(q, k, require=np.array([1, 0]))
        n_unc = int(nunc.item())
        if n_unc:
            idx.search_exact_device(q, k, s_, i_, torch.nonzero(flags != 1).flatten().to(torch.int32),
                                    require=np.array([1, 0]))
        ts, ti = torch_topk_filtered(idx.xn, q, k, allowed)
        n_allowed = int(allowed.sum())
        assert torch.equal(ti < 0, i_ < 0) and torch.equal(torch.isneginf(ts), torch.isneginf(s_))
        full = min(k, n_allowed)
        if full:
            rep = bench.compare_topk_device(s_[:, :full], i_[:, :full], ts[:, :full], ti[:, :full])
            assert rep["ok"], rep
        assert bool(allowed[i_[i_ >= 0]].all())
        print(f"s={s} nq={nq}: {n_allowed} allowed rows, {n_unc} uncertified")
        if n_allowed >= k:
            assert n_unc == 0


def test_different_masks_per_query():
    rng = np.random.default_rng(12)
    N, D, nq, k = 200_000, 384, 64, 10
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    labels[rng.random(N) < 0.2] = 0
    bits = [1 << int(b) for b in rng.integers(0, 32, 4 * nq)]
    req = np.zeros((nq, 2), np.int64)
    for r in range(nq):
        kind = r % 4
        if kind == 1:
            req[r] = [bits[4 * r] | bits[4 * r + 1], 0]
        elif kind == 2:
            req[r] = [0, bits[4 * r] | bits[4 * r + 2]]
        elif kind == 3:
            req[r] = [bits[4 * r] | bits[4 * r + 1] | bits[4 * r + 2], bits[4 * r + 3]]
    req[5] = [0xFFFFFFFF, 0]                                # nothing but all-ones labels: padded, exact re-run
    labels[:3] = 0xFFFFFFFF
    check(build(x, labels), x, q, k, labels, req, expect_certified=False)


def test_adversarial_labels_each_query_only_its_bottom_percent():
    """Query j may only return rows labelled with bit j: its own bottom 1 % by score.  The answer must be exact.

    Such queries are not certified by the scan, and the test pins down why.  The best allowed rows of a query sit at
    its 1st percentile, in the bulk of the score distribution, where ~500k rows of this catalog fall per unit of score,
    not in the sparse top tail the candidate budget is sized for.  The certificate needs every allowed row within eps
    (the bf16 error bound) of the K-th allowed score among the candidates.  That is thousands of rows here, while the
    plan keeps a few hundred.  So the finalize kernel reports reason 8 (the K-th score does not clear the bound) and
    nothing else: no overflow, no score mismatch.  The query is re-run exactly."""
    import bench
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200 import _native, ops
    g = torch.Generator(device="cuda").manual_seed(31)
    N, D, nq, k = 1_000_000, 384, 32, 10
    x = torch.randn((N, D), device=dev(), generator=g)
    q = torch.randn((nq, D), device=dev(), generator=g)
    idx = pkg.FlatIPIndex.adopt(x)
    qn = q / (q.norm(dim=1, keepdim=True) + 1e-8)
    labels = torch.zeros(N, device=dev(), dtype=torch.int64)
    for j in range(nq):
        bottom = torch.topk(idx.xn @ qn[j], N // 100, largest=False).indices
        labels[bottom] |= 1 << j
    idx.set_labels(labels)
    req = np.stack([np.array([1 << j for j in range(nq)], np.int64), np.zeros(nq, np.int64)], 1)
    s, i, flags, nunc = idx.search_device(q, k, require=req)
    thr = torch.empty(nq, device=dev())
    cnt = torch.empty(nq, device=dev(), dtype=torch.int32)
    ws = idx._workspace(nq, k)
    _native.check(_native.load().tt_flat_debug_read(ws.data_ptr(), N, D, nq, k, thr.data_ptr(), cnt.data_ptr(),
                                                    ops._stream()), "tt_flat_debug_read")
    n_unc = int(nunc.item())
    reasons = sorted(set(flags.tolist()))
    print(f"adversarial bottom-1% labels: {n_unc}/{nq} uncertified, flags {reasons}, candidates per query "
          f"{int(cnt.min())}-{int(cnt.max())}, finite thresholds {int(torch.isfinite(thr).sum())}/{nq}")
    assert set(reasons) <= {1, -8}, reasons
    assert int(cnt.min()) >= k and int(cnt.max()) <= 4096          # the threshold worked; only the bound did not clear
    if n_unc:
        idx.search_exact_device(q, k, s, i, torch.nonzero(flags != 1).flatten().to(torch.int32), require=req)
    for j in range(nq):
        allowed = (labels >> j) & 1 == 1
        ts, ti = torch_topk_filtered(idx.xn, q[j:j + 1], k, allowed)
        rep = bench.compare_topk_device(s[j:j + 1], i[j:j + 1], ts, ti)
        assert rep["ok"], (j, rep)


def test_fewer_allowed_rows_than_k_pad_and_never_leak():
    rng = np.random.default_rng(3)
    N, D, nq, k = 1000, 64, 4, 20
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = np.zeros(N, np.uint64)
    labels[[7, 100, 555, 901, 999]] = 1
    labels[:500] |= 2
    req = np.array([[1, 0], [4, 0], [2, 0], [0, 3]], np.int64)
    idx = build(x, labels)
    check(idx, x, q, k, labels, req, expect_certified=False)
    s, i, _ = idx.search_checked_device(torch.from_numpy(q).to(dev()), k, require=req)
    s, i = s.cpu().numpy(), i.cpu().numpy()
    assert sorted(i[0, :5].tolist()) == [7, 100, 555, 901, 999] and (i[0, 5:] == -1).all() and np.isneginf(s[0, 5:]).all()
    assert (i[1] == -1).all() and np.isneginf(s[1]).all()
    # the always-exact path alone, with a row selection: the masks are those of the QUERY row
    es, ei = idx.search_exact_device(torch.from_numpy(q).to(dev()), k, require=req)
    assert np.array_equal(ei.cpu().numpy(), i)
    sel = torch.tensor([2, 0], device=dev(), dtype=torch.int32)
    ss = torch.zeros((nq, k), device=dev())
    si = torch.zeros((nq, k), device=dev(), dtype=torch.int64)
    idx.search_exact_device(torch.from_numpy(q).to(dev()), k, ss, si, sel, require=req)
    assert np.array_equal(si.cpu().numpy()[[2, 0]], i[[2, 0]])


@pytest.mark.parametrize("N,D,nq,k", [(200_000, 384, 64, 10), (2_000, 64, 20, 10), (200_000, 384, 1, 10)])
def test_filter_with_exclusion_list(N, D, nq, k):
    rng = np.random.default_rng(N + 5)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = bit0_labels(rng, N, 0.1)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    top = search_filtered(xn, qn, 25, labels, [1, 0])[1]      # each query's own best ALLOWED rows ...
    ex = np.concatenate([top, rng.integers(0, N, (nq, 25)), np.full((nq, 2), -1)], 1).astype(np.int64)
    check(build(x, labels), x, q, k, labels, [1, 0], ex)


@pytest.mark.parametrize("N,D,nq,k", [(200_000, 384, 64, 10), (10_000, 64, 300, 10), (1_000_000, 384, 1, 10)])
def test_trivial_filter_through_the_filtered_kernel_is_bit_identical(N, D, nq, k):
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200 import _native, ops
    g = torch.Generator(device="cuda").manual_seed(N + nq)
    x = torch.randn((N, D), device=dev(), generator=g)
    q = torch.randn((nq, D), device=dev(), generator=g)
    idx = pkg.FlatIPIndex.adopt(x)
    idx.set_labels(torch.randint(0, 1 << 32, (N,), device=dev(), generator=g) | 1)
    s0, i0, f0, _ = idx.search_device(q, k)
    lib = _native.load()
    for req in (torch.zeros((nq, 2), device=dev(), dtype=torch.int32),          # (0, 0) through the FILTER kernels
                torch.tensor([[1, 0]] * nq, device=dev(), dtype=torch.int32)):  # a mask every row satisfies
        s1 = torch.empty_like(s0); i1 = torch.empty_like(i0); f1 = torch.empty_like(f0)
        nunc = torch.empty(1, device=dev(), dtype=torch.int32)
        ws = idx._workspace(nq, k)
        _native.check(lib.tt_flat_search_filtered(
            q.data_ptr(), nq, idx.xn.data_ptr(), idx.xh.data_ptr(), idx.stats.data_ptr(), N, D, k, 0, s1.data_ptr(),
            i1.data_ptr(), f1.data_ptr(), nunc.data_ptr(), idx.labels.data_ptr(), req.data_ptr(), 0, 0, ws.data_ptr(),
            ws.numel(), ops._stream()), "tt_flat_search_filtered")
        assert torch.equal(s0, s1) and torch.equal(i0, i1) and torch.equal(f0, f1)
    # the Python surfaces route (0, 0) to the plain search
    s2, i2, _ = idx.search_checked_device(q, k, require=np.zeros(2, np.int64))
    s3, i3, _ = idx.search_checked_device(q, k)
    assert torch.equal(s2, s3) and torch.equal(i2, i3)


def test_labels_changed_between_searches_and_add_after_set_labels():
    rng = np.random.default_rng(41)
    N, D, nq, k = 50_000, 64, 16, 10
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    labels = bit0_labels(rng, N, 0.3)
    idx = build(x, labels)
    check(idx, x, q, k, labels, [1, 0])
    # in-place update of the rows the first search returned: they are no longer in stock
    first = idx.search_checked_device(torch.from_numpy(q).to(dev()), k, require=[1, 0])[1].cpu().numpy()
    rows = np.unique(first)
    idx.set_labels(np.zeros(rows.size, np.int64), rows=rows)
    labels[rows] = 0
    check(idx, x, q, k, labels, [1, 0])
    assert not np.isin(idx.search_checked_device(torch.from_numpy(q).to(dev()), k, require=[1, 0])[1].cpu().numpy(), rows).any()
    # add with labels (grows the storage), then without (new rows get 0)
    x2 = rng.standard_normal((30_000, D)).astype(np.float32)
    l2 = bit0_labels(rng, 30_000, 0.5)
    idx.add(x2, labels=l2)
    x3 = rng.standard_normal((5_000, D)).astype(np.float32)
    idx.add(torch.from_numpy(x3).to(dev()))
    xa = np.concatenate([x, x2, x3])
    la = np.concatenate([labels, l2, np.zeros(5_000, np.uint64)])
    assert idx.ntotal == xa.shape[0] and np.array_equal(idx.labels.cpu().numpy().view(np.uint32), la.astype(np.uint32))
    check(idx, xa, q, k, la, [1, 0])
    check(idx, xa, q, k, la, [0, 0])
    # a fresh index never given labels refuses a filter
    with pytest.raises(ValueError, match="set_labels"):
        build(x).search_device(torch.from_numpy(q).to(dev()), k, require=[1, 0])
    # host surfaces
    s, i = idx.search(q, k, require=np.array([1, 0]))
    rs, ri = search_filtered(fo.normalize_rows(xa), fo.normalize_rows(q), k, la, [1, 0])
    assert np.array_equal(i, ri)


# ---- Python surfaces --------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["weighted_avg", "attention"])
def test_retrieval_pipeline_require_any_with_exclude_history(method):
    import two_tower_model_v2_b200 as pkg
    from oracle import buyer_tower_oracle as bo
    rng = np.random.default_rng(23)
    N, D, B, S, k = 30000, 384, 16, 50, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    ids = [f"p{i}" for i in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, ids)
    cats = rng.integers(0, 8, N)
    labels = (1 << cats).astype(np.int64)                     # one category bit per item
    db.set_labels(labels)
    torch.manual_seed(3)
    tower = pkg.BuyerTower(D, method).to(dev())
    pipe = pkg.RetrievalPipeline(tower, db)
    events = ["view", "add_to_cart", "purchase"]
    rows = rng.integers(0, N, (B, S))
    ev = rng.integers(0, 3, (B, S))
    lens = rng.integers(1, S + 1, B)
    batch = [[{"product_id": ids[rows[b, s]], "event_type": events[ev[b, s]]} for s in range(lens[b])] for b in range(B)]
    want_any = np.array([(1 << int(rng.integers(0, 8))) | (1 << int(rng.integers(0, 8))) for _ in range(B)], np.int64)
    got = pipe.retrieve_batch(batch, k, exclude_history=True, require_any=want_any)
    xn = fo.normalize_rows(cat)
    wts = np.array([1.0, 5.0, 10.0], np.float32)
    for b in range(B):
        hist = {ids[r] for r in rows[b, :lens[b]]}
        assert not hist & {p for p, _ in got[b]}, f"buyer {b}: a history item was returned"
        assert all(labels[int(p[1:])] & want_any[b] for p, _ in got[b]), f"buyer {b}: a disallowed item"
        x = xn[rows[b, :lens[b]]][None]
        w = wts[ev[b, :lens[b]]][None]
        if method == "weighted_avg":
            emb = bo.weighted_average(x, w)
        else:
            emb = bo.attention_aggregation(x, w, *[p.detach().cpu().numpy() for p in tower.attention.parameters()])
        rs, ri = search_filtered(xn, fo.normalize_rows(emb), k, labels, [0, want_any[b]], rows[b:b + 1, :lens[b]])
        assert [p for p, _ in got[b]] == [ids[i] for i in ri[0]], f"buyer {b}"
        assert np.allclose([s for _, s in got[b]], rs[0], atol=1e-5)
    one = pipe.retrieve(batch[0], k, exclude_history=True, require_any=int(want_any[0]))
    assert [p for p, _ in one] == [p for p, _ in got[0]]



def test_vector_database_labels_by_product_id():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(9)
    N, D, nq, k = 5000, 96, 6, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    pids = [f"item-{i}" for i in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, pids)
    plain = db.retrieve_batch(q, k)
    # everything in stock (bit 0), except the two best items of every query
    db.set_labels(np.ones(N, np.int64))
    out = sorted({p for r in range(nq) for p, _ in plain[r][:2]})
    db.set_labels(np.zeros(len(out), np.int64), product_ids=out)
    labels = np.ones(N, np.uint64)
    labels[[db.id_to_index[p] for p in out]] = 0
    got = db.retrieve_batch(q, k, require_all=1)
    rs, ri = search_filtered(fo.normalize_rows(cat), fo.normalize_rows(q), k, labels, [1, 0])
    for r in range(nq):
        assert [p for p, _ in got[r]] == [pids[i] for i in ri[r]]
        assert not set(out) & {p for p, _ in got[r]}
    one = db.retrieve(q[0], k, require_all=1, exclude=[got[0][0][0]])
    assert [p for p, _ in one] == [p for p, _ in got[0][1:]] + [one[-1][0]] and len(one) == k
    assert db.retrieve_batch(q, k, require_all=0) == plain
    with pytest.raises(ValueError):
        db.set_labels([1], product_ids=["no-such-item"])


# ---- full size ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [0.1, 0.01])
def test_full_size_10m_nq4096_k100_every_query(s):
    """The benched shape with a filter of selectivity s: every query against the chunked fp32 torch checker over the
    allowed rows."""
    import bench
    torch.cuda.empty_cache()
    N, D, nq, k = 10_000_000, 384, 4096, 100
    index, _, _ = bench.make_shard(N, D, 1, 0)
    try:
        g = torch.Generator(device="cuda").manual_seed(4323)
        allowed = torch.rand(N, device="cuda", generator=g) < s
        index.set_labels(allowed.to(torch.int32))
        q = torch.randn((nq, D), device="cuda", generator=g)
        req = np.array([1, 0])
        out, i, flags, nunc = index.search_device(q, k, require=req)
        n_bad = int(nunc.item())
        if n_bad:
            index.search_exact_device(q, k, out, i, torch.nonzero(flags != 1).flatten().to(torch.int32), require=req)
        print(f"10M x 384, nq {nq}, K {k}, s {s}: {n_bad} uncertified queries")
        assert n_bad <= max(1, nq // 1000)
        assert int(i.min()) >= 0 and bool(allowed[i].all())
        ts, tix = torch_topk_filtered(index.xn, q, k, allowed)
        rep = bench.compare_topk_device(out, i, ts, tix)
        assert rep["ok"], rep
    finally:
        del index
        torch.cuda.empty_cache()
