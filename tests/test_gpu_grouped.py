"""GPU: grouped search (tt_flat_search_grouped, tt_flat_search_exact_grouped) against the group oracle on every route
of the planner, over group layouts from one group per row to groups that follow the scores, composed with exclusion
lists and label filters, in the identity cases bit for bit against the plain search, and through the Python surfaces."""
import ctypes

import numpy as np
import pytest
import torch

from group_oracle import grouped_search, group_of, walk
from oracle import flat_ip_oracle as fo

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def build(x, groups=None, labels=None):
    import two_tower_model_v2_b200 as pkg
    idx = pkg.FlatIPIndex(x.shape[1])
    idx.add(x)
    if groups is not None:
        idx.set_groups(groups)
    if labels is not None:
        idx.set_labels(labels)
    return idx


def plan(N, D, nq, K):
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    assert _native.load().tt_flat_plan_describe(N, D, nq, K, out) == 0
    return {"supported": out[0], "use_threshold": out[6], "route_exact": out[7]}


def check(idx, x, q, k, groups, m, labels=None, req=None, ex=None):
    """search_checked_device with the cap against the group oracle; returns the number of re-run queries."""
    kw = {"max_per_group": m}
    if ex is not None:
        kw["exclude"] = torch.from_numpy(ex).to(dev())
    if req is not None:
        kw["require"] = req
    s, i, n_bad = idx.search_checked_device(torch.from_numpy(q).to(dev()), k, **kw)
    s, i = s.cpu().numpy(), i.cpu().numpy()
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rs, ri = grouped_search(xn, qn, k, groups, m, labels, req, ex)
    ok, msg = fo.compare_topk(s, i, rs, ri, xn, qn)
    assert ok, msg
    g = group_of(groups, i)
    for r in range(q.shape[0]):
        got = g[r][(i[r] >= 0) & (g[r] >= 0)]
        assert (np.unique(got, return_counts=True)[1] <= m).all(), f"query {r}: a group exceeds its cap"
        if ex is not None:
            assert not np.isin(i[r][i[r] >= 0], ex[r]).any(), f"query {r} returned an excluded row"
    return n_bad


def unit(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


# ---- shapes -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,D", [(7, 32), (2000, 100), (50_000, 384), (300_000, 768)])
@pytest.mark.parametrize("K", [1, 10, 100, 1000])
def test_shapes(N, D, K):
    rng = np.random.default_rng(N + D + K)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((3, D)).astype(np.float32)
    groups = rng.integers(0, 10_000, N)
    idx = build(x, groups)
    k = min(K, N)
    for m in (1, 2, 5, 64):
        check(idx, x, q, k, groups, m)


def test_wide_rows_run_the_exact_route():
    rng = np.random.default_rng(5)
    N, D = 20_000, 1536
    assert not plan(N, D, 4, 10)["supported"]
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((4, D)).astype(np.float32)
    groups = rng.integers(-300, 300, N)
    idx = build(x, groups)
    for m in (1, 5):
        assert check(idx, x, q, 10, np.where(groups >= 0, groups, -1), m) == 0


def test_route_exact_and_every_row_a_candidate():
    rng = np.random.default_rng(6)
    # K a large fraction of N (route_exact), and a catalog of at most 16384 rows (every row is a candidate)
    for N, D, K in ((40_000, 64, 2048), (3000, 128, 500)):
        p = plan(N, D, 4, K)
        x = rng.standard_normal((N, D)).astype(np.float32)
        q = rng.standard_normal((4, D)).astype(np.float32)
        groups = rng.integers(0, 50, N)          # m * 50 < K for small m: the tail is padding
        idx = build(x, groups)
        for m in (1, 3, 64):
            n_bad = check(idx, x, q, K, groups, m)
            if not p["use_threshold"] and not p["route_exact"]:
                assert n_bad == 0, "a short answer over every row is certified"


# ---- group layouts ------------------------------------------------------------------------------------------
def layout(name, rng, x):
    N = x.shape[0]
    if name == "few":
        return rng.integers(0, 12, N)                   # m * G < K: the tail is (-inf, -1)
    if name == "random10k":
        return rng.integers(0, 10_000, N)
    if name == "one_per_row":
        return np.arange(N)
    if name == "ungrouped":
        return np.full(N, -1)
    if name == "30pct_ungrouped":
        g = rng.integers(0, 2000, N)
        g[rng.random(N) < 0.3] = -1
        return g
    if name == "correlated":
        dirs = unit(rng, 500, x.shape[1])
        return np.argmax(fo.normalize_rows(x) @ dirs.T, axis=1)
    raise ValueError(name)


@pytest.mark.parametrize("name", ["few", "random10k", "one_per_row", "ungrouped", "30pct_ungrouped", "correlated"])
@pytest.mark.parametrize("m", [1, 2])
def test_layouts(name, m):
    rng = np.random.default_rng(sum(map(ord, name)) + m)
    N, D = 50_000, 384
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = np.concatenate([rng.standard_normal((4, D)), x[rng.integers(0, N, 4)]]).astype(np.float32)
    groups = layout(name, rng, x)
    idx = build(x, groups)
    check(idx, x, q, 100, groups, m)


def test_duplicate_rows_across_and_within_groups():
    rng = np.random.default_rng(11)
    N, D = 50_000, 128
    x = rng.standard_normal((N, D)).astype(np.float32)
    base = rng.integers(0, N, 40)
    for j, b in enumerate(base):                 # 40 rows copied 30 times each
        x[N - 30 * (j + 1):N - 30 * j] = x[b]
    groups = rng.integers(0, 5000, N)
    groups[N - 1200:] = rng.integers(0, 3, 1200)   # copies split over 3 groups and shared within them
    q = x[base[:6]] + 0.01 * rng.standard_normal((6, D)).astype(np.float32)
    idx = build(x, groups)
    for m in (1, 2, 5):
        check(idx, x, q, 100, groups, m)


# ---- composition ------------------------------------------------------------------------------------------------
def test_exclusions_and_filters_compose():
    rng = np.random.default_rng(12)
    N, D, nq, K = 60_000, 384, 6, 100
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    groups = rng.integers(0, 300, N)
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    idx = build(x, groups, labels)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    # lists that name every group's best row, padded, up to 1024 entries
    full_s, full_i = fo.search(xn, qn, 4000)
    ex = np.full((nq, 1024), -1, np.int64)
    for r in range(nq):
        _, first = np.unique(group_of(groups, full_i[r]), return_index=True)
        best = full_i[r][np.sort(first)][:300]
        extra = rng.integers(0, N, 1024 - best.size - 10)
        ex[r, :best.size] = best
        ex[r, best.size:best.size + extra.size] = extra
    req = np.array([[0, 0], [1, 0], [0, 6], [3, 0], [0, 0], [1 << 31, 0]], np.int64)
    for m in (1, 2):
        check(idx, x, q, K, groups, m, ex=ex)
        check(idx, x, q, K, groups, m, labels=labels, req=req)
        check(idx, x, q, K, groups, m, labels=labels, req=req, ex=ex)


# ---- identity cases ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["own_group", "ungrouped", "m_ge_k"])
@pytest.mark.parametrize("mode", ["plain", "excl", "filtered"])
def test_identity_cases_are_bit_identical(case, mode):
    rng = np.random.default_rng(13)
    N, D, nq = 200_000, 384, 64
    K = 50 if case == "m_ge_k" else 100
    m = 64 if case == "m_ge_k" else 1
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    groups = {"own_group": np.arange(N), "ungrouped": np.full(N, -1), "m_ge_k": rng.integers(0, 20, N)}[case]
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    idx = build(x, groups, labels)
    kw = {}
    if mode in ("excl", "filtered"):
        kw["exclude"] = torch.from_numpy(rng.integers(-1, N, (nq, 40))).to(dev())
    if mode == "filtered":
        kw["require"] = np.array([1, 0], np.int64)
    qd = torch.from_numpy(q).to(dev())
    ps, pi, pf, _ = idx.search_device(qd, K, **kw)
    gs, gi, gf, _ = idx.search_device(qd, K, max_per_group=m, **kw)
    both = ((pf == 1) & (gf == 1)).cpu().numpy()
    assert both.sum() >= nq // 2
    assert torch.equal(ps[both], gs[both]) and torch.equal(pi[both], gi[both])
    a_s, a_i, _ = idx.search_checked_device(qd, K, **kw)
    b_s, b_i, _ = idx.search_checked_device(qd, K, max_per_group=m, **kw)
    assert torch.equal(a_i, b_i)


# ---- tensor path against exact path -------------------------------------------------------------------------
def test_tensor_path_matches_exact_path():
    rng = np.random.default_rng(14)
    N, D, nq, K = 300_000, 384, 128, 100
    x = rng.standard_normal((N, D)).astype(np.float32)
    dirs = unit(rng, 2000, D)
    groups = np.argmax(fo.normalize_rows(x) @ dirs.T, axis=1)
    idx = build(x, groups)
    qd = torch.from_numpy(rng.standard_normal((nq, D)).astype(np.float32)).to(dev())
    ex = torch.from_numpy(rng.integers(-1, N, (nq, 16))).to(dev())
    for m in (1, 3):
        s, i, f, _ = idx.search_device(qd, K, max_per_group=m, exclude=ex)
        es, ei = idx.search_exact_device(qd, K, max_per_group=m, exclude=ex)
        ok = f == 1
        assert int(ok.sum()) > 0
        assert torch.equal(i[ok], ei[ok])
        assert float((s[ok] - es[ok]).abs().max()) <= 1e-5


# ---- certificate rejection ------------------------------------------------------------------------------------
def test_crowded_group_fails_the_certificate_and_reruns_exactly():
    rng = np.random.default_rng(15)
    N, D, K = 100_000, 256, 100
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((2, D)).astype(np.float32)
    x[:20_000] = q[0] + 0.3 * rng.standard_normal((20_000, D)).astype(np.float32)   # query 0's neighbourhood ...
    groups = rng.integers(1, 10_000, N)
    groups[:20_000] = 0                                                                # ... is one brand
    idx = build(x, groups)
    qd = torch.from_numpy(q).to(dev())
    _, _, f, _ = idx.search_device(qd, K, max_per_group=1)
    assert int(f[0]) <= 0, "the candidates of query 0 are one group: its first pass cannot be certified"
    assert check(idx, x, q, K, groups, 1) >= 1


# ---- large batch ------------------------------------------------------------------------------------------------
def test_large_batch_against_exact_and_torch():
    import bench
    N, D, nq, K, m = 1_000_000, 384, 4096, 100, 2
    g = torch.Generator(device=dev()).manual_seed(16)
    xn = torch.randn((N, D), device=dev(), generator=g)
    import two_tower_model_v2_b200 as pkg
    idx = pkg.FlatIPIndex.adopt(xn)
    groups = torch.randint(0, 50_000, (N,), device=dev(), generator=g)
    idx.set_groups(groups)
    q = torch.randn((nq, D), device=dev(), generator=g)
    s, i, n_bad = idx.search_async(q, K, max_per_group=m).result()
    sample = torch.arange(0, nq, 128, device=dev(), dtype=torch.int32)
    es, ei = torch.full_like(s, float("nan")), torch.full_like(i, -2)
    idx.search_exact_device(q, K, es, ei, sample, max_per_group=m)
    assert torch.equal(i[sample.long()], ei[sample.long()])
    # fp32 torch checker: sgemm over every row, the walk on the host
    ts, ti = bench.torch_flat_topk(idx.xn, q[sample.long()], 4000)
    ws, wi = walk(ts.cpu().numpy(), ti.cpu().numpy(), groups.cpu().numpy(), m, K)
    rep = bench.compare_topk_device(s[sample.long()], i[sample.long()], torch.from_numpy(ws).to(dev()),
                                    torch.from_numpy(wi).to(dev()))
    assert rep["ok"], rep


# ---- public API -------------------------------------------------------------------------------------------------
def test_vector_database_retrieve_batch_with_brands():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(17)
    N, D, nq, k = 20_000, 128, 8, 20
    cat = rng.standard_normal((N, D)).astype(np.float32)
    pids = [f"p{i}" for i in range(N)]
    brands = [None if r % 7 == 0 else f"brand-{r % 311}" for r in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, pids)
    db.set_groups(brands)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    got = db.retrieve_batch(q, k, max_per_group=1)
    keys = np.array([-1 if b is None else int(b.split("-")[1]) for b in brands])
    rs, ri = grouped_search(fo.normalize_rows(cat), fo.normalize_rows(q), k, keys, 1)
    for r in range(nq):
        assert [p for p, _ in got[r]] == [pids[i] for i in ri[r]]
        named = [brands[int(p[1:])] for p, _ in got[r] if brands[int(p[1:])] is not None]
        assert len(named) == len(set(named))


def test_retrieval_pipeline_exclude_history_and_cap():
    import two_tower_model_v2_b200 as pkg
    from oracle import buyer_tower_oracle as bo
    rng = np.random.default_rng(18)
    N, D, B, S, k = 30_000, 384, 12, 40, 10
    cat = rng.standard_normal((N, D)).astype(np.float32)
    ids = [f"p{i}" for i in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, ids)
    sellers = rng.integers(0, 40, N)
    db.set_groups(sellers.tolist())
    torch.manual_seed(3)
    tower = pkg.BuyerTower(D, "weighted_avg").to(dev())
    pipe = pkg.RetrievalPipeline(tower, db)
    events = ["view", "add_to_cart", "purchase"]
    rows = rng.integers(0, N, (B, S))
    ev = rng.integers(0, 3, (B, S))
    lens = rng.integers(1, S + 1, B)
    batch = [[{"product_id": ids[rows[b, s]], "event_type": events[ev[b, s]]} for s in range(lens[b])] for b in range(B)]
    got = pipe.retrieve_batch(batch, k, exclude_history=True, max_per_group=2)
    xn = fo.normalize_rows(cat)
    wts = np.array([1.0, 5.0, 10.0], np.float32)
    for b in range(B):
        emb = bo.weighted_average(xn[rows[b, :lens[b]]][None], wts[ev[b, :lens[b]]][None])
        rs, ri = grouped_search(xn, fo.normalize_rows(emb), k, sellers, 2, exclude=rows[b:b + 1, :lens[b]])
        assert [p for p, _ in got[b]] == [ids[i] for i in ri[0]], f"buyer {b}"
        assert np.allclose([s for _, s in got[b]], rs[0], atol=1e-5)
    one = pipe.retrieve(batch[0], k, exclude_history=True, max_per_group=2)
    assert [p for p, _ in one] == [p for p, _ in got[0]]


def test_groups_follow_add_and_renumber_sparse_keys():
    rng = np.random.default_rng(19)
    N, D = 5000, 64
    x = rng.standard_normal((N, D)).astype(np.float32)
    keys = rng.choice(np.array([3, 1 << 40, 7, -5, 99_999_999_999]), N)
    idx = build(x, keys)
    assert idx.n_groups == 4 and idx.groups.dtype == torch.int32
    more = rng.standard_normal((100, D)).astype(np.float32)
    idx.add(more)
    assert (idx.groups[N:] == -1).all()
    keys2 = np.concatenate([np.where(keys >= 0, keys, -1), np.full(100, -1)])
    q = rng.standard_normal((3, D)).astype(np.float32)
    check(idx, np.concatenate([x, more]), q, 50, group_of_keys(keys2), 2)
    idx.set_groups(np.array([7, 7]), rows=np.array([N, N + 1]))
    keys2[[N, N + 1]] = 7
    check(idx, np.concatenate([x, more]), q, 50, group_of_keys(keys2), 1)


def group_of_keys(keys):
    """Dense ids of raw keys, as the index renumbers them (negative = ungrouped)."""
    out = np.full(keys.shape, -1, np.int64)
    pos = keys >= 0
    out[pos] = np.unique(keys[pos], return_inverse=True)[1]
    return out
