"""GPU: range search (tt_flat_range_search, tt_flat_range_search_exact) against the fp64-judged range oracle on every
route of the planner, against the top-K search, through the overflow re-runs, with label filters and exclusion lists,
through VectorDatabase.retrieve_above, and at the benched catalog size."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import flat_ip_oracle as fo
from range_oracle import check_range

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


def plan(N, D, nq):
    from two_tower_model_v2_b200 import _native
    out = (ctypes.c_int32 * 16)()
    assert _native.load().tt_flat_plan_describe(N, D, nq, 1, out) == 0
    return {"supported": out[0], "block": out[1]}


def radii_at_ranks(xn, qn, ranks):
    """Per query: a radius between the fp64 scores of ranks r and r+1 (r = 0: above the best row), so that about r rows
    qualify and no row sits on the radius."""
    s = np.sort(qn.astype(np.float64) @ xn.astype(np.float64).T, axis=1)[:, ::-1]
    out = np.empty(qn.shape[0])
    for i, r in enumerate(ranks):
        out[i] = s[i, 0] + 0.01 if r == 0 else 0.5 * (s[i, r - 1] + s[i, min(r, s.shape[1] - 1)])
    return out.astype(np.float32)


def run(idx, q, radius, L, **kw):
    counts, s, i, n_t, n_x = idx.range_search_async(torch.from_numpy(q).to(dev()), radius, L, **kw).result()
    return counts.cpu().numpy(), s.cpu().numpy(), i.cpu().numpy(), n_t, n_x


ROUTES = [  # name, N, D, nq
    ("every_row_fits", 2_000, 64, 20),
    ("single_tiling", 200_000, 384, 64),
    ("single_nq1", 200_000, 384, 1),
    ("pair_tiling", 200_000, 384, 200),
    ("d768_streamed_query_blocks", 100_000, 768, 150),
    ("d30", 20_000, 30, 8),
    ("unsupported_d1536", 3_000, 1536, 5),
]


@pytest.mark.parametrize("name,N,D,nq", ROUTES, ids=[r[0] for r in ROUTES])
def test_routes_match_range_oracle(name, N, D, nq):
    p = plan(N, D, nq)
    if name == "unsupported_d1536":
        assert p["supported"] == 0
    elif name == "pair_tiling" or name.startswith("d768"):
        assert p["block"] == 256
    rng = np.random.default_rng(N + nq)
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    L = 500
    ranks = [(0, 4, 1000, 1500)[r % 4] for r in range(nq)]       # none, a few, about 1000 (> L), more than L
    rad = radii_at_ranks(xn, qn, ranks)
    idx = build(x)
    c, s, i, n_t, n_x = run(idx, q, rad, L)
    ok, msg = check_range(c, s, i, xn, qn, rad, L)
    assert ok, f"{name}: {msg}"
    assert n_x == 0 or name == "unsupported_d1536", f"{name}: {n_x} queries needed the exact path"
    print(f"{name}: counts {sorted(set(c.tolist()))[:6]}..., tensor re-runs {n_t}, exact re-runs {n_x}")


def test_agrees_with_topk_search_bit_for_bit():
    rng = np.random.default_rng(21)
    N, D, nq, L = 200_000, 384, 96, 100
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rad = radii_at_ranks(xn, qn, [(300, 100, 40, 1, 0)[r % 5] for r in range(nq)])
    idx = build(x)
    c, s, i, _, _ = run(idx, q, rad, L)
    qd = torch.from_numpy(q).to(dev())
    ts, ti, _ = idx.search_checked_device(qd, L)
    ts, ti = ts.cpu().numpy(), ti.cpu().numpy()
    for r in range(nq):
        m = min(int(c[r]), L)
        assert np.array_equal(i[r, :m], ti[r, :m]) and np.array_equal(s[r, :m], ts[r, :m]), f"query {r}"
    k = int(c[c < L].max()) + 3
    ks, ki, _ = idx.search_checked_device(qd, k)
    ks, ki = ks.cpu().numpy(), ki.cpu().numpy()
    for r in np.flatnonzero(c < L):
        m = int(c[r])
        assert np.array_equal(i[r, :m], ki[r, :m]) and np.array_equal(s[r, :m], ks[r, :m]), f"query {r} (k={k})"


def _clustered(rng, N, D, nq, n_dup):
    """A random catalog with, for each query, n_dup rows q + noise of growing size: their scores spread from ~0.93 down
    to ~0.3 (nearly all above a radius of 0.2), far more candidates than the default budget holds."""
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    qn = fo.normalize_rows(q)
    for j in range(nq):
        sig = np.linspace(0.02, 0.15, n_dup, dtype=np.float32)[:, None]
        rows = slice(1000 + j * n_dup, 1000 + (j + 1) * n_dup)
        x[rows] = qn[j] + sig * rng.standard_normal((n_dup, D)).astype(np.float32)
    return x, q


def test_overflow_reruns_on_the_tensor_path():
    rng = np.random.default_rng(33)
    N, D, nq, L = 300_000, 384, 4, 1000
    x, q = _clustered(rng, N, D, nq, 60_000)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    idx = build(x)
    _, _, _, flags, need, _ = idx.range_search_device(torch.from_numpy(q).to(dev()), 0.2, L)
    assert bool(((-flags) & 1 == 1).all()), flags                     # every query's candidates overflowed
    c, s, i, n_t, n_x = run(idx, q, 0.2, L)
    ok, msg = check_range(c, s, i, xn, qn, 0.2, L)
    assert ok, msg
    assert (c >= 50_000).all() and n_t == nq and n_x == 0, (c, n_t, n_x)
    # a workspace budget too small for even one query's re-run: the exact path serves them
    idx.RANGE_WS_BUDGET = 1 << 19
    c2, s2, i2, n_t2, n_x2 = run(idx, q, 0.2, L)
    assert n_x2 == nq and n_t2 == 0
    assert np.array_equal(c2, c) and check_range(c2, s2, i2, xn, qn, 0.2, L)[0]


def test_overflow_reruns_from_a_large_batch():
    """A first pass over 300 queries (CTA-pair tiling, few catalog slices) whose 4 clustered queries overflow: their
    re-run plans for 4 queries and slices the catalog more finely, and its segments must still hold them."""
    rng = np.random.default_rng(34)
    N, D, nq, L = 300_000, 384, 300, 1000
    x, q4 = _clustered(rng, N, D, 4, 60_000)
    q = np.concatenate([q4, rng.standard_normal((nq - 4, D)).astype(np.float32)])
    assert plan(N, D, nq)["block"] == 256
    idx = build(x)
    _, _, _, flags, _, _ = idx.range_search_device(torch.from_numpy(q).to(dev()), 0.2, L)
    fl = flags.cpu().numpy()
    assert ((-fl[:4]) & 1 == 1).all() and (fl[4:] == 1).all(), fl[:8]
    c, s, i, n_t, n_x = run(idx, q, 0.2, L)
    assert n_t == 4 and n_x == 0, (n_t, n_x)
    sel = np.r_[0:4, 4:nq:37]
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q[sel])
    ok, msg = check_range(c[sel], s[sel], i[sel], xn, qn, 0.2, L)
    assert ok, msg
    assert (c[:4] >= 50_000).all(), c[:4]


def test_huge_band_exact_count():
    rng = np.random.default_rng(44)
    N, D, nq, L = 200_000, 384, 6, 2000
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    rad = radii_at_ranks(xn, qn, [N // 2] * nq)                       # the median: half the catalog qualifies
    c, s, i, n_t, n_x = run(build(x), q, rad, L)
    ok, msg = check_range(c, s, i, xn, qn, rad, L)
    assert ok, msg
    assert (np.abs(c - N // 2) <= 2).all(), c
    print(f"huge band: counts {c.tolist()}, tensor re-runs {n_t}, exact re-runs {n_x}")


def test_filters_and_exclusions_compose():
    rng = np.random.default_rng(55)
    N, D, nq, L = 200_000, 384, 40, 300
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    req = np.zeros((nq, 2), np.int64)
    req[::2, 0] = 1
    req[1::4, 1] = 6
    # every query excludes its 20 best rows; query 0's list covers its whole range result
    top = fo.search(xn, qn, 40)[1]
    ex = np.full((nq, 64), -1, np.int64)
    ex[:, :20] = top[:, :20]
    ex[0, :40] = top[0]
    rad = radii_at_ranks(xn, qn, [(30, 600, 40)[r % 3] for r in range(nq)])
    rad[0] = radii_at_ranks(xn, qn[:1], [40])[0]
    idx = build(x, labels)
    c, s, i, n_t, n_x = run(idx, q, rad, L, exclude=torch.from_numpy(ex).to(dev()), require=req)
    ok, msg = check_range(c, s, i, xn, qn, rad, L, labels, req, ex)
    assert ok, msg
    assert c[0] == 0 and (i[0] == -1).all()                           # the whole top is excluded: nothing, not counted
    assert n_x == 0


def test_exact_path_equals_tensor_path():
    rng = np.random.default_rng(66)
    N, D, nq, L = 100_000, 256, 24, 400
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    labels = rng.integers(0, 4, N).astype(np.uint64)
    rad = radii_at_ranks(xn, qn, [(10, 600, 200)[r % 3] for r in range(nq)])
    idx = build(x, labels)
    qd = torch.from_numpy(q).to(dev())
    ex = torch.from_numpy(fo.search(xn, qn, 5)[1]).to(dev())
    req = np.array([1, 0])
    c, s, i, flags, _, nunc = idx.range_search_device(qd, rad, L, exclude=ex, require=req)
    assert int(nunc.item()) == 0
    args = idx._range_args(qd, rad, L, ex, req)
    ce, se, ie = torch.empty_like(c), torch.empty_like(s), torch.empty_like(i)
    idx._range_exact(*args, ce, se, ie, torch.arange(nq, device=dev(), dtype=torch.int32))
    assert torch.equal(c, ce) and torch.equal(i < 0, ie < 0)
    pad = lambda t: torch.where(torch.isneginf(t), torch.zeros_like(t), t).cpu().numpy()    # the shared (-inf, -1) tails
    ok, msg = fo.compare_topk(pad(s), i.cpu().numpy(), pad(se), ie.cpu().numpy(), xn, qn)
    assert ok, msg
    assert check_range(ce.cpu().numpy(), se.cpu().numpy(), ie.cpu().numpy(), xn, qn, rad, L, labels, [1, 0],
                       ex.cpu().numpy())[0]


def test_retrieve_above_maps_products_exclusions_and_labels():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(77)
    N, D, nq = 5_000, 64, 3
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    pids = [f"sku{j}" for j in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(x, pids)
    labels = rng.integers(0, 2, N).astype(np.uint64)
    db.set_labels(labels)
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    ex = [[pids[j] for j in fo.search(xn, qn[r:r + 1], 3)[1][0]] + ["unknown"] for r in range(nq)]
    res = db.retrieve_above(q, 0.25, 100, exclude=ex, require_all=1)
    s64 = qn.astype(np.float64) @ xn.astype(np.float64).T
    for r in range(nq):
        want = [j for j in np.argsort(-s64[r], kind="stable") if s64[r, j] > 0.25 and labels[j] == 1
                and pids[j] not in ex[r]][:100]
        assert [p for p, _ in res[r]] == [pids[j] for j in want]
        assert all(abs(v - s64[r, j]) < 1e-5 for (_, v), j in zip(res[r], want))
    assert db.retrieve_above(q[0], 2.0) == [[]]


def test_full_size_10m_against_device_checker():
    """10M x 384 (generated as bench.py does), nq 1024, radius per query between its 500th and 501st exact scores: every
    query's count and list against a device fp32 checker (chunked sgemm with TF32 off, counting and top-k)."""
    import bench
    torch.cuda.empty_cache()
    index, _, _ = bench.make_shard(10_000_000, 384, 1, 0)
    try:
        nq, L = 1024, 1000
        q = torch.randn((nq, 384), device=dev(), generator=torch.Generator(device="cuda").manual_seed(99))
        ts, ti = bench.torch_flat_topk(index.xn, q, 501)
        rad = 0.5 * (ts[:, 499] + ts[:, 500])
        c, s, i, n_t, n_x = index.range_search_async(q, rad, L).result()
        # device checker: fp32 sgemm (TF32 off) over 1M-row chunks, rows above the radius counted
        qn = q / (q.norm(dim=1, keepdim=True) + 1e-8)
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        cnt = torch.zeros(nq, device=dev(), dtype=torch.int64)
        near = torch.zeros(nq, device=dev(), dtype=torch.int64)
        for lo in range(0, index.ntotal, 1 << 20):
            sc = qn @ index.xn[lo:lo + (1 << 20)].T
            cnt += (sc > rad[:, None]).sum(1)
            near += ((sc - rad[:, None]).abs() <= 1e-6).sum(1)
        torch.backends.cuda.matmul.allow_tf32 = prev
        assert bool(((c - cnt).abs() <= near).all()), "counts differ outside ties at the radius"
        m = int(c.min())
        assert m >= 490 and bool((c <= L).all())
        rep = bench.compare_topk_device(s[:, :m], i[:, :m], ts[:, :m], ti[:, :m])
        assert rep["ok"], rep
        assert bool((i[torch.arange(L, device=dev())[None, :] >= c[:, None]] == -1).all())
        print(f"10M x 384 nq {nq}: counts {int(c.min())}..{int(c.max())}, tensor re-runs {n_t}, exact re-runs {n_x}")
    finally:
        del index
        torch.cuda.empty_cache()
