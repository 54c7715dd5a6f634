"""GPU: range search on the sharded catalog - tt_range_merge against its numpy restatement bit for bit, shards emulated
on one device against FlatIPIndex.range_search_async on the whole catalog (filters, exclusions, an overflowing shard), the
public API and both /retrieve pipelines at world size 1, and a 2-GPU sharded range /retrieve."""
import numpy as np
import pytest
import torch

from oracle import flat_ip_oracle as fo
from range_oracle import check_range
from test_gpu_range import _clustered, radii_at_ranks
from test_sharded_range_host import range_merge_oracle

pytestmark = pytest.mark.gpu


def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


# ---- tt_range_merge alone ------------------------------------------------------------------------------------
def random_records(G, nq, L, seed, short_uncertified=False):
    """[G, nbytes] records of sorted runs: scores on a 1/64 grid (many ties, broken by id), ids unique per query, run
    lengths 0, L, or random (counts beyond L for full runs), garbage after each run's end, a few uncertified flags.
    Query 0 has runs adding up to exactly L.  short_uncertified: every third query has one rank flagged -2 whose count
    exceeds its listed rows."""
    from two_tower_model_v2_b200.sharded import range_record_layout, range_record_views
    rng = np.random.default_rng(seed)
    lay = range_record_layout(nq, L)
    buf = torch.zeros((G, lay.nbytes), dtype=torch.uint8)
    c, s, i, f = (t.numpy() for t in range_record_views(buf, lay, nq, L))
    M = 1 << 22
    perm = rng.permutation(M)[:G * L].astype(np.int64)
    n = rng.choice([0, L, -1], size=(G, nq), p=[0.2, 0.3, 0.5])
    n = np.where(n < 0, rng.integers(0, L + 1, (G, nq)), n)
    n[:, 0] = 0
    n[0, 0] = L // 2 if G > 1 else L
    if G > 1:
        n[1, 0] = L - L // 2
    for r in range(nq):
        ids = ((perm + r * 7919) % M).reshape(G, L)
        for g in range(G):
            m = int(n[g, r])
            sc = (rng.integers(-64, 64, m) / 64.0).astype(np.float32)
            order = np.lexsort((ids[g, :m], -sc.astype(np.float64)))
            s[g, r, :m], i[g, r, :m] = sc[order], ids[g, :m][order]
            s[g, r, m:], i[g, r, m:] = 7.0, 5                      # not a (-inf, -1) tail: the merge must not read it
            c[g, r] = m if m < L else L + int(rng.integers(0, 1000))
    f[:] = np.where(rng.random((G, nq)) < 0.05, rng.choice([-1, -4, -8, 0], (G, nq)), 1)
    if short_uncertified:
        # what tt_flat_range_search writes for a query it could not rank (reason 2): the exact count, or more, with a
        # list shorter than min(count, L) - here none at all - beside ranks with real rows
        for r in range(1, nq, 3):
            g = r % G
            f[g, r], c[g, r] = -2, L + 5
            s[g, r], i[g, r] = -np.inf, -1
            if r % 2 and L > 2:                                    # a short list of real rows ahead of the tail
                s[g, r, :2], i[g, r, :2] = 0.5, [3, 4]
    return buf, lay, n.sum(0)


MERGE_CASES = [(1, 1, 1), (1, 100, 37), (2, 100, 512), (3, 1, 37), (3, 16384, 1), (2, 16384, 37), (8, 1, 512),
               (8, 100, 512), (8, 1000, 37), (8, 16384, 37)]


@pytest.mark.parametrize("G,L,nq", MERGE_CASES)
def test_range_merge_matches_restatement_bit_for_bit(G, L, nq):
    from two_tower_model_v2_b200 import ops
    buf, lay, listed = random_records(G, nq, L, seed=G * 1000 + L + nq)
    got = ops.range_merge(buf.to(dev()), lay, nq, L)
    want = range_merge_oracle(buf, lay, nq, L)
    for a, b in zip(got[:4], want[:4]):
        assert torch.equal(a.cpu(), b)
    assert int(got[4].item()) == int(want[4].item())
    assert listed[0] == L                                           # runs adding up to exactly L


@pytest.mark.parametrize("G,L,nq", [(2, 8, 37), (2, 100, 512), (3, 1000, 37), (8, 16384, 37), (1, 100, 37)])
def test_range_merge_drops_runs_of_uncertified_ranks(G, L, nq):
    """A rank that did not certify a query may report a count its list does not hold (the list ends early in (-inf, -1)
    tail keys, all equal): its run is merged with length 0, the query comes out uncertified, and no other query's row
    or position >= L is touched."""
    from two_tower_model_v2_b200 import ops
    buf, lay, _ = random_records(G, nq, L, seed=G * 7 + L + nq, short_uncertified=True)
    got = ops.range_merge(buf.to(dev()), lay, nq, L)
    want = range_merge_oracle(buf, lay, nq, L)
    for a, b in zip(got[:4], want[:4]):
        assert torch.equal(a.cpu(), b)
    assert int(got[4].item()) == int(want[4].item())
    assert bool((got[3][1::3] != 1).all())


# ---- shards emulated on one device ---------------------------------------------------------------------------
def shard_views(full, G):
    """G FlatIPIndex shards that view the rows of `full` (no copy; the whole catalog's error statistics)."""
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


def emulated_sharded_range(full, G, q, rad, L, exclude=None, require=None):
    """The sharded schedule with every rank on this device: first pass into each shard's record, merge, then for the
    merged-uncertified queries each shard's re-run of its own rows, a second record of those queries, merge, scatter.
    -> (counts, scores, ids, merged first-pass flags, per-shard (n_tensor, n_exact))."""
    from two_tower_model_v2_b200 import ops
    from two_tower_model_v2_b200.sharded import range_record_layout, range_record_views
    from two_tower_model_v2_b200.vector_db import LabelMasks
    shards = shard_views(full, G)
    nq = q.shape[0]
    rad_t = full._radii(rad, nq)
    req = None if require is None else full._requires(require, nq)
    lay = range_record_layout(nq, L)
    gathered = torch.zeros((G, lay.nbytes), dtype=torch.uint8, device=dev())
    needs = []
    kw = {} if exclude is None else {"exclude": exclude}
    if req is not None:
        kw["require"] = LabelMasks(req)
    for g, idx in enumerate(shards):
        needs.append(idx.range_shard_into(q, rad_t, L, *range_record_views(gathered[g], lay, nq, L), **kw))
    c, s, i, flags, _ = ops.range_merge(gathered, lay, nq, L)
    flags = flags.clone()
    rows = torch.nonzero(flags != 1).flatten().cpu().numpy()
    reruns = []
    if rows.size:
        sel = torch.from_numpy(rows).to(dev())
        lay2 = range_record_layout(rows.size, L)
        g2 = torch.zeros((G, lay2.nbytes), dtype=torch.uint8, device=dev())
        for g, idx in enumerate(shards):
            cl, sl, il, fl = range_record_views(gathered[g], lay, nq, L)
            reruns.append(idx.range_rerun(q, rad_t, L, exclude, req, cl, sl, il, fl, needs[g], rows=rows))
            c2, s2, i2, f2 = range_record_views(g2[g], lay2, rows.size, L)
            c2.copy_(cl[sel])
            s2.copy_(sl[sel])
            i2.copy_(il[sel])
            f2.copy_(fl[sel])
        mc, ms, mi, mf, _ = ops.range_merge(g2, lay2, rows.size, L)
        assert bool((mf == 1).all())
        c[sel], s[sel], i[sel] = mc, ms, mi
    return c, s, i, flags, reruns


CASES = ["plain", "filter", "filter+excl", "overflow"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("G", [2, 3, 4])
def test_emulated_shards_equal_the_single_index(G, case):
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(G * 10 + CASES.index(case))
    if case == "overflow":
        N, D, nq, L = 300_000, 384, 4, 1000
        x, q = _clustered(rng, N, D, nq, 60_000)                 # each query's 60 000 near rows fill one or two shards
        rad = np.full(nq, 0.2, np.float32)
    else:
        N, D, nq, L = 150_000, 128, 48, 500
        x = rng.standard_normal((N, D)).astype(np.float32)
        q = rng.standard_normal((nq, D)).astype(np.float32)
        rad = radii_at_ranks(fo.normalize_rows(x), fo.normalize_rows(q), [(0, 100, 1200)[r % 3] for r in range(nq)])
    xn, qn = fo.normalize_rows(x), fo.normalize_rows(q)
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    full = pkg.FlatIPIndex(D)
    full.add(x)
    full.set_labels(labels)
    req = ex = None
    if case.startswith("filter"):
        req = np.zeros((nq, 2), np.int64)
        req[::2, 0] = 1
        req[1::4, 1] = 6
    if case.endswith("excl"):
        ex = np.concatenate([fo.search(xn, qn, 30)[1], rng.integers(0, N, (nq, 10)), np.full((nq, 2), -1)], 1)
    qd = torch.from_numpy(q).to(dev())
    exd = None if ex is None else torch.from_numpy(ex).to(dev())
    c, s, i, flags, reruns = emulated_sharded_range(full, G, qd, rad, L, exd, req)
    kw = {} if exd is None else {"exclude": exd}
    fc, fs, fi, n_t, n_x = full.range_search_async(qd, rad, L, require=req, **kw).result()
    _, _, _, fflags, _, _ = full.range_search_device(qd, rad, L, require=req, **kw)
    assert torch.equal(c, fc)
    ok = ((flags == 1) | ((-flags) & 1 == 1)) & ((fflags == 1) | ((-fflags) & 1 == 1))     # neither side went exact
    if any(r[1] for r in reruns):
        ok &= flags == 1
    if n_x:
        ok &= fflags == 1
    assert torch.equal(i[ok], fi[ok]) and torch.equal(s[ok], fs[ok])
    good, msg = check_range(c.cpu().numpy(), s.cpu().numpy(), i.cpu().numpy(), xn, qn, rad, L,
                            None if req is None else labels, req, ex)
    assert good, msg
    if case == "overflow":
        assert bool(((-flags) & 1 == 1).all()) and all(r[1] == 0 for r in reruns), (flags, reruns)
        assert sum(r[0] for r in reruns) >= nq and bool(ok.all())
    print(f"G {G} {case}: counts {int(c.min())}..{int(c.max())}, merged uncertified {int((flags != 1).sum())}, "
          f"shard re-runs {reruns}, single re-runs {n_t}/{n_x}")


# ---- public API at world size 1 ------------------------------------------------------------------------------
def test_sharded_range_api_world1_equals_single_index():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(81)
    N, D, nq, L = 60_000, 384, 24, 300
    x = rng.standard_normal((N, D)).astype(np.float32)
    q = rng.standard_normal((nq, D)).astype(np.float32)
    local = pkg.FlatIPIndex(D)
    local.add(x)
    sharded = pkg.ShardedFlatIPIndex(local, N)
    labels = rng.integers(0, 4, N).astype(np.int64)
    sharded.set_labels(labels)
    rad = radii_at_ranks(fo.normalize_rows(x), fo.normalize_rows(q), [(5, 200, 600)[r % 3] for r in range(nq)])
    qd = torch.from_numpy(q).to(dev())
    ex = torch.from_numpy(fo.search(fo.normalize_rows(x), fo.normalize_rows(q), 4)[1]).to(dev())
    for kw in ({}, {"require": np.array([1, 0])}, {"exclude": ex, "require": np.array([0, 2])}):
        c, s, i, n = sharded.range_search_device(qd, rad, L, **kw)
        fc, fs, fi, _, _ = local.range_search_async(qd, rad, L, **kw).result()
        assert torch.equal(c, fc) and torch.equal(i, fi) and torch.equal(s, fs) and n == 0
    hkw = {"exclude": ex.cpu().numpy(), "require": np.array([1, 0])}
    got = sharded.range_search(q, 0.1, 200, **hkw)
    want = local.range_search(q, 0.1, 200, **hkw)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    # two batches in flight, then the results
    p1 = sharded.range_search_async(qd, rad, L)
    p2 = sharded.range_search_async(qd, 0.2, 50)
    c2, _, i2, _ = p2.result()
    c1, _, i1, _ = p1.result()
    assert torch.equal(i1, local.range_search_async(qd, rad, L).result()[2])
    assert torch.equal(i2, local.range_search_async(qd, 0.2, 50).result()[2])


@pytest.mark.parametrize("method", ["weighted_avg", "attention"])
def test_retrieve_above_pipelines_world1(method):
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(25)
    N, D, B, S, L = 30_000, 384, 12, 30, 200
    cat = rng.standard_normal((N, D)).astype(np.float32)
    pids = [f"p{j}" for j in range(N)]
    db = pkg.VectorDatabase(D)
    db.build_index(cat, pids)
    labels = (1 << rng.integers(0, 4, N)).astype(np.int64)
    db.set_labels(labels)
    torch.manual_seed(4)
    tower = pkg.BuyerTower(D, method).to(dev())
    pipe = pkg.RetrievalPipeline(tower, db)
    batch = [[{"product_id": pids[int(j)], "event_type": ("view", "purchase")[t % 2], "timestamp": t}
              for t, j in enumerate(rng.integers(0, N, int(rng.integers(1, S))))] for _ in range(B)]
    want_any = np.array([(1 << int(rng.integers(0, 4))) | 1 for _ in range(B)], np.int64)
    got = pipe.retrieve_above_batch(batch, 0.05, L, exclude_history=True, require_any=want_any)
    idx, w, _ = pipe.encode_histories(batch)
    emb = pipe.encode_device(torch.from_numpy(idx).to(dev()), torch.from_numpy(w).to(dev()))
    hist = [[pids[j] for j in row if j >= 0] for row in idx]
    want = db.retrieve_above(emb.cpu().numpy(), 0.05, L, exclude=hist, require_any=want_any)
    assert got == want and sum(len(g) for g in got) > B
    # one request alone: pooled on its own (a batch of one may round the pooled embedding differently)
    idx1, w1, _ = pipe.encode_histories(batch[:1])
    emb1 = pipe.encode_device(torch.from_numpy(idx1).to(dev()), torch.from_numpy(w1).to(dev()))
    want1 = db.retrieve_above(emb1.cpu().numpy(), 0.05, L, exclude=hist[:1], require_any=int(want_any[0]))
    assert pipe.retrieve_above(batch[0], 0.05, L, exclude_history=True, require_any=int(want_any[0])) == want1[0]
    assert [p for p, _ in want1[0]] == [p for p, _ in want[0]]
    # the sharded pipeline at world size 1 (owner-computes pooling) equals the single index searched with its own pooled
    # embedding; with weighted_avg that embedding is the single-device pipeline's, so the results are too
    sharded = pkg.ShardedFlatIPIndex(db.index, N)
    sharded.set_labels(labels)
    spipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    idx_d, w_d = torch.from_numpy(idx).to(dev()), torch.from_numpy(w).to(dev())
    sc, ss, si, _ = spipe.retrieve_above_device_async(idx_d, w_d, 0.05, L, exclude_history=True,
                                                      require_any=want_any).result()
    req = np.stack([np.zeros(B, np.int64), want_any], 1)
    oc, os_, oi, _, _ = db.index.range_search_async(spipe.encode_device(idx_d, w_d), 0.05, L, exclude=idx_d,
                                                    require=req).result()
    assert torch.equal(sc, oc) and torch.equal(si, oi) and torch.equal(ss, os_)
    if method == "weighted_avg":
        pc, ps, pi, _, _ = pipe.retrieve_above_device_async(idx_d, w_d, 0.05, L, exclude_history=True,
                                                            require_any=want_any).result()
        assert torch.equal(sc, pc) and torch.equal(si, pi) and torch.allclose(ss, ps, atol=1e-6)
    lims, D_, I_, _ = spipe.retrieve_above_host_async(idx_d.cpu().pin_memory(), w_d.cpu().pin_memory(), 0.05, L,
                                                      exclude_history=True, require_any=want_any).result()
    si_h = si.cpu().numpy()
    assert all(np.array_equal(I_[lims[b]:lims[b + 1]], si_h[b][:lims[b + 1] - lims[b]]) for b in range(B))


# ---- two GPUs ------------------------------------------------------------------------------------------------
def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_range_retrieve_worker(rank, world, port, out_dir):
    import os
    import torch.distributed as dist
    import two_tower_model_v2_b200 as pkg
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    N, D, B, S, L = 2_000_000, 384, 64, 40, 1000
    g = torch.Generator(device="cuda").manual_seed(93)
    x = torch.randn((N, D), device="cuda", generator=g)
    idx_h = torch.randint(0, N, (B, S), device="cuda", generator=g)
    w_h = torch.rand((B, S), device="cuda", generator=g)
    labels = 1 << torch.randint(0, 8, (N,), device="cuda", generator=g)
    want_any = (1 << torch.randint(0, 8, (B,), generator=torch.Generator().manual_seed(3))).numpy() | 1
    lo, hi = pkg.shard_bounds(N, world, rank)
    local = pkg.FlatIPIndex.adopt(x[lo:hi].clone())
    local.id_offset = lo
    torch.manual_seed(5)
    tower = pkg.BuyerTower(D, "weighted_avg").cuda()
    sharded = pkg.ShardedFlatIPIndex(local, N)
    sharded.set_labels(labels)
    spipe = pkg.ShardedRetrievalPipeline(tower, sharded)
    pend = [spipe.retrieve_above_device_async(idx_h, w_h, m, L, exclude_history=True, require_any=want_any)
            for m in (0.05, 0.12)]
    outs = [p.result() for p in pend]
    if rank == 0:
        full = pkg.FlatIPIndex.adopt(x)
        full.set_labels(labels)
        emb = tower.forward_gather(full.xn, idx_h, w_h, None)
        req = np.stack([np.zeros(B, np.int64), want_any.astype(np.int64)], 1)
        ref = [full.range_search_async(emb, m, L, exclude=idx_h, require=req).result() for m in (0.05, 0.12)]
        np.savez(os.path.join(out_dir, "r0.npz"), c=np.stack([o[0].cpu().numpy() for o in outs]),
                 i=np.stack([o[2].cpu().numpy() for o in outs]), s=np.stack([o[1].cpu().numpy() for o in outs]),
                 fc=np.stack([r[0].cpu().numpy() for r in ref]), fi=np.stack([r[2].cpu().numpy() for r in ref]),
                 fs=np.stack([r[1].cpu().numpy() for r in ref]))
    sharded.close()
    dist.destroy_process_group()


def test_sharded_range_retrieve_on_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    mp.spawn(_sharded_range_retrieve_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r = np.load(tmp_path / "r0.npz")
    assert np.array_equal(r["c"], r["fc"]) and (r["c"][0] > 1000).any() and (r["c"][1] < 1000).any()
    assert np.array_equal(r["i"], r["fi"]) and np.allclose(r["s"], r["fs"], atol=1e-6)
