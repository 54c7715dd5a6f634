"""CPU: range search on the sharded catalog without a GPU - the argument checks of tt_range_merge, the range record
layout and chunking, argument validation before any collective, and ShardedFlatIPIndex.range_search_async at world size
2 (gloo) with range-oracle stand-ins for the local searches and a numpy restatement of tt_range_merge."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import flat_ip_oracle as fo
from range_oracle import range_search
from test_sharded_filter_host import _LabelledStandIn


def range_merge_oracle(gathered, lay, nq, L):
    """numpy restatement of tt_range_merge -> (counts, scores, ids, flags, n_uncertified [1]) torch tensors.  A rank's
    run holds min(count, L) entries if the rank certified the query, none otherwise."""
    from two_tower_model_v2_b200.sharded import range_record_views
    cg, sg, ig, fg = (t.cpu().numpy() for t in range_record_views(gathered.cpu(), lay, nq, L))
    counts = cg.sum(0).astype(np.int64)
    out_s, out_i = np.full((nq, L), -np.inf, np.float32), np.full((nq, L), -1, np.int64)
    flags = np.ones(nq, np.int32)
    for r in range(nq):
        n = np.where(fg[:, r] == 1, np.clip(cg[:, r], 0, L), 0)
        s = np.concatenate([sg[g, r, :n[g]] for g in range(cg.shape[0])])
        i = np.concatenate([ig[g, r, :n[g]] for g in range(cg.shape[0])])
        order = np.lexsort((i, -s.astype(np.float64)))[:L]
        out_s[r, :order.size], out_i[r, :order.size] = s[order], i[order]
        f = fg[:, r]
        if (f != 1).any():
            flags[r] = -int(np.bitwise_or.reduce(np.where(f < 0, -f, 0)))
    nunc = torch.tensor([int((flags != 1).sum())], dtype=torch.int32)
    return (torch.from_numpy(counts), torch.from_numpy(out_s), torch.from_numpy(out_i), torch.from_numpy(flags), nunc)


# ---- the C-ABI ------------------------------------------------------------------------------------------------
def test_range_merge_arguments_are_checked_without_a_gpu(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    p = ctypes.c_void_p(256)          # never dereferenced: the argument checks come first
    cases = [  # gathered, stride, off_counts, off_scores, off_ids, off_flags, G, nq, L, out, what
        (None, 4096, 0, 16, 64, 128, 2, 1, 10, p, "null pointer"),
        (p, 4096, 0, 16, 64, 128, 2, 1, 10, None, "null pointer"),
        (p, 4096, 0, 16, 64, 128, 0, 1, 10, p, "1 <= G <= 64"),
        (p, 4096, 0, 16, 64, 128, 65, 1, 10, p, "1 <= G <= 64"),
        (p, 4096, 0, 16, 64, 128, 2, 1, 0, p, "TT_FLAT_RANGE_MAX_RESULTS"),
        (p, 4096, 0, 16, 64, 128, 2, 1, 16385, p, "TT_FLAT_RANGE_MAX_RESULTS"),
        (p, 4096, 4, 16, 64, 128, 2, 1, 10, p, "misaligned"),
        (p, 4096, 0, 18, 64, 128, 2, 1, 10, p, "misaligned"),
        (p, 4096, 0, 16, 68, 128, 2, 1, 10, p, "misaligned"),
        (p, 4096, 0, 16, 64, 130, 2, 1, 10, p, "misaligned"),
        (p, 4100, 0, 16, 64, 128, 2, 1, 10, p, "misaligned"),
        (ctypes.c_void_p(260), 4096, 0, 16, 64, 128, 2, 1, 10, p, "misaligned"),
        (p, 4096, 0, 16, 64, 128, 2, -1, 10, p, "nq >= 0"),
    ]
    for gth, stride, oc, os_, oi, of, G, nq, L, out, what in cases:
        rc = lib.tt_range_merge(gth, stride, oc, os_, oi, of, G, nq, L, out, p, p, p, p, None)
        assert rc == 1 and what in _native.last_error(), (what, _native.last_error())


def test_range_merge_binding_matches_the_header():
    import re
    from pathlib import Path
    from two_tower_model_v2_b200 import _native
    text = (Path(__file__).resolve().parents[1] / "include" / "tt_b200.h").read_text()
    decl = re.search(r"int tt_range_merge\((.*?)\);", re.sub(r"/\*.*?\*/", "", text, flags=re.S), re.S).group(1)
    assert len(decl.split(",")) == len(_native.SIGNATURES["tt_range_merge"][1]) == 15


def test_range_record_layout_is_aligned_and_views_round_trip():
    from two_tower_model_v2_b200.sharded import range_record_layout, range_record_views
    for nq, L in ((1, 1), (3, 7), (37, 100), (5, 16384)):
        lay = range_record_layout(nq, L)
        assert all(o % 16 == 0 for o in lay)
        assert lay.nbytes >= nq * (8 + 12 * L + 4)
        buf = torch.zeros((2, lay.nbytes), dtype=torch.uint8)
        c, s, i, f = range_record_views(buf, lay, nq, L)
        assert c.shape == (2, nq) and s.shape == (2, nq, L) and i.shape == (2, nq, L) and f.shape == (2, nq)
        rng = np.random.default_rng(nq)
        want = (rng.integers(-5, 1 << 40, (2, nq)), rng.standard_normal((2, nq, L)).astype(np.float32),
                rng.integers(-1, 1 << 40, (2, nq, L)), rng.integers(-15, 2, (2, nq)).astype(np.int32))
        for view, w in zip((c, s, i, f), want):
            view.copy_(torch.from_numpy(w))
        for view, w in zip(range_record_views(buf.clone(), lay, nq, L), want):      # fields do not overlap
            assert np.array_equal(view.numpy(), w)
        one = range_record_views(buf[1], lay, nq, L)
        assert np.array_equal(one[1].numpy(), want[1][1])


def test_range_chunks_fit_the_exchange_budget():
    from two_tower_model_v2_b200.sharded import RANGE_EXCHANGE_BUDGET, range_chunk_rows, range_record_layout
    for nq, L, G in ((4096, 16384, 8), (4096, 1000, 8), (1, 16384, 64), (100, 100, 2), (4096, 16384, 1)):
        c = range_chunk_rows(nq, L, G)
        assert 1 <= c <= nq and c == range_chunk_rows(nq, L, G)
        assert c == 1 or G * range_record_layout(c, L).nbytes <= RANGE_EXCHANGE_BUDGET
        assert c == nq or G * range_record_layout(c + 1, L).nbytes > RANGE_EXCHANGE_BUDGET
    assert range_chunk_rows(4096, 16384, 8) < 4096 and range_chunk_rows(4096, 100, 8) == 4096
    assert range_chunk_rows(10, 100, 2, budget=2 * range_record_layout(3, 100).nbytes) == 3


# ---- stand-in local index -------------------------------------------------------------------------------------
class _RangeOracleIndex(_LabelledStandIn):
    """A FlatIPIndex stand-in on a CPU rank: the first pass and the re-run search the shard with the range oracle
    (GLOBAL exclusion ids, the masks of a LabelMasks).  `fail` lists (call, query) pairs whose first pass reports the
    query uncertified with a count its empty list does not hold; `reruns` logs the query rows each re-run completed."""

    def __init__(self, xn_shard, id_offset, fail=()):
        super().__init__(xn_shard.shape[0], id_offset)
        self.xn, self.d, self.device = xn_shard, xn_shard.shape[1], torch.device("cpu")
        self.fail, self.calls, self.reruns = set(fail), 0, []

    def _radii(self, radius, nq):
        from two_tower_model_v2_b200.vector_db import FlatIPIndex
        return FlatIPIndex._radii(self, radius, nq)

    def _search(self, q, rad, L, excl, req):
        qn = fo.normalize_rows(q.numpy())
        ex = None
        if excl is not None:
            e = excl.numpy()
            ex = np.where((e >= self.id_offset) & (e < self.id_offset + self.n), e - self.id_offset, -1)
        labels = None if req is None else self.labels.view(np.uint32)
        c, s, i = range_search(self.xn, qn, rad.numpy(), L, labels, None if req is None else req.numpy(), ex)
        return c, s, np.where(i >= 0, i + self.id_offset, -1)

    def range_shard_into(self, q, rad, L, counts, scores, ids, flags, *, exclude=None, require=None):
        c, s, i = self._search(q, rad, L, exclude, None if require is None else require.words)
        f = np.ones(q.shape[0], np.int32)
        for call, r in self.fail:
            if call == self.calls:
                f[r], c[r], s[r], i[r] = -2, c[r] + L + 5, -np.inf, -1      # a count its (empty) list does not hold
        self.calls += 1
        for view, v in zip((counts, scores, ids, flags), (c, s, i, f)):
            view.copy_(torch.from_numpy(v))
        return torch.ones(q.shape[0], dtype=torch.int32)

    def range_rerun(self, q, rad, L, excl, req, counts, scores, ids, flags, need, rows=None):
        rows = np.asarray(rows)
        rows = rows[flags.numpy()[rows] != 1]
        self.reruns.append(rows.tolist())
        if rows.size:
            sel = torch.from_numpy(rows)
            c, s, i = self._search(q[sel], rad[sel], L, None if excl is None else excl[sel],
                                   None if req is None else req[sel])
            counts[sel], scores[sel], ids[sel] = torch.from_numpy(c), torch.from_numpy(s), torch.from_numpy(i)
            flags[sel] = 1
        return rows.size, 0

    def post_flag(self, status):
        return int(status[0])

    def read_flag(self, token):
        return token


def test_bad_arguments_raise_before_any_collective():
    import two_tower_model_v2_b200 as pkg
    rng = np.random.default_rng(1)
    local = _RangeOracleIndex(fo.normalize_rows(rng.standard_normal((20, 8)).astype(np.float32)), 0)
    sh = pkg.ShardedFlatIPIndex(local, 20)

    def no_collective(*a, **k):
        raise AssertionError("a collective was reached")
    sh._validate = sh._exchange = no_collective
    q = torch.zeros((3, 8))
    bad = [dict(radius=float("nan")), dict(radius=np.zeros(2)), dict(radius="0.5"),
           dict(max_results=0), dict(max_results=16385), dict(max_results=2.0),
           dict(require=np.array([1, 0])),                                  # no label words yet
           dict(exclude=torch.zeros((2, 4), dtype=torch.int64)), dict(exclude=torch.zeros((3, 4), dtype=torch.int32)),
           dict(exclude=np.zeros((3, 4), np.int64)), dict(exclude=torch.zeros((3, 1025), dtype=torch.int64))]
    for kw in bad:
        args = dict(radius=0.5, max_results=10)
        args.update(kw)
        with pytest.raises(ValueError):
            sh.range_search_async(q, args.pop("radius"), args.pop("max_results"), **args)
    sh.set_labels(np.ones(20, np.int64))
    for req in (np.zeros((3, 3), np.int64), np.array([[1, 0]] * 2), np.array([[-1, 0]] * 3)):
        with pytest.raises(ValueError):
            sh.range_search_async(q, 0.5, 10, require=req)
    with pytest.raises(ValueError, match="expected queries"):
        sh.range_search_async(torch.zeros((3, 5)), 0.5, 10)


# ---- world size 2 ---------------------------------------------------------------------------------------------
N, D, NQ = 800, 16, 6


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _data():
    rng = np.random.default_rng(7)                      # the same catalog, queries, labels and lists on every rank
    xn = fo.normalize_rows(rng.standard_normal((N, D)).astype(np.float32))
    q = rng.standard_normal((NQ, D)).astype(np.float32)
    qn = fo.normalize_rows(q)
    labels = rng.integers(0, 1 << 24, N, dtype=np.int64) << 8
    labels |= (rng.random(N) < 0.5).astype(np.int64) << 1
    labels[:N // 2] |= 4                                   # bit 2: every row of shard 0, none of shard 1
    s = np.sort(qn.astype(np.float64) @ xn.astype(np.float64).T, axis=1)[:, ::-1]

    def at(r):                                             # radius per query between its rank r and r + 1 scores
        return (0.5 * (s[:, r - 1] + s[:, r])).astype(np.float32)
    top = fo.search(xn, qn, 8)[1]
    ex = np.concatenate([top, np.full((NQ, 3), -1), np.full((NQ, 1), 10 * N)], 1).astype(np.int64)
    req = np.array([[2, 0], [0, 0], [4, 0], [2, 4], [0, 2 | 4], [2, 0]], np.int64)
    cases = {  # name: (radius, L, require, exclude)
        "split": (at(30), 50, None, None),
        "one_shard": (at(200), 400, np.array([4, 0]), None),
        "over_L": (at(200), 40, None, None),
        "zero": (2.0, 10, None, None),
        "small_shards": (-1.5, 600, None, None),
        "filter_excl": (at(100), 30, req, ex),
        "per_query_radius": (np.array([2.0, -1.5, 0.0, 0.3, 0.1, 0.5], np.float32), 300, None, None),
    }
    return xn, q, labels, cases


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import two_tower_model_v2_b200 as pkg
    xn, q, labels, cases = _data()
    lo, hi = pkg.shard_bounds(N, world, rank)
    out = {}
    for name, (rad, L, req, ex) in cases.items():
        local = _RangeOracleIndex(xn[lo:hi], lo)
        sharded = pkg.ShardedFlatIPIndex(local, N, range_merge=range_merge_oracle)
        sharded.set_labels(labels)
        kw = {} if ex is None else {"exclude": torch.from_numpy(ex)}
        c, s, i, n = sharded.range_search_device(torch.from_numpy(q), rad, L, require=req, **kw)
        out[name] = (c.numpy(), s.numpy(), i.numpy(), n, local.reruns)
    # two batches in flight before .result(), then a batch whose query 2 rank 1 does not certify
    local = _RangeOracleIndex(xn[lo:hi], lo, fail=[(2, 2)] if rank == 1 else [])
    sharded = pkg.ShardedFlatIPIndex(local, N, range_merge=range_merge_oracle)
    sharded.set_labels(labels)
    p1 = sharded.range_search_async(torch.from_numpy(q), cases["split"][0], 50)
    p2 = sharded.range_search_async(torch.from_numpy(q), cases["over_L"][0], 40)
    p3 = sharded.range_search_async(torch.from_numpy(q), cases["over_L"][0], 40)
    for name, p in (("in_flight_1", p2), ("in_flight_0", p1), ("uncertified", p3)):
        c, s, i, n = p.result()
        out[name] = (c.numpy(), s.numpy(), i.numpy(), n, list(local.reruns))
    np.savez(os.path.join(out_dir, f"r{rank}.npz"),
             **{f"{k}_{f}": np.asarray(v[j], dtype=object if f == "reruns" else None)
                for k, v in out.items() for j, f in enumerate(("c", "s", "i", "n", "reruns"))})
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def world2(tmp_path_factory):
    d = tmp_path_factory.mktemp("range_gloo")
    mp.spawn(_worker, args=(2, _free_port(), str(d)), nprocs=2, join=True)
    return [np.load(d / f"r{r}.npz", allow_pickle=True) for r in range(2)]


def _check(world2, name, rad, L, req=None, ex=None):
    xn, q, labels, _ = _data()
    want_c, want_s, want_i = range_search(xn, fo.normalize_rows(q), rad, L, None if req is None else labels.astype(np.uint64),
                                          req, ex)
    for g in world2:
        assert np.array_equal(g[f"{name}_c"], want_c), name
        assert np.array_equal(g[f"{name}_i"], want_i), name
        assert np.allclose(g[f"{name}_s"], want_s, atol=1e-6) and np.array_equal(np.isneginf(g[f"{name}_s"]),
                                                                                  np.isneginf(want_s)), name
    return want_c, want_i


@pytest.mark.parametrize("name", ["split", "one_shard", "over_L", "zero", "small_shards", "filter_excl",
                                  "per_query_radius"])
def test_world2_equals_the_range_oracle(world2, name):
    _, _, labels, cases = _data()
    rad, L, req, ex = cases[name]
    c, i = _check(world2, name, rad, L, req, ex)
    for g in world2:
        assert int(g[f"{name}_n"]) == 0 and g[f"{name}_reruns"].tolist() == []
    lists = [i[r][i[r] >= 0] for r in range(NQ)]
    if name == "split":
        assert all((x < N // 2).any() and (x >= N // 2).any() for x in lists) and (c < L).all()
    elif name == "one_shard":
        assert all((x < N // 2).all() for x in lists) and (c > 0).all()
    elif name == "over_L":
        assert (c > L).all() and all((x < N // 2).any() and (x >= N // 2).any() for x in lists)
    elif name == "zero":
        assert (c == 0).all() and (i == -1).all()
    elif name == "small_shards":
        assert (c == N).all() and all(x.size == L for x in lists)
    elif name == "filter_excl":
        for r in range(NQ):
            assert not np.isin(lists[r], ex[r]).any()
            a, y = req[r]
            assert ((labels[lists[r]] & a) == a).all() and (y == 0 or (labels[lists[r]] & y != 0).all())
    elif name == "per_query_radius":
        assert c[0] == 0 and c[1] == N


def test_world2_two_batches_in_flight(world2):
    _, _, _, cases = _data()
    _check(world2, "in_flight_0", cases["split"][0], 50)
    _check(world2, "in_flight_1", cases["over_L"][0], 40)


def test_world2_uncertified_query_is_rerun_by_its_rank_only(world2):
    _, _, _, cases = _data()
    _check(world2, "uncertified", cases["over_L"][0], 40)
    r0, r1 = world2
    assert int(r0["uncertified_n"]) == int(r1["uncertified_n"]) == 1
    assert r0["uncertified_reruns"].tolist() == [[]]          # rank 0 joins the second exchange with its first-pass row
    assert r1["uncertified_reruns"].tolist() == [[2]]
