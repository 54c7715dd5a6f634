"""CPU: label filters on the sharded search without a GPU - the argument checks of the shard C-ABI calls,
ShardedFlatIPIndex.set_labels, and the serial, two-phase and pipelined schedules at world size 2 (gloo) with filtered
oracle stand-ins for the local searches."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from filter_oracle import search_filtered
from oracle import flat_ip_oracle as fo


def test_shard_filter_arguments_are_checked_without_a_gpu(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    p = ctypes.c_void_p(256)          # never dereferenced: the argument checks come first
    odd4, odd8 = ctypes.c_void_p(260), ctypes.c_void_p(260)
    for labels, req, what in [(None, p, "null labels or require"), (p, None, "null labels or require"),
                              (odd4, p, "16-byte aligned"), (p, odd8, "8-byte aligned")]:
        rc = lib.tt_flat_search_shard_filtered(p, 1, p, p, p, 1000, 64, 10, 0, p, p, p, p, p, labels, req, None, 0, p,
                                               1 << 20, None)
        assert rc == 1 and what in _native.last_error(), _native.last_error()
        rc = lib.tt_flat_shard_sample_filtered(p, 1, p, p, 1000, 2000, 64, 10, labels, req, p, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error(), _native.last_error()
        rc = lib.tt_flat_shard_search_filtered(1, p, p, 1000, 2000, 64, 10, 0, p, 2, p, p, p, p, p, labels, req, None, 0,
                                               p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error(), _native.last_error()
    rc = lib.tt_flat_search_shard_filtered(p, 1, p, p, p, 1000, 64, 10, 0, p, p, p, p, None, p, p, None, 0, p, 1 << 20, None)
    assert rc == 1 and "null bound" in _native.last_error()


# ---- stand-ins ---------------------------------------------------------------------------------------------
class _LabelledStandIn:
    """The label state of a FlatIPIndex on the host: words are allocated (zero-filled) on the first set_labels."""

    def __init__(self, n, id_offset):
        self.n, self.id_offset, self.labels = n, id_offset, None

    @property
    def ntotal(self):
        return self.n

    def set_labels(self, labels, rows=None):
        from two_tower_model_v2_b200.vector_db import u32_words
        w = u32_words(labels, "labels")            # the value checks of FlatIPIndex.set_labels
        if self.labels is None:
            self.labels = np.zeros(self.ntotal, np.int32)
        if rows is None:
            assert w.shape == (self.ntotal,)
            self.labels[:] = w
        else:
            self.labels[np.asarray(rows)] = w


def _words(x):
    return np.asarray(x, np.int64) & 0xFFFFFFFF


def test_set_labels_slices_and_routes_global_rows():
    import two_tower_model_v2_b200 as pkg
    N, G = 10, 3
    bounds = [pkg.shard_bounds(N, G, r) for r in range(G)]       # [0, 4), [4, 8), [8, 10)
    full = np.array([1, 2, 3, 4, 5, 6, 7, 8, 0xFFFFFFFF, 10], np.int64)
    locals_ = [_LabelledStandIn(hi - lo, lo) for lo, hi in bounds]
    for loc in locals_:
        pkg.ShardedFlatIPIndex(loc, N).set_labels(full)
    for (lo, hi), loc in zip(bounds, locals_):
        assert _words(loc.labels).tolist() == full[lo:hi].tolist()
    # rows= routes each word to the shard that owns the row; a shard that gets no word still ends up with zeros
    rows, words = np.array([5, 1, 6]), np.array([50, 10, 0xFFFFFFFE], np.int64)
    locals_ = [_LabelledStandIn(hi - lo, lo) for lo, hi in bounds]
    for loc in locals_:
        pkg.ShardedFlatIPIndex(loc, N).set_labels(words, rows=torch.from_numpy(rows))
    assert _words(locals_[0].labels).tolist() == [0, 10, 0, 0]
    assert _words(locals_[1].labels).tolist() == [0, 50, 0xFFFFFFFE, 0]
    assert locals_[2].labels is not None and _words(locals_[2].labels).tolist() == [0, 0]
    # an in-place update keeps the other words
    pkg.ShardedFlatIPIndex(locals_[1], N).set_labels([7], rows=[4])
    assert _words(locals_[1].labels).tolist() == [7, 50, 0xFFFFFFFE, 0]
    sh = pkg.ShardedFlatIPIndex(_LabelledStandIn(4, 0), N)
    for labels, rows in ((np.zeros(9, np.int64), None), (np.zeros(2, np.int64), np.array([0])),
                         (np.zeros(1, np.int64), np.array([10])), (np.zeros(1, np.int64), np.array([-1])),
                         (np.array([1 << 32]), np.array([0])), (np.zeros(1, np.int64), np.array([0.0]))):
        with pytest.raises(ValueError):
            sh.set_labels(labels, rows)


def test_set_labels_passes_bit_31_words_to_a_flat_index():
    """Through the real FlatIPIndex.set_labels checks (storage stubbed): words with bit 31 set, whole array and rows=."""
    import two_tower_model_v2_b200 as pkg
    from two_tower_model_v2_b200.vector_db import FlatIPIndex

    class _Shell(FlatIPIndex):
        def __init__(self, n, id_offset):
            self.d, self.device, self.id_offset = 4, torch.device("cpu"), id_offset
            self.xn, self.labels, self._labels_store, self.stored = torch.zeros((n, 4)), None, None, []

        def _store_labels(self, words, rows):
            self.stored.append((_words(words).tolist(), None if rows is None else rows.tolist()))

    a, b = _Shell(2, 0), _Shell(2, 2)
    for loc in (a, b):
        pkg.ShardedFlatIPIndex(loc, 4).set_labels(np.array([1, 0xFFFFFFFF, 0x80000000, 7], np.int64))
        pkg.ShardedFlatIPIndex(loc, 4).set_labels(np.array([0x80000000, 0xFFFFFFFF]), rows=[1, 2])
        pkg.ShardedFlatIPIndex(loc, 4).set_labels(torch.tensor([0xFFFFFFFF]), rows=torch.tensor([3]))
    assert a.stored == [([1, 0xFFFFFFFF], None), ([0x80000000], [1]), ([], [])]
    assert b.stored == [([0x80000000, 7], None), ([0xFFFFFFFF], [0]), ([0xFFFFFFFF], [1])]


def test_filter_without_labels_and_bad_masks_raise_before_any_collective():
    import two_tower_model_v2_b200 as pkg
    sh = pkg.ShardedFlatIPIndex(_LabelledStandIn(4, 0), 4)       # no process group: a collective would raise otherwise
    q = torch.zeros((3, 8))
    with pytest.raises(ValueError, match="set_labels"):
        sh.search_async(q, 2, require=np.array([1, 0]))
    with pytest.raises(ValueError, match="set_labels"):
        sh.search_exact_device(q, 2, require=np.array([1, 0]))
    for bad in (np.zeros((3, 3), np.int64), np.array([[1, 0]] * 2), np.array([[-1, 0]] * 3)):
        with pytest.raises(ValueError):
            sh._requires(bad, 3, q.device)
    assert sh._requires(np.zeros((3, 2), np.int64), 3, q.device) is None
    assert sh._requires(None, 3, q.device) is None
    sh.local.device, sh.local.d = q.device, 8
    with pytest.raises(ValueError):              # the sliced call checks its masks before the query all-gather
        sh.search_host_sliced_async(np.zeros((3, 8), np.float32), 2, require=np.array([[1, 0]] * 2))


def test_label_masks_of_the_wrong_shape_are_rejected():
    from two_tower_model_v2_b200.vector_db import FlatIPIndex, LabelMasks
    idx = FlatIPIndex.__new__(FlatIPIndex)
    idx.device, idx.labels = torch.device("cpu"), torch.zeros(5, dtype=torch.int32)
    ok = torch.ones((3, 2), dtype=torch.int32)
    assert idx._requires(LabelMasks(ok), 3) is ok
    for bad in (torch.ones((2, 2), dtype=torch.int32), torch.ones((3, 2), dtype=torch.int64), torch.ones((2, 3), dtype=torch.int32).t()):
        with pytest.raises(ValueError, match="LabelMasks"):
            idx._requires(LabelMasks(bad), 3)


class _FilterOracleIndex(_LabelledStandIn):
    """A FlatIPIndex stand-in on a CPU rank: every local call searches the shard with filter_oracle.search_filtered
    (GLOBAL exclusion ids, the masks of a LabelMasks) and records which call saw a filter.  A shard with fewer than k
    allowed rows pads with (-inf, -1) and flags -2, as the kernels do."""

    def __init__(self, xn_shard, id_offset, rank=0, world=1):
        super().__init__(xn_shard.shape[0], id_offset)
        self.xn, self.rank, self.world = xn_shard, rank, world
        self.exact_calls, self.saw, self.q = 0, [], {}

    def _search(self, q, k, exclude, require):
        qn = fo.normalize_rows(q.numpy())
        req = np.zeros((qn.shape[0], 2), np.int64) if require is None else require.words.numpy()
        ex = None
        if exclude is not None:
            e = exclude.numpy()
            ex = np.where((e >= self.id_offset) & (e < self.id_offset + self.n), e - self.id_offset, -1)
        labels = self.labels if self.labels is not None else np.zeros(self.n, np.int32)
        s, i = search_filtered(self.xn, qn, k, labels.view(np.uint32), req, ex)
        return s, np.where(i >= 0, i + self.id_offset, -1)

    def search_shard_into(self, q, k, scores, ids, bound, flags, *, exclude=None, require=None):
        self.saw.append(("shard", require is not None))
        s, i = self._search(q, k, exclude, require)
        scores[:, :k] = torch.from_numpy(s)
        ids[:, :k] = torch.from_numpy(i)
        bound.fill_(float("-inf"))
        flags.copy_(torch.from_numpy(np.where((i < 0).any(1), -2, 1).astype(np.int32)))

    def search_exact_into(self, q, k, scores, ids, qsel, *, exclude=None, require=None):
        self.exact_calls += 1
        self.saw.append(("exact", require is not None))
        rows = qsel.long()
        req = None if require is None else type(require)(require.words[rows])
        s, i = self._search(q[rows], k, None if exclude is None else exclude[rows], req)
        scores[rows, :k] = torch.from_numpy(s)
        ids[rows, :k] = torch.from_numpy(i)

    # the two-phase contract
    def shard_plan_ok(self, n_total, nq, k, n_local_min):
        return n_local_min >= k

    def shard_sample(self, q, k, n_total, topr, slot=0, *, exclude=None, require=None):
        self.saw.append(("sample", require is not None))
        self.q[slot] = q
        topr.fill_(float(self.rank))

    def shard_search_into(self, nq, k, n_total, topr_g, scores, ids, bound, flags, slot=0, *, exclude=None, require=None):
        assert [float(topr_g[g, 0, 0]) for g in range(self.world)] == [float(g) for g in range(self.world)]
        self.search_shard_into(self.q[slot], k, scores, ids, bound, flags, exclude=exclude, require=require)
        self.saw[-1] = ("global", require is not None)

    # status words of the pipelined schedule (host stand-ins of the pinned ring)
    def post_flag(self, status):
        return status.clone().tolist() if isinstance(status, torch.Tensor) else int(status)

    def read_flag(self, token):
        return token


def _merge_status(gathered, lay, nq, K, nunc=None):
    from test_sharded_gloo import _merge_oracle
    s, i, f, n = _merge_oracle(gathered, lay, nq, K)
    if nunc is not None:
        nunc.fill_(n)
    return s, i, f, n


class _GlooExchange:
    """Stands in for P2PExchange: `push` all-gathers the record over gloo at once and returns its sequence number,
    `wait` hands back the gathered [G, nbytes] buffer."""

    def __init__(self, world):
        self.world, self.seq, self.got = world, [0, 0, 0], {}

    def push(self, ch, src):
        out = torch.empty((self.world, src.numel()), dtype=torch.uint8)
        dist.all_gather_into_tensor(out.view(-1), src.contiguous())
        self.seq[ch] += 1
        self.got[(ch, self.seq[ch])] = out
        return self.seq[ch]

    def wait(self, ch, seq, status):
        return self.got.pop((ch, seq))

    def all_gather(self, ch, src, status):
        return self.wait(ch, self.push(ch, src), status)


# ---- world size 2 ---------------------------------------------------------------------------------------------
N, D, NQ, K = 800, 16, 6, 10
REQ = np.array([[0, 0],          # no filter
                [2, 0],          # ~30 % of the rows, both shards
                [4, 0],          # rows of shard 0 only
                [8, 0],          # no row at all
                [16, 0],         # 4 rows, 2 per shard: fewer than k
                [0, 2 | 4]], np.int64)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _data(with_excl):
    rng = np.random.default_rng(0)                      # the same catalog, queries, labels and lists on every rank
    xn = fo.normalize_rows(rng.standard_normal((N, D)).astype(np.float32))
    q = rng.standard_normal((NQ, D)).astype(np.float32)
    labels = rng.integers(0, 1 << 24, N, dtype=np.int64) << 8                     # noise in bits 8-31
    labels |= (rng.random(N) < 0.3).astype(np.int64) << 1
    labels[:N // 2] |= (rng.random(N // 2) < 0.5).astype(np.int64) << 2
    labels[[1, 2, N - 3, N - 2]] |= 16
    ex = None
    if with_excl:                                       # each query's own 5 best allowed rows, random rows, padding
        top = search_filtered(xn, fo.normalize_rows(q), 5, labels, REQ)[1]
        ex = np.concatenate([top, rng.integers(0, N, (NQ, 4)), np.full((NQ, 2), -1)], 1).astype(np.int64)
        ex[0, -1] = 10 * N
    return xn, q, labels, ex


def _worker(rank, world, port, out_dir, mode, with_excl, by_rows):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import two_tower_model_v2_b200 as pkg
    from test_sharded_gloo import _FlagOnceMerge
    xn, q, labels, ex = _data(with_excl)
    lo, hi = pkg.shard_bounds(N, world, rank)
    local = _FilterOracleIndex(xn[lo:hi], lo, rank, world)
    if mode == "serial":
        local.shard_plan_ok = None              # no global-threshold plan: every shard picks its own threshold
    merge = _FlagOnceMerge() if mode == "two_phase" else _merge_status
    sharded = pkg.ShardedFlatIPIndex(local, N, merge=merge)
    if by_rows:
        rows = np.flatnonzero(labels)
        sharded.set_labels(labels[rows], rows=rows)
    else:
        sharded.set_labels(labels)
    kw = {} if ex is None else {"exclude": torch.from_numpy(ex)}
    reqs = [REQ]
    if mode == "pipelined":
        ex_ = _GlooExchange(world)
        sharded._p2p_for = lambda *a: ex_
        reqs = [REQ, np.roll(REQ, 1, 0), np.array([2, 0])]
        pending = [sharded.search_async(torch.from_numpy(q), K, require=r, **kw) for r in reqs]
        outs = [p.result() for p in pending]
    else:
        outs = [sharded.search_device(torch.from_numpy(q), K, require=REQ, **kw)]
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), s=np.stack([o[0].numpy() for o in outs]),
             i=np.stack([o[1].numpy() for o in outs]), n_bad=np.array([o[2] for o in outs]),
             reqs=np.stack([np.broadcast_to(r, (NQ, 2)) for r in reqs]), exact_calls=local.exact_calls,
             saw=np.array([f"{a}:{b}" for a, b in local.saw]))
    dist.destroy_process_group()


def _run(tmp_path, mode, with_excl=False, by_rows=False):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), mode, with_excl, by_rows), nprocs=world, join=True)
    xn, q, labels, ex = _data(with_excl)
    outs = [np.load(tmp_path / f"r{r}.npz") for r in range(world)]
    for g in outs:
        for b in range(g["i"].shape[0]):
            rs, ri = search_filtered(xn, fo.normalize_rows(q), K, labels, g["reqs"][b], ex)
            assert np.array_equal(g["i"][b], ri), b
            assert np.allclose(g["s"][b], rs, atol=1e-6) and np.array_equal(np.isneginf(g["s"][b]), np.isneginf(rs))
    return outs, labels


def _common(outs, labels):
    g = outs[0]
    i = g["i"][0]
    assert (i[2][i[2] >= 0] < N // 2).all() and (i[2] >= 0).all()       # shard 0 holds every allowed row
    assert (i[3] == -1).all()                                            # nothing allowed
    assert sorted(i[4, :4].tolist()) == [1, 2, N - 3, N - 2] and (i[4, 4:] == -1).all()
    for r in range(NQ):
        got = i[r][i[r] >= 0]
        assert ((labels[got] & REQ[r, 0]) == REQ[r, 0]).all() and (REQ[r, 1] == 0 or (labels[got] & REQ[r, 1] != 0).all())


def test_serial_path_filters(tmp_path):
    outs, labels = _run(tmp_path, "serial")
    _common(outs, labels)
    for g in outs:
        # the two short queries (no row / 4 rows) fail the "k rows" check of the merge: ONE exact re-run, with masks
        assert g["n_bad"].tolist() == [2] and int(g["exact_calls"]) == 1
        assert set(g["saw"].tolist()) == {"shard:True", "exact:True"}


def test_two_phase_path_filters_with_rows_set_by_id(tmp_path):
    outs, labels = _run(tmp_path, "two_phase", by_rows=True)
    _common(outs, labels)
    for g in outs:
        assert g["n_bad"].tolist() == [3] and int(g["exact_calls"]) == 1     # + query 2, forced by the merge stand-in
        assert set(g["saw"].tolist()) == {"sample:True", "global:True", "exact:True"}


def test_two_phase_path_filter_plus_exclusions(tmp_path):
    xn, q, labels, ex = _data(True)
    outs, _ = _run(tmp_path, "two_phase", with_excl=True)
    for g in outs:
        for r in range(NQ):
            assert not np.isin(g["i"][0][r][g["i"][0][r] >= 0], ex[r]).any()
        assert set(g["saw"].tolist()) == {"sample:True", "global:True", "exact:True"}


def test_pipelined_schedule_filters(tmp_path):
    outs, labels = _run(tmp_path, "pipelined", with_excl=True)
    for g in outs:
        assert g["n_bad"].tolist()[:2] == [2, 2]          # the two short queries of each masked batch
        assert int(g["exact_calls"]) == 2 + (g["n_bad"][2] > 0)
        saw = g["saw"].tolist()
        assert saw.count("sample:True") == 3 and saw.count("global:True") == 3 and "exact:True" in saw
