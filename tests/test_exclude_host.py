"""CPU: exclusion lists (tt_flat_search_excl & co.) without a GPU - the masked reference search, the argument checks
of the C-ABI, and the sharded plumbing (world size 2, gloo) with oracle stand-ins for the local searches."""
import ctypes
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from exclusion_oracle import search_excluding
from oracle import flat_ip_oracle as fo


def _brute_force(xn, qn, k, exclude):
    s = qn.astype(np.float32) @ xn.astype(np.float32).T
    out_s = np.full((qn.shape[0], k), -np.inf, np.float32)
    out_i = np.full((qn.shape[0], k), -1, np.int64)
    for r in range(qn.shape[0]):
        allowed = np.setdiff1d(np.arange(xn.shape[0]), exclude[r])
        order = allowed[np.lexsort((allowed, -s[r, allowed]))][:k]
        out_s[r, :len(order)], out_i[r, :len(order)] = s[r, order], order
    return out_s, out_i


def test_masked_search_equals_brute_force():
    rng = np.random.default_rng(5)
    N, D, nq, k = 700, 16, 7, 12
    xn = fo.normalize_rows(rng.standard_normal((N, D)).astype(np.float32))
    qn = fo.normalize_rows(rng.standard_normal((nq, D)).astype(np.float32))
    top = fo.search(xn, qn, 40)[1]
    ex = np.full((nq, 60), -1, np.int64)
    ex[0, :30] = top[0, :30]                                  # the query's own best rows
    ex[1, :5] = [top[1, 0], top[1, 0], 5000, -7, top[1, 3]]   # duplicates, out of range, below 0
    ex[2, :] = rng.integers(0, N, 60)                         # random rows
    ex[3, :40] = top[3, :40]
    ex6 = np.concatenate([ex, np.full((nq, N), -1, np.int64)], 1)
    ex6[6, :N - 5] = np.arange(5, N)                          # 5 allowed rows < k
    for exclude in (ex, ex6):
        got = search_excluding(xn, qn, k, exclude, block=256)
        want = _brute_force(xn, qn, k, exclude)
        assert np.array_equal(got[1], want[1])
        assert np.allclose(got[0], want[0], atol=1e-6)
    got = search_excluding(xn, qn, k, ex6)
    assert got[1][6, :5].tolist() == fo.search(xn[:5], qn[6:7], 5)[1][0].tolist()
    assert (got[1][6, 5:] == -1).all() and np.isneginf(got[0][6, 5:]).all()
    # no list: the plain oracle
    s, i = search_excluding(xn, qn, k, np.full((nq, 0), -1, np.int64))
    rs, ri = fo.search(xn, qn, k)
    assert np.array_equal(i, ri) and np.array_equal(s, rs)


def test_exclusion_arguments_are_checked_without_a_gpu(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    p = ctypes.c_void_p(256)          # never dereferenced: the argument checks come first
    for E, excl, what in [(1025, p, "TT_FLAT_MAX_EXCLUDE"), (-1, p, "TT_FLAT_MAX_EXCLUDE"), (3, None, "null exclusion")]:
        rc = lib.tt_flat_search_excl(p, 1, p, p, p, 1000, 64, 10, 0, p, p, p, p, excl, E, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error()
        rc = lib.tt_flat_search_shard_excl(p, 1, p, p, p, 1000, 64, 10, 0, p, p, p, p, p, excl, E, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error()
        rc = lib.tt_flat_shard_search_excl(1, p, p, 1000, 2000, 64, 10, 0, p, 2, p, p, p, p, p, excl, E, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error()
        rc = lib.tt_flat_search_exact_excl(p, 1, None, 1, p, 1000, 64, 10, 0, p, p, excl, E, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error()
    assert lib.tt_flat_search_excl_workspace_bytes(1_000_000, 384, 16, 10, 1025) == 0
    # E = 0 sizes the plain search; E > 0 plans the scan for K_plan = min(K + E, N, TT_FLAT_MAX_K)
    assert lib.tt_flat_search_excl_workspace_bytes(1_000_000, 384, 16, 10, 0) == lib.tt_flat_search_workspace_bytes(1_000_000, 384, 16, 10)
    assert lib.tt_flat_search_excl_workspace_bytes(1_000_000, 384, 16, 10, 100) == lib.tt_flat_search_workspace_bytes(1_000_000, 384, 16, 110)
    assert lib.tt_flat_search_excl_workspace_bytes(500, 64, 4, 10, 1000) == lib.tt_flat_search_workspace_bytes(500, 64, 4, 500)
    assert _native.plan_k(100, 50, 10_000_000) == 150 and _native.plan_k(2000, 1000, 10**7) == _native.TT_FLAT_MAX_K
    assert _native.plan_k(10, 1000, 300) == 300


# ---- sharded plumbing, world size 2 ------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class _ExclOracleIndex:
    """Stands in for FlatIPIndex on a CPU rank: search_shard_into / search_exact_into with exclusion lists of
    GLOBAL ids.  A shard with fewer than k allowed rows pads with (-inf, -1) and flags -2, as the kernel does."""

    def __init__(self, xn_shard, id_offset):
        self.xn, self.id_offset = xn_shard, id_offset
        self.exact_calls, self.saw_exclude = 0, []

    @property
    def ntotal(self):
        return self.xn.shape[0]

    def _search(self, q, k, exclude):
        s, i = fo.search(self.xn, fo.normalize_rows(q.numpy()), min(k + exclude.shape[1], self.ntotal))
        from exclusion_oracle import filter_topk
        return filter_topk(s, i + self.id_offset, exclude.numpy(), k)

    def search_shard_into(self, q, k, scores, ids, bound, flags, *, exclude):
        self.saw_exclude.append("shard")
        s, i = self._search(q, k, exclude)
        scores[:, :k] = torch.from_numpy(s)
        ids[:, :k] = torch.from_numpy(i)
        bound.fill_(float("-inf"))
        flags.copy_(torch.from_numpy(np.where((i < 0).any(1), -2, 1).astype(np.int32)))

    def search_exact_into(self, q, k, scores, ids, qsel, *, exclude):
        self.exact_calls += 1
        rows = qsel.long()
        s, i = self._search(q[rows], k, exclude[rows])
        scores[rows, :k] = torch.from_numpy(s)
        ids[rows, :k] = torch.from_numpy(i)


class _ExclGlobalThresholdIndex(_ExclOracleIndex):
    """Adds the two-phase contract; records the K the plan checks were asked about."""

    def __init__(self, xn_shard, id_offset, rank, world):
        super().__init__(xn_shard, id_offset)
        self.rank, self.world, self.q, self.plan_ks = rank, world, None, []

    def shard_plan_ok(self, n_total, nq, k, n_local_min):
        self.plan_ks.append(k)
        return n_local_min >= k

    def shard_sample(self, q, k, n_total, topr, slot=0, *, exclude):
        self.q = q
        topr.fill_(float(self.rank))

    def shard_search_into(self, nq, k, n_total, topr_g, scores, ids, bound, flags, slot=0, *, exclude):
        assert [float(topr_g[g, 0, 0]) for g in range(self.world)] == [float(g) for g in range(self.world)]
        self.search_shard_into(self.q, k, scores, ids, bound, flags, exclude=exclude)
        self.saw_exclude[-1] = "global"


def _data(N, D, nq, k):
    rng = np.random.default_rng(0)                      # same catalog, queries and lists on every rank
    xn = fo.normalize_rows(rng.standard_normal((N, D)).astype(np.float32))
    q = rng.standard_normal((nq, D)).astype(np.float32)
    top = fo.search(xn, fo.normalize_rows(q), 2 * k)[1]
    E = 24
    ex = np.full((nq, E), -1, np.int64)
    for r in range(nq):
        ex[r, :k] = top[r, :k]                          # the query's own top k: rows of both shards
    ex[0, k:k + 4] = [0, N - 1, 10 * N, ex[0, 0]]       # first / last row, out of range, a duplicate
    ex[1, :] = -1                                       # nothing to exclude for this query
    return xn, q, ex


def _worker(rank, world, port, N, D, nq, k, out_dir, two_phase, short_query):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import two_tower_model_v2_b200 as pkg
    from test_sharded_gloo import _FlagOnceMerge, _merge_oracle
    xn, q, ex = _data(N, D, nq, k)
    if short_query:                                     # query 3 keeps 4 rows, 2 on each shard: fewer than k
        keep = [1, 2, N - 3, N - 2]
        ex = np.concatenate([ex, np.full((nq, N - 4), -1, np.int64)], 1)
        ex[3, :] = -1
        ex[3, :N - 4] = np.setdiff1d(np.arange(N), keep)
    lo, hi = pkg.shard_bounds(N, world, rank)
    local = _ExclGlobalThresholdIndex(xn[lo:hi], lo, rank, world) if two_phase else _ExclOracleIndex(xn[lo:hi], lo)
    sharded = pkg.ShardedFlatIPIndex(local, N, merge=_FlagOnceMerge() if two_phase else _merge_oracle)
    s, i, n_bad = sharded.search_device(torch.from_numpy(q), k, exclude=torch.from_numpy(ex))
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), s=s.numpy(), i=i.numpy(), n_bad=n_bad, exact_calls=local.exact_calls,
             paths=np.array(local.saw_exclude), plan_ks=np.array(getattr(local, "plan_ks", []), np.int64), ex=ex)
    dist.destroy_process_group()


def _expect(tmp_path, N, D, nq, k, world):
    xn, q, _ = _data(N, D, nq, k)
    ex = np.load(tmp_path / "r0.npz")["ex"]
    rs, ri = search_excluding(xn, fo.normalize_rows(q), k, ex)
    outs = [np.load(tmp_path / f"r{r}.npz") for r in range(world)]
    for g in outs:
        assert np.array_equal(g["i"], ri)
        assert np.allclose(g["s"], rs, atol=1e-6) and np.array_equal(np.isneginf(g["s"]), np.isneginf(rs))
        for r in range(nq):                              # no listed id anywhere in the result
            assert not np.isin(g["i"][r][g["i"][r] >= 0], ex[r]).any()
    return outs, ri


def test_sharded_serial_path_with_exclusions(tmp_path):
    N, D, nq, k, world = 801, 16, 6, 10, 2
    mp.spawn(_worker, args=(world, _free_port(), N, D, nq, k, str(tmp_path), False, True), nprocs=world, join=True)
    outs, ri = _expect(tmp_path, N, D, nq, k, world)
    assert ri[3, :4].tolist() != [-1] * 4 and (ri[3, 4:] == -1).all()
    for g in outs:
        # the short query fails the "k rows" check of the merge and is re-run exactly once, with its list
        assert int(g["n_bad"]) == 1 and int(g["exact_calls"]) == 1
        assert set(g["paths"].tolist()) == {"shard"}


def test_sharded_two_phase_path_with_exclusions(tmp_path):
    N, D, nq, k, world = 800, 16, 6, 10, 2
    mp.spawn(_worker, args=(world, _free_port(), N, D, nq, k, str(tmp_path), True, False), nprocs=world, join=True)
    outs, _ = _expect(tmp_path, N, D, nq, k, world)
    for g in outs:
        assert int(g["n_bad"]) == 1 and int(g["exact_calls"]) == 1      # query 2, forced by the merge stand-in
        assert set(g["paths"].tolist()) == {"global"}
        assert set(g["plan_ks"].tolist()) == {k + 24}                    # planned for K_plan = k + E
