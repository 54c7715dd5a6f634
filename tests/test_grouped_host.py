"""CPU: the group-cap oracle, argument validation of max_per_group and group keys, VectorDatabase's key mapping and the
C-ABI argument errors of tt_flat_search_grouped / tt_flat_search_exact_grouped (no GPU needed)."""
import numpy as np
import pytest

from group_oracle import per_group_top_m, walk


def tie_heavy_order(rng, nq, n, n_groups, allowed_frac):
    """Random orderings with many tied scores (ties broken by id), part of the rows not allowed (-1 tail)."""
    s = np.full((nq, n), -np.inf, np.float32)
    i = np.full((nq, n), -1, np.int64)
    for r in range(nq):
        rows = np.flatnonzero(rng.random(n) < allowed_frac)
        sc = rng.integers(0, 6, rows.size).astype(np.float32)
        o = np.lexsort((rows, -sc))
        s[r, :rows.size], i[r, :rows.size] = sc[o], rows[o]
    groups = rng.integers(-2, n_groups, n)
    groups[rng.random(n) < 0.1] = n_groups + 5        # ids out of range are ungrouped too
    return s, i, groups


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("m,k", [(1, 1), (1, 10), (2, 7), (3, 50), (64, 20)])
def test_oracle_restatements_agree(seed, m, k):
    rng = np.random.default_rng(seed)
    s, i, groups = tie_heavy_order(rng, 4, 300, [1, 3, 40][seed % 3], 0.7)
    groups = np.where(groups >= [1, 3, 40][seed % 3], -1, groups)
    a = walk(s, i, groups, m, k)
    b = per_group_top_m(s, i, groups, m, k)
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])


def test_walk_identity_cases():
    rng = np.random.default_rng(7)
    s, i, _ = tie_heavy_order(rng, 3, 200, 5, 0.8)
    k = 30
    plain = (s[:, :k], i[:, :k])
    for groups, m in ((np.arange(200), 1), (np.full(200, -1), 1), (rng.integers(0, 3, 200), k)):
        gs, gi = walk(s, i, groups, m, k)
        assert np.array_equal(gi, plain[1]) and np.array_equal(gs, plain[0])


def test_walk_pads_when_groups_run_out():
    s = np.array([[5, 4, 3, 2, 1]], np.float32)
    i = np.array([[0, 1, 2, 3, 4]], np.int64)
    gs, gi = walk(s, i, np.array([0, 0, 0, 1, 1]), 1, 4)
    assert gi.tolist() == [[0, 3, -1, -1]] and np.isneginf(gs[0, 2:]).all()


def bare_index(n=3, d=4):
    """A FlatIPIndex shell with n CPU rows, enough for the host-side validation (no device work)."""
    import torch
    from two_tower_model_v2_b200.vector_db import FlatIPIndex
    idx = FlatIPIndex.__new__(FlatIPIndex)
    idx.d = d
    idx.xn = idx._xn_store = torch.zeros((n, d))
    idx.groups = None
    idx.n_groups = 0
    idx._group_keys_store = idx._groups_store = None
    return idx


@pytest.mark.parametrize("bad", [0, 65, -1, 2.0, True, "3", np.float32(2)])
def test_max_per_group_validation(bad):
    import torch
    idx = bare_index()
    idx.groups = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(ValueError):
        idx._group_cap(bad)


def test_max_per_group_accepts_range_and_needs_groups():
    import torch
    idx = bare_index()
    assert idx._group_cap(None) is None
    with pytest.raises(ValueError, match="set_groups"):
        idx._group_cap(2)
    idx.groups = torch.zeros(3, dtype=torch.int32)
    assert idx._group_cap(1) == 1 and idx._group_cap(np.int64(64)) == 64


@pytest.mark.parametrize("keys,rows", [(np.array([1.5, 2.0, 3.0]), None), (np.array([True, False, True]), None),
                                       (np.array([1, 2]), None), (np.array([[1, 2, 3]]), None),
                                       (np.array([1, 2]), np.array([0])), (np.array([1]), np.array([3])),
                                       (np.array([1]), np.array([-1])), (np.array([1]), np.array([0.0]))])
def test_group_key_validation(keys, rows):
    idx = bare_index()
    with pytest.raises(ValueError):
        idx.set_groups(keys, rows=rows)


class _RecordingIndex:
    def __init__(self):
        self.calls = []

    def set_groups(self, keys, rows=None):
        self.calls.append((np.asarray(keys).copy(), None if rows is None else np.asarray(rows).copy()))


def make_db(pids):
    from two_tower_model_v2_b200.vector_db import VectorDatabase
    db = VectorDatabase(4)
    db.index = _RecordingIndex()
    db.product_ids = list(pids)
    db.id_to_index = {p: r for r, p in enumerate(pids)}
    return db


def test_database_maps_group_values_to_keys():
    db = make_db(["a", "b", "c", "d", "e"])
    db.set_groups(["acme", None, "zeta", "acme", 17])
    keys, rows = db.index.calls[-1]
    assert rows is None and keys.dtype == np.int64
    assert keys[1] == -1 and keys[0] == keys[3] and len({keys[0], keys[2], keys[4]}) == 3 and (keys[[0, 2, 4]] >= 0).all()
    db.set_groups(["zeta", None], product_ids=["e", "a"])      # the same value keeps its key across calls
    keys2, rows2 = db.index.calls[-1]
    assert rows2.tolist() == [4, 0] and keys2[0] == keys[2] and keys2[1] == -1


def test_database_unknown_product_changes_nothing():
    db = make_db(["a", "b"])
    with pytest.raises(ValueError, match="unknown"):
        db.set_groups(["x", "y"], product_ids=["a", "nope"])
    with pytest.raises(ValueError):
        db.set_groups(["x"], product_ids=["a", "b"])
    assert db.index.calls == []


def test_c_abi_argument_errors(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    buf = np.zeros(4, np.int32)
    grp = buf.ctypes.data
    common = (None, 1, None, None, None, 4, 8, 1, 0, None, None, None, None)

    def grouped(groups, n_groups, m, labels=None, require=None):
        return lib.tt_flat_search_grouped(*common, groups, n_groups, m, labels, require, None, 0, None, 0, None)

    def exact(groups, n_groups, m, labels=None, require=None):
        return lib.tt_flat_search_exact_grouped(None, 1, None, 1, None, 4, 8, 1, 0, None, None, labels, require, None, 0,
                                                groups, n_groups, m, None, 0, None)

    for call in (grouped, exact):
        assert call(None, 1, 1) == 1 and "null groups" in _native.last_error()
        assert call(grp, 1, 0) == 1 and "max_per_group" in _native.last_error()
        assert call(grp, 1, _native.TT_FLAT_MAX_PER_GROUP + 1) == 1 and "max_per_group" in _native.last_error()
        assert call(grp, -1, 1) == 1 and "n_groups" in _native.last_error()
        assert call(grp, 1, 1, labels=grp) == 1 and "both NULL" in _native.last_error()


def test_workspace_sizes(native_lib):
    lib = native_lib
    # tensor-core plan: the exclusion search's workspace; exact route (D > 1024): the exact path's plus the group state
    assert lib.tt_flat_search_grouped_workspace_bytes(1_000_000, 384, 128, 100, 0, 5000) == \
        lib.tt_flat_search_excl_workspace_bytes(1_000_000, 384, 128, 100, 0)
    assert lib.tt_flat_search_grouped_workspace_bytes(100_000, 1536, 4, 10, 3, 5000) == \
        lib.tt_flat_search_exact_grouped_workspace_bytes(100_000, 1536, 4, 10, 5000)
    base = lib.tt_flat_search_exact_workspace_bytes(100_000, 384, 8, 10)
    assert lib.tt_flat_search_exact_grouped_workspace_bytes(100_000, 384, 8, 10, 0) == base
    assert lib.tt_flat_search_exact_grouped_workspace_bytes(100_000, 384, 8, 10, 5000) >= base + 8 * 5000 * 16
    assert lib.tt_flat_search_grouped_workspace_bytes(100_000, 384, 4, 10, 0, -1) == 0
