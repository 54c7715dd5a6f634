"""CPU: range search (tt_flat_range_search & co.) without a GPU - the range oracle on hand-built cases, the argument
checks of the C-ABI and of the Python surface, and the assembly of faiss's (lims, D, I) layout."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import flat_ip_oracle as fo
from range_oracle import check_range, range_search


def _unit(rows):
    return fo.normalize_rows(np.asarray(rows, np.float32))


def test_strictly_greater_and_ties_at_the_radius():
    xn = _unit([[1, 0], [1, 0], [0, 1], [1, 1], [-1, 0]])
    qn = _unit([[1, 0]])
    c, s, i = range_search(xn, qn, 1.0, 4)          # rows 0 and 1 score exactly 1.0: not above it
    assert c.tolist() == [0] and (i == -1).all() and np.isneginf(s).all()
    c, s, i = range_search(xn, qn, 0.5, 4)          # ties ordered by ascending id
    assert c.tolist() == [3] and i[0].tolist() == [0, 1, 3, -1] and s[0, :2].tolist() == [1.0, 1.0]
    c, s, i = range_search(xn, qn, 0.0, 4)          # row 2 scores exactly 0: not above it
    assert c.tolist() == [3]


def test_count_beyond_L_and_below_minus_one():
    rng = np.random.default_rng(3)
    xn = _unit(rng.standard_normal((500, 8)))
    qn = _unit(rng.standard_normal((4, 8)))
    c, s, i = range_search(xn, qn, 0.0, 10)
    s32 = qn @ xn.T
    assert c.tolist() == (s32 > 0).sum(1).tolist() and (c > 10).all()
    rs, ri = fo.search(xn, qn, 10)
    assert np.array_equal(i, ri) and np.array_equal(s, rs)            # truncated to the best L
    c, s, i = range_search(xn, qn, -1.5, 16)                           # every row qualifies
    assert c.tolist() == [500] * 4 and (i >= 0).all()
    c, s, i = range_search(xn, qn, [2.0, 0.0, 2.0, 0.99], 10)         # nothing above the radius for queries 0 and 2
    assert c[0] == 0 and c[2] == 0 and (i[[0, 2]] == -1).all()
    ok, msg = check_range(c, s, i, xn, qn, [2.0, 0.0, 2.0, 0.99], 10)
    assert ok, msg


def test_labels_and_exclusions_compose():
    rng = np.random.default_rng(5)
    xn = _unit(rng.standard_normal((300, 6)))
    qn = _unit(rng.standard_normal((3, 6)))
    labels = rng.integers(0, 4, 300).astype(np.uint64)
    ex = np.full((3, 5), -1, np.int64)
    top = fo.search(xn, qn, 5)[1]
    ex[:, :3] = top[:, :3]
    ex[1, 3] = 10_000                                                  # ids outside the catalog are ignored
    c, s, i = range_search(xn, qn, 0.1, 400, labels, [1, 0], ex)
    s32 = qn @ xn.T
    for r in range(3):
        ok = (labels & 1) == 1
        ok[ex[r][(ex[r] >= 0) & (ex[r] < 300)]] = False
        assert c[r] == int(((s32[r] > np.float32(0.1)) & ok).sum())
        got = i[r, :c[r]]
        assert ok[got].all() and not np.isin(got, ex[r]).any()
    assert check_range(c, s, i, xn, qn, 0.1, 400, labels, [1, 0], ex)[0]
    # the checker catches a counted excluded row and a missing row
    bad = c.copy()
    bad[0] += 2
    assert not check_range(bad, s, i, xn, qn, 0.1, 400, labels, [1, 0], ex)[0]
    s2, i2 = s.copy(), i.copy()
    i2[0, 0] = ex[0, 0]
    assert not check_range(c, s2, i2, xn, qn, 0.1, 400, labels, [1, 0], ex)[0]


def test_range_arguments_are_checked_without_a_gpu(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    p = ctypes.c_void_p(256)          # never dereferenced: the argument checks come first
    odd = ctypes.c_void_p(260)
    cases = [  # labels, require, L, E, excl, N, workspace, what
        (p, None, 10, 0, None, 1000, p, "both NULL or both non-NULL"),
        (None, p, 10, 0, None, 1000, p, "both NULL or both non-NULL"),
        (odd, p, 10, 0, None, 1000, p, "16-byte aligned"),
        (p, odd, 10, 0, None, 1000, p, "8-byte aligned"),
        (None, None, 0, 0, None, 1000, p, "TT_FLAT_RANGE_MAX_RESULTS"),
        (None, None, 16385, 0, None, 1000, p, "TT_FLAT_RANGE_MAX_RESULTS"),
        (None, None, 10, 1025, p, 1000, p, "TT_FLAT_MAX_EXCLUDE"),
        (None, None, 10, 3, None, 1000, p, "null exclusion"),
        (None, None, 10, 0, None, 1 << 31, p, "2^31"),
        (None, None, 10, 0, None, 1000, None, "null"),
    ]
    for labels, req, L, E, excl, N, ws, what in cases:
        rc = lib.tt_flat_range_search(p, 1, p, p, p, N, 64, p, L, 0, p, p, p, p, p, p, labels, req, excl, E, ws, 1 << 20, None)
        assert rc == 1 and what in _native.last_error(), (what, _native.last_error())
        rc = lib.tt_flat_range_search_exact(p, 1, None, 1, p, N, 64, p, L, 0, p, p, p, labels, req, excl, E, ws, 1 << 20, None)
        assert rc == 1 and what in _native.last_error(), (what, _native.last_error())
    rc = lib.tt_flat_range_search(p, 1, p, odd, p, 1000, 64, p, 10, 0, p, p, p, p, p, p, None, None, None, 0, p, 1 << 20, None)
    assert rc == 1 and "Xh must be 16-byte aligned" in _native.last_error()
    rc = lib.tt_flat_range_search(p, 1, p, p, p, 1000, 64, None, 10, 0, p, p, p, p, p, p, None, None, None, 0, p, 1 << 20, None)
    assert rc == 1 and "null pointer" in _native.last_error()
    # workspace sizing: more candidate budget, more room; unsupported widths size the exact path
    small = lib.tt_flat_range_workspace_bytes(1_000_000, 384, 64, 1024)
    large = lib.tt_flat_range_workspace_bytes(1_000_000, 384, 64, 65536)
    assert 0 < small < large
    assert lib.tt_flat_range_workspace_bytes(1000, 1536, 4, 100) == lib.tt_flat_range_exact_workspace_bytes(1000, 1536, 4, 16384)
    assert lib.tt_flat_range_workspace_bytes(0, 384, 4, 100) == 0


def _cpu_index(n=10, d=4):
    """A FlatIPIndex shell on the host: enough state for the argument checks that run before any device work."""
    from two_tower_model_v2_b200.vector_db import FlatIPIndex
    idx = FlatIPIndex.__new__(FlatIPIndex)
    idx.d, idx.device = d, torch.device("cpu")
    idx.xn = torch.zeros((n, d))
    idx.labels = None
    idx._labels_store = None
    return idx


def test_radius_and_max_results_validation():
    from two_tower_model_v2_b200.vector_db import range_max_results
    idx = _cpu_index()
    q = torch.zeros((3, 4))
    for bad in (float("nan"), float("inf"), -float("inf"), 1e39, np.array([0.1, np.nan, 0.2]), np.zeros(2), np.zeros((3, 1)),
                np.array([True, False, True]), "0.5", None, torch.tensor([0.1, float("inf"), 0.0])):
        with pytest.raises(ValueError):
            idx.range_search_device(q, bad, 10)
    for bad in (0, 16385, -1, 2.0, True, "10", None):
        with pytest.raises(ValueError):
            range_max_results(bad)
        with pytest.raises(ValueError):
            idx.range_search_device(q, 0.5, bad)
    assert range_max_results(1) == 1 and range_max_results(np.int64(16384)) == 16384
    assert idx._radii(0.25, 3).tolist() == [0.25] * 3
    assert idx._radii(np.array([1, 2, 3], np.int64), 3).tolist() == [1.0, 2.0, 3.0]
    with pytest.raises(ValueError, match="expected queries"):
        idx.range_search_device(torch.zeros((3, 5)), 0.5, 10)
    with pytest.raises(ValueError, match="set_labels"):
        idx.range_search_device(q, 0.5, 10, require=np.array([1, 0]))


def test_csr_assembly_from_padded_results():
    from two_tower_model_v2_b200.vector_db import range_csr
    counts = np.array([0, 2, 5, 3])
    s = np.array([[-np.inf] * 3, [0.9, 0.8, -np.inf], [0.7, 0.6, 0.5], [1.0, 0.9, 0.1]], np.float32)
    i = np.array([[-1] * 3, [4, 2, -1], [7, 8, 9], [1, 3, 0]], np.int64)
    lims, D, I = range_csr(counts, s, i)
    assert lims.tolist() == [0, 0, 2, 5, 8] and lims.dtype == np.int64
    assert I.tolist() == [4, 2, 7, 8, 9, 1, 3, 0] and D.dtype == np.float32 and I.dtype == np.int64
    assert D.tolist() == pytest.approx([0.9, 0.8, 0.7, 0.6, 0.5, 1.0, 0.9, 0.1])
    lims, D, I = range_csr(np.zeros(0, np.int64), np.zeros((0, 4), np.float32), np.zeros((0, 4), np.int64))
    assert lims.tolist() == [0] and D.size == 0 and I.size == 0


def test_rerun_groups_fit_the_budget():
    from two_tower_model_v2_b200.vector_db import range_rerun_groups
    need = np.array([5, 100, 7, 3, 2000, 50])
    ws = lambda n, need_max: n * need_max * 10 * 8
    groups = range_rerun_groups(np.array([0, 1, 2, 4, 5]), need, ws, 10_000)
    assert [g.tolist() for g in groups] == [[0, 2], [5], [1], [4]]   # ascending need; 2000 x 10 x 8 alone exceeds
    assert all(ws(len(g), int(need[g].max())) <= 10_000 for g in groups[:-1])
    assert range_rerun_groups(np.zeros(0, np.int64), need, ws, 10_000) == []


def test_rerun_segments_hold_the_fullest_first_pass_segment(native_lib):
    """A re-run plans for its own (smaller) number of queries, which often slices the catalog more finely than the first
    pass did (10M rows: 9 slices at nq 4096, 148 for up to 128 queries): its segments must still hold need candidates,
    and the first pass's whole per-query total spread over the re-run's slices."""
    from two_tower_model_v2_b200.vector_db import _plan_slices
    idx = _cpu_index(n=10_000_000, d=384)
    idx.xn = torch.empty((10_000_000, 0))          # only the row count is read
    idx.d = 384
    for nq_first in (4096, 1024, 512, 200, 1):
        s_first = _plan_slices(10_000_000, 384, nq_first)
        for n in (1, 4, 64, 300):
            if n > nq_first:
                continue
            s_new = _plan_slices(10_000_000, 384, n)
            for need in (300, 5000):
                seg = 2 * idx._rerun_budget(n, need, s_first) / s_new     # the segment make_range_plan sizes
                assert seg >= 2 * need and seg >= 2 * need * s_first / s_new, (nq_first, n, need, s_first, s_new)
    assert _plan_slices(10_000_000, 384, 4096) < _plan_slices(10_000_000, 384, 1)
