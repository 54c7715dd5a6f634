"""CPU: label filters (tt_flat_search_filtered & co.) without a GPU - the masked reference search, the mask semantics,
and the argument checks of the C-ABI and of the Python surfaces."""
import ctypes

import numpy as np
import pytest
import torch

from exclusion_oracle import search_excluding
from filter_oracle import allows, search_filtered
from oracle import flat_ip_oracle as fo


def test_mask_semantics():
    lab = np.array([0, 1, 2, 3, 0xFFFFFFFF, 0x80000000, 0x80000001, 6], np.uint64)
    assert allows(lab, 0, 0).all()                                   # (0, 0) allows every row, label 0 included
    assert allows(lab, 1, 0).tolist() == [False, True, False, True, True, False, True, False]
    assert allows(lab, 0, 6).tolist() == [False, False, True, True, True, False, False, True]
    assert allows(lab, 3, 0).tolist() == [False, False, False, True, True, False, False, False]
    assert allows(lab, 1, 6).tolist() == [False, False, False, True, True, False, False, False]
    assert allows(lab, 0xFFFFFFFF, 0).tolist() == [False, False, False, False, True, False, False, False]
    assert allows(lab, 0, 0xFFFFFFFF).tolist() == [False, True, True, True, True, True, True, True]
    assert allows(lab, 0x80000000, 1).tolist() == [False, False, False, False, True, False, True, False]


def _brute_force(xn, qn, k, labels, req, exclude=None):
    s = qn.astype(np.float32) @ xn.astype(np.float32).T
    out_s = np.full((qn.shape[0], k), -np.inf, np.float32)
    out_i = np.full((qn.shape[0], k), -1, np.int64)
    for r in range(qn.shape[0]):
        ok = allows(labels, req[r][0], req[r][1])
        if exclude is not None:
            ok[exclude[r][(exclude[r] >= 0) & (exclude[r] < xn.shape[0])]] = False
        rows = np.flatnonzero(ok)
        order = rows[np.lexsort((rows, -s[r, rows]))][:k]
        out_s[r, :len(order)], out_i[r, :len(order)] = s[r, order], order
    return out_s, out_i


def test_masked_search_equals_brute_force():
    rng = np.random.default_rng(8)
    N, D, nq, k = 900, 16, 9, 12
    xn = fo.normalize_rows(rng.standard_normal((N, D)).astype(np.float32))
    qn = fo.normalize_rows(rng.standard_normal((nq, D)).astype(np.float32))
    labels = rng.integers(0, 1 << 32, N, dtype=np.uint64)
    labels[:50] = 0
    req = np.array([[0, 0], [1, 0], [0, 6], [3, 12], [0xFFFFFFFF, 0], [1 << 31, 0], [5, 0], [0, 1], [2, 2]], np.int64)
    rare = np.zeros(N, np.uint64)
    rare[[3, 10, 700]] = 1 << 20                    # 3 allowed rows < k for query 5's mask on this label set
    for lab, r in ((labels, req), (rare | labels & ~np.uint64(1 << 20), np.array([[1 << 20, 0]] * nq))):
        got = search_filtered(xn, qn, k, lab, r)
        want = _brute_force(xn, qn, k, lab, r)
        assert np.array_equal(got[1], want[1]) and np.allclose(got[0], want[0], atol=1e-6)
    got = search_filtered(xn, qn, k, rare | labels & ~np.uint64(1 << 20), [1 << 20, 0])
    assert sorted(got[1][0, :3].tolist()) == [3, 10, 700] and (got[1][:, 3:] == -1).all() and np.isneginf(got[0][:, 3:]).all()
    # (0, 0) is the plain oracle; a mask nothing satisfies pads everything
    s, i = search_filtered(xn, qn, k, labels, [0, 0])
    rs, ri = fo.search(xn, qn, k)
    assert np.array_equal(i, ri) and np.array_equal(s, rs)
    s, i = search_filtered(xn, qn, k, np.zeros(N, np.uint64), [1, 0])
    assert (i == -1).all() and np.isneginf(s).all()
    # composed with exclusion lists: allowed and not listed
    top = fo.search(xn, qn, 40)[1]
    ex = np.full((nq, 30), -1, np.int64)
    ex[:, :20] = top[:, :20]
    ex[1, 20:23] = [N + 5, -3, top[1, 0]]
    got = search_filtered(xn, qn, k, labels, req, ex)
    want = _brute_force(xn, qn, k, labels, req, ex)
    assert np.array_equal(got[1], want[1]) and np.allclose(got[0], want[0], atol=1e-6)
    s, i = search_filtered(xn, qn, k, labels, [0, 0], ex)
    rs, ri = search_excluding(xn, qn, k, ex)
    assert np.array_equal(i, ri)


def test_filter_arguments_are_checked_without_a_gpu(native_lib):
    from two_tower_model_v2_b200 import _native
    lib = native_lib
    p = ctypes.c_void_p(256)          # never dereferenced: the argument checks come first
    odd = ctypes.c_void_p(260)
    for labels, req, E, excl, what in [(None, p, 0, None, "null labels or require"), (p, None, 0, None, "null labels or require"),
                                       (odd, p, 0, None, "16-byte aligned"), (p, ctypes.c_void_p(260), 0, None, "8-byte aligned"),
                                       (p, p, 1025, p, "TT_FLAT_MAX_EXCLUDE"), (p, p, 3, None, "null exclusion")]:
        rc = lib.tt_flat_search_filtered(p, 1, p, p, p, 1000, 64, 10, 0, p, p, p, p, labels, req, excl, E, p, 1 << 20, None)
        assert rc == 1 and what in _native.last_error(), _native.last_error()
        if "aligned" not in what:
            rc = lib.tt_flat_search_exact_filtered(p, 1, None, 1, p, 1000, 64, 10, 0, p, p, labels, req, excl, E, p, 1 << 20, None)
            assert rc == 1 and what in _native.last_error(), _native.last_error()


def test_label_and_mask_validation():
    from two_tower_model_v2_b200.vector_db import require_masks, u32_words
    w = u32_words(np.array([0, 1, 0xFFFFFFFF], np.int64), "labels")
    assert w.dtype == np.int32 and w.view(np.uint32).tolist() == [0, 1, 0xFFFFFFFF]
    assert u32_words(np.array([5], np.uint32), "labels").tolist() == [5]
    for bad in (np.array([-1]), np.array([1 << 32]), np.array([0.5]), np.array([True])):
        with pytest.raises(ValueError):
            u32_words(bad, "labels")
    assert require_masks(0, 0, 4) is None
    assert require_masks([0, 0, 0], 0, 3) is None
    m = require_masks(1, [0, 2, 0xFFFFFFFF], 3)
    assert m.shape == (3, 2) and m.view(np.uint32).tolist() == [[1, 0], [1, 2], [1, 0xFFFFFFFF]]
    with pytest.raises(ValueError):
        require_masks([1, 2], 0, 3)
    with pytest.raises(ValueError):
        require_masks(-1, 0, 1)
    with pytest.raises(ValueError):
        require_masks(0, 1 << 32, 1)


def _cpu_index(n=10, d=4):
    """A FlatIPIndex shell on the host: enough state for the argument checks that run before any device work."""
    from two_tower_model_v2_b200.vector_db import FlatIPIndex
    idx = FlatIPIndex.__new__(FlatIPIndex)
    idx.d, idx.device = d, torch.device("cpu")
    idx.xn = torch.zeros((n, d))
    idx.labels = None
    idx._labels_store = None
    return idx


def test_filter_on_an_unlabelled_index_and_bad_shapes_are_rejected():
    idx = _cpu_index()
    q = torch.zeros((3, 4))
    with pytest.raises(ValueError, match="set_labels"):
        idx.search_device(q, 2, require=np.array([1, 0]))
    for bad in (np.zeros((3, 3), np.int64), np.zeros((2, 2), np.int64) + 1, np.array([1, 2, 3]), np.array([[-1, 0]] * 3)):
        with pytest.raises(ValueError):
            idx._requires(bad, 3)
    assert idx._requires(np.zeros((3, 2), np.int64), 3) is None        # (0, 0) everywhere: the plain search
    assert idx._requires(None, 3) is None
    for labels, rows in ((np.zeros(9, np.int64), None), (np.zeros(2, np.int64), np.array([0])),
                         (np.array([1 << 32] * 10), None), (np.zeros(1, np.int64), np.array([10])),
                         (np.zeros(1, np.int64), np.array([0.0]))):
        with pytest.raises(ValueError):
            idx.set_labels(labels, rows)


def test_set_labels_by_unknown_product_id_changes_nothing():
    from two_tower_model_v2_b200 import VectorDatabase

    class _Recorder:
        ntotal = 3

        def __init__(self):
            self.calls = []

        def set_labels(self, labels, rows=None):
            self.calls.append((np.asarray(labels).tolist(), None if rows is None else rows.tolist()))

    db = VectorDatabase(4)
    with pytest.raises(ValueError, match="Index not built"):
        db.set_labels([1, 2, 3])
    db.index = _Recorder()
    db.product_ids = ["a", "b", "c"]
    db.id_to_index = {"a": 0, "b": 1, "c": 2}
    with pytest.raises(ValueError, match="unknown product ids"):
        db.set_labels([1, 2], ["a", "nope"])
    assert db.index.calls == []
    db.set_labels([7, 9], ["c", "a"])
    db.set_labels([1, 2, 3])
    assert db.index.calls == [([7, 9], [2, 0]), ([1, 2, 3], None)]
