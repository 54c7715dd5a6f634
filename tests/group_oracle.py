"""Group-cap restatements of the exact search, for the tests of tt_flat_search_grouped & co.

Built on the unchanged IndexFlatIP oracle (oracle/flat_ip_oracle.py) and on the exclusion and filter oracles: they
give the full (score desc, id asc) ordering of the rows a query may return, and the cap is applied to it twice,
independently:
  - `walk`: the contract as written, one row at a time: take a row if it is ungrouped or fewer than m rows of its group
    were taken before it, stop after k takes;
  - `per_group_top_m`: keep each group's first m rows (and every ungrouped row), then the first k of what is kept.
Both give (scores f32 [nq, k'], ids i64 [nq, k']), k' = min(k, N), (-inf, -1) padded.
"""
import numpy as np

from exclusion_oracle import search_excluding
from filter_oracle import search_filtered
from oracle import flat_ip_oracle as fo


def allowed_order(xn, qn, labels=None, require=None, exclude=None):
    """Every allowed, not excluded row of each query in (fp32 score desc, id asc) order: (scores, ids) [nq, N], with a
    (-inf, -1) tail after the allowed rows."""
    n = xn.shape[0]
    if labels is not None:
        return search_filtered(xn, qn, n, labels, require, exclude)
    if exclude is not None:
        return search_excluding(xn, qn, n, exclude)
    return fo.search(xn, qn, n)


def group_of(groups, ids):
    """Group of each id (-1 = ungrouped, and for the padding id -1)."""
    g = np.asarray(groups, np.int64)
    out = np.where(ids >= 0, g[np.maximum(ids, 0)], -1)
    return np.where(out >= 0, out, -1)


def walk(order_s, order_i, groups, m, k):
    """The contract's walk over full orderings -> (scores [nq, k], ids [nq, k])."""
    nq = order_i.shape[0]
    out_s = np.full((nq, k), -np.inf, np.float32)
    out_i = np.full((nq, k), -1, np.int64)
    for r in range(nq):
        taken, used = 0, {}
        for s, i, g in zip(order_s[r], order_i[r], group_of(groups, order_i[r])):
            if taken == k or i < 0:
                break
            if g >= 0:
                if used.get(g, 0) >= m:
                    continue
                used[g] = used.get(g, 0) + 1
            out_s[r, taken], out_i[r, taken] = s, i
            taken += 1
    return out_s, out_i


def per_group_top_m(order_s, order_i, groups, m, k):
    """The top-k of the rows that rank among the first m of their own group -> (scores [nq, k], ids [nq, k])."""
    nq, n = order_i.shape
    out_s = np.full((nq, k), -np.inf, np.float32)
    out_i = np.full((nq, k), -1, np.int64)
    for r in range(nq):
        valid = order_i[r] >= 0
        g = group_of(groups, order_i[r])
        pos = np.arange(n)
        by_group = np.lexsort((pos, g))          # grouped by id, each group in walk order
        gs = g[by_group]
        start = np.r_[0, np.flatnonzero(np.diff(gs)) + 1]
        rank = np.empty(n, np.int64)
        rank[by_group] = pos - np.repeat(start, np.diff(np.r_[start, n]))
        keep = np.flatnonzero(valid & ((g < 0) | (rank < m)))[:k]
        out_s[r, :keep.size] = order_s[r, keep]
        out_i[r, :keep.size] = order_i[r, keep]
    return out_s, out_i


def grouped_search(xn, qn, k, groups, m, labels=None, require=None, exclude=None):
    """The exact grouped top-k of already-normalised operands (the walk; k clamped to N)."""
    k = min(k, xn.shape[0])
    s, i = allowed_order(xn, qn, labels, require, exclude)
    return walk(s, i, groups, m, k)
