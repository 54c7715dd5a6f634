"""Range-search restatement (tt_flat_range_search & co.) for the tests, on top of the filter and exclusion oracles.

faiss's inner-product range_search returns every row whose score is STRICTLY greater than the radius.  Here a query sees
the rows its label masks allow minus its exclusion list (filter_oracle.search_filtered, which composes
exclusion_oracle): its count is the number of those rows scoring > radius, and its list is the best min(count, L) of
them, score descending, id ascending, padded with (-inf, -1).  `check_range` judges a result on fp64 scores: a row within
`tie` of the radius may fall on either side, and ids may differ only inside score ties.
"""
import numpy as np

from filter_oracle import allows, search_filtered


def _allowed(n, labels, req, excl_row):
    ok = np.ones(n, bool) if labels is None else allows(labels, req[0], req[1])
    if excl_row is not None:
        e = np.asarray(excl_row, np.int64)
        ok[e[(e >= 0) & (e < n)]] = False
    return ok


def _masks(nq, require):
    return np.broadcast_to(np.asarray([0, 0] if require is None else require, np.int64) & 0xFFFFFFFF, (nq, 2))


def range_search(xn, qn, radius, L, labels=None, require=None, exclude=None):
    """-> (counts i64 [nq], scores f32 [nq, L], ids i64 [nq, L]) with fp32 scores (qn @ xn.T)."""
    nq, n = qn.shape[0], xn.shape[0]
    rad = np.broadcast_to(np.asarray(radius, np.float32), (nq,))
    req = _masks(nq, require)
    lab = np.zeros(n, np.uint64) if labels is None else labels
    top_s, top_i = search_filtered(xn, qn, min(L, n), lab, req, exclude)
    s32 = qn.astype(np.float32) @ xn.astype(np.float32).T
    counts = np.zeros(nq, np.int64)
    out_s = np.full((nq, L), -np.inf, np.float32)
    out_i = np.full((nq, L), -1, np.int64)
    for r in range(nq):
        ok = _allowed(n, labels, req[r], None if exclude is None else exclude[r])
        counts[r] = int(((s32[r] > rad[r]) & ok).sum())
        keep = np.flatnonzero((top_i[r] >= 0) & (top_s[r] > rad[r]))[:L]
        out_s[r, :keep.size] = top_s[r, keep]
        out_i[r, :keep.size] = top_i[r, keep]
    return counts, out_s, out_i


def check_range(counts, scores, ids, xn, qn, radius, L, labels=None, require=None, exclude=None, score_tol=1e-5,
                tie=1e-6, id_offset=0):
    """(ok, message) for a device result, judged on fp64 scores.  xn / qn: the normalised fp32 rows and queries."""
    counts, scores, ids = np.asarray(counts), np.asarray(scores), np.asarray(ids)
    nq, n = qn.shape[0], xn.shape[0]
    rad = np.broadcast_to(np.asarray(radius, np.float64), (nq,))
    req = _masks(nq, require)
    if scores.shape != (nq, L) or ids.shape != (nq, L) or counts.shape != (nq,):
        return False, f"shapes {counts.shape} {scores.shape} {ids.shape}"
    for r in range(nq):
        ok = _allowed(n, labels, req[r], None if exclude is None else exclude[r])
        s64 = xn.astype(np.float64) @ qn[r].astype(np.float64)
        s64[~ok] = -np.inf
        lo, hi = int((s64 > rad[r] + tie).sum()), int((s64 > rad[r] - tie).sum())
        c = int(counts[r])
        if not lo <= c <= hi:
            return False, f"query {r}: count {c} outside [{lo}, {hi}]"
        m = min(c, L)
        got = ids[r, :m] - id_offset
        if (ids[r, m:] != -1).any() or not np.isneginf(scores[r, m:]).all():
            return False, f"query {r}: the tail after {m} entries is not (-inf, -1)"
        if m == 0:
            continue
        if got.min() < 0 or got.max() >= n or np.unique(got).size != m:
            return False, f"query {r}: ids out of range or repeated"
        if not np.isfinite(s64[got]).all():
            return False, f"query {r}: returned a disallowed or excluded row"
        if (s64[got] <= rad[r] - tie).any():
            return False, f"query {r}: returned a row at or below the radius"
        if np.abs(scores[r, :m] - s64[got]).max() > score_tol:
            return False, f"query {r}: score error {np.abs(scores[r, :m] - s64[got]).max():.3e}"
        if (np.diff(scores[r, :m].astype(np.float64)) > 0).any():
            return False, f"query {r}: scores not sorted descending"
        # nothing better was left out: every row not returned scores at most the last returned one (up to a tie), and
        # with fewer than L returned, no row clearly above the radius was left out
        rest = s64.copy()
        rest[got] = -np.inf
        floor = s64[got].min() if m == L else rad[r]
        if rest.max() > floor + tie:
            return False, f"query {r}: row {int(rest.argmax())} ({rest.max():.7f}) left out above {floor:.7f}"
        # order: positions may swap only inside ties
        if (np.diff(s64[got]) > tie).any():
            return False, f"query {r}: order differs outside a tie"
    return True, "ok"
