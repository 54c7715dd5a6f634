"""Label-filter restatements of the exact search, for the tests of tt_flat_search_filtered & co.

Built on the unchanged IndexFlatIP oracle (oracle/flat_ip_oracle.py) and the exclusion oracle: a query sees only the
rows its masks allow, so the masked result is the oracle's search over that subset of rows, with the subset's
positions mapped back to row ids (score descending, id ascending, (-inf, -1) padded when fewer than k rows are
allowed).  Queries with the same masks share one search.
"""
import numpy as np

from exclusion_oracle import search_excluding

U32 = np.uint32


def allows(labels, require_all, require_any):
    """Row r is allowed iff (labels[r] & all) == all and (any == 0 or (labels[r] & any) != 0).  u32 semantics."""
    lab = np.asarray(labels).astype(np.uint64) & 0xFFFFFFFF
    a, y = int(require_all) & 0xFFFFFFFF, int(require_any) & 0xFFFFFFFF
    ok = (lab & a) == a
    if y:
        ok &= (lab & y) != 0
    return ok


def search_filtered(xn, qn, k, labels, require, exclude=None):
    """fo.search over the rows query i's masks require[i] = (all, any) allow, minus its exclusion list (ids < 0 or
    outside the catalog are ignored) -> (scores f32 [nq, k'], ids i64 [nq, k']), k' = min(k, N)."""
    nq, n = qn.shape[0], xn.shape[0]
    k = min(k, n)
    req = np.broadcast_to(np.asarray(require, dtype=np.int64) & 0xFFFFFFFF, (nq, 2))
    ex = None if exclude is None else np.asarray(exclude, dtype=np.int64).reshape(nq, -1)
    out_s = np.full((nq, k), -np.inf, np.float32)
    out_i = np.full((nq, k), -1, np.int64)
    groups = {}
    for r in range(nq):
        groups.setdefault((int(req[r, 0]), int(req[r, 1])), []).append(r)
    for (a, y), rows in groups.items():
        sub = np.flatnonzero(allows(labels, a, y))
        if sub.size == 0:
            continue
        rows = np.asarray(rows)
        if ex is None:
            sub_ex = np.full((rows.size, 0), -1, np.int64)
        else:   # global ids -> positions in `sub` (-1 for ids the subset does not hold)
            e = ex[rows]
            pos = np.searchsorted(sub, e)
            hit = (e >= 0) & (pos < sub.size) & (sub[np.minimum(pos, sub.size - 1)] == e)
            sub_ex = np.where(hit, pos, -1)
        s, i = search_excluding(xn[sub], qn[rows], k, sub_ex)
        kk = s.shape[1]
        out_s[rows, :kk] = s
        out_i[rows, :kk] = np.where(i >= 0, sub[np.maximum(i, 0)], -1)
    return out_s, out_i


def torch_topk_filtered(xn, q, k, allowed):
    """bench.torch_flat_topk (fp32 sgemm + torch.topk on the device) over the rows `allowed` (bool [N], one mask for
    every query), ids mapped back and (-inf, -1) padded to k; device tensors."""
    import torch

    import bench
    idx = torch.nonzero(allowed).flatten()
    s = torch.full((q.shape[0], k), float("-inf"), device=q.device)
    i = torch.full((q.shape[0], k), -1, device=q.device, dtype=torch.int64)
    if idx.numel():
        ts, ti = bench.torch_flat_topk(xn[idx], q, k)
        s[:, :ts.shape[1]] = ts
        i[:, :ts.shape[1]] = idx[ti]
    return s, i
