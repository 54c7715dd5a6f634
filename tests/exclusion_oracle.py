"""Exclusion-aware restatements of the exact search, for the tests of tt_flat_search_excl & co.

Both are built on the unchanged IndexFlatIP oracle (oracle/flat_ip_oracle.py) and on bench.torch_flat_topk: at most
E distinct rows are excluded per query, so the exact top-(k + E) over all rows holds the exact top-k over the allowed
rows.  Dropping the excluded ids from it and keeping the first k gives the masked result, ordered like the library
(score descending, id ascending), padded with (-inf, -1) when fewer than k rows are allowed.
"""
import numpy as np

from oracle import flat_ip_oracle as fo


def filter_topk(scores, ids, exclude, k):
    """(scores, ids) [nq, k + E] sorted lists minus the ids of exclude[q] -> [nq, k], (-inf, -1) padded."""
    scores, ids = np.asarray(scores), np.asarray(ids)
    ex = np.asarray(exclude, dtype=np.int64).reshape(ids.shape[0], -1)
    out_s = np.full((ids.shape[0], k), -np.inf, np.float32)
    out_i = np.full((ids.shape[0], k), -1, np.int64)
    for r in range(ids.shape[0]):
        keep = np.flatnonzero((ids[r] >= 0) & ~np.isin(ids[r], ex[r]))[:k]
        out_s[r, :len(keep)] = scores[r, keep]
        out_i[r, :len(keep)] = ids[r, keep]
    return out_s, out_i


def search_excluding(xn, qn, k, exclude, block=65536):
    """fo.search over the rows query i does not list in exclude[i] (entries < 0 or >= N are ignored)."""
    n = xn.shape[0]
    k = min(k, n)
    ex = np.asarray(exclude, dtype=np.int64).reshape(qn.shape[0], -1)
    s, i = fo.search(xn, qn, min(k + ex.shape[1], n), block=block)
    return filter_topk(s, i, ex, k)


def torch_topk_excluding(xn, q, k, exclude):
    """bench.torch_flat_topk (fp32 sgemm + torch.topk on the device) with the listed rows masked; device tensors."""
    import torch

    import bench
    E = exclude.shape[1]
    s, i = bench.torch_flat_topk(xn, q, k + E)
    hit = (i[:, :, None] == exclude[:, None, :]).any(2)
    # stable: allowed entries keep their order, excluded ones move behind them
    order = torch.sort(hit.to(torch.int8), dim=1, stable=True).indices[:, :k]
    s, i, hit = torch.gather(s, 1, order), torch.gather(i, 1, order), torch.gather(hit, 1, order)
    return s.masked_fill(hit, float("-inf")), i.masked_fill(hit, -1)
