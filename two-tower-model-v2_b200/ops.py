"""PyTorch ops over the C-ABI: `torch.ops.tt.*`, CUDA only.

Each op allocates its outputs with torch (device memory + current stream are torch's job: plumbing)
and hands raw pointers to libtt_b200.so.  There is no CPU or Meta implementation on purpose.
"""
from __future__ import annotations

from typing import Tuple

import torch

from . import _native


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"tt_b200: `{name}` must be a CUDA tensor (no CPU fallback); got {t.device}")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


@torch.library.custom_op("tt::pool_weighted", mutates_args=(), device_types="cuda")
def pool_weighted(x: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """buyer_tower.py:43-68 — x [B,S,D], w [B,S] -> [B,D]."""
    B, S, D = x.shape
    out = torch.empty((B, D), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _native.check(_native.load().tt_pool_weighted(x.data_ptr(), w.data_ptr(), out.data_ptr(), B, S, D, _stream()),
                      "tt_pool_weighted")
    return out


@torch.library.custom_op("tt::pool_weighted_gather", mutates_args=(), device_types="cuda")
def pool_weighted_gather(table: torch.Tensor, idx: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """Same as pool_weighted with rows x[b,s] = table[idx[b,s]] (idx out of range = zero row)."""
    N, D = table.shape
    B, S = idx.shape
    out = torch.empty((B, D), device=table.device, dtype=torch.float32)
    with torch.cuda.device(table.device):
        _native.check(_native.load().tt_pool_weighted_gather(table.data_ptr(), N, idx.data_ptr(), w.data_ptr(),
                                                             out.data_ptr(), B, S, D, _stream()),
                      "tt_pool_weighted_gather")
    return out


@torch.library.custom_op("tt::attention_logits", mutates_args=(), device_types="cuda")
def attention_logits(x: torch.Tensor, W1: torch.Tensor, b1: torch.Tensor, W2: torch.Tensor,
                     b2: torch.Tensor) -> torch.Tensor:
    """buyer_tower.py:85-86 — x [R,D] -> logits [R] = W2.relu(W1 x + b1) + b2 (fp32)."""
    R, D = x.shape
    H = W1.shape[0]
    out = torch.empty((R,), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _native.check(_native.load().tt_attention_logits(x.data_ptr(), R, D, W1.data_ptr(), b1.data_ptr(),
                                                         W2.data_ptr(), b2.data_ptr(), H, out.data_ptr(), _stream()),
                      "tt_attention_logits")
    return out


@torch.library.custom_op("tt::pool_attention", mutates_args=(), device_types="cuda")
def pool_attention(x: torch.Tensor, logits: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """buyer_tower.py:89-99 — softmax_s(logits*w)-weighted sum + L2 normalise."""
    B, S, D = x.shape
    out = torch.empty((B, D), device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        _native.check(_native.load().tt_pool_attention(x.data_ptr(), logits.data_ptr(), w.data_ptr(), out.data_ptr(),
                                                       B, S, D, _stream()), "tt_pool_attention")
    return out


@torch.library.custom_op("tt::pool_attention_fused", mutates_args=(), device_types="cuda")
def pool_attention_fused(x: torch.Tensor, w: torch.Tensor, W1: torch.Tensor, b1: torch.Tensor, W2: torch.Tensor,
                         b2: torch.Tensor) -> torch.Tensor:
    """buyer_tower.py:70-101 in one kernel / one pass over x — x [B,S,D], w [B,S], MLP params -> [B,D]."""
    B, S, D = x.shape
    H = W1.shape[0]
    lib = _native.load()
    out = torch.empty((B, D), device=x.device, dtype=torch.float32)
    ws = torch.empty(max(int(lib.tt_pool_attention_fused_workspace_bytes(max(B, 1), S, D, H)), 256), device=x.device,
                     dtype=torch.uint8)
    with torch.cuda.device(x.device):
        _native.check(lib.tt_pool_attention_fused(x.data_ptr(), w.data_ptr(), W1.data_ptr(), b1.data_ptr(), W2.data_ptr(),
                                                  b2.data_ptr(), H, out.data_ptr(), B, S, D, ws.data_ptr(), ws.numel(),
                                                  _stream()), "tt_pool_attention_fused")
    return out


@torch.library.custom_op("tt::pool_attention_gather", mutates_args=(), device_types="cuda")
def pool_attention_gather(table: torch.Tensor, row_logits: torch.Tensor, zero_row_logit: float,
                          idx: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    N, D = table.shape
    B, S = idx.shape
    out = torch.empty((B, D), device=table.device, dtype=torch.float32)
    with torch.cuda.device(table.device):
        _native.check(_native.load().tt_pool_attention_gather(table.data_ptr(), N, row_logits.data_ptr(),
                                                              float(zero_row_logit), idx.data_ptr(), w.data_ptr(),
                                                              out.data_ptr(), B, S, D, _stream()),
                      "tt_pool_attention_gather")
    return out


def pool_backward(x: torch.Tensor, w: torch.Tensor, logits, g: torch.Tensor, need_dx: bool = True):
    """Backward of the pooling op (tt_pool_backward): -> (dx [B,S,D] or None, dw [B,S], dlogit [B,S] or None)."""
    B, S, D = x.shape
    dx = torch.empty_like(x) if need_dx else None
    dw = torch.empty((B, S), device=x.device, dtype=torch.float32)
    dlogit = torch.empty((B, S), device=x.device, dtype=torch.float32) if logits is not None else None
    with torch.cuda.device(x.device):
        _native.check(_native.load().tt_pool_backward(
            x.data_ptr(), w.data_ptr(), 0 if logits is None else logits.data_ptr(), g.data_ptr(),
            0 if dx is None else dx.data_ptr(), dw.data_ptr(), 0 if dlogit is None else dlogit.data_ptr(), B, S, D,
            _stream()), "tt_pool_backward")
    return dx, dw, dlogit


def infonce_forward(buyer: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, temperature: float):
    """InfoNCE forward (tt_infonce_forward): buyer/pos f32 [B,D], neg f32 [B,M,D] -> (loss [1], row_loss [B], lse [B])."""
    B, D = buyer.shape
    M = neg.shape[1]
    loss = torch.empty(1, device=buyer.device, dtype=torch.float32)
    row_loss = torch.empty(B, device=buyer.device, dtype=torch.float32)
    lse = torch.empty(B, device=buyer.device, dtype=torch.float32)
    with torch.cuda.device(buyer.device):
        _native.check(_native.load().tt_infonce_forward(buyer.data_ptr(), pos.data_ptr(), neg.data_ptr() if M else 0, B, M, D,
                                                        float(temperature), loss.data_ptr(), row_loss.data_ptr(), lse.data_ptr(),
                                                        _stream()), "tt_infonce_forward")
    return loss, row_loss, lse


def infonce_backward(buyer: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, lse: torch.Tensor, grad_loss: torch.Tensor,
                     temperature: float):
    """InfoNCE backward (tt_infonce_backward): grad_loss f32 [1] on the device -> (d_buyer [B,D], d_pos [B,D], d_neg [B,M,D])."""
    B, D = buyer.shape
    M = neg.shape[1]
    lib = _native.load()
    d_buyer, d_pos, d_neg = torch.empty_like(buyer), torch.empty_like(pos), torch.empty_like(neg)
    ws = torch.empty(max(int(lib.tt_infonce_workspace_bytes(B)), 256), device=buyer.device, dtype=torch.uint8)
    with torch.cuda.device(buyer.device):
        _native.check(lib.tt_infonce_backward(buyer.data_ptr(), pos.data_ptr(), neg.data_ptr() if M else 0, lse.data_ptr(),
                                              grad_loss.data_ptr(), B, M, D, float(temperature), d_buyer.data_ptr(),
                                              d_pos.data_ptr(), d_neg.data_ptr() if M else 0, ws.data_ptr(), ws.numel(),
                                              _stream()), "tt_infonce_backward")
    return d_buyer, d_pos, d_neg


def pool_partial_gather(table: torch.Tensor, row_lo: int, n_total: int, owns_invalid: bool, row_logits, zero_row_logit: float,
                        idx: torch.Tensor, w: torch.Tensor, partial: torch.Tensor = None) -> torch.Tensor:
    """Owner-computes partial pooling over this rank's rows of a sharded item table -> partial f32 [B, D+4]
    (tt_pool_partial_gather); row_logits None = weighted_avg."""
    n_local, D = table.shape
    B, S = idx.shape
    if partial is None:
        partial = torch.empty((B, D + 4), device=table.device, dtype=torch.float32)
    with torch.cuda.device(table.device):
        _native.check(_native.load().tt_pool_partial_gather(
            table.data_ptr(), n_local, int(row_lo), int(n_total), 1 if owns_invalid else 0,
            0 if row_logits is None else row_logits.data_ptr(), float(zero_row_logit), idx.data_ptr(), w.data_ptr(),
            partial.data_ptr(), B, S, D, _stream()), "tt_pool_partial_gather")
    return partial


def pool_partial_merge(partials_g: torch.Tensor, attention: bool) -> torch.Tensor:
    """All-gathered partials f32 [G, B, D+4] -> L2-normalised buyer embeddings [B, D] (tt_pool_partial_merge)."""
    G, B, D2 = partials_g.shape
    out = torch.empty((B, D2 - 4), device=partials_g.device, dtype=torch.float32)
    with torch.cuda.device(partials_g.device):
        _native.check(_native.load().tt_pool_partial_merge(partials_g.data_ptr(), G, 1 if attention else 0, out.data_ptr(),
                                                           B, D2 - 4, _stream()), "tt_pool_partial_merge")
    return out


@torch.library.custom_op("tt::topk_merge", mutates_args=(), device_types="cuda")
def topk_merge(scores_g: torch.Tensor, ids_g: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """[G,nq,K] per-shard sorted lists -> [nq,K] (score desc, id asc)."""
    G, nq, K = scores_g.shape
    scores = torch.empty((nq, K), device=scores_g.device, dtype=torch.float32)
    ids = torch.empty((nq, K), device=scores_g.device, dtype=torch.int64)
    with torch.cuda.device(scores_g.device):
        _native.check(_native.load().tt_topk_merge(scores_g.data_ptr(), ids_g.data_ptr(), G, nq, K,
                                                   scores.data_ptr(), ids.data_ptr(), _stream()), "tt_topk_merge")
    return scores, ids


@torch.library.custom_op("tt::flat_build", mutates_args=("xn", "xh", "stats"), device_types="cuda")
def flat_build(x: torch.Tensor, xn: torch.Tensor, xh: torch.Tensor, stats: torch.Tensor, row0: int,
               normalize: bool) -> None:
    """vector_db.py:44-54 — rows of x -> xn[row0:] (f32, x/(||x||+1e-8) if normalize) and xh[row0:] (bf16 shadow);
    folds the error-bound norms into stats f32[4].  x may alias xn[row0:row0+rows]."""
    rows, D = x.shape
    with torch.cuda.device(x.device):
        _native.check(_native.load().tt_flat_build(x.data_ptr(), rows, D, 1 if normalize else 0, xn.data_ptr(),
                                                   xh.data_ptr(), row0, stats.data_ptr(), _stream()), "tt_flat_build")


@torch.library.custom_op("tt::flat_search", mutates_args=(), device_types="cuda")
def flat_search(q: torch.Tensor, xn: torch.Tensor, xh: torch.Tensor, stats: torch.Tensor, k: int,
                id_offset: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """vector_db.py:152-160 / :189-197 — exact top-k of q f32 [nq,D] (un-normalised) against the index arrays ->
    (scores f32 [nq,k], ids i64 [nq,k], flags i32 [nq], n_uncertified i32 [1]); rows with flags != 1 must be
    re-run through tt::flat_search_exact (FlatIPIndex.search_checked_device does both)."""
    nq, D = q.shape
    N = xn.shape[0]
    lib = _native.load()
    dev = q.device
    scores = torch.empty((nq, k), device=dev, dtype=torch.float32)
    ids = torch.empty((nq, k), device=dev, dtype=torch.int64)
    flags = torch.empty((max(nq, 1),), device=dev, dtype=torch.int32)
    nunc = torch.empty((1,), device=dev, dtype=torch.int32)
    ws = torch.empty(max(int(lib.tt_flat_search_workspace_bytes(N, D, max(nq, 1), k)), 256), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        _native.check(lib.tt_flat_search(q.data_ptr(), nq, xn.data_ptr(), xh.data_ptr(), stats.data_ptr(), N, D, k, id_offset,
                                         scores.data_ptr(), ids.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                                         ws.data_ptr(), ws.numel(), _stream()), "tt_flat_search")
    return scores, ids, flags[:nq].clone(), nunc


@torch.library.custom_op("tt::flat_search_exact", mutates_args=(), device_types="cuda")
def flat_search_exact(q: torch.Tensor, xn: torch.Tensor, k: int, id_offset: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Always-exact fp32 path (CUDA-core scoring + radix select) for every row of q."""
    nq, D = q.shape
    N = xn.shape[0]
    lib = _native.load()
    dev = q.device
    scores = torch.empty((nq, k), device=dev, dtype=torch.float32)
    ids = torch.empty((nq, k), device=dev, dtype=torch.int64)
    ws = torch.empty(max(int(lib.tt_flat_search_exact_workspace_bytes(N, D, nq, k)), 256), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        _native.check(lib.tt_flat_search_exact(q.data_ptr(), nq, 0, nq, xn.data_ptr(), N, D, k, id_offset, scores.data_ptr(),
                                               ids.data_ptr(), ws.data_ptr(), ws.numel(), _stream()), "tt_flat_search_exact")
    return scores, ids


def shard_merge(gathered: torch.Tensor, off_scores: int, off_ids: int, off_bound: int, off_flags: int, nq: int, K: int,
                nunc: torch.Tensor = None):
    """[G, record bytes] all-gathered shard records -> (scores [nq,K], ids [nq,K], flags [nq], n_uncertified [1])
    with the global exactness certificate (tt_shard_merge)."""
    G, stride = gathered.shape
    dev = gathered.device
    scores = torch.empty((nq, K), device=dev, dtype=torch.float32)
    ids = torch.empty((nq, K), device=dev, dtype=torch.int64)
    flags = torch.empty((max(nq, 1),), device=dev, dtype=torch.int32)
    if nunc is None:
        nunc = torch.empty((1,), device=dev, dtype=torch.int32)
    stride = gathered.stride(0)
    with torch.cuda.device(dev):
        _native.check(_native.load().tt_shard_merge(gathered.data_ptr(), stride, off_scores, off_ids, off_bound, off_flags,
                                                    G, nq, K, scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                                                    nunc.data_ptr(), _stream()), "tt_shard_merge")
    return scores, ids, flags[:nq], nunc


def range_merge(gathered: torch.Tensor, layout, nq: int, L: int, nunc: torch.Tensor = None):
    """[G, record bytes] all-gathered range records (sharded.range_record_layout) -> (counts [nq] i64, scores [nq, L],
    ids [nq, L], flags [nq], n_uncertified [1]): the summed counts and the best min(count, L) rows of the union
    (tt_range_merge)."""
    G = gathered.shape[0]
    dev = gathered.device
    counts = torch.empty((nq,), device=dev, dtype=torch.int64)
    scores = torch.empty((nq, L), device=dev, dtype=torch.float32)
    ids = torch.empty((nq, L), device=dev, dtype=torch.int64)
    flags = torch.empty((max(nq, 1),), device=dev, dtype=torch.int32)
    if nunc is None:
        nunc = torch.empty((1,), device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        _native.check(_native.load().tt_range_merge(gathered.data_ptr(), gathered.stride(0), layout.off_counts,
                                                    layout.off_scores, layout.off_ids, layout.off_flags, G, nq, L,
                                                    counts.data_ptr(), scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                                                    nunc.data_ptr(), _stream()), "tt_range_merge")
    return counts, scores, ids, flags[:nq], nunc


__all__ = ["shard_merge", "range_merge", "flat_build", "flat_search", "flat_search_exact", "pool_weighted", "pool_weighted_gather", "attention_logits", "pool_attention",
           "pool_attention_gather", "pool_attention_fused", "pool_backward", "infonce_forward", "infonce_backward", "pool_partial_gather", "pool_partial_merge", "topk_merge", "_f32c", "_stream"]
