"""`/retrieve` hot path kept on the device (SURVEY.md §8f-1).

The reference serves a request as `encoder.encode_buyer(interactions)` -> `.cpu().numpy()` ->
`vector_db.retrieve(embedding, k)` (src/api/server.py:241-244): every history item is re-encoded through
the text tower on every request (src/inference/encoder.py:276-292) and the pooled embedding takes a host
round trip before the search.  The catalog rows ARE those item embeddings (the same ItemTower output,
encoder.py:235-240), so here a request is: history product ids -> catalog row indices (host dict) ->
fused gather + pooling + L2 norm out of the device-resident fp32 table (tt_pool_*_gather) -> exact top-K
(tt_flat_search) with the pooled embedding never leaving the device.

History semantics follow encode_buyer: sort by timestamp when every interaction has one, keep the last
`max_interaction_history` (configs/config.yaml:14), event weights through get_event_weight.  One deliberate
difference: a product id that is not in the catalog pools as an all-zero row here (and is counted in the
`unknown` result of encode_histories), whereas the reference would encode the empty text for it.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .buyer_tower import BuyerTower
from .config import DEFAULT_EVENT_WEIGHTS, get_event_weight
from ._native import TT_FLAT_RANGE_MAX_RESULTS
from .vector_db import PendingSearch, VectorDatabase, range_csr, require_masks


class RetrievalPipeline:
    def __init__(self, buyer_tower: BuyerTower, vector_db: VectorDatabase, config: Optional[Dict[str, Any]] = None,
                 max_interaction_history: int = 100):
        if vector_db.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        self.tower = buyer_tower
        self.db = vector_db
        self.index = vector_db.index
        self.config = config if config is not None else {"event_weights": dict(DEFAULT_EVENT_WEIGHTS)}
        self.max_history = int(max_interaction_history)
        self.table = self.index.xn                              # [N, D] fp32, device resident
        self.item_logits = buyer_tower.precompute_item_logits(self.table)   # None in weighted_avg mode
        self._pins: Dict[Tuple[int, int], Tuple[torch.Tensor, torch.Tensor]] = {}

    # -- host side: interactions -> (row indices, weights), padded with (-1, 0) ---------------------
    def encode_histories(self, batch: Sequence[Sequence[Dict[str, Any]]]) -> Tuple[np.ndarray, np.ndarray, int]:
        lens, rows_all, w_all, unknown = [], [], [], 0
        for interactions in batch:
            if all(it.get("timestamp") is not None for it in interactions):
                interactions = sorted(interactions, key=lambda x: x["timestamp"])       # encoder.py:263-264
            interactions = interactions[-self.max_history:]                             # encoder.py:267-268
            rows = [self.db.id_to_index.get(it["product_id"], -1) for it in interactions]
            unknown += sum(1 for r in rows if r < 0)
            rows_all.append(rows)
            w_all.append([float(get_event_weight(it["event_type"], self.config)) for it in interactions])
            lens.append(len(rows))
        S = max(max(lens, default=0), 1)
        idx = np.full((len(batch), S), -1, np.int64)
        w = np.zeros((len(batch), S), np.float32)
        for b, (rows, ws) in enumerate(zip(rows_all, w_all)):
            idx[b, :len(rows)] = rows
            w[b, :len(ws)] = ws
        return idx, w, unknown

    # -- device side ------------------------------------------------------------------------------
    def encode_device(self, indices: torch.Tensor, weights: torch.Tensor) -> torch.Tensor:
        """history rows i64 [B,S] + weights f32 [B,S] (device) -> buyer embeddings [B,D] (device)."""
        return self.tower.forward_gather(self.table, indices, weights, self.item_logits)

    def retrieve_device_async(self, indices: torch.Tensor, weights: torch.Tensor, k: int, *,
                              exclude_history: bool = False, require_all=0, require_any=0,
                              max_per_group: Optional[int] = None) -> PendingSearch:
        """exclude_history: the pooled history rows `indices` (-1 padded; the last `max_interaction_history`
        interactions when they come from encode_histories) are also the exclusion list of the search, so no buyer
        is shown the items they have just viewed, carted or bought.  No extra host-to-device copy.
        require_all / require_any: label masks (scalars or one per buyer, host values): only items whose label word
        (VectorDatabase.set_labels) has every bit of require_all and, unless require_any is 0, one bit of require_any.
        max_per_group: at most that many items of one group (VectorDatabase.set_groups: a brand, a seller) per buyer."""
        k = min(k, self.index.ntotal)                                                  # vector_db.py:159
        req = require_masks(require_all, require_any, int(indices.shape[0]))
        emb = self.encode_device(indices, weights)
        kw = {} if req is None else {"require": req}
        if exclude_history:
            kw["exclude"] = indices.to(device=self.index.device, dtype=torch.int64).contiguous()
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        return self.index.search_async(emb, k, **kw)

    def retrieve_above_device_async(self, indices: torch.Tensor, weights: torch.Tensor, min_score,
                                    max_results: int = TT_FLAT_RANGE_MAX_RESULTS, *, exclude_history: bool = False,
                                    require_all=0, require_any=0) -> PendingSearch:
        """Relevance floor instead of a fixed k: every item scoring strictly above `min_score` (a float, or one per
        buyer), best first, at most `max_results` per buyer.  `.result()` -> (counts [B] i64, scores [B, L], rows [B, L]
        i64, n_rerun_tensor, n_rerun_exact) as FlatIPIndex.range_search_async; counts[b] items qualified, the first
        min(counts[b], L) are listed, the tail is (-inf, -1).  exclude_history, require_all, require_any as in
        retrieve_device_async: excluded and disallowed items are neither listed nor counted."""
        req = require_masks(require_all, require_any, int(indices.shape[0]))
        emb = self.encode_device(indices, weights)
        kw = {} if req is None else {"require": req}
        if exclude_history:
            kw["exclude"] = indices.to(device=self.index.device, dtype=torch.int64).contiguous()
        return self.index.range_search_async(emb, min_score, max_results, **kw)

    def _stage(self, batch: Sequence[Sequence[Dict[str, Any]]]):
        """Padded history rows / weights of a batch, copied to the device through pinned buffers."""
        idx, w, _ = self.encode_histories(batch)
        key = idx.shape
        pins = self._pins.get(key)
        if pins is None:
            if len(self._pins) > 16:
                self._pins.clear()
            pins = self._pins[key] = (torch.empty(key, dtype=torch.int64, pin_memory=True),
                                      torch.empty(key, dtype=torch.float32, pin_memory=True))
        pins[0].copy_(torch.from_numpy(idx))
        pins[1].copy_(torch.from_numpy(w))
        dev = self.index.device
        return pins[0].to(dev, non_blocking=True), pins[1].to(dev, non_blocking=True)

    def retrieve_arrays(self, batch: Sequence[Sequence[Dict[str, Any]]], k: int = 10, *, exclude_history: bool = False,
                        require_all=0, require_any=0, max_per_group: Optional[int] = None):
        """-> (scores f32 [B,k'], row indices i64 [B,k']) numpy; one H2D of the padded history, one D2H.
        exclude_history: leave out the buyer's last `max_interaction_history` interacted items; require_all /
        require_any: label masks (see retrieve_device_async); a buyer with fewer than k' allowed items gets (-inf, -1)
        at the tail; max_per_group: group cap (see retrieve_device_async)."""
        idx_dev, w_dev = self._stage(batch)
        pending = self.retrieve_device_async(idx_dev, w_dev, k, exclude_history=exclude_history,
                                             require_all=require_all, require_any=require_any,
                                             max_per_group=max_per_group)
        scores, ids, _ = pending.result()
        return scores.cpu().numpy(), ids.cpu().numpy()

    def retrieve(self, interactions: Sequence[Dict[str, Any]], k: int = 10, *,
                 exclude_history: bool = False, require_all=0, require_any=0,
                 max_per_group: Optional[int] = None) -> List[Tuple[str, float]]:
        """One request, the shape of server.py:241-244 -> [(product_id, score)] in descending score.
        exclude_history: never return the items of the buyer's last `max_interaction_history` interactions.
        require_all / require_any: label masks; max_per_group: group cap (see retrieve_device_async)."""
        scores, ids = self.retrieve_arrays([interactions], k, exclude_history=exclude_history, require_all=require_all,
                                           require_any=require_any, max_per_group=max_per_group)
        pids = self.db.product_ids
        return [(pids[i], float(s)) for i, s in zip(ids[0].tolist(), scores[0].tolist()) if 0 <= i < len(pids)]

    def retrieve_batch(self, batch: Sequence[Sequence[Dict[str, Any]]], k: int = 10, *,
                       exclude_history: bool = False, require_all=0, require_any=0,
                       max_per_group: Optional[int] = None) -> List[List[Tuple[str, float]]]:
        """exclude_history: as in retrieve, per buyer; require_all / require_any: scalars or one value per buyer;
        max_per_group: group cap (see retrieve_device_async)."""
        scores, ids = self.retrieve_arrays(batch, k, exclude_history=exclude_history, require_all=require_all,
                                           require_any=require_any, max_per_group=max_per_group)
        pids = self.db.product_ids
        n = len(pids)
        return [[(pids[i], s) for i, s in zip(ri, rs) if 0 <= i < n] for rs, ri in zip(scores.tolist(), ids.tolist())]

    def retrieve_above_batch(self, batch: Sequence[Sequence[Dict[str, Any]]], min_score,
                             max_results: int = TT_FLAT_RANGE_MAX_RESULTS, *, exclude_history: bool = False,
                             require_all=0, require_any=0) -> List[List[Tuple[str, float]]]:
        """Per buyer, every product scoring strictly above `min_score` (a float or one per buyer), best first, at most
        `max_results`.  exclude_history, require_all, require_any as in retrieve_batch."""
        idx_dev, w_dev = self._stage(batch)
        counts, scores, ids, _, _ = self.retrieve_above_device_async(
            idx_dev, w_dev, min_score, max_results, exclude_history=exclude_history, require_all=require_all,
            require_any=require_any).result()
        lims, s, r = range_csr(counts.cpu().numpy(), scores.cpu().numpy(), ids.cpu().numpy())
        pids = self.db.product_ids
        s, r = s.tolist(), r.tolist()
        return [[(pids[i], v) for i, v in zip(r[lims[b]:lims[b + 1]], s[lims[b]:lims[b + 1]])] for b in range(len(batch))]

    def retrieve_above(self, interactions: Sequence[Dict[str, Any]], min_score,
                       max_results: int = TT_FLAT_RANGE_MAX_RESULTS, *, exclude_history: bool = False, require_all=0,
                       require_any=0) -> List[Tuple[str, float]]:
        """One request -> [(product_id, score)] of every product scoring strictly above `min_score`, best first, at most
        `max_results` (see retrieve_above_batch)."""
        return self.retrieve_above_batch([interactions], min_score, max_results, exclude_history=exclude_history,
                                         require_all=require_all, require_any=require_any)[0]


class ShardedRetrievalPipeline:
    """The `/retrieve` path over a catalog sharded across GPUs (BASELINE config C5; one process per GPU, every rank
    calls the same methods with the same batch - the front-end replicates or slices requests as it does queries).

    The item table of the pooling IS the sharded catalog (fp32 rows `xn` of the local FlatIPIndex), so the pooling is
    owner-computes: each rank reduces the history rows it owns into a partial record per buyer (tt_pool_partial_gather:
    weighted sums are linear, the attention softmax merges like an online softmax), ONE all-gather of the [B, D+4]
    records over NVLink (our peer-memory push/wait kernels, or NCCL) and tt_pool_partial_merge give every rank the
    buyer embeddings, which go straight into the sharded exact search (ShardedFlatIPIndex.search_async).
    History row ids are GLOBAL catalog rows; ids outside [0, n_total) pool as all-zero rows (zero-padded history).
    """

    def __init__(self, buyer_tower: BuyerTower, sharded_index, group=None):
        import torch.distributed as dist
        self.tower = buyer_tower
        self.sharded = sharded_index
        self.local = sharded_index.local
        self.group = group
        self.n_total = sharded_index.n_total
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.attention = buyer_tower.aggregation_method == "attention"
        if buyer_tower.aggregation_method not in ("attention", "weighted_avg"):
            raise ValueError(f"Unknown aggregation method: {buyer_tower.aggregation_method}")
        self.table = self.local.xn
        self.row_lo = int(self.local.id_offset)
        self.item_logits = buyer_tower.precompute_item_logits(self.table)      # logits of the LOCAL rows
        self.zero_row_logit = buyer_tower.zero_row_logit() if self.attention else 0.0
        self._bufs = {}

    def encode_device(self, indices: torch.Tensor, weights: torch.Tensor, k_for_exchange: int = 100) -> torch.Tensor:
        """history rows i64 [B,S] (global ids) + weights f32 [B,S], replicated on every rank -> buyer embeddings [B,D]
        on every rank."""
        import torch.distributed as dist
        from . import ops
        idx = indices.to(device=self.table.device, dtype=torch.int64).contiguous()
        w = ops._f32c(weights.to(self.table.device), "weights")
        B, D = idx.shape[0], self.table.shape[1]
        key = (B, self.world)
        bufs = self._bufs.get(key)
        if bufs is None:
            if len(self._bufs) > 8:
                self._bufs.clear()
            bufs = self._bufs[key] = (torch.empty((B, D + 4), device=self.table.device, dtype=torch.float32),
                                      torch.empty((self.world, B, D + 4), device=self.table.device, dtype=torch.float32))
        partial, gathered = bufs
        ops.pool_partial_gather(self.table, self.row_lo, self.n_total, self.rank == 0, self.item_logits,
                                self.zero_row_logit, idx, w, partial)
        if self.world == 1:
            gathered = partial.view(1, B, D + 4)
        else:
            p2p = None
            if self.table.is_cuda:
                from .sharded import record_layout
                p2p = self.sharded._p2p_for(B, k_for_exchange, self.table.device, self.world, record_layout(B, k_for_exchange))
            if p2p is not None and len(p2p.nbytes) > 2:
                status = self.sharded._bufs.setdefault(("status", B, k_for_exchange, self.world),
                                                       torch.zeros(2, dtype=torch.int32, device=self.table.device))
                g = p2p.all_gather(2, partial.view(torch.uint8).view(-1), status)
                gathered = g.view(torch.float32).view(self.world, B, D + 4)
            else:
                dist.all_gather_into_tensor(gathered.view(-1), partial.view(-1), group=self.group)
        return ops.pool_partial_merge(gathered, self.attention)

    def retrieve_device_async(self, indices: torch.Tensor, weights: torch.Tensor, k: int, *,
                              exclude_history: bool = False, require_all=0, require_any=0) -> PendingSearch:
        """exclude_history: the pooled history rows (global ids, -1 padded; the last `max_interaction_history`
        interactions when built by RetrievalPipeline.encode_histories) are the exclusion list of the search.
        require_all / require_any: label masks, scalars or one per buyer, as in RetrievalPipeline (the words come from
        ShardedFlatIPIndex.set_labels)."""
        k = min(k, self.n_total)                                                       # vector_db.py:159
        req = require_masks(require_all, require_any, int(indices.shape[0]))
        emb = self.encode_device(indices, weights, k)
        kw = {} if req is None else {"require": req}
        if exclude_history:
            kw["exclude"] = indices.to(device=self.table.device, dtype=torch.int64).contiguous()
        return self.sharded.search_async(emb, k, **kw)

    def retrieve_host_async(self, idx_host: torch.Tensor, w_host: torch.Tensor, k: int, *,
                            exclude_history: bool = False, require_all=0, require_any=0) -> PendingSearch:
        """Pinned host tensors in (history rows / weights of the WHOLE batch, the same on every rank), numpy out.
        exclude_history: as in retrieve_device_async (the copied history rows are the list); require_all /
        require_any: label masks as in retrieve_device_async."""
        dev = self.table.device
        idx_dev, w_dev = idx_host.to(dev, non_blocking=True), w_host.to(dev, non_blocking=True)
        pending = self.retrieve_device_async(idx_dev, w_dev, k, exclude_history=exclude_history,
                                             require_all=require_all, require_any=require_any)

        def finish():
            s, i, n_bad = pending.result()
            return s.cpu().numpy(), i.cpu().numpy(), n_bad
        return PendingSearch(finish)

    def retrieve_above_device_async(self, indices: torch.Tensor, weights: torch.Tensor, min_score,
                                    max_results: int = TT_FLAT_RANGE_MAX_RESULTS, *, exclude_history: bool = False,
                                    require_all=0, require_any=0) -> PendingSearch:
        """Relevance floor over the sharded catalog: owner-computes pooling (encode_device), then
        ShardedFlatIPIndex.range_search_async.  `.result()` -> (counts [B] i64, scores [B, L], ids [B, L] GLOBAL rows,
        n_rerun), the same on every rank.  exclude_history / require_all / require_any as in retrieve_device_async."""
        req = require_masks(require_all, require_any, int(indices.shape[0]))
        emb = self.encode_device(indices, weights)
        kw = {} if req is None else {"require": req}
        if exclude_history:
            kw["exclude"] = indices.to(device=self.table.device, dtype=torch.int64).contiguous()
        return self.sharded.range_search_async(emb, min_score, max_results, **kw)

    def retrieve_above_host_async(self, idx_host: torch.Tensor, w_host: torch.Tensor, min_score,
                                  max_results: int = TT_FLAT_RANGE_MAX_RESULTS, *, exclude_history: bool = False,
                                  require_all=0, require_any=0) -> PendingSearch:
        """Pinned host tensors in (the WHOLE batch, the same on every rank) -> `.result()` = faiss's (lims, D, I) numpy
        layout of retrieve_above_device_async's result (I: global rows) and n_rerun."""
        dev = self.table.device
        idx_dev, w_dev = idx_host.to(dev, non_blocking=True), w_host.to(dev, non_blocking=True)
        pending = self.retrieve_above_device_async(idx_dev, w_dev, min_score, max_results,
                                                   exclude_history=exclude_history, require_all=require_all,
                                                   require_any=require_any)

        def finish():
            c, s, i, n_bad = pending.result()
            lims, D, I = range_csr(c.cpu().numpy(), s.cpu().numpy(), i.cpu().numpy())
            return lims, D, I, n_bad
        return PendingSearch(finish)
