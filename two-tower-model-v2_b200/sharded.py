"""Catalog sharding across GPUs (north_star (3); the reference has no multi-device path).

One process per GPU.  Rank r owns the contiguous catalog rows [lo_r, hi_r); every rank searches its
shard for the replicated query batch and writes its result straight into one byte record

    { scores f32[nq,K] | ids i64[nq,K] | bound f32[nq] | flags i32[nq] }

(ids are global row numbers; lists shorter than K are padded with score -inf / id -1).  ONE
all-gather of the records (NCCL over NVLink/NVSwitch) and a merge kernel (tt_shard_merge) produce the
global top-K on every rank together with a *global* exactness certificate: the merged K-th score must
clear, on every shard, the bound of the rows that shard did not rescore in fp32.  Queries that fail it
(rare) are re-run through the always-exact fp32 path on every shard and merged again.

The local search and the merge are injectable so that the pack / exchange / fallback logic is testable
on CPU with the gloo backend (tests/test_sharded_gloo.py).
"""
from __future__ import annotations

from typing import Callable, NamedTuple, Optional, Tuple

import os

import torch
import torch.distributed as dist


def shard_bounds(n_total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous block partition: rank r owns [r*ceil(N/G), min(N, (r+1)*ceil(N/G)))."""
    if world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("bad world_size/rank")
    per = -(-n_total // world_size)
    lo = min(n_total, rank * per)
    hi = min(n_total, lo + per)
    return lo, hi


class RecordLayout(NamedTuple):
    """Byte offsets of one rank's record (every field 16-byte aligned)."""
    off_scores: int
    off_ids: int
    off_bound: int
    off_flags: int
    nbytes: int


def record_layout(nq: int, k: int) -> RecordLayout:
    def up(x):
        return (x + 15) // 16 * 16
    o_scores = 0
    o_ids = up(o_scores + nq * k * 4)
    o_bound = up(o_ids + nq * k * 8)
    o_flags = up(o_bound + nq * 4)
    return RecordLayout(o_scores, o_ids, o_bound, o_flags, up(o_flags + nq * 4))


def record_views(buf: torch.Tensor, lay: RecordLayout, nq: int, k: int):
    """Typed views (scores, ids, bound, flags) into a uint8 record (or a [G, nbytes] stack of records)."""
    lead = buf.shape[:-1]

    def field(off, n, dtype, shape):
        size = torch.empty((), dtype=dtype).element_size()
        return buf[..., off:off + n * size].view(dtype).view(*lead, *shape)
    return (field(lay.off_scores, nq * k, torch.float32, (nq, k)), field(lay.off_ids, nq * k, torch.int64, (nq, k)),
            field(lay.off_bound, nq, torch.float32, (nq,)), field(lay.off_flags, nq, torch.int32, (nq,)))


def _merge_cuda(gathered: torch.Tensor, lay: RecordLayout, nq: int, k: int, nunc: Optional[torch.Tensor] = None):
    from . import ops
    return ops.shard_merge(gathered, lay.off_scores, lay.off_ids, lay.off_bound, lay.off_flags, nq, k, nunc)


class _RawCudaBuffer:
    """__cuda_array_interface__ over a raw device pointer (uint8), for a zero-copy torch view."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3,
                                         "strides": None}


class P2PExchange:
    """All-gather of fixed-size records over NVLink peer memory with our own kernels (tt_p2p_push /
    tt_p2p_wait) instead of NCCL.

    Every rank owns one device buffer holding, per channel, NSLOT receive areas [NSLOT][G][nbytes] and flags
    int32 [NSLOT][G] (slot = sequence number mod NSLOT).  `push` and `wait` are separate so that a caller can defer
    the wait: the pipelined sharded search pushes batch j's record, scans batch j+1 and only then waits for the
    peers' records of batch j (by then they have long arrived).  With the 3-stage pipeline of ShardedFlatIPIndex a
    slot is overwritten no earlier than three exchanges later, after a wait that proves every peer has consumed it.  The buffers are mapped into every rank through CUDA IPC handles exchanged once over
    the process group (tt_p2p_alloc / tt_p2p_open); afterwards an exchange is two kernel launches
    on the caller's stream and no host synchronisation: push my record into my slot on every peer and raise
    my sequence flag there; wait (one warp, acquire loads, bounded by a time-out) until every rank's flag for
    this sequence number is up.  `status[1]` turns non-zero if a wait timed out.
    """

    NSLOT = 4

    def __init__(self, channel_bytes, device: torch.device, group=None, timeout_s: float = 20.0):
        from . import _native
        self.lib = _native.load()
        self.check = _native.check
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.device = device
        self.timeout_s = timeout_s
        G = self.world
        self.nbytes = [int(b) for b in channel_bytes]
        assert all(b % 16 == 0 for b in self.nbytes)
        self.recv_off, self.flag_off = [], []
        off = 0
        for b in self.nbytes:
            self.recv_off.append(off)
            off += self.NSLOT * G * b
            off = (off + 255) // 256 * 256
        for _ in self.nbytes:
            self.flag_off.append(off)
            off += self.NSLOT * G * 4
            off = (off + 255) // 256 * 256
        import ctypes
        self._ctypes = ctypes
        self.total_bytes = off
        self.base, self.peer_base, self.buf = None, [], None

        def agree(ok: bool) -> bool:
            """Every rank leaves each set-up stage together: MIN over the ranks' success flags."""
            t = torch.tensor([1 if ok else 0], device=device, dtype=torch.int32)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
            return bool(int(t.item()))

        # stage 1: allocate the receive buffer
        ptr, handle, err = ctypes.c_void_p(), ctypes.create_string_buffer(64), None
        try:
            with torch.cuda.device(device):
                self.check(self.lib.tt_p2p_alloc(off, ctypes.byref(ptr), handle), "tt_p2p_alloc")
            self.base = int(ptr.value)
        except Exception as e:
            err = e
        if not agree(err is None):
            self._abort()
            raise RuntimeError(f"P2PExchange: receive-buffer allocation failed on some rank ({err!r} here)")
        # stage 2: exchange the IPC handles and map every peer
        handles = [None] * G
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        self.peer_base = [None] * G
        try:
            for r in range(G):
                if r == self.rank:
                    self.peer_base[r] = self.base
                    continue
                p = ctypes.c_void_p()
                with torch.cuda.device(device):
                    self.check(self.lib.tt_p2p_open(ctypes.create_string_buffer(handles[r], 64), ctypes.byref(p)), "tt_p2p_open")
                self.peer_base[r] = int(p.value)
        except Exception as e:
            err = e
        if not agree(err is None):
            dist.barrier(group=group)       # nobody frees a buffer a peer may still be mapping
            self._abort()
            raise RuntimeError(f"P2PExchange: mapping a peer's buffer failed on some rank ({err!r} here)")
        # zero-copy torch view of the local buffer (kernels downstream take torch tensors)
        self.buf = torch.as_tensor(_RawCudaBuffer(self.base, off), device=device)
        self.done = torch.zeros(len(self.nbytes), dtype=torch.int32, device=device)
        self.seq = [0] * len(self.nbytes)
        self._ptr_arrays = {}
        dist.barrier(group=group)       # every rank has mapped every buffer before the first push

    def _abort(self) -> None:
        """Local clean-up of a failed set-up: unmap whatever peers were opened, free the own buffer."""
        with torch.cuda.device(self.device):
            for r, p in enumerate(self.peer_base):
                if p is not None and r != self.rank:
                    self.lib.tt_p2p_close(self._ctypes.c_void_p(p))
            if self.base is not None:
                self.lib.tt_p2p_free(self._ctypes.c_void_p(self.base))
        self.base, self.peer_base, self.buf = None, [], None

    def close(self) -> None:
        """Collective: every rank calls it after its last exchange.  Order matters for CUDA IPC: all ranks finish
        their work, every rank unmaps the peers' buffers, and only then does anybody free its own buffer."""
        if getattr(self, "base", None) is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        with torch.cuda.device(self.device):
            for r, p in enumerate(self.peer_base):
                if r != self.rank:
                    self.lib.tt_p2p_close(self._ctypes.c_void_p(p))
        dist.barrier(group=self.group)
        with torch.cuda.device(self.device):
            self.buf = None
            self.lib.tt_p2p_free(self._ctypes.c_void_p(self.base))
        self.base, self.peer_base = None, []

    def _ptrs(self, ch: int, slot: int):
        key = (ch, slot)
        arr = self._ptr_arrays.get(key)
        if arr is None:
            G, b = self.world, self.nbytes[ch]
            c = self._ctypes
            dst = (c.c_void_p * G)(*[p + self.recv_off[ch] + (slot * G + self.rank) * b for p in self.peer_base])
            flg = (c.c_void_p * G)(*[p + self.flag_off[ch] + (slot * G + self.rank) * 4 for p in self.peer_base])
            arr = self._ptr_arrays[key] = (dst, flg)
        return arr

    def push(self, ch: int, src: torch.Tensor) -> int:
        """Copies this rank's record (uint8 [nbytes[ch]], 16-byte aligned) into its slot on every peer and raises its
        sequence flag there (one kernel on the current stream).  Returns the sequence number to `wait` for."""
        G, b = self.world, self.nbytes[ch]
        assert src.numel() * src.element_size() == b
        self.seq[ch] += 1
        seq = self.seq[ch]
        dst, flg = self._ptrs(ch, seq % self.NSLOT)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            self.check(self.lib.tt_p2p_push(src.data_ptr(), b, dst, flg, G, seq, self.done[ch:ch + 1].data_ptr(), stream),
                       "tt_p2p_push")
        return seq

    def wait(self, ch: int, seq: int, status: torch.Tensor) -> torch.Tensor:
        """One-warp kernel on the current stream: returns once every rank's record `seq` has landed here -> uint8
        [G, nbytes[ch]] view of this rank's receive slot, valid for kernels enqueued after this call."""
        G, b = self.world, self.nbytes[ch]
        slot = seq % self.NSLOT
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            my_flags = self.base + self.flag_off[ch] + slot * G * 4
            self.check(self.lib.tt_p2p_wait(my_flags, G, seq, self.timeout_s, status[1:2].data_ptr(), stream), "tt_p2p_wait")
        o = self.recv_off[ch] + slot * G * b
        return self.buf[o:o + G * b].view(G, b)

    def all_gather(self, ch: int, src: torch.Tensor, status: torch.Tensor) -> torch.Tensor:
        """push + wait back to back."""
        return self.wait(ch, self.push(ch, src), status)


class ShardedFlatIPIndex:
    """A FlatIPIndex per rank over its row block + all-gather/merge search.

    `local_index` provides `ntotal`, `search_shard_into(q, k_local, scores, ids, bound, flags)` and
    `search_exact_into(q, k_local, scores, ids, qsel)`, both writing the first k_local columns of the
    [nq,k] record views (see FlatIPIndex).
    `merge(gathered[G,nbytes] uint8, layout, nq, k) -> (scores, ids, flags, n_uncertified)`.
    """

    MAX_P2P_SHAPES = 4

    def __init__(self, local_index, n_total: int, group=None, merge: Optional[Callable] = None, exchange: str = "auto"):
        if n_total >= 1 << 32:
            raise ValueError("sharded catalogs are limited to 2^32 - 1 rows (merge keys carry 32-bit ids)")
        self.local = local_index
        self._n_local_min = None
        self.n_total = int(n_total)
        self.group = group
        self._merge = merge if merge is not None else _merge_cuda
        self._bufs = {}
        self._p2p = {}
        # "p2p": our push/wait kernels over NVLink peer memory; "nccl": torch.distributed all-gather.
        # "auto" tries p2p on CUDA and falls back to nccl if the IPC set-up fails.
        self.exchange = os.environ.get("TT_B200_EXCHANGE", exchange)
        self.exchange_used = None
        self.pipelined = os.environ.get("TT_B200_SHARD_PIPELINE", "1") != "0"
        self._inflight = []

    @property
    def ntotal(self) -> int:
        return self.n_total

    def _buffers(self, nq: int, k: int, device, world: int):
        key = (nq, k, world)
        b = self._bufs.get(key)
        if b is None:
            lay = record_layout(nq, k)
            rec = torch.zeros(lay.nbytes, dtype=torch.uint8, device=device)
            gathered = torch.zeros((world, lay.nbytes), dtype=torch.uint8, device=device)
            if len(self._bufs) > 8:
                self._bufs.clear()
            b = self._bufs[key] = (lay, rec, gathered)
        return b

    def _exchange(self, rec: torch.Tensor, gathered: torch.Tensor, world: int):
        if world == 1:
            gathered[0].copy_(rec)
        else:
            dist.all_gather_into_tensor(gathered.view(-1), rec, group=self.group)

    def close(self) -> None:
        """Releases the peer-memory exchanges (every rank, after its last search has completed)."""
        self.flush()
        for ex in self._p2p.values():
            if ex is not None:
                ex.close()
        self._p2p.clear()

    def _p2p_for(self, nq: int, k: int, device, world: int, lay: RecordLayout):
        """The P2PExchange for this (nq, k) shape (channel 0: top-r lists, channel 1: result records, channel 2: pooling
        partials of the sharded /retrieve path), or None
        when the NCCL path is to be used.  Created collectively: every rank reaches this with the same shape."""
        if world == 1 or device.type != "cuda" or self.exchange == "nccl" or self._merge is not _merge_cuda:
            self.exchange_used = self.exchange_used or "nccl"
            return None
        key = (nq, k, world)
        if key in self._p2p:
            self._p2p[key] = self._p2p.pop(key)       # most recently used last
        if key not in self._p2p:
            from ._native import TT_SHARD_TOPR
            # Bounded: a server with many batch shapes must not keep one IPC buffer set per shape for ever.  Every
            # rank sees the same sequence of shapes, so evicting the least recently used one is collective-safe.
            while len(self._p2p) >= self.MAX_P2P_SHAPES:
                self.flush()          # no batch may still be using the exchange that is about to be closed
                old_key = next(iter(self._p2p))
                old = self._p2p.pop(old_key)
                if old is not None:
                    old.close()
            ok, ex = 1, None
            try:
                d = getattr(self.local, "d", None)
                chans = [nq * TT_SHARD_TOPR * 4, lay.nbytes]
                if d is not None and d % 4 == 0:     # channel 2: pooling partials [nq, d+4] f32 of the sharded /retrieve path
                    chans.append(nq * (d + 4) * 4)
                ex = P2PExchange(chans, device, self.group)
            except Exception as e:     # IPC not permitted, no peer access, ...
                if self.exchange == "p2p":
                    raise
                self._p2p_error = repr(e)
                ok = 0
            flag = torch.tensor([ok], device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)     # all ranks take the same path
            self._p2p[key] = ex if int(flag.item()) == 1 else None
            self.exchange_used = "p2p" if self._p2p[key] is not None else "nccl"
        return self._p2p[key]

    def _validate(self, world: int, device) -> None:
        """Once, collectively: the shards must add up to n_total, and every rank learns the smallest shard so that
        all ranks take the same branch (global threshold vs per-shard) whatever partition the caller loaded."""
        if self._n_local_min is not None:
            return
        n_local = int(self.local.ntotal)
        if world > 1:
            t = torch.tensor([n_local, -n_local], device=device, dtype=torch.int64)
            tot = torch.tensor([n_local], device=device, dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM, group=self.group)
            n_min, n_max, total = int(t[0]), -int(t[1]), int(tot[0])
        else:
            n_min = n_max = total = n_local
        if total != self.n_total:
            raise ValueError(f"shards hold {total} rows in total but n_total = {self.n_total}")
        self._n_local_min, self._n_local_max = n_min, n_max

    def _global_threshold(self, world: int, nq: int, k: int, exclude) -> bool:
        """Whether all ranks take the one-threshold plan.  A function of replicated values only (n_total, the
        smallest shard, nq, k and the exclusion list width), so every rank decides alike.  With E exclusions per
        query the plan is made for K_plan = min(k + E, n_total, TT_FLAT_MAX_K)."""
        n_local_min = self._n_local_min if self._n_local_min is not None else self.local.ntotal
        plan_ok = getattr(self.local, "shard_plan_ok", None)
        if exclude is not None:
            from ._native import plan_k
            k = plan_k(k, exclude.shape[1], self.n_total)
        return world > 1 and n_local_min >= k and plan_ok is not None and plan_ok(self.n_total, nq, k, max(n_local_min, 0))

    @staticmethod
    def _kw(exclude):
        """Keyword arguments of the local calls: none without a list, so stand-ins that predate it keep working."""
        return {} if exclude is None else {"exclude": exclude}

    def _local_search(self, q: torch.Tensor, k: int, k_local: int, world: int, views, p2p=None, status=None,
                      exclude=None) -> None:
        """Fills this rank's record.  With every shard holding >= k rows and a plan for it, all ranks use ONE
        threshold estimated from a sample of the whole catalog (a small all-gather of per-rank top-r sampled
        scores): candidates per rank drop to ~1/G of the single-device count.  Otherwise each shard picks its
        own threshold."""
        scores, ids, bound, flags = views
        nq = q.shape[0]
        kw = self._kw(exclude)
        if self._global_threshold(world, nq, k, exclude):
            from ._native import TT_SHARD_TOPR
            key = ("topr", nq, world)
            bufs = self._bufs.get(key)
            if bufs is None:
                bufs = self._bufs[key] = (torch.empty((nq, TT_SHARD_TOPR), device=q.device, dtype=torch.float32),
                                          torch.empty((world, nq, TT_SHARD_TOPR), device=q.device, dtype=torch.float32))
            topr, topr_g = bufs
            self.local.shard_sample(q, k, self.n_total, topr, **kw)
            if p2p is not None:
                topr_g = p2p.all_gather(0, topr.view(torch.uint8).view(-1), status).view(torch.float32).view(world, nq, TT_SHARD_TOPR)
            else:
                dist.all_gather_into_tensor(topr_g.view(-1), topr.view(-1), group=self.group)
            self.local.shard_search_into(nq, k, self.n_total, topr_g, scores, ids, bound, flags, **kw)
        else:
            self.local.search_shard_into(q, k_local, scores, ids, bound, flags, **kw)

    def search_async(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None):
        """Enqueues the sharded search of one batch and returns a PendingSearch; `.result()` looks at the global
        certificate later (no host sync between consecutive batches).

        With the peer-memory exchange and the one-threshold plan the batches run as a 3-stage software pipeline on the
        caller's stream, so that no rank ever idles in a wait kernel for a slower peer:
            call j :  A(j)   sample pass of batch j, push of its top-r lists
                      B(j-1) wait for the peers' lists of j-1, threshold, main scan, finalize, push of the record
                      C(j-2) wait for the peers' records of j-2, merge + global certificate
        `.result()` of a batch first enqueues whatever stages it (and every older batch) still misses.  Every rank
        issues the same calls in the same order, so the exchanges pair up.  A caller that keeps three batches in
        flight gets the full overlap; with fewer the stages simply run back to back.

        `exclude` (i64 [nq, E], GLOBAL ids, -1 = padding, replicated on every rank like q): the exact top-k over the
        rows query i does not list; with fewer than k allowed rows the tail is (-inf, -1)."""
        from .vector_db import PendingSearch
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        nq = q.shape[0]
        if exclude is not None and exclude.shape[1] == 0:
            exclude = None
        self._validate(world, q.device)
        lay, rec, gathered = self._buffers(nq, k, q.device, world)
        k_local = min(k, self.local.ntotal)
        p2p = self._p2p_for(nq, k, q.device, world, lay)
        global_thr = self._global_threshold(world, nq, k, exclude)
        if p2p is not None and global_thr and self.pipelined:
            return self._search_pipelined(q, k, nq, world, lay, rec, p2p, exclude)
        self.flush()          # never interleave the two schedules
        views = record_views(rec, lay, nq, k)
        scores, ids, bound, flags = views
        if k_local < k:   # shard smaller than k: pad so every rank contributes [nq,k]
            scores.fill_(float("-inf"))
            ids.fill_(-1)
        if p2p is not None:
            status = self._bufs.setdefault(("status", nq, k, world), torch.zeros(2, dtype=torch.int32, device=q.device))
            self._local_search(q, k, k_local, world, views, p2p, status, exclude)
            gathered = p2p.all_gather(1, rec, status)
            s, i, fl, n_unc = self._merge(gathered, lay, nq, k, status[0:1])
            n_unc = status
        else:
            self._local_search(q, k, k_local, world, views, exclude=exclude)
            self._exchange(rec, gathered, world)
            s, i, fl, n_unc = self._merge(gathered, lay, nq, k)
        post = getattr(self.local, "post_flag", None)
        token = post(n_unc) if post is not None else None
        return PendingSearch(lambda: self._finish(q, k, s, i, fl, n_unc, token, exclude))

    def _finish(self, q, k, s, i, fl, n_unc, token, exclude=None):
        # identical on every rank: all ranks merged the same records
        st = self.local.read_flag(token) if token is not None else int(n_unc)
        if isinstance(st, list):
            if st[1]:
                raise RuntimeError(f"sharded search: peer exchange {st[1]} timed out (a rank is missing)")
            st = st[0]
        n_bad = st
        if not n_bad:
            return s, i, 0
        # Re-run the flagged queries alone (this rank's record buffer may already hold a later batch):
        # exact fp32 search of every shard, a small exchange, merge, scatter into the result.
        rows = torch.nonzero(fl != 1).flatten()
        kw = {} if exclude is None else {"exclude": exclude[rows].contiguous()}
        s2, i2 = self.search_exact_device(q[rows].contiguous(), k, **kw)
        s[rows] = s2
        i[rows] = i2
        return s, i, n_bad

    # -- 3-stage pipeline -----------------------------------------------------------------------------------------
    NSLOT = 3      # batches in flight: workspaces / status words are per slot

    def _search_pipelined(self, q, k, nq, world, lay, rec, p2p, exclude=None):
        from ._native import TT_SHARD_TOPR
        from .vector_db import PendingSearch
        self._pipe_seq = getattr(self, "_pipe_seq", 0) + 1
        slot = self._pipe_seq % self.NSLOT
        dev = q.device
        topr = self._bufs.setdefault(("topr1", nq, world), torch.empty((nq, TT_SHARD_TOPR), device=dev, dtype=torch.float32))
        status = self._bufs.setdefault(("status", nq, k, world, slot), torch.zeros(2, dtype=torch.int32, device=dev))
        b = {"q": q, "k": k, "nq": nq, "world": world, "lay": lay, "rec": rec, "p2p": p2p, "slot": slot, "status": status,
             "stage": 0, "out": None, "exclude": exclude}
        # stage A: sample pass + push of the top-r lists (no wait)
        self.local.shard_sample(q, k, self.n_total, topr, slot, **self._kw(exclude))
        b["seq0"] = p2p.push(0, topr.view(torch.uint8).view(-1))
        b["stage"] = 1
        self._inflight.append(b)
        # advance the older batches by one stage each, oldest first
        if len(self._inflight) >= 3:
            self._advance(self._inflight[-3], 3)
        if len(self._inflight) >= 2:
            self._advance(self._inflight[-2], 2)
        return PendingSearch(lambda: self._finish_pipelined(b))

    def _advance(self, b, to_stage: int) -> None:
        from ._native import TT_SHARD_TOPR
        p2p, nq, k, world, lay = b["p2p"], b["nq"], b["k"], b["world"], b["lay"]
        if b["stage"] < 2 <= to_stage:          # stage B
            topr_g = p2p.wait(0, b["seq0"], b["status"]).view(torch.float32).view(world, nq, TT_SHARD_TOPR)
            scores, ids, bound, flags = record_views(b["rec"], lay, nq, k)
            self.local.shard_search_into(nq, k, self.n_total, topr_g, scores, ids, bound, flags, b["slot"],
                                         **self._kw(b["exclude"]))
            b["seq1"] = p2p.push(1, b["rec"])
            b["stage"] = 2
        if b["stage"] < 3 <= to_stage:          # stage C
            gathered = p2p.wait(1, b["seq1"], b["status"])
            s, i, fl, _ = self._merge(gathered, lay, nq, k, b["status"][0:1])
            post = getattr(self.local, "post_flag", None)
            b["out"] = (s, i, fl, post(b["status"]) if post is not None else None)
            b["stage"] = 3

    def flush(self) -> None:
        """Enqueues every stage still missing of every batch in flight (oldest first)."""
        for b in list(self._inflight):
            self._advance(b, 3)
        self._inflight = [b for b in self._inflight if b["stage"] < 3]

    def _finish_pipelined(self, b):
        if b["stage"] < 3:
            for older in list(self._inflight):
                self._advance(older, 3)
                if older is b:
                    break
        self._inflight = [x for x in self._inflight if x["stage"] < 3]
        s, i, fl, token = b["out"]
        return self._finish(b["q"], b["k"], s, i, fl, b["status"], token, b["exclude"])

    def search_exact_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None):
        """Always-exact fp32 path over the sharded catalog (collective: every rank calls it with the same q):
        fp32 exact search of every shard, one exchange of the records (NCCL / plain copy), merge.  Serves the
        queries the global certificate rejects and the parity checks of bench.py / tests.  With `exclude` a query
        may have fewer than k allowed rows: its merged list then ends in (-inf, -1), which is exact here."""
        if exclude is not None and exclude.shape[1] == 0:
            exclude = None
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        nsel = q.shape[0]
        k_local = min(k, self.local.ntotal)
        lay2 = record_layout(nsel, k)
        rec2 = torch.zeros(lay2.nbytes, dtype=torch.uint8, device=q.device)
        gathered2 = torch.zeros((world, lay2.nbytes), dtype=torch.uint8, device=q.device)
        s_l, i_l, b_l, f_l = record_views(rec2, lay2, nsel, k)
        s_l.fill_(float("-inf"))
        i_l.fill_(-1)
        b_l.fill_(float("-inf"))
        f_l.fill_(1)
        if k_local > 0:
            self.local.search_exact_into(q, k_local, s_l, i_l, torch.arange(nsel, device=q.device, dtype=torch.int32),
                                         **self._kw(exclude))
        self._exchange(rec2, gathered2, world)
        s2, i2, fl2, n_unc2 = self._merge(gathered2, lay2, nsel, k)
        if exclude is None:
            if int(n_unc2):
                raise RuntimeError("sharded search: queries still uncertified after the exact re-run")
        elif bool(((fl2 != 1) & (fl2 != -2)).any()):     # -2 alone: fewer than k allowed rows, exact as padded
            raise RuntimeError("sharded search: queries still uncertified after the exact re-run")
        return s2, i2

    def search_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None):
        """q replicated on every rank -> global (scores, ids) [nq,k] on every rank, and the number of
        queries that failed the global certificate and were re-run through the exact path."""
        return self.search_async(q, k, **self._kw(exclude)).result()

    def search_host_async(self, q, k: int, *, exclude=None):
        """numpy in / numpy out round trip (pinned staging), asynchronous; `.result()` -> (scores, ids, n_rerun).
        `exclude`: numpy int64 [nq, E] global ids (see search_async)."""
        from .vector_db import host_search_async
        return host_search_async(self, self.search_async, self.local.device, self.local.d, q, k, exclude=exclude)

    def search_host_sliced_async(self, q_local, k: int):
        """Serving layout for G ranks fronting one sharded catalog: every rank submits ITS share of the batch
        (numpy [nq_local, D], the same row count on every rank).  The shares are all-gathered on the device (rank
        order = batch order), the whole batch is searched as usual, and each rank gets back the results of its own
        rows: host copies are nq_local*D*4 bytes in and nq_local*k*12 bytes out per rank instead of the whole batch
        on every rank.  `.result()` -> (scores [nq_local,k], ids [nq_local,k], n_rerun) numpy."""
        import numpy as np
        from .vector_db import PendingSearch
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        rank = dist.get_rank(self.group) if dist.is_initialized() else 0
        dev, d = self.local.device, self.local.d
        q_local = np.ascontiguousarray(q_local, dtype=np.float32)
        if q_local.ndim != 2 or q_local.shape[1] != d:
            raise ValueError(f"expected queries [nq_local, {d}], got {q_local.shape}")
        nl = q_local.shape[0]
        rings = self.__dict__.setdefault("_sliced_rings", {})
        ring = rings.get((nl, k))
        if ring is None:
            if len(rings) > 8:
                rings.clear()
            ring = rings[(nl, k)] = {"next": 0, "sets": [
                (torch.empty((nl, d), dtype=torch.float32, pin_memory=True),
                 torch.empty((nl, k), dtype=torch.float32, pin_memory=True),
                 torch.empty((nl, k), dtype=torch.int64, pin_memory=True)) for _ in range(3)]}
        slot = ring["next"]
        hq, hs, hi = ring["sets"][slot]
        ring["next"] = (slot + 1) % 3
        evs = ring.setdefault("h2d_done", [None] * 3)
        if evs[slot] is not None:
            evs[slot].synchronize()      # the previous user's H2D copy of this staging set has been consumed
        hq.copy_(torch.from_numpy(q_local))
        stream = torch.cuda.current_stream(dev)
        with torch.cuda.device(dev):
            dq_local = hq.to(dev, non_blocking=True)
            evs[slot] = torch.cuda.Event()
            evs[slot].record(stream)
            dq_all = torch.empty((world, nl, d), device=dev, dtype=torch.float32)    # fresh: the exact re-run may need it later
            if world > 1:
                dist.all_gather_into_tensor(dq_all.view(-1), dq_local.view(-1), group=self.group)
            else:
                dq_all[0].copy_(dq_local)
            pending = self.search_async(dq_all.view(world * nl, d), k)

        def finish():
            scores, ids, n_bad = pending.result()
            st = torch.cuda.current_stream(dev)
            with torch.cuda.device(dev):
                hs.copy_(scores[rank * nl:(rank + 1) * nl], non_blocking=True)
                hi.copy_(ids[rank * nl:(rank + 1) * nl], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(st)
            ev.synchronize()
            return hs.numpy().copy(), hi.numpy().copy(), n_bad
        return PendingSearch(finish)
