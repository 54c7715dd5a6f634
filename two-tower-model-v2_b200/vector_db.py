"""Vector database: drop-in for the reference `src/inference/vector_db.py:10-231`.

`VectorDatabase` keeps the reference's constructor, attributes (`embedding_dim`, `index`,
`product_ids`, `id_to_index`, `index_to_id`), methods, argument meaning, return types and
exceptions.  `faiss.IndexFlatIP` is replaced by `FlatIPIndex`, a device-resident exact
inner-product index searched by hand-written sm_100a kernels through the C-ABI
(tt_flat_build / tt_flat_search / tt_flat_search_exact).  No faiss, no CPU search path.

Beyond the reference surface (SURVEY.md §8f-2/3): `search_batch` returns (scores, ids) arrays
without building Python tuples, and load/save read and write the FAISS flat-index file layout
(`IxFI`) so artefacts of `scripts/build_index.py` interoperate.
"""
from __future__ import annotations

import json
import struct
from pathlib import Path
from typing import Dict, List, NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import _native, ops

# ---------------------------------------------------------------------------------------------
# FAISS flat-index file (`faiss.write_index` of an IndexFlatIP; reference call sites vector_db.py:77,117).
# faiss is not vendored under /root/reference and not installable here, so the layout below restates upstream faiss
# (faiss/impl/index_write.cpp: `write_index` -> fourcc "IxFI" for METRIC_INNER_PRODUCT, `write_index_header`
# -> d, ntotal, two dummies (1 << 20), is_trained, metric_type; then the storage as `WRITEXBVECTOR(codes)` / in
# releases before 1.7.1 `WRITEVECTOR(xb)`: a u64 count of 4-byte units followed by the raw fp32 rows; faiss/impl/io_macros.h)
# and has NOT been checked against a file written by a real faiss (see INTEGRATION.md "Before production").  The
# reader therefore refuses everything it does not recognise exactly, loudly, instead of guessing:
#   u32 fourcc "IxFI" | i32 d | i64 ntotal | i64 dummy | i64 dummy | u8 is_trained | i32 metric_type (0 = inner
#   product) | u64 n_floats (= ntotal * d) | f32[n_floats] row-major rows | end of file
_FOURCC_IXFI = struct.unpack("<I", b"IxFI")[0]
_HDR = struct.Struct("<IiqqqBiQ")   # 45 bytes, little endian, unpadded
_OTHER_FAISS_FOURCC = {b"IxF2": "IndexFlatL2", b"IxFl": "IndexFlat (other metric)", b"IwFl": "IndexIVFFlat",
                       b"IxMp": "IndexIDMap", b"IxM2": "IndexIDMap2", b"IHNf": "IndexHNSWFlat", b"IxPq": "IndexPQ",
                       b"IwPQ": "IndexIVFPQ", b"IxSQ": "IndexScalarQuantizer", b"IxPT": "IndexPreTransform"}


def write_flat_ip_file(path: str, rows: np.ndarray) -> None:
    rows = np.ascontiguousarray(rows, dtype="<f4")
    n, d = rows.shape
    with open(path, "wb") as f:
        f.write(_HDR.pack(_FOURCC_IXFI, d, n, 1 << 20, 1 << 20, 1, 0, n * d))
        f.write(rows.tobytes())


def read_flat_ip_file(path: str) -> np.ndarray:
    import os
    with open(path, "rb") as f:
        hdr = f.read(_HDR.size)
        if len(hdr) != _HDR.size:
            raise ValueError(f"{path}: truncated flat index header")
        fourcc, d, n, _, _, trained, metric, nfl = _HDR.unpack(hdr)
        if fourcc != _FOURCC_IXFI:
            tag = hdr[:4]
            kind = _OTHER_FAISS_FOURCC.get(tag)
            what = f"a faiss {kind} file" if kind else f"fourcc {tag!r}"
            raise ValueError(f"{path}: not an IndexFlatIP file ({what}); only the flat inner-product index the reference "
                             f"builds (faiss.IndexFlatIP, vector_db.py:48) is supported")
        if metric != 0 or nfl != n * d or d <= 0 or n < 0 or trained not in (0, 1):
            raise ValueError(f"{path}: inconsistent flat index header (d={d}, ntotal={n}, floats={nfl}, metric={metric}, "
                             f"is_trained={trained})")
        expect = _HDR.size + 4 * n * d
        actual = os.fstat(f.fileno()).st_size
        if actual < expect:
            raise ValueError(f"{path}: truncated flat index payload ({actual} bytes, header promises {expect})")
        if actual > expect:
            raise ValueError(f"{path}: {actual - expect} unexpected bytes after the fp32 rows - not the plain IndexFlatIP "
                             f"layout this reader knows; refusing to guess")
        data = np.fromfile(f, dtype="<f4", count=n * d)
    if data.size != n * d:
        raise ValueError(f"{path}: truncated flat index payload")
    return data.reshape(n, d)


# ---------------------------------------------------------------------------------------------
# Native shard file (SURVEY.md §8f-3): everything a rank needs to serve its block of catalog rows without
# re-normalising or re-rounding - the fp32 rows faiss would store, their bf16 shadow (pitch Dp) and the error-bound
# statistics - so an N-GPU server loads G files in parallel straight into device memory.
#   magic "TTB2SHRD" | u32 version | u32 d | u32 dp | u64 rows | u64 id_offset | u64 n_total | f32 stats[4] |
#   pad to 64 bytes | f32 xn[rows*d] | u16 xh[rows*dp]   (little endian)
_SHARD_MAGIC = b"TTB2SHRD"
_SHARD_HDR = struct.Struct("<8sIIIQQQ4f")
_SHARD_HDR_BYTES = 64


def write_native_shard(path: str, xn: np.ndarray, xh_bits: np.ndarray, stats: np.ndarray, id_offset: int = 0,
                       n_total: Optional[int] = None) -> None:
    """xn f32 [rows,d]; xh_bits u16 [rows,dp] (the bf16 bit patterns); stats f32 [4]."""
    xn = np.ascontiguousarray(xn, dtype="<f4")
    xh_bits = np.ascontiguousarray(xh_bits, dtype="<u2")
    rows, d = xn.shape
    if xh_bits.shape[0] != rows or xh_bits.shape[1] < d or xh_bits.shape[1] % 64 != 0:
        raise ValueError(f"bf16 shadow shape {xh_bits.shape} does not match rows [{rows},{d}] (pitch must be a multiple of 64)")
    st = np.asarray(stats, dtype="<f4").reshape(4)
    hdr = _SHARD_HDR.pack(_SHARD_MAGIC, 1, d, xh_bits.shape[1], rows, int(id_offset),
                          int(rows if n_total is None else n_total), *st.tolist())
    with open(path, "wb") as f:
        f.write(hdr.ljust(_SHARD_HDR_BYTES, b"\0"))
        f.write(xn.tobytes())
        f.write(xh_bits.tobytes())


def read_native_shard(path: str):
    """-> (xn f32 [rows,d], xh_bits u16 [rows,dp], stats f32 [4], id_offset, n_total); validates header and sizes."""
    with open(path, "rb") as f:
        hdr = f.read(_SHARD_HDR_BYTES)
        if len(hdr) != _SHARD_HDR_BYTES:
            raise ValueError(f"{path}: truncated shard header")
        magic, version, d, dp, rows, id_offset, n_total, s0, s1, s2, s3 = _SHARD_HDR.unpack(hdr[:_SHARD_HDR.size])
        if magic != _SHARD_MAGIC or version != 1:
            raise ValueError(f"{path}: not a tt_b200 shard file (magic {magic!r}, version {version})")
        if d <= 0 or dp < d or dp % 64 != 0 or n_total < rows:
            raise ValueError(f"{path}: inconsistent shard header (d={d}, dp={dp}, rows={rows}, n_total={n_total})")
        xn = np.fromfile(f, dtype="<f4", count=rows * d)
        xh = np.fromfile(f, dtype="<u2", count=rows * dp)
    if xn.size != rows * d or xh.size != rows * dp:
        raise ValueError(f"{path}: truncated shard payload")
    return xn.reshape(rows, d), xh.reshape(rows, dp), np.array([s0, s1, s2, s3], np.float32), int(id_offset), int(n_total)


# ---------------------------------------------------------------------------------------------
# Label filters (tt_flat_search_filtered): one u32 label word per row, masks {all, any} per query.  Both travel as int32
# tensors holding the u32 bit patterns.
_U32_LIMIT = 1 << 32


def u32_words(values, what: str):
    """Integer values in [0, 2^32) -> int32 words with the same bits: a numpy array for host input, a tensor on the same
    device for a CUDA tensor.  int32 / uint32 tensors are taken as raw words; any other integer input is range-checked
    (an int64 CUDA tensor with one device-to-host read)."""
    if isinstance(values, torch.Tensor) and values.is_cuda:
        if values.dtype == torch.int32:
            return values
        if values.dtype == torch.uint32:
            return values.view(torch.int32)
        if values.dtype != torch.int64:
            raise ValueError(f"{what} must be an integer tensor (int64, int32 or uint32), got {values.dtype}")
        if bool(((values < 0) | (values >= _U32_LIMIT)).any()):
            raise ValueError(f"{what} must be in [0, 2^32)")
        return torch.where(values >= (1 << 31), values - _U32_LIMIT, values).to(torch.int32)
    if isinstance(values, torch.Tensor):
        values = values.numpy()
    arr = np.asarray(values)
    if arr.size == 0:
        arr = arr.astype(np.int64)
    if arr.dtype == np.bool_ or not np.issubdtype(arr.dtype, np.integer):
        raise ValueError(f"{what} must hold integers in [0, 2^32), got dtype {arr.dtype}")
    if arr.size and (int(arr.min()) < 0 or int(arr.max()) >= _U32_LIMIT):
        raise ValueError(f"{what} must be in [0, 2^32), got values in [{int(arr.min())}, {int(arr.max())}]")
    return arr.astype(np.uint32).view(np.int32)          # a fresh contiguous copy (0-d input stays 0-d)


def require_masks(require_all, require_any, nq: int) -> Optional[np.ndarray]:
    """(all, any) masks, each a scalar or one value per query -> int32 words [nq, 2], or None when every query's masks
    are (0, 0) (no filter)."""
    cols = []
    for name, v in (("require_all", require_all), ("require_any", require_any)):
        w = u32_words(v, name)
        if w.ndim > 1 or (w.ndim == 1 and w.shape[0] != nq):
            raise ValueError(f"{name} must be a scalar or one value per query ({nq}), got shape {w.shape}")
        cols.append(np.broadcast_to(w, (nq,)))
    req = np.ascontiguousarray(np.stack(cols, 1))
    return req if req.any() else None


class LabelMasks(NamedTuple):
    """Label masks already validated: int32 [nq, 2] on the index's device, at least one of them not (0, 0).
    ShardedFlatIPIndex normalises `require` into this once per batch, so that the per-shard calls of that batch neither
    validate the masks again nor read them back to the host (which would stall the pipelined schedule)."""
    words: torch.Tensor


# ---------------------------------------------------------------------------------------------
# Range search helpers (host side)
def range_max_results(max_results) -> int:
    """max_results -> int in [1, TT_FLAT_RANGE_MAX_RESULTS]; anything else raises ValueError."""
    if isinstance(max_results, (bool, np.bool_)) or not isinstance(max_results, (int, np.integer)):
        raise ValueError(f"max_results must be an integer, got {type(max_results).__name__}")
    if not 1 <= int(max_results) <= _native.TT_FLAT_RANGE_MAX_RESULTS:
        raise ValueError(f"max_results must be in [1, {_native.TT_FLAT_RANGE_MAX_RESULTS}], got {max_results}")
    return int(max_results)


def range_csr(counts: np.ndarray, scores: np.ndarray, ids: np.ndarray):
    """Padded per-query range results (counts [nq]; scores / ids [nq, L], best first, (-inf, -1) tail) -> faiss's
    range_search layout (lims i64 [nq + 1], D f32 [total], I i64 [total]); query i keeps min(counts[i], L) entries."""
    counts = np.asarray(counts, np.int64)
    scores, ids = np.asarray(scores), np.asarray(ids)
    n = np.minimum(counts, scores.shape[1])
    lims = np.zeros(counts.shape[0] + 1, np.int64)
    np.cumsum(n, out=lims[1:])
    keep = np.arange(scores.shape[1])[None, :] < n[:, None]
    return lims, scores[keep].astype(np.float32), ids[keep].astype(np.int64)


def range_rerun_groups(rows: np.ndarray, need: np.ndarray, ws_bytes, budget_bytes: int):
    """The overflowed query rows of a range search, in re-run groups: ascending need, each group as large as its
    workspace ws_bytes(n_queries, largest_need) fits budget_bytes.  A row that does not fit alone forms a group of one."""
    rows = np.asarray(rows, np.int64)
    order = rows[np.argsort(np.asarray(need)[rows], kind="stable")]
    groups, cur = [], []
    for r in order.tolist():
        if cur and ws_bytes(len(cur) + 1, int(need[r])) > budget_bytes:
            groups.append(np.array(cur, np.int64))
            cur = []
        cur.append(r)
    if cur:
        groups.append(np.array(cur, np.int64))
    return groups


def _plan_slices(n: int, d: int, nq: int) -> int:
    """Catalog slices of the scan plan for nq queries (the range search keeps the top-K planner's slices)."""
    import ctypes
    out = (ctypes.c_int32 * 16)()
    _native.check(_native.load().tt_flat_plan_describe(n, d, nq, 1, out), "tt_flat_plan_describe")
    return int(out[13])


# ---------------------------------------------------------------------------------------------
class _FlagRing:
    """A few pinned int32 slots: the status words of a search (uncertified count[, exchange time-out]) are
    copied into one of them asynchronously, so the host can look at them later without draining the stream.
    The completion event is recorded on the stream of the STATUS TENSOR's device (the index's device), not on
    the calling thread's current device: a worker thread that never called set_device still waits for the right
    stream.  A slot recycled before it was read (more than `n` searches in flight) is detected and raised."""
    WIDTH = 2

    def __init__(self, n: int = 64):
        self.host = torch.zeros((n, self.WIDTH), dtype=torch.int32, pin_memory=True)
        self.n, self.next = n, 0
        self.gen = [0] * n

    def post(self, status_dev: torch.Tensor):
        slot = self.next
        self.next = (self.next + 1) % self.n
        self.gen[slot] += 1
        w = int(status_dev.numel())
        stream = torch.cuda.current_stream(status_dev.device)
        with torch.cuda.stream(stream):
            self.host[slot, :w].copy_(status_dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
        return slot, ev, w, self.gen[slot]

    def read(self, slot: int, ev, w: int = 1, gen: int = None):
        ev.synchronize()
        if gen is not None and self.gen[slot] != gen:
            raise RuntimeError(f"tt_b200: more than {self.n} searches in flight: the status slot of this search was recycled")
        vals = self.host[slot, :w].tolist()
        return vals[0] if w == 1 else vals


class PendingSearch:
    """Result of an asynchronous search.  `result()` waits for THIS search only (not for work enqueued
    after it), re-runs uncertified queries through the exact path and returns (scores, ids, n_rerun)."""

    def __init__(self, finish):
        self._finish = finish
        self._out = None

    def result(self):
        if self._out is None:
            self._out = self._finish()
            self._finish = None
        return self._out


# ---------------------------------------------------------------------------------------------
class FlatIPIndex:
    """Device-resident exact inner-product index (stands where faiss.IndexFlatIP stood).

    HBM layout: `xn` f32 [N, D] (what faiss would store) + `xh` bf16 [N, Dp] (streamed by the
    tensor-core scan, Dp = D rounded up to 64) + `stats` f32 [4] (error-bound norms).
    """

    def __init__(self, d: int, device: Optional[torch.device] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("tt_b200 FlatIPIndex needs a CUDA device (there is no CPU search path)")
        self.d = int(d)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.dp = int(_native.load().tt_flat_pitch(self.d))
        self.xn: Optional[torch.Tensor] = None
        self.xh: Optional[torch.Tensor] = None
        self._xn_store: Optional[torch.Tensor] = None     # capacity >= ntotal rows; xn / xh are its leading views
        self._xh_store: Optional[torch.Tensor] = None
        self.stats = torch.zeros(4, device=self.device, dtype=torch.float32)
        self.id_offset = 0
        self.labels: Optional[torch.Tensor] = None        # int32 [N] (u32 label words) once set_labels was called
        self._labels_store: Optional[torch.Tensor] = None
        self.groups: Optional[torch.Tensor] = None        # int32 [N] dense group ids (-1 = ungrouped) once set_groups ran
        self.n_groups = 0
        self._group_keys_store: Optional[torch.Tensor] = None   # int64 [capacity] raw keys as given to set_groups
        self._groups_store: Optional[torch.Tensor] = None
        self._ws: Dict[Tuple[int, int], torch.Tensor] = {}
        self._exact_ws: Optional[torch.Tensor] = None
        self._ring: Optional[_FlagRing] = None

    # -- size ------------------------------------------------------------------------------
    @property
    def ntotal(self) -> int:
        return 0 if self.xn is None else int(self.xn.shape[0])

    # -- build -----------------------------------------------------------------------------
    def _alloc(self, n: int) -> None:
        """Makes room for n rows.  The first build allocates exactly n rows (a 10M-row catalog must not be over-
        allocated); later `add` calls grow the storage geometrically (x1.5), so appending m batches copies
        O(total) rows instead of O(m * total)."""
        old = self.ntotal
        cap = 0 if self._xn_store is None else int(self._xn_store.shape[0])
        if n > cap:
            new_cap = n if old == 0 else max(n, cap + cap // 2)
            xn = torch.empty((new_cap, self.d), device=self.device, dtype=torch.float32)
            xh = torch.empty((new_cap, self.dp), device=self.device, dtype=torch.bfloat16)
            if old:
                xn[:old].copy_(self.xn)
                xh[:old].copy_(self.xh)
            self._xn_store, self._xh_store = xn, xh
        self.xn, self.xh = self._xn_store[:n], self._xh_store[:n]
        if self._labels_store is not None:             # labels stay aligned with the rows; new rows get 0
            if self._labels_store.shape[0] < self._xn_store.shape[0]:
                lab = torch.zeros(self._xn_store.shape[0], device=self.device, dtype=torch.int32)
                lab[:old].copy_(self._labels_store[:old])
                self._labels_store = lab
            self._labels_store[old:n].zero_()
            self.labels = self._labels_store[:n]
        if self._groups_store is not None:             # so do groups; new rows are ungrouped
            if self._groups_store.shape[0] < self._xn_store.shape[0]:
                keys = torch.full((self._xn_store.shape[0],), -1, device=self.device, dtype=torch.int64)
                keys[:old].copy_(self._group_keys_store[:old])
                dense = torch.full((self._xn_store.shape[0],), -1, device=self.device, dtype=torch.int32)
                dense[:old].copy_(self._groups_store[:old])
                self._group_keys_store, self._groups_store = keys, dense
            self._group_keys_store[old:n].fill_(-1)
            self._groups_store[old:n].fill_(-1)
            self.groups = self._groups_store[:n]
        self._ws.clear()
        self._exact_ws = None

    def _build_rows(self, row0: int, rows: int, normalize: bool) -> None:
        """Normalises xn[row0:row0+rows] in place and writes the bf16 shadow rows."""
        lib = _native.load()
        src = self.xn[row0:row0 + rows]
        with torch.cuda.device(self.device):
            _native.check(lib.tt_flat_build(src.data_ptr(), rows, self.d, 1 if normalize else 0,
                                            self.xn.data_ptr(), self.xh.data_ptr(), row0, self.stats.data_ptr(),
                                            ops._stream()), "tt_flat_build")

    def add(self, x, normalize: bool = True, chunk_rows: int = 1 << 17, labels=None) -> None:
        """Appends rows (numpy [n,d] or a torch tensor on any device).  `labels` (n values in [0, 2^32), see
        set_labels) are the new rows' label words; without them the new rows of a labelled index get 0."""
        if labels is not None:
            n_new = x.shape[0]
            words = u32_words(labels, "labels")
            if tuple(words.shape) != (n_new,):
                raise ValueError(f"expected {n_new} label words, got shape {tuple(words.shape)}")
            row0 = self.ntotal
            self.add(x, normalize, chunk_rows)
            self._store_labels(words, torch.arange(row0, row0 + n_new))
            return
        if isinstance(x, np.ndarray):
            if x.ndim != 2 or x.shape[1] != self.d:
                raise ValueError(f"expected [n, {self.d}] rows, got {x.shape}")
            n = x.shape[0]
            row0 = self.ntotal
            self._alloc(row0 + n)
            for s in range(0, n, chunk_rows):
                e = min(n, s + chunk_rows)
                host = torch.from_numpy(np.ascontiguousarray(x[s:e], dtype=np.float32))
                self.xn[row0 + s:row0 + e].copy_(host, non_blocking=False)
                self._build_rows(row0 + s, e - s, normalize)
        else:
            if x.dim() != 2 or x.shape[1] != self.d:
                raise ValueError(f"expected [n, {self.d}] rows, got {tuple(x.shape)}")
            n = x.shape[0]
            row0 = self.ntotal
            self._alloc(row0 + n)
            for s in range(0, n, chunk_rows):
                e = min(n, s + chunk_rows)
                self.xn[row0 + s:row0 + e].copy_(x[s:e].to(torch.float32))
                self._build_rows(row0 + s, e - s, normalize)

    @classmethod
    def adopt(cls, xn: torch.Tensor, normalize: bool = True, chunk_rows: int = 1 << 20) -> "FlatIPIndex":
        """Takes ownership of a CUDA f32 [N,D] tensor and normalises it in place (no second fp32 copy;
        used for catalogs generated or loaded directly on the device)."""
        if not (xn.is_cuda and xn.dtype == torch.float32 and xn.dim() == 2 and xn.is_contiguous()):
            raise ValueError("adopt() needs a contiguous CUDA float32 [N,D] tensor")
        self = cls(xn.shape[1], xn.device)
        self.xn = self._xn_store = xn
        self.xh = self._xh_store = torch.empty((xn.shape[0], self.dp), device=xn.device, dtype=torch.bfloat16)
        for s in range(0, xn.shape[0], chunk_rows):
            self._build_rows(s, min(chunk_rows, xn.shape[0] - s), normalize)
        return self

    def save_native(self, path: str, n_total: Optional[int] = None) -> None:
        """Writes this index (one rank's shard) as a native shard file: no re-normalisation on load."""
        write_native_shard(path, self.xn.cpu().numpy(), self.xh.view(torch.int16).cpu().numpy().view(np.uint16),
                           self.stats.cpu().numpy(), self.id_offset, n_total)

    @classmethod
    def load_native(cls, path: str, device: Optional[torch.device] = None) -> "FlatIPIndex":
        """Loads a native shard file straight into device memory (rows, bf16 shadow and statistics as stored)."""
        xn, xh, stats, id_offset, _ = read_native_shard(path)
        self = cls(xn.shape[1], device)
        if xh.shape[1] != self.dp:
            raise ValueError(f"{path}: bf16 pitch {xh.shape[1]} does not match this build's pitch {self.dp}")
        self.xn = self._xn_store = torch.from_numpy(xn).to(self.device)
        self.xh = self._xh_store = torch.from_numpy(xh.view(np.int16)).to(self.device).view(torch.bfloat16)
        self.stats = torch.from_numpy(stats).to(self.device)
        self.id_offset = id_offset
        return self

    # -- label words -----------------------------------------------------------------------
    def set_labels(self, labels, rows=None) -> None:
        """Sets the u32 label word of every row (`labels` [ntotal]), or of the listed `rows` only (in-place update;
        `labels` then has one value per listed row).  numpy or CUDA input, values in [0, 2^32); int32 / uint32 tensors
        are taken as raw words.  Stream-ordered: a search enqueued after this call sees the new words.  Rows that never
        got a label have the word 0.  Labels are serving state: save / load do not store them."""
        if self.ntotal == 0:
            raise ValueError("empty index")
        words = u32_words(labels, "labels")
        if rows is None:
            if tuple(words.shape) != (self.ntotal,):
                raise ValueError(f"expected one label word per row ({self.ntotal}), got shape {tuple(words.shape)}")
        else:
            r = rows if isinstance(rows, torch.Tensor) else torch.from_numpy(np.asarray(rows))
            if r.dim() != 1 or r.dtype not in (torch.int64, torch.int32) or tuple(words.shape) != (r.shape[0],):
                raise ValueError(f"rows must be a 1-D integer array with one entry per label word, got rows "
                                 f"{r.dtype} {tuple(r.shape)} and labels {tuple(words.shape)}")
            if r.numel() and (int(r.min()) < 0 or int(r.max()) >= self.ntotal):
                raise ValueError(f"rows must be in [0, {self.ntotal})")
        self._store_labels(words, None if rows is None else r)

    def _store_labels(self, words, rows: Optional[torch.Tensor]) -> None:
        """Writes validated int32 words (numpy or CUDA) to all rows, or to the given rows."""
        w = torch.from_numpy(words) if isinstance(words, np.ndarray) else words
        with torch.cuda.device(self.device):
            if self._labels_store is None:
                self._labels_store = torch.zeros(self._xn_store.shape[0], device=self.device, dtype=torch.int32)
                self.labels = self._labels_store[:self.ntotal]
            if rows is None:
                self.labels.copy_(w.to(self.device))
            else:
                self.labels.index_copy_(0, rows.to(self.device, torch.int64), w.to(self.device))

    # -- groups --------------------------------------------------------------------------------
    def set_groups(self, keys, rows=None) -> None:
        """Sets the group key (a brand, a seller) of every row (`keys` [ntotal]), or of the listed `rows` only (`keys`
        then has one value per listed row): int64 values, numpy or CUDA.  A negative key means ungrouped.  Keys may be
        sparse (64-bit seller ids): the index renumbers the non-negative keys of all rows densely on every call.  A
        search with `max_per_group=m` returns at most m rows of one group.  Rows added later are ungrouped.  Groups are
        serving state: save / load do not store them."""
        if self.ntotal == 0:
            raise ValueError("empty index")
        k = keys if isinstance(keys, torch.Tensor) else torch.from_numpy(np.asarray(keys))
        if k.dtype not in (torch.int64, torch.int32, torch.int16, torch.int8, torch.uint8):
            raise ValueError(f"group keys must be integers, got {k.dtype}")
        if rows is None:
            if tuple(k.shape) != (self.ntotal,):
                raise ValueError(f"expected one group key per row ({self.ntotal}), got shape {tuple(k.shape)}")
        else:
            r = rows if isinstance(rows, torch.Tensor) else torch.from_numpy(np.asarray(rows))
            if r.dim() != 1 or r.dtype not in (torch.int64, torch.int32) or tuple(k.shape) != (r.shape[0],):
                raise ValueError(f"rows must be a 1-D integer array with one entry per group key, got rows "
                                 f"{r.dtype} {tuple(r.shape)} and keys {tuple(k.shape)}")
            if r.numel() and (int(r.min()) < 0 or int(r.max()) >= self.ntotal):
                raise ValueError(f"rows must be in [0, {self.ntotal})")
        k = k.to(self.device, torch.int64)
        with torch.cuda.device(self.device):
            if self._group_keys_store is None:
                cap = self._xn_store.shape[0]
                self._group_keys_store = torch.full((cap,), -1, device=self.device, dtype=torch.int64)
                self._groups_store = torch.full((cap,), -1, device=self.device, dtype=torch.int32)
            raw = self._group_keys_store[:self.ntotal]
            if rows is None:
                raw.copy_(k)
            else:
                raw.index_copy_(0, r.to(self.device, torch.int64), k)
            grouped = raw >= 0
            uniq, inv = torch.unique(raw[grouped], return_inverse=True)
            dense = self._groups_store[:self.ntotal]
            dense.fill_(-1)
            dense[grouped] = inv.to(torch.int32)
            self.groups = dense
            self.n_groups = int(uniq.numel())

    def _group_cap(self, max_per_group) -> Optional[int]:
        """Validates a per-group cap -> the int, or None (no cap: the plain search runs)."""
        if max_per_group is None:
            return None
        if isinstance(max_per_group, (bool, np.bool_)) or not isinstance(max_per_group, (int, np.integer)):
            raise ValueError(f"max_per_group must be an int, got {type(max_per_group).__name__}")
        if not 1 <= int(max_per_group) <= _native.TT_FLAT_MAX_PER_GROUP:
            raise ValueError(f"max_per_group must be in [1, {_native.TT_FLAT_MAX_PER_GROUP}], got {max_per_group}")
        if self.groups is None:
            raise ValueError("a group cap needs group keys: call set_groups() first")
        return int(max_per_group)

    def _requires(self, require, nq: int) -> Optional[torch.Tensor]:
        """Validates per-query label masks (CUDA or numpy [nq, 2] = {all, any}, or [2] for every query) -> int32 [nq, 2]
        on this device, or None when every query's masks are (0, 0): the unfiltered search runs."""
        if require is None:
            return None
        if isinstance(require, LabelMasks):
            w = require.words
            if tuple(w.shape) != (nq, 2) or w.dtype != torch.int32 or w.device != self.device or not w.is_contiguous():
                raise ValueError(f"LabelMasks must hold contiguous int32 [nq={nq}, 2] words on {self.device}, got "
                                 f"{w.dtype} {tuple(w.shape)} on {w.device}")
            if self.labels is None:
                raise ValueError("a label filter needs label words: call set_labels() first")
            return w
        w = u32_words(require, "require")
        if tuple(w.shape) not in ((2,), (nq, 2)):
            raise ValueError(f"require must be [nq={nq}, 2] or [2] ({{all, any}} masks), got shape {tuple(w.shape)}")
        if not bool(w.any()):
            return None
        if self.labels is None:
            raise ValueError("a label filter needs label words: call set_labels() first")
        if isinstance(w, np.ndarray):
            w = torch.from_numpy(w)
        return w.to(self.device).expand(nq, 2).contiguous()

    def rows_host(self) -> np.ndarray:
        """The stored fp32 rows (what faiss.write_index would serialise)."""
        return self.xn.cpu().numpy()

    # -- search ----------------------------------------------------------------------------
    def _exclusions(self, exclude, nq: int) -> Optional[torch.Tensor]:
        """Validates an exclusion list (CUDA i64 [nq, E], ids in this index's result id space, -1 padded) -> the
        contiguous tensor, or None when there is nothing to exclude (E == 0 runs the plain search)."""
        if exclude is None:
            return None
        if not (isinstance(exclude, torch.Tensor) and exclude.is_cuda and exclude.dtype == torch.int64
                and exclude.dim() == 2 and exclude.shape[0] == nq):
            raise ValueError(f"exclude must be a CUDA int64 tensor [nq={nq}, E], got "
                             f"{getattr(exclude, 'dtype', type(exclude))} {tuple(getattr(exclude, 'shape', ()))}")
        if exclude.shape[1] > _native.TT_FLAT_MAX_EXCLUDE:
            raise ValueError(f"at most {_native.TT_FLAT_MAX_EXCLUDE} exclusions per query, got {exclude.shape[1]}")
        if exclude.shape[1] == 0:
            return None
        return exclude.to(self.device).contiguous()

    def _workspace(self, nq: int, k: int, n_excl: int = 0) -> torch.Tensor:
        key = (nq, k) if n_excl == 0 else (nq, k, "excl", n_excl)
        ws = self._ws.get(key)
        if ws is None:
            lib = _native.load()
            nbytes = int(lib.tt_flat_search_workspace_bytes(self.ntotal, self.d, nq, k) if n_excl == 0 else
                         lib.tt_flat_search_excl_workspace_bytes(self.ntotal, self.d, nq, k, n_excl))
            ws = torch.empty(max(nbytes, 256), device=self.device, dtype=torch.uint8)
            if len(self._ws) > 8:
                self._ws.clear()
            self._ws[key] = ws
        return ws

    def _group_workspace(self, nq: int, k: int, n_excl: int) -> torch.Tensor:
        key = (nq, k, "group", n_excl, self.n_groups)
        ws = self._ws.get(key)
        if ws is None:
            nbytes = int(_native.load().tt_flat_search_grouped_workspace_bytes(self.ntotal, self.d, nq, k, n_excl,
                                                                               self.n_groups))
            ws = torch.empty(max(nbytes, 256), device=self.device, dtype=torch.uint8)
            if len(self._ws) > 8:
                self._ws.clear()
            self._ws[key] = ws
        return ws

    def search_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None, require=None,
                      max_per_group: Optional[int] = None):
        """Asynchronous search of CUDA f32 queries [nq,D] on the current stream.

        Returns (scores [nq,k] f32, ids [nq,k] i64, flags [nq] i32, n_uncertified [1] i32) device
        tensors; rows with flags != 1 (1 = certified exact, <= 0 = -(reason bits), see include/tt_b200.h) must be
        passed to `search_exact_device` (`search_checked_device` / `search_async` do both).
        `exclude` (CUDA i64 [nq, E], E <= 1024, ids as returned, -1 = padding): the top-k over the rows query i does
        not list in exclude[i]; with fewer than k allowed rows the tail is (-inf, -1).
        `require` (CUDA or numpy [nq, 2] = {all, any} u32 masks, or [2] for every query): only rows whose label word
        has every bit of `all` and, unless any == 0, one bit of `any` (see set_labels); composes with `exclude`.
        `max_per_group` (int in [1, 64], needs set_groups): at most that many rows of one group, taken best first; the
        rows a group cannot take make room for the next best rows (see tt_flat_search_grouped).
        """
        if self.ntotal == 0:
            raise ValueError("empty index")
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected queries [nq, {self.d}], got {tuple(q.shape)}")
        if not 1 <= k <= min(self.ntotal, _native.TT_FLAT_MAX_K):
            raise ValueError(f"k must be in [1, min(ntotal, {_native.TT_FLAT_MAX_K})], got {k}")
        req = self._requires(require, q.shape[0])
        cap = self._group_cap(max_per_group)
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        scores = torch.empty((nq, k), device=self.device, dtype=torch.float32)
        ids = torch.empty((nq, k), device=self.device, dtype=torch.int64)
        flags = torch.empty((max(nq, 1),), device=self.device, dtype=torch.int32)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if cap is not None:
                E = 0 if excl is None else excl.shape[1]
                ws = self._group_workspace(max(nq, 1), k, E)
                _native.check(lib.tt_flat_search_grouped(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, scores.data_ptr(), ids.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    self.groups.data_ptr(), self.n_groups, cap, 0 if req is None else self.labels.data_ptr(),
                    0 if req is None else req.data_ptr(), 0 if excl is None else excl.data_ptr(), E, ws.data_ptr(),
                    ws.numel(), ops._stream()), "tt_flat_search_grouped")
            elif req is not None:
                E = 0 if excl is None else excl.shape[1]
                ws = self._workspace(max(nq, 1), k, E)
                _native.check(lib.tt_flat_search_filtered(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, scores.data_ptr(), ids.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    self.labels.data_ptr(), req.data_ptr(), 0 if excl is None else excl.data_ptr(), E, ws.data_ptr(),
                    ws.numel(), ops._stream()), "tt_flat_search_filtered")
            elif excl is None:
                ws = self._workspace(max(nq, 1), k)
                _native.check(lib.tt_flat_search(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, scores.data_ptr(), ids.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_search")
            else:
                E = excl.shape[1]
                ws = self._workspace(max(nq, 1), k, E)
                _native.check(lib.tt_flat_search_excl(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, scores.data_ptr(), ids.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    excl.data_ptr(), E, ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_search_excl")
        return scores, ids, flags[:nq], nunc

    def search_exact_device(self, q: torch.Tensor, k: int, scores: Optional[torch.Tensor] = None,
                            ids: Optional[torch.Tensor] = None, qsel: Optional[torch.Tensor] = None, *,
                            exclude: Optional[torch.Tensor] = None, require=None, max_per_group: Optional[int] = None):
        """Always-exact fp32 path; with `qsel` (i32 query rows) only those rows of scores/ids are rewritten.
        `exclude` [nq, E] and `require` [nq, 2] are indexed by query row (qsel[i]), as in search_device;
        `max_per_group` as in search_device."""
        req = self._requires(require, q.shape[0])
        cap = self._group_cap(max_per_group)
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        if scores is None:
            scores = torch.empty((nq, k), device=self.device, dtype=torch.float32)
            ids = torch.empty((nq, k), device=self.device, dtype=torch.int64)
        nsel = nq if qsel is None else int(qsel.numel())
        lib = _native.load()
        need = int(lib.tt_flat_search_exact_workspace_bytes(self.ntotal, self.d, nsel, k) if cap is None else
                   lib.tt_flat_search_exact_grouped_workspace_bytes(self.ntotal, self.d, nsel, k, self.n_groups))
        if self._exact_ws is None or self._exact_ws.numel() < need:
            self._exact_ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        with torch.cuda.device(self.device):
            if cap is not None:
                _native.check(lib.tt_flat_search_exact_grouped(
                    q.data_ptr(), nq, 0 if qsel is None else qsel.data_ptr(), nsel, self.xn.data_ptr(), self.ntotal,
                    self.d, k, self.id_offset, scores.data_ptr(), ids.data_ptr(),
                    0 if req is None else self.labels.data_ptr(), 0 if req is None else req.data_ptr(),
                    0 if excl is None else excl.data_ptr(), 0 if excl is None else excl.shape[1],
                    self.groups.data_ptr(), self.n_groups, cap, self._exact_ws.data_ptr(), self._exact_ws.numel(),
                    ops._stream()), "tt_flat_search_exact_grouped")
            elif req is not None:
                _native.check(lib.tt_flat_search_exact_filtered(
                    q.data_ptr(), nq, 0 if qsel is None else qsel.data_ptr(), nsel, self.xn.data_ptr(), self.ntotal,
                    self.d, k, self.id_offset, scores.data_ptr(), ids.data_ptr(), self.labels.data_ptr(), req.data_ptr(),
                    0 if excl is None else excl.data_ptr(), 0 if excl is None else excl.shape[1],
                    self._exact_ws.data_ptr(), self._exact_ws.numel(), ops._stream()), "tt_flat_search_exact_filtered")
            elif excl is None:
                _native.check(lib.tt_flat_search_exact(
                    q.data_ptr(), nq, 0 if qsel is None else qsel.data_ptr(), nsel, self.xn.data_ptr(), self.ntotal,
                    self.d, k, self.id_offset, scores.data_ptr(), ids.data_ptr(), self._exact_ws.data_ptr(),
                    self._exact_ws.numel(), ops._stream()), "tt_flat_search_exact")
            else:
                _native.check(lib.tt_flat_search_exact_excl(
                    q.data_ptr(), nq, 0 if qsel is None else qsel.data_ptr(), nsel, self.xn.data_ptr(), self.ntotal,
                    self.d, k, self.id_offset, scores.data_ptr(), ids.data_ptr(), excl.data_ptr(), excl.shape[1],
                    self._exact_ws.data_ptr(), self._exact_ws.numel(), ops._stream()), "tt_flat_search_exact_excl")
        return scores, ids

    def search_shard_into(self, q: torch.Tensor, k: int, scores: torch.Tensor, ids: torch.Tensor,
                          bound: torch.Tensor, flags: torch.Tensor, *, exclude: Optional[torch.Tensor] = None,
                          require=None) -> None:
        """Shard-local search for ShardedFlatIPIndex (tt_flat_search_shard): fills the caller's record views.
        scores/ids are [nq, k_record] with k_record >= k; only the first k columns of each row are written.
        `exclude` holds GLOBAL ids (ids of other shards are ignored here); `require`: label masks as in search_device,
        tested against this shard's label words."""
        req = self._requires(require, q.shape[0])
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        direct = scores.shape[1] == k and scores.is_contiguous() and ids.is_contiguous()
        s_out = scores if direct else torch.empty((nq, k), device=self.device, dtype=torch.float32)
        i_out = ids if direct else torch.empty((nq, k), device=self.device, dtype=torch.int64)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if req is not None:
                E = 0 if excl is None else excl.shape[1]
                ws = self._workspace(max(nq, 1), k, E)
                _native.check(lib.tt_flat_search_shard_filtered(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, s_out.data_ptr(), i_out.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    bound.data_ptr(), self.labels.data_ptr(), req.data_ptr(), 0 if excl is None else excl.data_ptr(), E,
                    ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_search_shard_filtered")
            elif excl is None:
                ws = self._workspace(max(nq, 1), k)
                _native.check(lib.tt_flat_search_shard(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, s_out.data_ptr(), i_out.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    bound.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_search_shard")
            else:
                ws = self._workspace(max(nq, 1), k, excl.shape[1])
                _native.check(lib.tt_flat_search_shard_excl(
                    q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                    k, self.id_offset, s_out.data_ptr(), i_out.data_ptr(), flags.data_ptr(), nunc.data_ptr(),
                    bound.data_ptr(), excl.data_ptr(), excl.shape[1], ws.data_ptr(), ws.numel(), ops._stream()),
                    "tt_flat_search_shard_excl")
        if not direct:
            scores[:, :k].copy_(s_out)
            ids[:, :k].copy_(i_out)

    def search_exact_into(self, q: torch.Tensor, k: int, scores: torch.Tensor, ids: torch.Tensor,
                          qsel: torch.Tensor, *, exclude: Optional[torch.Tensor] = None, require=None) -> None:
        """Exact fp32 re-run of the query rows `qsel`, written into [nq, k_record] record views."""
        kw = {} if exclude is None else {"exclude": exclude}
        if require is not None:
            kw["require"] = require
        if scores.shape[1] == k and scores.is_contiguous() and ids.is_contiguous():
            self.search_exact_device(q, k, scores, ids, qsel, **kw)
            return
        s_tmp, i_tmp = self.search_exact_device(q, k, **kw)
        rows = qsel.long()
        scores[rows, :k] = s_tmp[rows]
        ids[rows, :k] = i_tmp[rows]

    def scan_scores_device(self, q: torch.Tensor) -> torch.Tensor:
        """Diagnostic: dense bf16 tensor-core scores [nq, N] exactly as the scan epilogue sees them
        (tt_flat_scan_scores; small catalogs only).  Rows never reported by the kernel read NaN."""
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        lib = _native.load()
        need = int(lib.tt_flat_scan_scores_workspace_bytes(self.ntotal, self.d, nq))
        ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        out = torch.empty((nq, self.ntotal), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            _native.check(lib.tt_flat_scan_scores(q.data_ptr(), nq, self.xh.data_ptr(), self.stats.data_ptr(),
                                                  self.ntotal, self.d, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                                  ops._stream()), "tt_flat_scan_scores")
        return out

    def search_async(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None,
                     require=None, max_per_group: Optional[int] = None) -> PendingSearch:
        """Enqueues a search and returns at once; `.result()` checks the certificate later, so a caller can
        keep the next batch's kernels queued behind this one (no idle GPU between batches).  `exclude`, `require`:
        see search_device; uncertified queries are re-run exactly with the same lists and masks.  (Masks in a CUDA
        tensor cost one device-to-host read to tell a filter from (0, 0); numpy masks cost none.)  `max_per_group`: see
        search_device; the re-runs keep the cap."""
        kw = {} if exclude is None else {"exclude": exclude}
        if require is not None:
            kw["require"] = require
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        scores, ids, flags, nunc = self.search_device(q, k, **kw)
        if self._ring is None:
            self._ring = _FlagRing()
        token = self._ring.post(nunc)

        def finish():
            n_bad = self._ring.read(*token)
            if n_bad:
                qsel = torch.nonzero(flags != 1).flatten().to(torch.int32)
                self.search_exact_device(q, k, scores, ids, qsel, **kw)
            return scores, ids, n_bad
        return PendingSearch(finish)

    def search_checked_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None, require=None,
                              max_per_group: Optional[int] = None):
        """search_device + re-run of uncertified queries through the exact path (one host sync)."""
        return self.search_async(q, k, exclude=exclude, require=require, max_per_group=max_per_group).result()

    # -- range search (tt_flat_range_search) -----------------------------------------------------
    # Bytes of workspace one range call takes at most: the first pass sizes its candidate budget to fit, and the
    # re-runs of overflowed queries run in groups that fit.
    RANGE_WS_BUDGET = 2 << 30

    def _radii(self, radius, nq: int) -> torch.Tensor:
        """A Python float (every query), or a numpy / CUDA [nq] array -> contiguous f32 [nq] on this device.  A bad shape
        or a non-finite radius (after the cast to f32) raises ValueError; a CUDA radius costs one device-to-host read."""
        if isinstance(radius, torch.Tensor):
            if radius.dim() != 1 or radius.shape[0] != nq or radius.dtype == torch.bool or radius.is_complex():
                raise ValueError(f"radius must be a float or a real [nq={nq}] array, got {radius.dtype} {tuple(radius.shape)}")
            r = radius.to(self.device, torch.float32).contiguous()
            if not bool(torch.isfinite(r).all()):
                raise ValueError("radius must be finite")
            return r
        a = np.asarray(radius) if not isinstance(radius, (float, int)) or isinstance(radius, bool) else np.float64(radius)
        if a.shape not in ((), (nq,)) or a.dtype == np.bool_ or not np.issubdtype(a.dtype, np.number) \
                or np.issubdtype(a.dtype, np.complexfloating):
            raise ValueError(f"radius must be a float or a real [nq={nq}] array, got {a.dtype} {a.shape}")
        with np.errstate(over="ignore"):                   # beyond the f32 range: inf, rejected below
            r = np.broadcast_to(a.astype(np.float32), (nq,)).copy()
        if not np.isfinite(r).all():
            raise ValueError("radius must be finite")
        return torch.from_numpy(r).to(self.device)

    def _range_args(self, q, radius, max_results, exclude, require):
        """Validates a range search before anything is launched -> (q, radius f32 [nq], L, exclude, masks)."""
        if self.ntotal == 0:
            raise ValueError("empty index")
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected queries [nq, {self.d}], got {tuple(q.shape)}")
        L = range_max_results(max_results)
        req = self._requires(require, q.shape[0])
        rad = self._radii(radius, q.shape[0])
        q = ops._f32c(q, "queries")
        return q, rad, L, self._exclusions(exclude, q.shape[0]), req

    def _range_workspace(self, nq: int, budget: int, cache: bool = True) -> torch.Tensor:
        """The workspace of a range call; cache=False (the re-runs, whose budgets vary with each batch) allocates one that
        is freed with the call instead of staying in the workspace cache."""
        key = ("range", nq, budget)
        ws = self._ws.get(key) if cache else None
        if ws is None:
            nbytes = int(_native.load().tt_flat_range_workspace_bytes(self.ntotal, self.d, nq, budget))
            ws = torch.empty(max(nbytes, 256), device=self.device, dtype=torch.uint8)
            if cache:
                if len(self._ws) > 8:
                    self._ws.clear()
                self._ws[key] = ws
        return ws

    def _rerun_budget(self, n: int, need: int, first_slices: int) -> int:
        """Candidate budget of a re-run of n overflowed queries whose fullest segment held `need` candidates in a first
        pass over `first_slices` catalog slices.  The re-run's plan slices the catalog for n queries, often into more
        slices; its segments (2 x budget / slices) must hold at least need candidates, and as many as the first pass's
        total for that query (at most need x first_slices) spread over the re-run's slices."""
        return need * max(first_slices, _plan_slices(self.ntotal, self.d, n))

    def _range_budget(self, nq: int, L: int) -> int:
        """Candidates per query the first pass makes room for: 2L, at least 16384, halved until the workspace fits."""
        lib = _native.load()
        b = max(2 * L, 16384)
        while b > 64 and lib.tt_flat_range_workspace_bytes(self.ntotal, self.d, nq, b) > self.RANGE_WS_BUDGET:
            b //= 2
        return b

    def _range_launch(self, q, rad, L: int, excl, req, budget: int, cache: bool = True, out=None):
        """`out`: the caller's contiguous (counts [nq], scores [nq, L], ids [nq, L], flags [nq]) to write into (nq >= 1)."""
        nq = q.shape[0]
        if out is not None:
            counts, scores, ids, flags = out
        else:
            counts = torch.empty((nq,), device=self.device, dtype=torch.int64)
            scores = torch.empty((nq, L), device=self.device, dtype=torch.float32)
            ids = torch.empty((nq, L), device=self.device, dtype=torch.int64)
            flags = torch.empty((max(nq, 1),), device=self.device, dtype=torch.int32)
        need = torch.empty((max(nq, 1),), device=self.device, dtype=torch.int32)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        ws = self._range_workspace(max(nq, 1), budget, cache)
        lib = _native.load()
        with torch.cuda.device(self.device):
            _native.check(lib.tt_flat_range_search(
                q.data_ptr(), nq, self.xn.data_ptr(), self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, self.d,
                rad.data_ptr(), L, self.id_offset, counts.data_ptr(), scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                need.data_ptr(), nunc.data_ptr(), 0 if req is None else self.labels.data_ptr(),
                0 if req is None else req.data_ptr(), 0 if excl is None else excl.data_ptr(),
                0 if excl is None else excl.shape[1], ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_range_search")
        return counts, scores, ids, flags[:nq], need[:nq], nunc

    def _range_exact(self, q, rad, L: int, excl, req, counts, scores, ids, qsel: torch.Tensor) -> None:
        """Exact fp32 re-run of the query rows qsel (i32, on this device) into counts / scores / ids."""
        lib = _native.load()
        nsel = int(qsel.numel())
        need = int(lib.tt_flat_range_exact_workspace_bytes(self.ntotal, self.d, nsel, L))
        if self._exact_ws is None or self._exact_ws.numel() < need:
            self._exact_ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        with torch.cuda.device(self.device):
            _native.check(lib.tt_flat_range_search_exact(
                q.data_ptr(), q.shape[0], qsel.data_ptr(), nsel, self.xn.data_ptr(), self.ntotal, self.d, rad.data_ptr(), L,
                self.id_offset, counts.data_ptr(), scores.data_ptr(), ids.data_ptr(),
                0 if req is None else self.labels.data_ptr(), 0 if req is None else req.data_ptr(),
                0 if excl is None else excl.data_ptr(), 0 if excl is None else excl.shape[1], self._exact_ws.data_ptr(),
                self._exact_ws.numel(), ops._stream()), "tt_flat_range_search_exact")

    def range_search_device(self, q: torch.Tensor, radius, max_results: int, *, exclude: Optional[torch.Tensor] = None,
                            require=None):
        """Asynchronous range search of CUDA f32 queries [nq, D] on the current stream: every row whose fp32 score is
        strictly greater than `radius` (a float, or a numpy / CUDA [nq] array; finite).

        Returns (counts [nq] i64, scores [nq, L] f32, ids [nq, L] i64, flags [nq] i32, need [nq] i32,
        n_uncertified [1] i32) device tensors, L = max_results (1 <= L <= 16384): counts[i] rows qualify, the best
        min(counts[i], L) of them come first (score desc, id asc), the tail is (-inf, -1).  Rows with flags != 1 are not
        certified (see include/tt_b200.h); `range_search_async` re-runs them.  `exclude` and `require` as in
        search_device: excluded and disallowed rows are never returned and never counted."""
        q, rad, L, excl, req = self._range_args(q, radius, max_results, exclude, require)
        return self._range_launch(q, rad, L, excl, req, self._range_budget(max(q.shape[0], 1), L))

    def range_search_async(self, q: torch.Tensor, radius, max_results: int = _native.TT_FLAT_RANGE_MAX_RESULTS, *,
                           exclude: Optional[torch.Tensor] = None, require=None) -> PendingSearch:
        """range_search_device, then `.result()` -> (counts, scores, ids, n_rerun_tensor, n_rerun_exact) with every query
        certified: queries whose candidates overflowed their segments are re-run through the tensor-core path with
        segments sized from `need`, in groups whose workspace fits RANGE_WS_BUDGET; a query that alone does not fit, and
        every other uncertified query, is re-run through the exact fp32 path with the same masks and list."""
        q, rad, L, excl, req = self._range_args(q, radius, max_results, exclude, require)
        nq = q.shape[0]
        counts, scores, ids, flags, need, nunc = self._range_launch(q, rad, L, excl, req,
                                                                    self._range_budget(max(nq, 1), L))
        if self._ring is None:
            self._ring = _FlagRing()
        token = self._ring.post(nunc)

        def finish():
            if not self._ring.read(*token):
                return counts, scores, ids, 0, 0
            n_tensor, n_exact = self.range_rerun(q, rad, L, excl, req, counts, scores, ids, flags, need)
            return counts, scores, ids, n_tensor, n_exact
        return PendingSearch(finish)

    def range_rerun(self, q, rad, L: int, excl, req, counts, scores, ids, flags, need, rows=None):
        """Completes a first range pass in place: the uncertified queries among `rows` (numpy query rows; None = all) are
        re-run through the tensor-core path with segments sized from `need`, in groups whose workspace fits
        RANGE_WS_BUDGET; a query that alone does not fit, and every other uncertified query, through the exact fp32 path.
        The completed rows' flags are set to 1.  q, rad, excl, req are the validated first-pass arguments (see _range_args) -> (n_rerun_tensor, n_rerun_exact)."""
        nq = q.shape[0]
        fl, nd = flags.cpu().numpy(), need.cpu().numpy()
        bad = fl != 1
        if rows is not None:
            sel_rows = np.zeros(nq, bool)
            sel_rows[np.asarray(rows, np.int64)] = True
            bad &= sel_rows
        over = np.flatnonzero(bad & ((-fl) & 1 == 1))
        exact = [np.flatnonzero(bad & ((-fl) & 1 == 0))]
        lib = _native.load()
        first_slices = _plan_slices(self.ntotal, self.d, max(nq, 1))

        def ws_bytes(n, need_max):
            return int(lib.tt_flat_range_workspace_bytes(self.ntotal, self.d, n,
                                                         self._rerun_budget(n, need_max, first_slices)))
        n_tensor = 0
        for g in range_rerun_groups(over, nd, ws_bytes, self.RANGE_WS_BUDGET):
            need_max = int(nd[g].max())
            if g.size == 1 and ws_bytes(1, need_max) > self.RANGE_WS_BUDGET:
                exact.append(g)
                continue
            sel = torch.from_numpy(g).to(self.device)
            c2, s2, i2, f2, _, _ = self._range_launch(
                q[sel].contiguous(), rad[sel].contiguous(), L, None if excl is None else excl[sel].contiguous(),
                None if req is None else req[sel].contiguous(), self._rerun_budget(g.size, need_max, first_slices),
                cache=False)
            ok = f2 == 1
            counts[sel[ok]], scores[sel[ok]], ids[sel[ok]] = c2[ok], s2[ok], i2[ok]
            exact.append(g[~ok.cpu().numpy()])
            n_tensor += g.size
        rows = np.concatenate(exact)
        if rows.size:
            self._range_exact(q, rad, L, excl, req, counts, scores, ids,
                              torch.from_numpy(rows.astype(np.int32)).to(self.device))
        done = np.flatnonzero(bad)
        if done.size:
            flags[torch.from_numpy(done).to(self.device)] = 1       # every completed row is now exact
        return n_tensor, int(rows.size)

    def range_shard_into(self, q: torch.Tensor, rad: torch.Tensor, L: int, counts, scores, ids, flags, *,
                         exclude: Optional[torch.Tensor] = None, require=None) -> torch.Tensor:
        """First pass of ShardedFlatIPIndex.range_search_async over this shard's rows, written into the caller's record
        views (counts [nq], scores / ids [nq, L], flags [nq], contiguous; nq >= 1) -> need [nq].  `rad`: validated f32
        [nq] radii on this device (no host read here); `exclude`: GLOBAL ids; `require`: label masks (a LabelMasks
        costs no host read).  Ids are row + id_offset."""
        req = self._requires(require, q.shape[0])
        q = ops._f32c(q, "queries")
        excl = self._exclusions(exclude, q.shape[0])
        return self._range_launch(q, rad, L, excl, req, self._range_budget(q.shape[0], L),
                                  out=(counts, scores, ids, flags))[4]

    def range_search(self, q: np.ndarray, radius, max_results: int = _native.TT_FLAT_RANGE_MAX_RESULTS, *,
                     exclude: Optional[np.ndarray] = None, require=None):
        """Host-to-host range search, the shape of faiss `index.range_search(q, radius)`: q f32 [nq, d] (un-normalised)
        -> (lims i64 [nq + 1], D f32 [total], I i64 [total]); query i's rows are I[lims[i]:lims[i+1]], best first, at
        most max_results of them (range_search_device's counts tell whether more qualified).  A row is returned iff its
        fp32 score is strictly greater than the radius (a float or one per query).  `exclude`: numpy int64 [nq, E] ids
        to leave out per query (-1 = padding); `require`: label masks as in search."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        if q.ndim != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected queries [nq, {self.d}], got {q.shape}")
        kw = {}
        if exclude is not None:
            exclude = np.ascontiguousarray(exclude, dtype=np.int64)
            if exclude.ndim != 2 or exclude.shape[0] != q.shape[0]:
                raise ValueError(f"expected exclusions [nq={q.shape[0]}, E], got {exclude.shape}")
            kw["exclude"] = torch.from_numpy(exclude).to(self.device)
        with torch.cuda.device(self.device):
            dq = torch.from_numpy(q).to(self.device)
            counts, scores, ids, _, _ = self.range_search_async(dq, radius, max_results, require=require, **kw).result()
            return range_csr(counts.cpu().numpy(), scores.cpu().numpy(), ids.cpu().numpy())

    def post_flag(self, nunc_dev: torch.Tensor):
        if self._ring is None:
            self._ring = _FlagRing()
        return self._ring.post(nunc_dev)

    def read_flag(self, token) -> int:
        return self._ring.read(*token)

    # -- sharded catalogs: one threshold for the whole catalog (tt_flat_shard_*) ---------------------
    def shard_plan_ok(self, n_total: int, nq: int, k: int, n_local_min: int) -> bool:
        return bool(_native.load().tt_flat_shard_plan_ok(int(n_local_min), int(n_total), self.d, int(nq), int(k)))

    def _shard_workspace(self, n_total: int, nq: int, k: int, slot: int = 0) -> torch.Tensor:
        key = ("shard", n_total, nq, k, slot)
        ws = self._ws.get(key)
        if ws is None:
            nbytes = int(_native.load().tt_flat_shard_workspace_bytes(self.ntotal, n_total, self.d, nq, k))
            ws = torch.empty(max(nbytes, 256), device=self.device, dtype=torch.uint8)
            if len(self._ws) > 12:
                self._ws.clear()
            self._ws[key] = ws
        return ws

    def shard_sample(self, q: torch.Tensor, k: int, n_total: int, topr: torch.Tensor, slot: int = 0, *,
                     exclude: Optional[torch.Tensor] = None, require=None) -> None:
        """Phase 1 of the sharded search: fills topr f32 [nq, TT_SHARD_TOPR] (this shard's largest sampled scores).
        `slot` selects the workspace (phase 2 of the same batch must use the same slot; batches in flight at the same
        time need different slots).  With `exclude` [nq, E] the sample is planned for K_plan = min(k + E, n_total,
        TT_FLAT_MAX_K); phase 2 must get the same list.  With `require` (label masks, see search_device) only the
        allowed rows are sampled; phase 2 must get the same masks."""
        req = self._requires(require, q.shape[0])
        if exclude is not None and exclude.shape[1] > 0:
            k = _native.plan_k(k, exclude.shape[1], n_total)
        q = ops._f32c(q, "queries")
        ws = self._shard_workspace(n_total, q.shape[0], k, slot)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if req is not None:
                _native.check(lib.tt_flat_shard_sample_filtered(
                    q.data_ptr(), q.shape[0], self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, n_total, self.d, k,
                    self.labels.data_ptr(), req.data_ptr(), topr.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()),
                    "tt_flat_shard_sample_filtered")
            else:
                _native.check(lib.tt_flat_shard_sample(
                    q.data_ptr(), q.shape[0], self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, n_total, self.d, k,
                    topr.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_shard_sample")

    def shard_search_into(self, nq: int, k: int, n_total: int, topr_g: torch.Tensor, scores: torch.Tensor,
                          ids: torch.Tensor, bound: torch.Tensor, flags: torch.Tensor, slot: int = 0, *,
                          exclude: Optional[torch.Tensor] = None, require=None) -> None:
        """Phase 2: global threshold from the gathered lists [G, nq, TT_SHARD_TOPR], main scan, finalize into
        the record views (scores/ids must be contiguous [nq,k]).  `exclude`, `require`: the list and the masks phase 1
        was given."""
        req = self._requires(require, nq)
        excl = self._exclusions(exclude, nq)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if req is not None:
                E = 0 if excl is None else excl.shape[1]
                ws = self._shard_workspace(n_total, nq, _native.plan_k(k, E, n_total), slot)
                _native.check(lib.tt_flat_shard_search_filtered(
                    nq, self.xn.data_ptr(), self.xh.data_ptr(), self.ntotal, n_total, self.d, k, self.id_offset,
                    topr_g.data_ptr(), topr_g.shape[0], scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                    nunc.data_ptr(), bound.data_ptr(), self.labels.data_ptr(), req.data_ptr(),
                    0 if excl is None else excl.data_ptr(), E, ws.data_ptr(), ws.numel(), ops._stream()),
                    "tt_flat_shard_search_filtered")
            elif excl is None:
                ws = self._shard_workspace(n_total, nq, k, slot)
                _native.check(lib.tt_flat_shard_search(
                    nq, self.xn.data_ptr(), self.xh.data_ptr(), self.ntotal, n_total, self.d, k, self.id_offset,
                    topr_g.data_ptr(), topr_g.shape[0], scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                    nunc.data_ptr(), bound.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_shard_search")
            else:
                ws = self._shard_workspace(n_total, nq, _native.plan_k(k, excl.shape[1], n_total), slot)
                _native.check(lib.tt_flat_shard_search_excl(
                    nq, self.xn.data_ptr(), self.xh.data_ptr(), self.ntotal, n_total, self.d, k, self.id_offset,
                    topr_g.data_ptr(), topr_g.shape[0], scores.data_ptr(), ids.data_ptr(), flags.data_ptr(),
                    nunc.data_ptr(), bound.data_ptr(), excl.data_ptr(), excl.shape[1], ws.data_ptr(), ws.numel(),
                    ops._stream()), "tt_flat_shard_search_excl")

    def search_host_async(self, q: np.ndarray, k: int, *, exclude: Optional[np.ndarray] = None,
                          require=None, max_per_group: Optional[int] = None) -> PendingSearch:
        """Host-to-host search, asynchronous: stages q through pinned memory, enqueues H2D + search + D2H and
        returns; `.result()` -> (scores, ids, n_rerun) numpy arrays.  Up to 3 calls may be in flight.
        `exclude`: numpy int64 [nq, E]; `require`: numpy [nq, 2] or [2] label masks; `max_per_group`: group cap (see
        search_device)."""
        return host_search_async(self, self.search_async, self.device, self.d, q, k, exclude=exclude, require=require,
                                 max_per_group=max_per_group)

    def search(self, q: np.ndarray, k: int, *, exclude: Optional[np.ndarray] = None,
               require=None, max_per_group: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Host-to-host search, the shape of faiss `index.search(q, k)`: q f32 [nq,d] (un-normalised:
        the device op applies q/(||q||+1e-8)) -> (scores f32 [nq,k], ids i64 [nq,k]).  `exclude`: numpy int64
        [nq, E] ids to leave out per query (-1 = padding); `require`: label masks {all, any} per query ([nq, 2] or
        [2]); `max_per_group`: at most that many rows per group (see set_groups); short results end in (-inf, -1)."""
        scores, ids, _ = self.search_host_async(q, k, exclude=exclude, require=require,
                                                max_per_group=max_per_group).result()
        return scores, ids


def host_search_async(owner, search_async, device, d: int, q: np.ndarray, k: int, depth: int = 3, *,
                      exclude: Optional[np.ndarray] = None, require=None,
                      max_per_group: Optional[int] = None) -> PendingSearch:
    """Shared host round trip of FlatIPIndex / ShardedFlatIPIndex: pinned staging buffers in a ring of `depth`
    sets per (nq, k) so that consecutive batches overlap their copies with the previous batch's kernels.
    `exclude` (numpy int64 [nq, E]) is copied to the device with the queries and passed on as `exclude=`; `require`
    (label masks, FlatIPIndex only) is passed on as `require=`, and `max_per_group` (FlatIPIndex only) as
    `max_per_group=`."""
    q = np.ascontiguousarray(q, dtype=np.float32)
    if q.ndim != 2 or q.shape[1] != d:
        raise ValueError(f"expected queries [nq, {d}], got {q.shape}")
    nq = q.shape[0]
    if exclude is not None:
        exclude = np.ascontiguousarray(exclude, dtype=np.int64)
        if exclude.ndim != 2 or exclude.shape[0] != nq:
            raise ValueError(f"expected exclusions [nq={nq}, E], got {exclude.shape}")
    if nq == 0:
        empty = (np.empty((0, k), np.float32), np.empty((0, k), np.int64), 0)
        return PendingSearch(lambda: empty)
    rings = owner.__dict__.setdefault("_host_rings", {})
    ring = rings.get((nq, k))
    if ring is None:
        if len(rings) > 8:
            rings.clear()
        ring = rings[(nq, k)] = {"next": 0, "sets": [
            (torch.empty((nq, d), dtype=torch.float32, pin_memory=True),
             torch.empty((nq, k), dtype=torch.float32, pin_memory=True),
             torch.empty((nq, k), dtype=torch.int64, pin_memory=True)) for _ in range(depth)]}
    slot = ring["next"]
    hq, hs, hi = ring["sets"][slot]
    ring["next"] = (slot + 1) % depth
    evs = ring.setdefault("h2d_done", [None] * depth)
    if evs[slot] is not None:
        evs[slot].synchronize()          # the previous user's H2D copy of this staging set has been consumed
    hq.copy_(torch.from_numpy(q))
    stream = torch.cuda.current_stream(device)
    with torch.cuda.device(device):
        dq = hq.to(device, non_blocking=True)
        evs[slot] = torch.cuda.Event()
        evs[slot].record(stream)
        kw = {} if exclude is None else {"exclude": torch.from_numpy(exclude).to(device)}
        if require is not None:
            kw["require"] = require
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        pending = search_async(dq, k, **kw)

    def finish():
        scores, ids, n_bad = pending.result()        # exact re-run (if any) is enqueued before the copies below
        st = torch.cuda.current_stream(device)
        with torch.cuda.device(device):
            hs.copy_(scores, non_blocking=True)
            hi.copy_(ids, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(st)
        ev.synchronize()
        return hs.numpy().copy(), hi.numpy().copy(), n_bad
    return PendingSearch(finish)


# ---------------------------------------------------------------------------------------------
class VectorDatabase:
    """Vector database for product retrieval (reference vector_db.py:10)."""

    def __init__(self, embedding_dim: int = 384):
        self.embedding_dim = embedding_dim
        self.index: Optional[FlatIPIndex] = None
        self.product_ids: Optional[List[str]] = None
        self.id_to_index: Optional[Dict[str, int]] = None
        self.index_to_id: Optional[Dict[int, str]] = None

    def build_index(self, embeddings: np.ndarray, product_ids: List[str]):
        """vector_db.py:25-61 — rows are L2-normalised (x / (||x|| + 1e-8)) and stored as f32."""
        n_products, dim = embeddings.shape
        if dim != self.embedding_dim:
            raise ValueError(f"Embedding dimension mismatch: expected {self.embedding_dim}, got {dim}")
        index = FlatIPIndex(self.embedding_dim)
        embeddings = np.asarray(embeddings)
        if embeddings.dtype == np.float64:
            # the reference normalises in the INPUT dtype and only then casts to f32 (vector_db.py:44-45,51)
            norms = np.linalg.norm(embeddings, axis=1, keepdims=True)
            index.add((embeddings / (norms + 1e-8)).astype(np.float32), normalize=False)
        else:
            index.add(embeddings, normalize=True)
        self.index = index
        self.product_ids = product_ids
        self.id_to_index = {pid: idx for idx, pid in enumerate(product_ids)}
        self.index_to_id = {idx: pid for idx, pid in enumerate(product_ids)}
        print(f"Built FAISS index with {n_products} products")

    def load_index(self, index_path: str, product_ids_path: Optional[str] = None,
                   mapping_path: Optional[str] = None):
        """vector_db.py:63-98 — rows are taken verbatim from the file (no re-normalisation)."""
        rows = read_flat_ip_file(index_path)
        if self.embedding_dim is not None and rows.shape[1] != self.embedding_dim:
            # faiss would load it and fail at the first search; say so at load time
            raise ValueError(f"Embedding dimension mismatch: expected {self.embedding_dim}, index file has {rows.shape[1]}")
        index = FlatIPIndex(rows.shape[1])
        index.add(rows, normalize=False)
        self.index = index
        self.embedding_dim = rows.shape[1] if self.embedding_dim is None else self.embedding_dim
        if product_ids_path:
            self.product_ids = np.load(product_ids_path, allow_pickle=True).tolist()
        else:
            self.product_ids = [f"product_{i}" for i in range(self.index.ntotal)]
        if mapping_path and Path(mapping_path).exists():
            with open(mapping_path, "r", encoding="utf-8") as f:
                self.id_to_index = json.load(f)
            self.index_to_id = {v: k for k, v in self.id_to_index.items()}
        else:
            self.id_to_index = {pid: idx for idx, pid in enumerate(self.product_ids)}
            self.index_to_id = {idx: pid for idx, pid in enumerate(self.product_ids)}
        print(f"Loaded FAISS index with {len(self.product_ids)} products")

    def save_index(self, index_path: str, product_ids_path: Optional[str] = None,
                   mapping_path: Optional[str] = None):
        """vector_db.py:100-128."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() first.")
        write_flat_ip_file(index_path, self.index.rows_host())
        if product_ids_path:
            np.save(product_ids_path, np.array(self.product_ids))
        if mapping_path and self.id_to_index:
            with open(mapping_path, "w", encoding="utf-8") as f:
                json.dump(self.id_to_index, f, ensure_ascii=False, indent=2)
        print(f"Saved FAISS index to {index_path}")

    # -- label words ---------------------------------------------------------------------------
    def set_labels(self, labels, product_ids: Optional[List[str]] = None) -> None:
        """Sets the u32 label words the `require` filters test (e.g. bit 0 = in stock, bits 1-31 = category groups):
        one per index row in index order, or one per listed product id.  An unknown product id raises ValueError and
        changes nothing.  Labels are serving state: save_index / load_index do not store them."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        if product_ids is None:
            self.index.set_labels(labels)
            return
        unknown = [p for p in product_ids if p not in self.id_to_index]
        if unknown:
            raise ValueError(f"{len(unknown)} unknown product ids, e.g. {unknown[:3]}")
        self.index.set_labels(labels, rows=np.array([self.id_to_index[p] for p in product_ids], np.int64))

    def set_groups(self, groups, product_ids: Optional[List[str]] = None) -> None:
        """Sets each product's group for `max_per_group` (a brand name, a seller id: any hashable value; None =
        ungrouped): one per index row in index order, or one per listed product id.  Equal values are one group.  An
        unknown product id raises ValueError and changes nothing.  Groups are serving state: save_index / load_index do
        not store them."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        groups = list(groups)
        rows = None
        if product_ids is not None:
            product_ids = list(product_ids)
            if len(product_ids) != len(groups):
                raise ValueError(f"expected one group per product id ({len(product_ids)}), got {len(groups)}")
            unknown = [p for p in product_ids if p not in self.id_to_index]
            if unknown:
                raise ValueError(f"{len(unknown)} unknown product ids, e.g. {unknown[:3]}")
            rows = np.array([self.id_to_index[p] for p in product_ids], np.int64)
        codes = self.__dict__.setdefault("_group_codes", {})
        keys = np.array([-1 if g is None else codes.setdefault(g, len(codes)) for g in groups], np.int64)
        self.index.set_groups(keys, rows=rows)

    # -- search --------------------------------------------------------------------------------
    def search_batch(self, query_embeddings: np.ndarray, k: int = 10, *,
                     exclude_rows: Optional[np.ndarray] = None, require=None,
                     max_per_group: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Array-returning retrieval: (scores f32 [nq,k'], row indices i64 [nq,k']) with k' = min(k, ntotal).
        `exclude_rows` int64 [nq, E] (-1 = padding): row indices query i must not return; `require` [nq, 2] or [2]:
        {all, any} label masks (see FlatIPIndex.search_device); `max_per_group`: at most that many rows per group (see
        set_groups); with fewer than k' rows to return the tail is (-inf, -1)."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        k = min(k, self.index.ntotal)   # vector_db.py:159
        kw = {} if exclude_rows is None else {"exclude": exclude_rows}
        if require is not None:
            kw["require"] = require
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        return self.index.search(np.asarray(query_embeddings), k, **kw)

    def _exclude_rows(self, lists, nq: int) -> Optional[np.ndarray]:
        """Product-id lists (one per query) -> row indices int64 [nq, E], -1 padded; unknown ids are dropped.
        None when nothing is left to exclude."""
        rows = [[r for r in (self.id_to_index.get(pid) for pid in ids) if r is not None and r >= 0] for ids in lists]
        E = max((len(r) for r in rows), default=0)
        if E == 0:
            return None
        out = np.full((nq, E), -1, np.int64)
        for i, r in enumerate(rows):
            out[i, :len(r)] = r
        return out

    def retrieve(self, query_embedding: np.ndarray, k: int = 10, *,
                 exclude: Optional[List[str]] = None, require_all=0, require_any=0,
                 max_per_group: Optional[int] = None) -> List[Tuple[str, float]]:
        """vector_db.py:130-169 — descending score; only query row 0 is returned, as in the reference.
        `exclude`: product ids that must not be returned (e.g. the buyer's own history); unknown ids are ignored.
        `require_all` / `require_any`: label masks (scalars, or one per query row): only products whose label word has
        every bit of require_all and, unless require_any is 0, one bit of require_any (see set_labels).
        `max_per_group`: at most that many products of one group (see set_groups)."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        query_embedding = np.asarray(query_embedding)
        if query_embedding.ndim == 1:
            query_embedding = query_embedding.reshape(1, -1)
        nq = query_embedding.shape[0]
        kw = {}
        req = require_masks(require_all, require_any, nq)
        if req is not None:
            kw["require"] = req
        if exclude is not None:
            kw["exclude_rows"] = self._exclude_rows([exclude] * nq, nq)
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        scores, indices = self.search_batch(query_embedding, k, **kw)
        results = []
        for idx, score in zip(indices[0], scores[0]):
            if 0 <= idx < len(self.product_ids):
                results.append((self.product_ids[idx], float(score)))
        return results

    def retrieve_batch(self, query_embeddings: np.ndarray, k: int = 10, *,
                       exclude: Optional[List[List[str]]] = None, require_all=0,
                       require_any=0, max_per_group: Optional[int] = None) -> List[List[Tuple[str, float]]]:
        """vector_db.py:171-209.  `exclude`: one list of product ids per query that it must not return.
        `require_all` / `require_any`: label masks, scalars or one per query (see retrieve); `max_per_group`: at most
        that many products of one group per query (see set_groups)."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        nq = np.asarray(query_embeddings).shape[0]
        kw = {}
        req = require_masks(require_all, require_any, nq)
        if req is not None:
            kw["require"] = req
        if exclude is not None:
            if len(exclude) != nq:
                raise ValueError(f"exclude needs one list per query ({nq}), got {len(exclude)}")
            kw["exclude_rows"] = self._exclude_rows(exclude, nq)
        if max_per_group is not None:
            kw["max_per_group"] = max_per_group
        scores, indices = self.search_batch(query_embeddings, k, **kw)
        pids = self.product_ids
        n = len(pids)
        all_results = []
        for query_scores, query_indices in zip(scores.tolist(), indices.tolist()):
            all_results.append([(pids[i], s) for i, s in zip(query_indices, query_scores) if 0 <= i < n])
        return all_results

    def retrieve_above(self, query_embeddings: np.ndarray, min_score, max_results: int = _native.TT_FLAT_RANGE_MAX_RESULTS,
                       *, exclude: Optional[List[List[str]]] = None, require_all=0,
                       require_any=0) -> List[List[Tuple[str, float]]]:
        """Every product whose score is strictly greater than `min_score` (a float, or one per query), best first, at
        most `max_results` per query: a relevance floor whose result size changes from query to query.  `exclude` and
        `require_all` / `require_any` as in retrieve_batch; excluded and disallowed products are never returned."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        q = np.asarray(query_embeddings)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        nq = q.shape[0]
        kw = {}
        req = require_masks(require_all, require_any, nq)
        if req is not None:
            kw["require"] = req
        if exclude is not None:
            if len(exclude) != nq:
                raise ValueError(f"exclude needs one list per query ({nq}), got {len(exclude)}")
            kw["exclude"] = self._exclude_rows(exclude, nq)
        lims, scores, rows = self.index.range_search(q, min_score, max_results, **kw)
        pids = self.product_ids
        n = len(pids)
        s, r = scores.tolist(), rows.tolist()
        return [[(pids[i], v) for i, v in zip(r[lims[j]:lims[j + 1]], s[lims[j]:lims[j + 1]]) if 0 <= i < n]
                for j in range(nq)]

    def get_embedding(self, product_id: str) -> Optional[np.ndarray]:
        """vector_db.py:211-231 — the reference returns None in every branch; kept."""
        return None
