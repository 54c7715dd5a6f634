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
from typing import Dict, List, Optional, Tuple

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

    def add(self, x, normalize: bool = True, chunk_rows: int = 1 << 17) -> None:
        """Appends rows (numpy [n,d] or a torch tensor on any device)."""
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

    def search_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None):
        """Asynchronous search of CUDA f32 queries [nq,D] on the current stream.

        Returns (scores [nq,k] f32, ids [nq,k] i64, flags [nq] i32, n_uncertified [1] i32) device
        tensors; rows with flags != 1 (1 = certified exact, <= 0 = -(reason bits), see include/tt_b200.h) must be
        passed to `search_exact_device` (`search_checked_device` / `search_async` do both).
        `exclude` (CUDA i64 [nq, E], E <= 1024, ids as returned, -1 = padding): the top-k over the rows query i does
        not list in exclude[i]; with fewer than k allowed rows the tail is (-inf, -1).
        """
        if self.ntotal == 0:
            raise ValueError("empty index")
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"expected queries [nq, {self.d}], got {tuple(q.shape)}")
        if not 1 <= k <= min(self.ntotal, _native.TT_FLAT_MAX_K):
            raise ValueError(f"k must be in [1, min(ntotal, {_native.TT_FLAT_MAX_K})], got {k}")
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        scores = torch.empty((nq, k), device=self.device, dtype=torch.float32)
        ids = torch.empty((nq, k), device=self.device, dtype=torch.int64)
        flags = torch.empty((max(nq, 1),), device=self.device, dtype=torch.int32)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if excl is None:
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
                            exclude: Optional[torch.Tensor] = None):
        """Always-exact fp32 path; with `qsel` (i32 query rows) only those rows of scores/ids are rewritten.
        `exclude` [nq, E] is indexed by query row (qsel[i]), as in search_device."""
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        if scores is None:
            scores = torch.empty((nq, k), device=self.device, dtype=torch.float32)
            ids = torch.empty((nq, k), device=self.device, dtype=torch.int64)
        nsel = nq if qsel is None else int(qsel.numel())
        lib = _native.load()
        need = int(lib.tt_flat_search_exact_workspace_bytes(self.ntotal, self.d, nsel, k))
        if self._exact_ws is None or self._exact_ws.numel() < need:
            self._exact_ws = torch.empty(need, device=self.device, dtype=torch.uint8)
        with torch.cuda.device(self.device):
            if excl is None:
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
                          bound: torch.Tensor, flags: torch.Tensor, *, exclude: Optional[torch.Tensor] = None) -> None:
        """Shard-local search for ShardedFlatIPIndex (tt_flat_search_shard): fills the caller's record views.
        scores/ids are [nq, k_record] with k_record >= k; only the first k columns of each row are written.
        `exclude` holds GLOBAL ids (ids of other shards are ignored here)."""
        q = ops._f32c(q, "queries")
        nq = q.shape[0]
        excl = self._exclusions(exclude, nq)
        direct = scores.shape[1] == k and scores.is_contiguous() and ids.is_contiguous()
        s_out = scores if direct else torch.empty((nq, k), device=self.device, dtype=torch.float32)
        i_out = ids if direct else torch.empty((nq, k), device=self.device, dtype=torch.int64)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if excl is None:
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
                          qsel: torch.Tensor, *, exclude: Optional[torch.Tensor] = None) -> None:
        """Exact fp32 re-run of the query rows `qsel`, written into [nq, k_record] record views."""
        kw = {} if exclude is None else {"exclude": exclude}
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

    def search_async(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None) -> PendingSearch:
        """Enqueues a search and returns at once; `.result()` checks the certificate later, so a caller can
        keep the next batch's kernels queued behind this one (no idle GPU between batches).  `exclude`: see
        search_device; uncertified queries are re-run exactly with the same lists."""
        kw = {} if exclude is None else {"exclude": exclude}
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

    def search_checked_device(self, q: torch.Tensor, k: int, *, exclude: Optional[torch.Tensor] = None):
        """search_device + re-run of uncertified queries through the exact path (one host sync)."""
        return self.search_async(q, k, **({} if exclude is None else {"exclude": exclude})).result()

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
                     exclude: Optional[torch.Tensor] = None) -> None:
        """Phase 1 of the sharded search: fills topr f32 [nq, TT_SHARD_TOPR] (this shard's largest sampled scores).
        `slot` selects the workspace (phase 2 of the same batch must use the same slot; batches in flight at the same
        time need different slots).  With `exclude` [nq, E] the sample is planned for K_plan = min(k + E, n_total,
        TT_FLAT_MAX_K); phase 2 must get the same list."""
        if exclude is not None and exclude.shape[1] > 0:
            k = _native.plan_k(k, exclude.shape[1], n_total)
        q = ops._f32c(q, "queries")
        ws = self._shard_workspace(n_total, q.shape[0], k, slot)
        with torch.cuda.device(self.device):
            _native.check(_native.load().tt_flat_shard_sample(
                q.data_ptr(), q.shape[0], self.xh.data_ptr(), self.stats.data_ptr(), self.ntotal, n_total, self.d, k,
                topr.data_ptr(), ws.data_ptr(), ws.numel(), ops._stream()), "tt_flat_shard_sample")

    def shard_search_into(self, nq: int, k: int, n_total: int, topr_g: torch.Tensor, scores: torch.Tensor,
                          ids: torch.Tensor, bound: torch.Tensor, flags: torch.Tensor, slot: int = 0, *,
                          exclude: Optional[torch.Tensor] = None) -> None:
        """Phase 2: global threshold from the gathered lists [G, nq, TT_SHARD_TOPR], main scan, finalize into
        the record views (scores/ids must be contiguous [nq,k]).  `exclude`: the list phase 1 was given."""
        excl = self._exclusions(exclude, nq)
        nunc = torch.empty((1,), device=self.device, dtype=torch.int32)
        lib = _native.load()
        with torch.cuda.device(self.device):
            if excl is None:
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

    def search_host_async(self, q: np.ndarray, k: int, *, exclude: Optional[np.ndarray] = None) -> PendingSearch:
        """Host-to-host search, asynchronous: stages q through pinned memory, enqueues H2D + search + D2H and
        returns; `.result()` -> (scores, ids, n_rerun) numpy arrays.  Up to 3 calls may be in flight.
        `exclude`: numpy int64 [nq, E] (see search_device)."""
        return host_search_async(self, self.search_async, self.device, self.d, q, k, exclude=exclude)

    def search(self, q: np.ndarray, k: int, *, exclude: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Host-to-host search, the shape of faiss `index.search(q, k)`: q f32 [nq,d] (un-normalised:
        the device op applies q/(||q||+1e-8)) -> (scores f32 [nq,k], ids i64 [nq,k]).  `exclude`: numpy int64
        [nq, E] ids to leave out per query (-1 = padding); short results end in (-inf, -1)."""
        scores, ids, _ = self.search_host_async(q, k, exclude=exclude).result()
        return scores, ids


def host_search_async(owner, search_async, device, d: int, q: np.ndarray, k: int, depth: int = 3, *,
                      exclude: Optional[np.ndarray] = None) -> PendingSearch:
    """Shared host round trip of FlatIPIndex / ShardedFlatIPIndex: pinned staging buffers in a ring of `depth`
    sets per (nq, k) so that consecutive batches overlap their copies with the previous batch's kernels.
    `exclude` (numpy int64 [nq, E]) is copied to the device with the queries and passed on as `exclude=`."""
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
        if exclude is None:
            pending = search_async(dq, k)
        else:
            pending = search_async(dq, k, exclude=torch.from_numpy(exclude).to(device))

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

    # -- search --------------------------------------------------------------------------------
    def search_batch(self, query_embeddings: np.ndarray, k: int = 10, *,
                     exclude_rows: Optional[np.ndarray] = None) -> Tuple[np.ndarray, np.ndarray]:
        """Array-returning retrieval: (scores f32 [nq,k'], row indices i64 [nq,k']) with k' = min(k, ntotal).
        `exclude_rows` int64 [nq, E] (-1 = padding): row indices query i must not return; with fewer than k' allowed
        rows the tail is (-inf, -1)."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        k = min(k, self.index.ntotal)   # vector_db.py:159
        if exclude_rows is None:
            return self.index.search(np.asarray(query_embeddings), k)
        return self.index.search(np.asarray(query_embeddings), k, exclude=exclude_rows)

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
                 exclude: Optional[List[str]] = None) -> List[Tuple[str, float]]:
        """vector_db.py:130-169 — descending score; only query row 0 is returned, as in the reference.
        `exclude`: product ids that must not be returned (e.g. the buyer's own history); unknown ids are ignored."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        query_embedding = np.asarray(query_embedding)
        if query_embedding.ndim == 1:
            query_embedding = query_embedding.reshape(1, -1)
        if exclude is not None:
            rows = self._exclude_rows([exclude] * query_embedding.shape[0], query_embedding.shape[0])
            scores, indices = self.search_batch(query_embedding, k, exclude_rows=rows)
        else:
            scores, indices = self.search_batch(query_embedding, k)
        results = []
        for idx, score in zip(indices[0], scores[0]):
            if 0 <= idx < len(self.product_ids):
                results.append((self.product_ids[idx], float(score)))
        return results

    def retrieve_batch(self, query_embeddings: np.ndarray, k: int = 10, *,
                       exclude: Optional[List[List[str]]] = None) -> List[List[Tuple[str, float]]]:
        """vector_db.py:171-209.  `exclude`: one list of product ids per query that it must not return."""
        if self.index is None:
            raise ValueError("Index not built. Call build_index() or load_index() first.")
        if exclude is not None:
            nq = np.asarray(query_embeddings).shape[0]
            if len(exclude) != nq:
                raise ValueError(f"exclude needs one list per query ({nq}), got {len(exclude)}")
            scores, indices = self.search_batch(query_embeddings, k, exclude_rows=self._exclude_rows(exclude, nq))
        else:
            scores, indices = self.search_batch(query_embeddings, k)
        pids = self.product_ids
        n = len(pids)
        all_results = []
        for query_scores, query_indices in zip(scores.tolist(), indices.tolist()):
            all_results.append([(pids[i], s) for i, s in zip(query_indices, query_scores) if 0 <= i < n])
        return all_results

    def get_embedding(self, product_id: str) -> Optional[np.ndarray]:
        """vector_db.py:211-231 — the reference returns None in every branch; kept."""
        return None
