"""ctypes binding of lib/libtt_b200.so (the C-ABI declared in include/tt_b200.h).

The product path has no fallback: if the shared library is missing this module raises at import
of the first op, and if there is no CUDA device every entry point returns TT_ERR_CUDA, which
`check` turns into a RuntimeError.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libtt_b200.so"

TT_FLAT_MAX_K = 2048
TT_SHARD_TOPR = 32
TT_FLAT_MAX_EXCLUDE = 1024
ABI_VERSION = 1


def plan_k(k: int, n_excl: int, n: int) -> int:
    """K_plan = min(K + E, N, TT_FLAT_MAX_K): the K a search with E exclusions per query plans its scan for
    (include/tt_b200.h); the global-threshold calls of a sharded search take it with N = N_total."""
    return min(int(k) + int(n_excl), int(n), TT_FLAT_MAX_K)

# name -> (restype, argtypes); mirrors include/tt_b200.h one to one
SIGNATURES = {
    "tt_abi_version": (c_int, []),
    "tt_last_error": (c_char_p, []),
    "tt_pool_weighted": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_pool_weighted_gather": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_attention_logits": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "tt_pool_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_pool_attention_gather": (c_int, [c_void_p, c_int64, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_pool_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_infonce_workspace_bytes": (c_size_t, [c_int]),
    "tt_infonce_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tt_infonce_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_pool_partial_gather": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_float, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int, c_int, c_void_p]),
    "tt_pool_partial_merge": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "tt_pool_attention_fused_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "tt_pool_attention_fused": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                        c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_flat_pitch": (c_int64, [c_int]),
    "tt_flat_build": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "tt_flat_search_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "tt_flat_search": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_flat_search_shard": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_flat_search_excl_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int, c_int]),
    "tt_flat_search_excl": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_flat_search_shard_excl": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                          c_size_t, c_void_p]),
    "tt_flat_shard_search_excl": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int64, c_void_p,
                                          c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                          c_void_p, c_size_t, c_void_p]),
    "tt_flat_search_exact_excl": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int64,
                                          c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "tt_flat_shard_plan_ok":(c_int, [c_int64, c_int64, c_int, c_int, c_int]),
    "tt_flat_shard_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_int, c_int]),
    "tt_flat_shard_sample": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p,
                                     c_void_p, c_size_t, c_void_p]),
    "tt_flat_shard_search": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int64, c_void_p, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_p2p_enable_peer": (c_int, [c_int]),
    "tt_p2p_alloc": (c_int, [c_size_t, c_void_p, c_void_p]),
    "tt_p2p_open": (c_int, [c_void_p, c_void_p]),
    "tt_p2p_close": (c_int, [c_void_p]),
    "tt_p2p_free": (c_int, [c_void_p]),
    "tt_p2p_push": (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_int32, c_void_p, c_void_p]),
    "tt_p2p_wait": (c_int, [c_void_p, c_int, c_int32, ctypes.c_double, c_void_p, c_void_p]),
    "tt_shard_merge": (c_int, [c_void_p, c_size_t, c_size_t, c_size_t, c_size_t, c_size_t, c_int, c_int, c_int,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tt_flat_search_exact_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "tt_flat_search_exact": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int64,
                                     c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tt_kernel_launch_count": (c_int64, []),
    "tt_profile_scan_arm": (c_int, [c_int]),
    "tt_profile_scan_read": (c_int, [c_void_p, c_int]),
    "tt_flat_plan_describe": (c_int, [c_int64, c_int, c_int, c_int, c_void_p]),
    "tt_flat_debug_read": (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "tt_flat_scan_scores_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "tt_flat_scan_scores": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_size_t,
                                    c_void_p]),
    "tt_topk_merge": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Loads the shared library once; raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("TT_B200_LIB", LIB_PATH))
    if not path.exists():
        raise NativeLibraryError(
            f"{path} not found: build it with `python two-tower-model-v2_b200/build.py` "
            "(or __graft_entry__.build()); there is no CPU/PyTorch fallback for these ops")
    lib = ctypes.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.tt_abi_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI mismatch: library {lib.tt_abi_version()} vs binding {ABI_VERSION}")
    _lib = lib
    return lib


def last_error() -> str:
    return load().tt_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = last_error()
        if rc == 1:
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
