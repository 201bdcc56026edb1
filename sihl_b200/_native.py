"""ctypes binding of ``libsihl_b200.so`` (``include/sihl_od.h``).

There is deliberately no fallback of any kind: if the shared library is missing
and cannot be built, importing the ops raises.  ``ctypes`` releases the GIL for
the duration of each call; every call only enqueues kernels on the stream it is
given.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import build as _build

_lock = threading.Lock()
_lib = None

P, I, I64, F = C.c_void_p, C.c_int, C.c_int64, C.c_float

_SIGNATURES = {
    "sihl_od_version": (C.c_int, []),
    "sihl_od_last_error_string": (C.c_char_p, []),
    "sihl_od_anchors": (I, [P, I, I, I, P, P, P, P]),
    "sihl_od_anchor_terms": (I, [P, I64, P, P]),
    "sihl_od_assign_select": (I, [P, P, I64, P, I, I, I, P, P, I, I, I, P, P, P, P, P]),
    "sihl_od_resolve_tiles": (I, [I64, P, P]),
    "sihl_od_assign_resolve": (I, [P, P, P, P, I, I64, I, I, P, P, P, P, P, P, P, P, P, I, P, P, P]),
    "sihl_od_assign_resolve_t": (I, [P, P, P, P, I, I64, I, I, P, P, I, P, P, P, P, P, P, P, I, P, P, P]),
    "sihl_od_pos_loss_tiles_exchange_t": (I, [P, P, P, I, I64, P, P, I, I, P, P, P, P, P, I, I, P, P, P, P, I, I, P]),
    "sihl_od_dense_decode_t": (I, [P, P, P, I, I, I64, I, P, P, I, I, F, P, I64, P, P, P, I, P]),
    "sihl_od_quad_matching": (I, [P, I64, P, P, I, I, I, P, P, P, P, P, P, P, P]),
    "sihl_od_pos_loss_tiles": (I, [P, P, P, I, I64, P, P, I, I, P, P, P, P, P, I, P, P, P, P]),
    "sihl_od_pos_loss_tiles_exchange": (I, [P, P, P, I, I64, P, P, I, I, P, P, P, P, P, I, P, P, P, P, I, I, P]),
    "sihl_od_exchange_region_bytes": (C.c_size_t, [I]),
    "sihl_od_exchange_create": (I, [I, I, P, P]),
    "sihl_od_exchange_open": (I, [P, P]),
    "sihl_od_exchange_close": (I, [P]),
    "sihl_od_exchange_destroy": (I, [P]),
    "sihl_od_exchange_barrier": (I, [P, I, I, P]),
    "sihl_od_exchange_set_timeout": (I, [P, I, C.c_uint64]),
    "sihl_od_exchange_status": (I, [P, I, P, P]),
    "sihl_od_loss_finalize": (I, [P, P, P]),
    "sihl_od_train_workspace_bytes": (C.c_size_t, [I, I64, I, I]),
    "sihl_od_train_assign": (I, [P, P, I64, P, I, I, I, P, P, P, I, I, I, P, P, P, I64, P, P, P, C.c_size_t, P]),
    "sihl_od_train_loss": (I, [P, P, P, P, I, I, I64, I, P, P, P, I64, P, P, P, I, I, P, P, P, P, P, P]),
    "sihl_od_train_loss_bwd": (I, [P, P, P, P, I, I, I64, I, P, P, P, I64, P, P, P, I, I, P, P, P, P, P, F, P, P, P, P, P]),
    "sihl_od_map_workspace_bytes": (C.c_size_t, [I, I, I]),
    "sihl_od_map_match": (I, [P, P, P, I, I, P, P, P, I, P, I, P, I, P, P, P, P, P, P]),
    "sihl_od_topk": (I, [P, I, I64, I, P, P, P]),
    "sihl_od_decode_rows": (I, [P, P, I, I, P, I, P, P, P, I, I, P, P, P, P, P]),
    "sihl_od_topk_t": (I, [P, I, I, I64, I, P, P, P]),
    "sihl_od_decode_rows_t": (I, [P, P, I, I, P, I, P, I, P, P, I, I, P, P, P, P, P]),
    "sihl_od_candidate_decode_t": (I, [P, P, P, I, I, I64, I, P, P, I, I, F, P, I64, P, P, P, I, P]),
    "sihl_od_dense_decode": (I, [P, P, P, I, I64, I, P, P, I, I, F, P, I64, P, P, P, I, P]),
    "sihl_od_candidate_decode": (I, [P, P, P, I, I64, I, P, P, I, I, F, P, I64, P, P, P, I, P]),
    "sihl_od_nms_workspace_bytes": (C.c_size_t, [I, I64]),
    "sihl_od_nms_topk": (I, [P, I64, P, P, P, I, F, I, P, P, P, P, P, I, P]),
    "sihl_od_nms_split_workspace_bytes": (C.c_size_t, [I, I64, I]),
    "sihl_od_nms_topk_split": (I, [P, I64, P, P, P, I, F, I, P, P, P, P, P, I, P]),
    "sihl_od_batched_nms_workspace_bytes": (C.c_size_t, [I64]),
    "sihl_od_batched_nms": (I, [P, P, P, P, I, I64, F, P, P, P, P]),
    "sihl_od_soft_nms_workspace_bytes": (C.c_size_t, [I, I64]),
    "sihl_od_soft_nms_topk": (I, [P, I64, P, P, P, I, I, F, F, F, I, P, P, P, P, P, I, P]),
    "sihl_od_batched_soft_nms_workspace_bytes": (C.c_size_t, [I64]),
    "sihl_od_batched_soft_nms": (I, [P, P, P, P, I, I64, I, F, F, F, I, P, P, P, P, P]),
    "sihl_od_mlp_hidden": (I, [P, I64, I, P, P, P, P, F, P, P]),
    "sihl_od_mlp_out": (I, [P, I64, I, P, P, I, I, P, P]),
    "sihl_od_mlp_hidden_train": (I, [P, I64, I, P, P, P, P, F, P, P, P, P]),
    "sihl_od_mlp_bwd_partial_rows": (I, []),
    "sihl_od_mlp_hidden_bwd_partial_rows": (I, []),
    "sihl_od_bf16_to_f32": (I, [P, I64, P, P]),
    "sihl_od_mlp_hidden_bwd": (I, [P, P, P, P, P, I64, I, P, P, I, P]),
    "sihl_od_lateral_rows": (I, [P, I, I, I64, P, P]),
    "sihl_od_rows_to_nchw": (I, [P, I, I, I64, P, P]),
    "sihl_od_mlp_hidden_bwd_rank1": (I, [P, P, P, P, P, P, I64, I, P, P, I, P]),
    "sihl_od_bn_bwd_colsums_map": (I, [P, I64, I64, I64, P, I64, I, P, I, P]),
    "sihl_od_bn_bwd_apply_map": (I, [P, I64, I64, I64, P, P, P, P, I64, I, P, P]),
    "sihl_od_rows_colsum": (I, [P, I64, I, P, I, P]),
    "sihl_od_bn_bwd_colsums": (I, [P, P, I64, I, P, I, P]),
    "sihl_od_bn_bwd_apply": (I, [P, P, P, P, P, I64, I, P, P]),
    "sihl_od_lateral_linear": (I, [P, I64, I, P, P, I64, I64, I64, P, P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class NativeError(RuntimeError):
    """A C-ABI call returned a non-zero status."""


def lib_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if the sources are newer) ``libsihl_b200.so``.  Raises if impossible."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.LIB_PATH
        if build_if_missing:
            try:
                path = _build.build()
            except Exception as exc:                       # nvcc absent or compile error
                if not os.path.exists(_build.LIB_PATH):
                    raise RuntimeError(
                        "libsihl_b200.so is missing and could not be built; the detection-head path has no "
                        f"CPU or PyTorch fallback ({exc})") from exc
                if not _build.is_fresh():
                    # a library exists but was built from OTHER sources than the ones in the tree: binding today's
                    # ctypes signatures to yesterday's ABI would be undefined behaviour on the GPU, not an error
                    raise RuntimeError(
                        "libsihl_b200.so is stale (its build stamp does not match csrc/ + include/) and the rebuild "
                        f"failed: {exc}") from exc
                path = _build.LIB_PATH
        if not os.path.exists(path):
            raise RuntimeError(f"{path} not found; run `python -m sihl_b200.build` (no fallback path exists)")
        lib = C.CDLL(path)
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = restype, argtypes
        _lib = lib
        return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().sihl_od_last_error_string()
        raise NativeError(f"{what} failed with status {status}: {msg.decode() if msg else '?'}")
