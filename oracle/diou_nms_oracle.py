"""numpy/ctypes front end of the DIoU-NMS oracle (``oracle/diou_nms_oracle.c``).

TEST INFRASTRUCTURE ONLY, beside ``od_oracle.py``: class-aware greedy NMS with the DIoU test of Zheng et al. (AAAI
2020), ``diou(kept, later) > thr``, and the dense postprocess that ends in it.  The C file is compiled with the flags of
``oracle/Makefile`` (fp32, ``-ffp-contract=off``) into ``oracle/_ref/``.
"""
from __future__ import annotations

import ctypes as C
import fcntl
import hashlib
import os
import subprocess

import numpy as np

from .od_oracle import _f32, _i64, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "diou_nms_oracle.c")
_LIB_PATH = os.path.join(_HERE, "_ref", "libdiou_nms_oracle.so")
_CFLAGS = ["-O2", "-std=c11", "-fPIC", "-shared", "-fvisibility=hidden", "-ffp-contract=off", "-fno-fast-math",
           "-Wall", "-Wextra"]
_lib = None


def build(force: bool = False) -> str:
    """Compile ``diou_nms_oracle.c`` (content-stamped and file-locked, as ``od_oracle.build``)."""
    with open(_SRC, "rb") as fh:
        fp = hashlib.sha256(fh.read() + " ".join(_CFLAGS).encode()).hexdigest()
    stamp = _LIB_PATH + ".stamp"

    def fresh():
        try:
            return os.path.exists(_LIB_PATH) and open(stamp).read().strip() == fp
        except OSError:
            return False

    if not force and fresh():
        return _LIB_PATH
    os.makedirs(os.path.dirname(_LIB_PATH), exist_ok=True)
    with open(os.path.join(os.path.dirname(_LIB_PATH), ".build_diou.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if force or not fresh():
            tmp = f"{_LIB_PATH}.tmp{os.getpid()}"
            subprocess.check_call([os.environ.get("CC", "gcc"), *_CFLAGS, "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, _LIB_PATH)
            with open(stamp, "w") as fh:
                fh.write(fp + "\n")
    return _LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_diou_pair.restype = C.c_float
        _lib.orc_batched_diou_nms.restype = C.c_int64
    return _lib


def diou_pair(a, b) -> np.float32:
    return np.float32(lib().orc_diou_pair(_p(_f32(a)), _p(_f32(b))))


def batched_diou_nms(boxes, scores, classes, diou_thr: float) -> np.ndarray:
    """Kept indices in (score desc, index asc) order."""
    boxes, scores, classes = _f32(boxes).reshape(-1, 4), _f32(scores), _i64(classes)
    n = len(scores)
    keep = np.empty(max(n, 1), np.int64)
    m = lib().orc_batched_diou_nms(_p(boxes), _p(scores), _p(classes), C.c_int64(n), C.c_float(diou_thr), _p(keep))
    return keep[:m].copy()


def dense_postprocess_diou(loc, cls, box_raw, offsets, scales, img_w, img_h, score_thr: float = 0.05,
                           diou_thr: float = 0.5, K: int = 100):
    """``od_oracle.dense_postprocess`` with DIoU-NMS -> (num_instances, scores, classes, boxes)."""
    loc, cls, box_raw = _f32(loc), _f32(cls), _f32(box_raw)
    B, A = loc.shape
    num = np.empty(B, np.int64)
    scores, classes, boxes = np.empty((B, K), np.float32), np.empty((B, K), np.int64), np.empty((B, K, 4), np.float32)
    lib().orc_dense_postprocess_diou(_p(loc), _p(cls), _p(box_raw), B, C.c_int64(A), cls.shape[-1], _p(_f32(offsets)),
                                     _p(_f32(scales)), int(img_w), int(img_h), C.c_float(score_thr), C.c_float(diou_thr),
                                     int(K), _p(num), _p(scores), _p(classes), _p(boxes))
    return num, scores, classes, boxes
