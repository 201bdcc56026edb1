"""References for the quadrilateral NMS: the host build of od_math.h's quad overlap and of the greedy quad NMS
(tests/host_quad_shim.cpp, compiled with -ffp-contract=off into a temporary directory), and an exact rational
restatement of the overlap (convex hull and convex-polygon intersection over fractions.Fraction) that shares no code
with it."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32
_shim = None


def shim() -> C.CDLL:
    global _shim
    if _shim is None:
        tmp = tempfile.mkdtemp(prefix="sihl_quad_shim_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libquad_shim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                               os.path.join(HERE, "host_quad_shim.cpp"), "-o", out])
        lib = C.CDLL(out)
        lib.shim_quad_iou_pairs.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
        lib.shim_quad_iou_pairs.restype = None
        lib.shim_batched_quad_nms.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_float, C.c_void_p]
        lib.shim_batched_quad_nms.restype = C.c_long
        _shim = lib
    return _shim


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def quad_iou_pairs(a, b) -> np.ndarray:
    """Host quad_iou of a[i] and b[i] (each [n, 4, 2] or [n, 8])."""
    a = np.ascontiguousarray(np.asarray(a, f32).reshape(-1, 8))
    b = np.ascontiguousarray(np.asarray(b, f32).reshape(-1, 8))
    assert a.shape == b.shape
    out = np.empty(len(a), f32)
    shim().shim_quad_iou_pairs(_ptr(a), _ptr(b), len(a), _ptr(out))
    return out


def quad_iou_matrix(a, b) -> np.ndarray:
    a = np.asarray(a, f32).reshape(-1, 8)
    b = np.asarray(b, f32).reshape(-1, 8)
    ia, ib = np.meshgrid(np.arange(len(a)), np.arange(len(b)), indexing="ij")
    return quad_iou_pairs(a[ia.ravel()], b[ib.ravel()]).reshape(len(a), len(b))


def batched_quad_nms(quads, scores, classes, thr) -> np.ndarray:
    """Greedy class-aware quad NMS on the host: kept indices in (score desc, index asc) order."""
    q = np.ascontiguousarray(np.asarray(quads, f32).reshape(-1, 8))
    s = np.ascontiguousarray(scores, f32)
    c = np.ascontiguousarray(classes, np.int64)
    keep = np.empty(max(len(q), 1), np.int64)
    m = shim().shim_batched_quad_nms(_ptr(q), _ptr(s), _ptr(c), len(q), float(thr), _ptr(keep))
    return keep[:m].copy()


# ---- exact reference ------------------------------------------------------------------------------------------------
def _cross(o, a, b):
    return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])


def exact_hull(quad):
    """Convex hull (CCW, no collinear points) of the quad's vertices as exact rationals."""
    pts = sorted({(Fraction(float(x)), Fraction(float(y))) for x, y in np.asarray(quad, f32).reshape(4, 2)})
    if len(pts) < 3:
        return pts
    lower, upper = [], []
    for p in pts:
        while len(lower) >= 2 and _cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    for p in reversed(pts):
        while len(upper) >= 2 and _cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    return lower[:-1] + upper[:-1]


def exact_area(poly):
    n = len(poly)
    return sum(poly[i][0] * poly[(i + 1) % n][1] - poly[(i + 1) % n][0] * poly[i][1] for i in range(n)) / 2 if n >= 3 else Fraction(0)


def _clip(poly, e0, e1):
    out = []
    n = len(poly)
    for i in range(n):
        p, q = poly[i], poly[(i + 1) % n]
        sp, sq = _cross(e0, e1, p), _cross(e0, e1, q)
        if sp >= 0:
            out.append(p)
        if (sp > 0 > sq) or (sp < 0 < sq):
            t = sp / (sp - sq)
            out.append((p[0] + t * (q[0] - p[0]), p[1] + t * (q[1] - p[1])))
    return out


def exact_iou(qa, qb) -> float:
    """IoU of the convex hulls of two quads, exactly, rounded once to float."""
    ha, hb = exact_hull(qa), exact_hull(qb)
    aa, ab = exact_area(ha), exact_area(hb)
    if aa <= 0 or ab <= 0:
        return 0.0
    poly = ha
    for i in range(len(hb)):
        if not poly:
            break
        poly = _clip(poly, hb[i], hb[(i + 1) % len(hb)])
    inter = exact_area(poly)
    return float(inter / (aa + ab - inter))


def rotated_rect(cx, cy, w, h, theta):
    """[4, 2] corners of a w x h rectangle centred at (cx, cy), rotated by theta, in CCW order (y up)."""
    c, s = np.cos(theta), np.sin(theta)
    dx = np.array([-w, w, w, -w]) / 2
    dy = np.array([-h, -h, h, h]) / 2
    return np.stack([cx + c * dx - s * dy, cy + s * dx + c * dy], 1)
