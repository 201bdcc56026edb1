"""Reference for the polygon-IoU COCO matching (sihl_od_quad_map_match): the host build of od_math.h's hull area and hull
IoU (tests/host_quad_map_shim.cpp, compiled with -ffp-contract=off into a temporary directory) and the COCOeval matching
loop on given IoUs and areas.

oracle/map_oracle.match_image restates COCOeval.evaluateImg with the box IoU and area built in.  match_image below is the
same loop over given IoUs and areas (tests/test_quad_map_oracle.py checks it equals map_oracle's on boxes), and
match_image_quads feeds it the shim's hull IoUs and hull areas, widened to double as the kernel does."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32
_shim = None


def shim() -> C.CDLL:
    global _shim
    if _shim is None:
        tmp = tempfile.mkdtemp(prefix="sihl_quad_map_shim_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libquad_map_shim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                               os.path.join(HERE, "host_quad_map_shim.cpp"), "-o", out])
        lib = C.CDLL(out)
        lib.shim_quad_hull_areas.argtypes = [C.c_void_p, C.c_long, C.c_void_p]
        lib.shim_quad_hull_areas.restype = None
        lib.shim_quad_iou_grid.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.c_void_p]
        lib.shim_quad_iou_grid.restype = None
        _shim = lib
    return _shim


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def quad_hull_areas(quads) -> np.ndarray:
    """Host hull area (fp32) of each quad ([n, 4, 2] or [n, 8])."""
    q = np.ascontiguousarray(np.asarray(quads, f32).reshape(-1, 8))
    out = np.empty(len(q), f32)
    shim().shim_quad_hull_areas(_ptr(q), len(q), _ptr(out))
    return out


def quad_iou_grid(a, b) -> np.ndarray:
    """Host [len(a), len(b)] fp32 quad_iou, each hull built once."""
    a = np.ascontiguousarray(np.asarray(a, f32).reshape(-1, 8))
    b = np.ascontiguousarray(np.asarray(b, f32).reshape(-1, 8))
    out = np.empty((len(a), len(b)), f32)
    shim().shim_quad_iou_grid(_ptr(a), len(a), _ptr(b), len(b), _ptr(out))
    return out


def match_image(det_scores, det_classes, gt_classes, ious, d_area, g_area, iou_thresholds, area_ranges):
    """COCOeval.evaluateImg of one image on precomputed ious [D, G] and areas (double).  Returns map_oracle.match_image's
    dict: order [K], dt_match [NA,T,K] by rank, dt_ignore [NA,T,K], gt_ignore [NA,G]."""
    det_scores = np.asarray(det_scores, np.float32)
    K, G, T, NA = len(det_scores), len(g_area), len(iou_thresholds), len(area_ranges)
    order = np.argsort(-det_scores.astype(np.float64), kind="mergesort")
    dt_match = -np.ones((NA, T, K), np.int32)
    dt_ignore = np.zeros((NA, T, K), np.uint8)
    gt_ignore = np.zeros((NA, G), np.uint8)
    for a, (lo, hi) in enumerate(area_ranges):
        gt_ignore[a] = (g_area < lo) | (g_area > hi)
        by_class = {}                                                              # gts of each class, ignored last
        for c in set(int(c) for c in gt_classes):
            by_class[c] = sorted([g for g in range(G) if gt_classes[g] == c], key=lambda g: gt_ignore[a, g])
        for t, thr in enumerate(iou_thresholds):
            taken = np.zeros(G, bool)
            for r, d in enumerate(order):
                gts = by_class.get(int(det_classes[d]), [])
                best, m = min(thr, 1 - 1e-10), -1
                for g in gts:
                    if taken[g]:
                        continue
                    if m > -1 and gt_ignore[a, m] == 0 and gt_ignore[a, g] == 1:
                        break
                    if ious[d, g] < best:
                        continue
                    best, m = ious[d, g], g
                if m == -1:
                    dt_ignore[a, t, r] = d_area[d] < lo or d_area[d] > hi
                    continue
                dt_ignore[a, t, r] = gt_ignore[a, m]
                dt_match[a, t, r] = m
                taken[m] = True
    return dict(order=order.astype(np.int32), dt_match=dt_match, dt_ignore=dt_ignore, gt_ignore=gt_ignore)


def match_image_quads(det_quads, det_scores, det_classes, gt_quads, gt_classes, iou_thresholds, area_ranges):
    """The quad oracle: match_image on the shim's hull IoUs and hull areas."""
    dq = np.asarray(det_quads, f32).reshape(-1, 8)
    gq = np.asarray(gt_quads, f32).reshape(-1, 8)
    ious = quad_iou_grid(dq, gq).astype(np.float64) if len(gq) else np.zeros((len(dq), 0))
    return match_image(det_scores, det_classes, gt_classes, ious, quad_hull_areas(dq).astype(np.float64),
                       quad_hull_areas(gq).astype(np.float64), iou_thresholds, area_ranges)
