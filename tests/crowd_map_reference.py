"""Reference for COCO's optional ground-truth annotations in the matching (sihl_od_map_match_crowd,
sihl_od_quad_map_match_crowd): ``iscrowd`` and ``area``, restated from pycocotools ``COCOeval._prepare`` /
``computeIoU`` / ``evaluateImg`` and torchmetrics 1.6 ``_get_coco_format``.  Neither library is installed here: parity
is UNPINNED, as for the rest of the COCO restatement (oracle/map_oracle.py).

Rules: a gt's range area is its annotated area when that is > 0, else the computed one (box: fp32 w and h multiplied
in double; quad: the hull area widened); a crowd gt is ignored in every area range; its overlap with a detection is
``maskUtils.iou(..., iscrowd=1)``, the intersection over the detection's area; it stays matchable after a match
(``if gtm[tind, gind] > 0 and not iscrowd[gind]: continue``), so a detection matched to it inherits its ignore flag.

``match_image`` is the COCOeval loop of oracle/map_oracle.py and tests/quad_map_reference.py with those two changes,
on given overlaps and areas; ``match_image_boxes`` / ``match_image_quads`` feed it the box overlaps of map_oracle plus
the box IoA below, or the host build of od_math.h's hull IoU and hull area (tests/quad_map_reference.py) plus its hull
IoA (tests/host_quad_ioa_shim.cpp, compiled with -ffp-contract=off into a temporary directory).  Without annotations
they give the tables of map_oracle.match_image and quad_map_reference.match_image_quads
(tests/test_map_crowd_oracle.py checks it)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import quad_map_reference as qm
from oracle import map_oracle as mo

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32
_shim = None


def shim() -> C.CDLL:
    global _shim
    if _shim is None:
        tmp = tempfile.mkdtemp(prefix="sihl_quad_ioa_shim_")
        atexit.register(shutil.rmtree, tmp, True)
        out = os.path.join(tmp, "libquad_ioa_shim.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                               os.path.join(HERE, "host_quad_ioa_shim.cpp"), "-o", out])
        lib = C.CDLL(out)
        lib.shim_quad_ioa_grid.argtypes = [C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.c_void_p]
        lib.shim_quad_ioa_grid.restype = None
        _shim = lib
    return _shim


def quad_ioa_grid(a, b) -> np.ndarray:
    """Host [len(a), len(b)] fp32 intersection of the hulls over the hull area of a's quad, each hull built once."""
    a = np.ascontiguousarray(np.asarray(a, f32).reshape(-1, 8))
    b = np.ascontiguousarray(np.asarray(b, f32).reshape(-1, 8))
    out = np.empty((len(a), len(b)), f32)
    shim().shim_quad_ioa_grid(a.ctypes.data_as(C.c_void_p), len(a), b.ctypes.data_as(C.c_void_p), len(b),
                              out.ctypes.data_as(C.c_void_p))
    return out


def box_ioa(d, g) -> np.ndarray:
    """maskUtils.iou for boxes with iscrowd = 1 (bbIou, union = the detection's area), double precision -> [D, G]."""
    d = np.asarray(d, np.float32).reshape(-1, 4); g = np.asarray(g, np.float32).reshape(-1, 4)
    dw, dh = mo._wh32(d); gw, gh = mo._wh32(g)
    dx, dy, gx, gy = d[:, 0].astype(np.float64), d[:, 1].astype(np.float64), g[:, 0].astype(np.float64), g[:, 1].astype(np.float64)
    out = np.zeros((len(d), len(g)))
    for i in range(len(d)):
        for j in range(len(g)):
            w = min(dx[i] + dw[i], gx[j] + gw[j]) - max(dx[i], gx[j])
            if w <= 0:
                continue
            h = min(dy[i] + dh[i], gy[j] + gh[j]) - max(dy[i], gy[j])
            if h <= 0:
                continue
            out[i, j] = w * h / (dw[i] * dh[i])
    return out


def _crowd(gt_crowd, G) -> np.ndarray:
    return np.zeros(G, bool) if gt_crowd is None else np.asarray(gt_crowd).reshape(-1) != 0


def range_areas(computed, gt_area) -> np.ndarray:
    """The area of each gt for the range test: the annotation where it is > 0 (NaN is not), else the computed one."""
    computed = np.asarray(computed, np.float64)
    if gt_area is None or computed.size == 0:
        return computed
    given = np.asarray(gt_area, np.float64).reshape(-1)
    return np.where(given > 0, given, computed)


def match_image(det_scores, det_classes, gt_classes, ious, d_area, g_area, iou_thresholds, area_ranges, gt_crowd=None):
    """COCOeval.evaluateImg of one image on precomputed overlaps [D, G] (the IoA in crowd columns) and range areas
    (double).  Returns map_oracle.match_image's dict: order [K], dt_match [NA,T,K] by rank, dt_ignore [NA,T,K],
    gt_ignore [NA,G]."""
    det_scores = np.asarray(det_scores, np.float32)
    K, G, T, NA = len(det_scores), len(g_area), len(iou_thresholds), len(area_ranges)
    crowd = _crowd(gt_crowd, G)
    order = np.argsort(-det_scores.astype(np.float64), kind="mergesort")
    dt_match = -np.ones((NA, T, K), np.int32)
    dt_ignore = np.zeros((NA, T, K), np.uint8)
    gt_ignore = np.zeros((NA, G), np.uint8)
    for a, (lo, hi) in enumerate(area_ranges):
        gt_ignore[a] = crowd | (g_area < lo) | (g_area > hi)
        by_class = {}                                                              # gts of each class, ignored last
        for c in set(int(c) for c in gt_classes):
            by_class[c] = sorted([g for g in range(G) if gt_classes[g] == c], key=lambda g: gt_ignore[a, g])
        for t, thr in enumerate(iou_thresholds):
            taken = np.zeros(G, bool)
            for r, d in enumerate(order):
                gts = by_class.get(int(det_classes[d]), [])
                best, m = min(thr, 1 - 1e-10), -1
                for g in gts:
                    if taken[g] and not crowd[g]:
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


def match_image_boxes(det_boxes, det_scores, det_classes, gt_boxes, gt_classes, iou_thresholds=mo.IOU_THRESHOLDS,
                      area_ranges=mo.AREA_RANGES, gt_crowd=None, gt_area=None):
    """The box oracle: map_oracle's box IoU (box_ioa in crowd columns) and box areas (annotated areas > 0 instead)."""
    K, G = len(det_scores), len(gt_boxes)
    crowd = _crowd(gt_crowd, G)
    ious = mo.box_iou(det_boxes, gt_boxes) if G else np.zeros((K, 0))
    if crowd.any():
        ious[:, crowd] = box_ioa(det_boxes, np.asarray(gt_boxes, np.float32).reshape(-1, 4)[crowd])
    g_area = range_areas(mo.box_area(gt_boxes) if G else np.zeros(0), gt_area)
    return match_image(det_scores, det_classes, gt_classes, ious, mo.box_area(det_boxes), g_area, iou_thresholds,
                       area_ranges, crowd)


def match_image_quads(det_quads, det_scores, det_classes, gt_quads, gt_classes, iou_thresholds=mo.IOU_THRESHOLDS,
                      area_ranges=mo.AREA_RANGES, gt_crowd=None, gt_area=None):
    """The quad oracle: the host hull IoU (hull IoA in crowd columns) and hull areas (annotated areas > 0 instead),
    widened to double as the kernels do."""
    dq = np.asarray(det_quads, f32).reshape(-1, 8)
    gq = np.asarray(gt_quads, f32).reshape(-1, 8)
    crowd = _crowd(gt_crowd, len(gq))
    ious = qm.quad_iou_grid(dq, gq).astype(np.float64) if len(gq) else np.zeros((len(dq), 0))
    if crowd.any():
        ious[:, crowd] = quad_ioa_grid(dq, gq[crowd]).astype(np.float64)
    g_area = range_areas(qm.quad_hull_areas(gq).astype(np.float64), gt_area)
    return match_image(det_scores, det_classes, gt_classes, ious, qm.quad_hull_areas(dq).astype(np.float64), g_area,
                       iou_thresholds, area_ranges, crowd)
