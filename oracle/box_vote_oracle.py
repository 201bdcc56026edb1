"""Class-aware box voting (merge-NMS) restated in numpy, as include/sihl_od.h defines it:

    for every kept box k of class c (keep sets from od_oracle.batched_nms / diou_nms_oracle.batched_diou_nms):
        V_k  = { j in the same list : class[j] == c and overlap(b_k, b_j) > thr }     k included; NaN never joins
        b'_k = sum_{j in V_k} s_j * b_j / sum_{j in V_k} s_j                           per coordinate
        b'_k = b_k when V_k is empty or the score sum is 0

overlap is the IoU of the hard NMS or the DIoU of DIoU-NMS, in fp32 and in the kernels' operator order (od_common.cuh
box_iou, od_math.h diou_pair).  The sums are exact (math.fsum over the fp64 products, each exact), then the quotient is
rounded to fp64 and once more to fp32.  The kernels sum in fp64 in another order, so a voted coordinate may differ from
this one in the last fp32 bit.

Test infrastructure only (numpy, CPU).  The thresholds are the fp32 values the C entry points receive.
"""
from __future__ import annotations

import math
from typing import Tuple

import numpy as np

from . import diou_nms_oracle as dno
from . import od_oracle as orc

f32 = np.float32
OVERLAPS = ("iou", "diou")


def overlap(kind: str, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """overlap(a, b[j]) of one box a [4] with boxes b [n,4] in fp32; NaN kept (two zero-area boxes)."""
    a = np.asarray(a, f32)
    b = np.asarray(b, f32).reshape(-1, 4)
    area_a = (a[2] - a[0]) * (a[3] - a[1])
    area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    w = np.fmax(f32(0), np.fmin(a[2], b[:, 2]) - np.fmax(a[0], b[:, 0]))
    h = np.fmax(f32(0), np.fmin(a[3], b[:, 3]) - np.fmax(a[1], b[:, 1]))
    inter = w * h
    with np.errstate(invalid="ignore", divide="ignore"):
        iou = inter / ((area_a + area_b) - inter)
        if kind == "iou":
            return iou.astype(f32)
        if kind != "diou":
            raise ValueError(kind)
        wi = np.fmax(f32(0), np.fmax(a[2], b[:, 2]) - np.fmin(a[0], b[:, 0]))
        hi = np.fmax(f32(0), np.fmax(a[3], b[:, 3]) - np.fmin(a[1], b[:, 1]))
        diag = ((wi * wi) + (hi * hi)) + f32(1e-7)
        dx = (a[0] + a[2]) / f32(2) - (b[:, 0] + b[:, 2]) / f32(2)
        dy = (a[1] + a[3]) / f32(2) - (b[:, 1] + b[:, 3]) / f32(2)
        cd = (dx * dx) + (dy * dy)
        return (iou - (cd / diag)).astype(f32)


def vote(box_k, cls_k, boxes, scores, classes, thr: float, kind: str) -> np.ndarray:
    """The voted box of one kept box (box_k, cls_k) over the list (boxes [n,4], scores [n], classes [n])."""
    box_k = np.asarray(box_k, f32)
    same = np.flatnonzero(np.asarray(classes) == cls_k)
    if same.size == 0:
        return box_k.copy()
    with np.errstate(invalid="ignore"):
        member = same[overlap(kind, box_k, boxes[same]) > f32(thr)]
    s = scores[member].astype(np.float64)
    total = math.fsum(s)
    if member.size == 0 or total == 0.0:
        return box_k.copy()
    b = boxes[member].astype(np.float64)
    return np.array([math.fsum(s * b[:, c]) / total for c in range(4)], np.float64).astype(f32)


def vote_boxes(boxes, scores, classes, keep, thr: float, kind: str = "iou") -> np.ndarray:
    """Voted boxes [len(keep), 4] of the kept indices of one list."""
    boxes, scores, classes = np.asarray(boxes, f32).reshape(-1, 4), np.asarray(scores, f32), np.asarray(classes, np.int64)
    out = np.empty((len(keep), 4), f32)
    for r, i in enumerate(np.asarray(keep, np.int64)):
        out[r] = vote(boxes[i], classes[i], boxes, scores, classes, thr, kind)
    return out


def batched_nms_vote(boxes, scores, classes, thr: float, kind: str = "iou") -> Tuple[np.ndarray, np.ndarray]:
    """(keep, voted boxes [len(keep), 4]): the keep set of the hard or DIoU oracle, then the vote."""
    boxes, scores, classes = np.asarray(boxes, f32).reshape(-1, 4), np.asarray(scores, f32), np.asarray(classes, np.int64)
    if kind == "iou":
        keep = orc.batched_nms(boxes, scores, classes, thr)
    elif kind == "diou":
        keep = dno.batched_diou_nms(boxes, scores, classes, thr)
    else:
        raise ValueError(kind)
    return keep, vote_boxes(boxes, scores, classes, keep, thr, kind)


def topk_vote(key, box, cls, count, thr: float, K: int, kind: str = "iou"):
    """The top-K entry on candidate lists (key [B, cap] uint64, box [B, cap, 4], cls [B, cap], count [B]): visit order
    (score desc, location asc) from the keys, the oracle's keep set, the first K survivors, their voted boxes.
    Returns (num_instances, scores, classes, boxes, boxes without voting), zero padded past num_instances."""
    key = np.asarray(key).view(np.uint64)
    B, cap = key.shape
    n = np.minimum(np.asarray(count, np.int64), cap)
    num = np.zeros(B, np.int64)
    scores, classes = np.zeros((B, K), f32), np.zeros((B, K), np.int64)
    voted, plain = np.zeros((B, K, 4), f32), np.zeros((B, K, 4), f32)
    for b in range(B):
        kb, bb, cb = key[b, :n[b]], np.asarray(box[b, :n[b]], f32), np.asarray(cls[b, :n[b]]).astype(np.int64)
        loc = np.uint64(0xFFFFFFFF) - (kb & np.uint64(0xFFFFFFFF))
        perm = np.argsort(loc, kind="stable")                              # index order = location order
        sc = (kb >> np.uint64(32)).astype(np.uint32).view(f32)
        sel = orc.batched_nms if kind == "iou" else dno.batched_diou_nms
        keep = perm[sel(bb[perm], sc[perm], cb[perm], thr)][:K]
        m = keep.size
        num[b] = m
        scores[b, :m], classes[b, :m], plain[b, :m] = sc[keep], cb[keep], bb[keep]
        voted[b, :m] = vote_boxes(bb, sc, cb, keep, thr, kind)
    return num, scores, classes, voted, plain
