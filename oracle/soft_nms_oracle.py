"""Class-aware Soft-NMS restated in numpy from the paper (Bodla et al., "Soft-NMS -- Improving Object Detection With
One Line of Code", ICCV 2017, Algorithm 1; the semantics of mmcv's soft_nms), as include/sihl_od.h defines it:

    s = scores (fp32); alive = boxes with s >= score_thr
    until max_out boxes are emitted or nothing is alive:
        m = alive box with the largest s; ties -> lowest index
        emit (m, s[m]); alive -= {m}
        for every alive j with class[j] == class[m]:
            iou = inter / ((area_m + area_j) - inter)        fp32; NaN (two empty boxes) -> 0
            linear:   w = 1 - iou if iou > iou_thr else 1    fp32
            gaussian: w = float32(exp(-iou^2 / sigma))       in fp64, rounded once
            s[j] = s[j] * w                                  fp32
            j dies once not (s[j] >= score_thr)

Test infrastructure only (numpy, CPU).  The thresholds and sigma are the fp32 values the C entry points receive.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

f32 = np.float32
METHODS = ("linear", "gaussian")


def box_iou(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """IoU of box a [4] with boxes b [n,4] in fp32, torchvision's CPU nms operator order; NaN mapped to 0."""
    a = a.astype(f32)
    b = b.astype(f32)
    area_a = (a[2] - a[0]) * (a[3] - a[1])
    area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    w = np.fmax(f32(0), np.fmin(a[2], b[:, 2]) - np.fmax(a[0], b[:, 0]))
    h = np.fmax(f32(0), np.fmin(a[3], b[:, 3]) - np.fmax(a[1], b[:, 1]))
    inter = w * h
    with np.errstate(invalid="ignore", divide="ignore"):
        iou = inter / ((area_a + area_b) - inter)
    return np.where(np.isnan(iou), f32(0), iou).astype(f32)


def weights(iou: np.ndarray, method: str, iou_thr: float, sigma: float) -> np.ndarray:
    if method == "linear":
        thr = f32(iou_thr)
        return np.where(iou > thr, f32(1) - iou, f32(1)).astype(f32)
    if method == "gaussian":
        i64 = iou.astype(np.float64)
        return np.exp(-(i64 * i64) / np.float64(f32(sigma))).astype(f32)
    raise ValueError(method)


def soft_nms(boxes, scores, classes, method: str, iou_thr: float = 0.3, sigma: float = 0.5, score_thr: float = 0.001,
             max_out: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
    """Returns (kept indices in selection order int64, their decayed scores fp32).  Ties go to the lowest index, so a
    caller that wants another tie order passes the boxes in that order."""
    boxes = np.asarray(boxes, f32).reshape(-1, 4)
    s = np.asarray(scores, f32).copy()
    classes = np.asarray(classes).astype(np.int64)
    n = s.shape[0]
    max_out = n if max_out is None else int(max_out)
    thr = f32(score_thr)
    alive = s >= thr
    keep, kept_scores = [], []
    while len(keep) < max_out:
        live = np.flatnonzero(alive)
        if live.size == 0:
            break
        m = int(live[np.argmax(s[live])])            # argmax returns the first of equal maxima: the lowest index
        keep.append(m)
        kept_scores.append(s[m])
        alive[m] = False
        j = live[(classes[live] == classes[m]) & (live != m)]
        if j.size == 0:
            continue
        s[j] = s[j] * weights(box_iou(boxes[m], boxes[j]), method, iou_thr, sigma)
        alive[j] = s[j] >= thr
    return np.asarray(keep, np.int64), np.asarray(kept_scores, f32)


def soft_nms_candidates(key, box, cls, method: str, iou_thr: float, sigma: float, score_thr: float, k: int):
    """The oracle on one image's candidate list as the dense decode writes it (uint64 key = score bits << 32 |
    ~location): ties between equal scores go to the lowest location.  Returns (num, scores [k], classes [k],
    boxes [k,4]) zero padded like sihl_od_soft_nms_topk."""
    key = np.asarray(key).view(np.uint64)
    loc = (~key & np.uint64(0xFFFFFFFF)).astype(np.int64)
    order = np.argsort(loc, kind="stable")
    score = (key >> np.uint64(32)).astype(np.uint32).view(f32)[order]
    b, c = np.asarray(box, f32).reshape(-1, 4)[order], np.asarray(cls)[order]
    idx, sc = soft_nms(b, score, c, method, iou_thr, sigma, score_thr, k)
    m = idx.size
    out_s, out_c, out_b = np.zeros(k, f32), np.zeros(k, np.int64), np.zeros((k, 4), f32)
    out_s[:m], out_c[:m], out_b[:m] = sc, c[idx], b[idx]
    return m, out_s, out_c, out_b
