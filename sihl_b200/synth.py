"""Synthetic inputs for the ObjectDetection-head hot path (SURVEY.md §8d).

Two generators with the same distributions:

* ``numpy`` (``np.random.RandomState`` — a frozen bit stream, so the committed
  golden fixtures can store a seed instead of the inputs) for tests and golden
  vectors;
* ``torch`` on a device (``torch.Generator``) for ``bench.py``.

Distributions (SURVEY.md §8d): level sizes from the image size, gt box sides
log-uniform in ``[8, 0.625*S]`` px with uniform centres, clamped to the image,
redrawn when a side collapses below 1 px, non-integer coordinates;
``loc_logits ~ N(-5, 1)`` (the head's initial bias, reference
``object_detection.py:58``), ``iou_preds ~ U(0,1)``, ``box_raw ~ N(0, 0.5^2)``,
``cls_logits ~ N(0, 1)``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np


def level_sizes(height: int, width: int, bottom_level: int = 3, top_level: int = 7,
                mode: str = "ceil") -> List[Tuple[int, int]]:
    """Feature-map sizes ``(h_l, w_l)`` for levels ``bottom..top``.

    ``mode="ceil"`` halves with ceil at every level (what stride-2 convs with
    padding produce: 320 -> 160, 80, 40, 20, 10, 5, 3), ``mode="floor"`` uses
    ``S // 2**l``.  The head itself never assumes either: it reads the sizes
    off the tensors it is given (reference ``object_detection.py:87``).
    """
    sizes = []
    for level in range(bottom_level, top_level + 1):
        if mode == "floor":
            sizes.append((max(height // 2 ** level, 1), max(width // 2 ** level, 1)))
        else:
            h, w = height, width
            for _ in range(level):
                h, w = (h + 1) // 2, (w + 1) // 2
            sizes.append((h, w))
    return sizes


def num_anchors(levels: Sequence[Tuple[int, int]]) -> int:
    return int(sum(h * w for h, w in levels))


def gt_boxes_np(rng: np.random.RandomState, n: int, height: int, width: int,
                min_side: float = 8.0, max_frac: float = 0.625) -> np.ndarray:
    """``n`` xyxy pixel boxes, fp32, non-lattice coordinates (SURVEY.md §3.4)."""
    out = np.zeros((n, 4), dtype=np.float32)
    s = float(min(height, width))
    lo, hi = math.log(min_side), math.log(max(max_frac * s, min_side * 1.5))
    i = 0
    while i < n:
        bw, bh = np.exp(rng.uniform(lo, hi, size=2))
        cx, cy = rng.uniform(0, width), rng.uniform(0, height)
        x1, y1 = max(cx - bw / 2, 0.0), max(cy - bh / 2, 0.0)
        x2, y2 = min(cx + bw / 2, float(width)), min(cy + bh / 2, float(height))
        box = np.array([x1, y1, x2, y2], dtype=np.float32)
        if box[2] - box[0] < 1.0 or box[3] - box[1] < 1.0:
            continue
        out[i] = box
        i += 1
    return out


@dataclass
class GtBatch:
    """Ragged ground truth in CSR form (what the C-ABI consumes)."""
    boxes: np.ndarray      # [sumG, 4] f32 xyxy px
    classes: np.ndarray    # [sumG] i64
    offsets: np.ndarray    # [B+1] i32

    @property
    def batch_size(self) -> int:
        return len(self.offsets) - 1

    def per_image(self):
        for b in range(self.batch_size):
            s, e = int(self.offsets[b]), int(self.offsets[b + 1])
            yield self.boxes[s:e], self.classes[s:e]


def gt_batch_np(seed: int, batch: int, height: int, width: int, num_classes: int,
                max_gt: int, ragged: bool = True, counts: Optional[Sequence[int]] = None,
                integer_coords: bool = False) -> GtBatch:
    """Ragged (``G_b ~ U{0..max_gt}``, image 0 empty when ``batch>1``) or full."""
    rng = np.random.RandomState(seed)
    if counts is None:
        if ragged:
            counts = [int(rng.randint(0, max_gt + 1)) for _ in range(batch)]
            if batch > 1:
                counts[0] = 0
            if batch > 2:
                counts[1] = max_gt
        else:
            counts = [max_gt] * batch
    boxes, classes = [], []
    for n in counts:
        b = gt_boxes_np(rng, n, height, width)
        if integer_coords:
            b = np.round(b).astype(np.float32)
        boxes.append(b)
        classes.append(rng.randint(0, num_classes, size=n).astype(np.int64))
    offsets = np.zeros(len(counts) + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(counts)
    return GtBatch(np.concatenate(boxes).reshape(-1, 4).astype(np.float32),
                   np.concatenate(classes).astype(np.int64), offsets)


@dataclass
class DenseMaps:
    loc_logits: np.ndarray   # [B, A]
    iou_preds: np.ndarray    # [B, A]
    box_raw: np.ndarray      # [B, A, 4]
    cls_logits: np.ndarray   # [B, A, C]


def dense_maps_np(seed: int, batch: int, anchors: int, num_classes: int,
                  loc_mean: float = -5.0, loc_std: float = 1.0) -> DenseMaps:
    rng = np.random.RandomState(seed)
    f32 = np.float32
    return DenseMaps(
        loc_logits=(loc_mean + loc_std * rng.standard_normal((batch, anchors))).astype(f32),
        iou_preds=rng.uniform(0, 1, (batch, anchors)).astype(f32),
        box_raw=(0.5 * rng.standard_normal((batch, anchors, 4))).astype(f32),
        cls_logits=rng.standard_normal((batch, anchors, num_classes)).astype(f32),
    )


def nms_candidates_np(seed: int, n: int, size: int, num_classes: int = 80):
    """NMS stress inputs (SURVEY.md §8d config[3]): sides U(4, 0.3*S), scores U(0.05,1)."""
    rng = np.random.RandomState(seed)
    w = rng.uniform(4, 0.3 * size, n)
    h = rng.uniform(4, 0.3 * size, n)
    cx, cy = rng.uniform(0, size, n), rng.uniform(0, size, n)
    boxes = np.stack([np.clip(cx - w / 2, 0, size), np.clip(cy - h / 2, 0, size),
                      np.clip(cx + w / 2, 0, size), np.clip(cy + h / 2, 0, size)], 1).astype(np.float32)
    bad = (boxes[:, 2] - boxes[:, 0] < 1) | (boxes[:, 3] - boxes[:, 1] < 1)
    boxes[bad] = np.array([0, 0, 8, 8], np.float32) + rng.uniform(0, size - 8, (int(bad.sum()), 1)).astype(np.float32)
    scores = rng.uniform(0.05, 1.0, n).astype(np.float32)
    classes = rng.randint(0, num_classes, n).astype(np.int64)
    return boxes, scores, classes


def quad_candidates_np(seed: int, n: int, size: int, num_classes: int = 80):
    """Quadrilateral NMS inputs: quads [n, 4, 2] f32 (four points (x, y) in [0, size]), scores U(0.05, 1) f32, classes
    int64.  Rotated rectangles (sides U(4, 0.15*S) x U(2, 0.05*S), any angle) with vertex jitter, in clusters of up to
    8 near-duplicates of one class (a detector's overlapping proposals) and, for a quarter of the clusters, a parallel
    neighbour shifted across its short side (slanted text lines: high AABB IoU, little or no polygon overlap)."""
    rng = np.random.RandomState(seed)
    quads = np.empty((n, 4, 2), np.float64)
    classes = np.empty(n, np.int64)
    i = 0
    while i < n:
        m = min(n - i, int(rng.randint(1, 9)))
        w, h = rng.uniform(4, 0.15 * size), rng.uniform(2, 0.05 * size)
        th = rng.uniform(-np.pi, np.pi)
        cx, cy = rng.uniform(0, size), rng.uniform(0, size)
        c, s = np.cos(th), np.sin(th)
        cls = rng.randint(0, num_classes)
        for k in range(m):
            if k == 1 and rng.rand() < 0.25:                      # parallel neighbour, one to two line heights away
                off = h * rng.uniform(1.0, 2.0)
                ccx, ccy, ww, hh = cx - s * off, cy + c * off, w, h
            else:                                                 # near-duplicate
                ccx, ccy = cx + rng.normal(0, 0.1 * h), cy + rng.normal(0, 0.1 * h)
                ww, hh = w * rng.uniform(0.9, 1.1), h * rng.uniform(0.9, 1.1)
            dx, dy = np.array([-ww, ww, ww, -ww]) / 2, np.array([-hh, -hh, hh, hh]) / 2
            q = np.stack([ccx + c * dx - s * dy, ccy + s * dx + c * dy], 1)
            quads[i] = q + rng.normal(0, 0.03 * hh, (4, 2))
            classes[i] = cls
            i += 1
    quads = np.clip(quads, 0, size).astype(np.float32)
    scores = rng.uniform(0.05, 1.0, n).astype(np.float32)
    return quads, scores, classes


def _rect_corners(cx, cy, w, h, th):
    """[..., 4, 2] corners of w x h rectangles centred at (cx, cy), rotated by th."""
    c, s = np.cos(th)[..., None], np.sin(th)[..., None]
    dx = np.array([-0.5, 0.5, 0.5, -0.5]) * w[..., None]
    dy = np.array([-0.5, -0.5, 0.5, 0.5]) * h[..., None]
    return np.stack([cx[..., None] + c * dx - s * dy, cy[..., None] + s * dx + c * dy], -1)


def quad_map_batch_np(seed: int, batch: int, k: int, gt_per_image: int, num_classes: int = 80, size: int = 1024,
                      counts=None):
    """Quad mAP inputs in the layout of ops.quad_map_match: ground truth = ``counts[b]`` (default ``gt_per_image``)
    rotated rectangles per image (long side log-uniform in [6, 0.2*S], aspect down to 1:20, any angle); detections
    [B, K] = jittered copies of a gt of the image (60%: centre, size, angle and vertices perturbed; 90% of them with the
    gt's class), parallel-line decoys (20%: a copy shifted across its short side by one to two line heights, so its
    AABB overlaps the gt's and its polygon barely or not) and random rectangles.  Scores are U(0, 1) rounded to two
    decimals (exact ties).  Returns det_quads [B,K,4,2] f32, det_scores [B,K] f32, det_classes [B,K] i64, gt_quads
    [sumG,4,2] f32, gt_classes [sumG] i64, gt_offsets [B+1] i32."""
    rng = np.random.RandomState(seed)
    counts = np.full(batch, gt_per_image, np.int64) if counts is None else np.asarray(counts, np.int64)
    offsets = np.zeros(batch + 1, np.int32)
    offsets[1:] = np.cumsum(counts)
    G = int(offsets[-1])
    gw = np.exp(rng.uniform(np.log(6.0), np.log(0.2 * size), G))
    gh = np.maximum(gw * rng.uniform(0.05, 1.0, G), 3.0)
    gth = rng.uniform(-np.pi, np.pi, G)
    gcx, gcy = rng.uniform(0.1 * size, 0.9 * size, G), rng.uniform(0.1 * size, 0.9 * size, G)
    gt_classes = rng.randint(0, num_classes, G).astype(np.int64)
    gt_quads = _rect_corners(gcx, gcy, gw, gh, gth)
    # detections: pick a gt of the image for each row (images without gt get random rectangles only)
    u = rng.uniform(0, 1, (batch, k))
    pick = offsets[:-1, None] + np.floor(rng.uniform(0, 1, (batch, k)) * np.maximum(counts, 1)[:, None]).astype(np.int64)
    has = (counts > 0)[:, None] & np.ones((batch, k), bool)
    pick = np.where(has, np.minimum(pick, max(G - 1, 0)), 0)
    copy, decoy = has & (u < 0.6), has & (u >= 0.6) & (u < 0.8)
    src = lambda a, fill: np.where(has, a[pick] if G else fill, fill)
    w, h, th = src(gw, 1.0), src(gh, 1.0), src(gth, 0.0)
    cx, cy = src(gcx, 0.0), src(gcy, 0.0)
    jw, jh = rng.uniform(0.9, 1.1, (batch, k)), rng.uniform(0.9, 1.1, (batch, k))
    w, h, th = w * jw, h * jh, th + rng.normal(0, 0.05, (batch, k))
    cx, cy = cx + rng.normal(0, 0.1, (batch, k)) * h, cy + rng.normal(0, 0.1, (batch, k)) * h
    off = h * rng.uniform(1.0, 2.0, (batch, k))
    cx, cy = np.where(decoy, cx - np.sin(th) * off, cx), np.where(decoy, cy + np.cos(th) * off, cy)
    rand = ~(copy | decoy)
    rw = np.exp(rng.uniform(np.log(6.0), np.log(0.2 * size), (batch, k)))
    w = np.where(rand, rw, w)
    h = np.where(rand, np.maximum(rw * rng.uniform(0.05, 1.0, (batch, k)), 3.0), h)
    th = np.where(rand, rng.uniform(-np.pi, np.pi, (batch, k)), th)
    cx = np.where(rand, rng.uniform(0.1 * size, 0.9 * size, (batch, k)), cx)
    cy = np.where(rand, rng.uniform(0.1 * size, 0.9 * size, (batch, k)), cy)
    det_quads = _rect_corners(cx, cy, w, h, th)
    det_quads = det_quads + rng.normal(0, 0.03, (batch, k, 4, 2)) * h[..., None, None] * copy[..., None, None]
    keep_cls = copy & (rng.uniform(0, 1, (batch, k)) < 0.9) | decoy
    det_classes = np.where(keep_cls, src(gt_classes, 0), rng.randint(0, num_classes, (batch, k))).astype(np.int64)
    det_scores = np.round(rng.uniform(0, 1, (batch, k)), 2).astype(np.float32)
    return (det_quads.astype(np.float32), det_scores, det_classes, gt_quads.astype(np.float32), gt_classes, offsets)


def map_crowd_batch_np(seed: int, batch: int, k: int, gt_per_image: int, num_classes: int = 80, geometry: str = "box",
                       size: int = 1024, counts=None, crowd_frac: float = 0.1):
    """mAP inputs with COCO's ``iscrowd`` / ``area`` annotations for ops.map_match (``geometry="box"``: the AABBs) or
    ops.quad_map_match (``"quad"``), built on :func:`quad_map_batch_np`.  About ``crowd_frac`` of the gts become crowd
    ("don't care") regions: large rectangles of 0.2 to 0.45 S a side, each with a cluster of up to 6 small same-class
    detections inside it.  ``gt_area``: 30% zeros and 5% negative (the computed area is used), 30% the gt's own
    area scaled by U(0.3, 3), the rest drawn near the 32^2 and 96^2 range boundaries (so gts move between small, medium and
    large).  Returns det [B,K,4] xyxy or [B,K,4,2], det_scores, det_classes, gt [sumG,4] or [sumG,4,2], gt_classes,
    gt_offsets, gt_crowd uint8 [sumG], gt_area float64 [sumG]."""
    if geometry not in ("box", "quad"):
        raise ValueError(f"geometry must be 'box' or 'quad', got {geometry!r}")
    dq, ds, dc, gq, gc, go = quad_map_batch_np(seed, batch, k, gt_per_image, num_classes, size, counts)
    rng = np.random.RandomState(seed + 7919)
    G = int(go[-1])
    crowd = (rng.uniform(0, 1, G) < crowd_frac).astype(np.uint8)
    for g in np.nonzero(crowd)[0]:
        b = int(np.searchsorted(go, g, side="right") - 1)
        cw, ch = rng.uniform(0.2, 0.45, 2) * size
        cx, cy = rng.uniform(0.25 * size, 0.75 * size, 2)
        th = rng.uniform(-np.pi, np.pi) if geometry == "quad" else 0.0
        gq[g] = _rect_corners(np.array(cx), np.array(cy), np.array(cw), np.array(ch), np.array(th))
        rows = rng.choice(k, size=min(6, k), replace=False)
        u, v = rng.uniform(-0.35, 0.35, (2, len(rows)))
        px, py = cx + np.cos(th) * u * cw - np.sin(th) * v * ch, cy + np.sin(th) * u * cw + np.cos(th) * v * ch
        w = rng.uniform(0.05, 0.2, len(rows)) * cw
        h = w * rng.uniform(0.3, 1.0, len(rows))
        dq[b, rows] = _rect_corners(px, py, w, h, th + rng.normal(0, 0.05, len(rows)))
        dc[b, rows] = gc[g]
    hull = np.abs(np.array([_shoelace(q) for q in gq.reshape(-1, 4, 2)])) if G else np.zeros(0)
    pick = rng.uniform(0, 1, G)
    near = np.where(rng.uniform(0, 1, G) < 0.5, 32.0, 96.0) ** 2 * rng.uniform(0.9, 1.1, G)
    gt_area = np.where(pick < 0.3, 0.0, np.where(pick < 0.35, -1.0, np.where(pick < 0.65, hull * rng.uniform(0.3, 3, G), near)))
    if geometry == "box":
        aabb = lambda q: np.concatenate([q.min(-2), q.max(-2)], -1).astype(np.float32)
        return aabb(dq), ds, dc, aabb(gq), gc, go, crowd, gt_area.astype(np.float64)
    return dq.astype(np.float32), ds, dc, gq.astype(np.float32), gc, go, crowd, gt_area.astype(np.float64)


def _shoelace(q) -> float:
    x, y = q[:, 0].astype(np.float64), q[:, 1].astype(np.float64)
    return 0.5 * float(np.dot(x, np.roll(y, -1)) - np.dot(y, np.roll(x, -1)))


# ----------------------------------------------------------------------------
# device-side generator for bench.py (torch imported lazily: synth is also used
# by numpy-only code)
# ----------------------------------------------------------------------------
def gt_batch_torch(gen, batch: int, height: int, width: int, num_classes: int, max_gt: int,
                   device, min_side: float = 8.0, max_frac: float = 0.625):
    """Full (``G_b == max_gt``) gt batch generated on ``device``.

    Returns ``(boxes [B*G,4] f32, classes [B*G] i64, offsets [B+1] i32)``.
    Boxes whose side collapses under 1 px after clamping are replaced by a
    centred box of the minimum side (the numpy generator redraws instead).
    """
    import torch
    n = batch * max_gt
    s = float(min(height, width))
    lo, hi = math.log(min_side), math.log(max(max_frac * s, min_side * 1.5))
    u = torch.rand((n, 4), generator=gen, device=device, dtype=torch.float64)
    bw = torch.exp(lo + (hi - lo) * u[:, 0])
    bh = torch.exp(lo + (hi - lo) * u[:, 1])
    cx, cy = u[:, 2] * width, u[:, 3] * height
    x1, y1 = (cx - bw / 2).clamp(min=0), (cy - bh / 2).clamp(min=0)
    x2, y2 = (cx + bw / 2).clamp(max=width), (cy + bh / 2).clamp(max=height)
    bad = ((x2 - x1) < 1) | ((y2 - y1) < 1)
    x1 = torch.where(bad, torch.full_like(x1, width / 2 - min_side / 2 + 0.37), x1)
    x2 = torch.where(bad, torch.full_like(x2, width / 2 + min_side / 2 + 0.37), x2)
    y1 = torch.where(bad, torch.full_like(y1, height / 2 - min_side / 2 + 0.41), y1)
    y2 = torch.where(bad, torch.full_like(y2, height / 2 + min_side / 2 + 0.41), y2)
    boxes = torch.stack([x1, y1, x2, y2], 1).to(torch.float32).contiguous()
    classes = torch.randint(0, num_classes, (n,), generator=gen, device=device, dtype=torch.int64)
    offsets = (torch.arange(batch + 1, device=device, dtype=torch.int32) * max_gt).contiguous()
    return boxes, classes, offsets


def dense_maps_torch(gen, batch: int, anchors: int, num_classes: int, device,
                     loc_mean: float = -5.0, loc_std: float = 1.0):
    import torch
    f32 = torch.float32
    loc = torch.randn((batch, anchors), generator=gen, device=device, dtype=f32) * loc_std + loc_mean
    iou = torch.rand((batch, anchors), generator=gen, device=device, dtype=f32)
    box = torch.randn((batch, anchors, 4), generator=gen, device=device, dtype=f32) * 0.5
    cls = torch.randn((batch, anchors, num_classes), generator=gen, device=device, dtype=f32)
    return loc, iou, box, cls
