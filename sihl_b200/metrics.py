"""Validation mAP with the detection <-> ground-truth matching on the GPU (SURVEY.md §8f N3).

The reference's head feeds ``torchmetrics.detection.mean_ap.MeanAveragePrecision(max_detection_thresholds=[1, 10, K],
backend="faster_coco_eval")`` (ref src/sihl/heads/object_detection.py:219-237, :245), which stores every batch and runs
COCOeval on the CPU at epoch end.  ``DetectionMAP`` keeps the interface the head uses (``to``, ``update``, ``compute``
-> dict with torchmetrics' scalar keys) but matches each batch right away with ``sihl_od_map_match`` (one CTA per image,
one greedy chain per IoU threshold x area range, fp64 box IoU) and keeps only the compact match tables; ``compute``
does COCOeval.accumulate / summarize on them — a few cumulative sums per category on the host.

``iou_type="quad"`` evaluates the QuadrilateralDetection head's four-vertex polygons instead of boxes: the matching is
``sihl_od_quad_map_match`` (the IoU of the convex hulls of the vertex sets, the hull's polygon area for the area ranges)
and everything after it is the same.

Targets may carry COCO's optional ``iscrowd`` and ``area`` keys, as torchmetrics and pycocotools read them; the matching
then runs through the ``_crowd`` entries (crowd regions and text datasets' "don't care" regions are ignored, and so are
the detections that land on them; an annotated area > 0 places a gt in the small / medium / large ranges).

Parity is UNPINNED: torchmetrics and faster_coco_eval are not installed where this was written; the algorithm is the
published COCOeval one (see oracle/map_oracle.py, which restates it independently for the tests).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
from torch import Tensor

from . import ops

RECALL_THRESHOLDS = np.linspace(0.0, 1.0, 101)


class DetectionMAP:
    """COCO mAP / mAR over everything passed to :meth:`update` since construction (or :meth:`reset`).  ``iou_type``:
    ``"bbox"`` (xyxy boxes, box IoU) or ``"quad"`` (quads ``[K, 4, 2]`` or ``[K, 8]``, polygon IoU of their hulls)."""

    IOU_TYPES = ("bbox", "quad")

    def __init__(self, max_detection_thresholds: Optional[Sequence[int]] = None,
                 iou_thresholds: Sequence[float] = ops.COCO_IOU_THRESHOLDS, sync_dist: bool = True,
                 iou_type: str = "bbox", **_ignored) -> None:
        if iou_type not in self.IOU_TYPES:
            raise ValueError(f"iou_type must be one of {self.IOU_TYPES}, got {iou_type!r}")
        self.iou_type = iou_type
        self.max_dets = sorted(int(m) for m in (max_detection_thresholds or (1, 10, 100)))
        self.iou_thresholds = tuple(float(t) for t in iou_thresholds)
        self.area_ranges = ops.COCO_AREA_RANGES
        self.sync_dist = sync_dist
        self.reset()

    # -- torchmetrics-compatible surface ------------------------------------------------------------------------
    def to(self, device) -> "DetectionMAP":
        return self

    def reset(self) -> None:
        self._batches: List[Dict[str, Tensor]] = []

    def update(self, preds: List[Dict[str, Tensor]], target: List[Dict[str, Tensor]]) -> None:
        """torchmetrics' signature (ref :230-236): per-image dicts ``scores`` / ``labels`` / ``boxes`` (xyxy px) and
        ``labels`` / ``boxes``.  Every image must carry the same number of detections (``forward`` returns K rows).
        With ``iou_type="quad"`` both read ``quads`` ([n, 4, 2] or [n, 8] px) in place of ``boxes``.  A target may also
        carry ``iscrowd`` (bool / integer) and ``area`` ([n] each, one value per ``labels`` entry); a missing key means
        zeros for that image, i.e. no crowd region and the computed area."""
        if self.iou_type == "quad":
            self._update_quads(preds, target)
            return
        scores = torch.stack([p["scores"] for p in preds])
        classes = torch.stack([p["labels"] for p in preds])
        boxes = torch.stack([p["boxes"] for p in preds])
        dev = scores.device
        counts = [int(t["boxes"].shape[0]) for t in target]
        gb = [t["boxes"].as_subclass(Tensor).reshape(-1, 4).to(device=dev, dtype=torch.float32) for t in target]
        gc = [t["labels"].as_subclass(Tensor).reshape(-1).to(device=dev, dtype=torch.int64) for t in target]
        gt_boxes = torch.cat(gb) if gb else torch.empty((0, 4), device=dev)
        gt_classes = torch.cat(gc) if gc else torch.empty((0,), dtype=torch.int64, device=dev)
        self.update_batch(scores, classes, boxes, gt_boxes, gt_classes, counts, **self._annotations(target, dev))

    def _update_quads(self, preds: List[Dict[str, Tensor]], target: List[Dict[str, Tensor]]) -> None:
        scores = torch.stack([p["scores"] for p in preds])
        classes = torch.stack([p["labels"] for p in preds])
        quads = torch.stack([p["quads"].reshape(-1, 8) for p in preds])
        dev = scores.device
        counts = [int(t["quads"].shape[0]) for t in target]
        gq = [t["quads"].as_subclass(Tensor).reshape(-1, 8).to(device=dev, dtype=torch.float32) for t in target]
        gc = [t["labels"].as_subclass(Tensor).reshape(-1).to(device=dev, dtype=torch.int64) for t in target]
        gt_quads = torch.cat(gq) if gq else torch.empty((0, 8), device=dev)
        gt_classes = torch.cat(gc) if gc else torch.empty((0,), dtype=torch.int64, device=dev)
        self.update_batch(scores, classes, quads, gt_quads, gt_classes, counts, **self._annotations(target, dev))

    @staticmethod
    def _annotations(target: List[Dict[str, Tensor]], dev) -> Dict[str, Optional[Tensor]]:
        """``gt_crowd`` / ``gt_area`` for :meth:`update_batch` from the targets' optional ``iscrowd`` / ``area``:
        None where no image has the key, otherwise concatenated with zeros for the images without it."""
        out: Dict[str, Optional[Tensor]] = {}
        for key, arg, dtype in (("iscrowd", "gt_crowd", torch.uint8), ("area", "gt_area", torch.float64)):
            if not any(key in t for t in target):
                out[arg] = None
                continue
            parts = []
            for i, t in enumerate(target):
                n = int(t["labels"].numel())
                if key not in t:
                    parts.append(torch.zeros(n, dtype=dtype, device=dev))
                    continue
                v = t[key].as_subclass(Tensor)
                if tuple(v.shape) != (n,):
                    raise ValueError(f"target {i}: {key!r} has shape {tuple(v.shape)}, labels has {n} entries")
                parts.append((v != 0).to(device=dev, dtype=dtype) if key == "iscrowd" else v.to(device=dev, dtype=dtype))
            out[arg] = torch.cat(parts) if parts else torch.empty((0,), dtype=dtype, device=dev)
        return out

    def update_batch(self, scores: Tensor, classes: Tensor, boxes: Tensor, gt_boxes: Tensor, gt_classes: Tensor,
                     gt_counts: Sequence[int], gt_crowd: Optional[Tensor] = None,
                     gt_area: Optional[Tensor] = None) -> None:
        """The batched form the drop-in head calls: detections [B,K,...] as ``forward`` returns them, ground truth
        concatenated with its per-image counts.  Enqueues the matching; nothing is synchronised.  With
        ``iou_type="quad"``, ``boxes`` / ``gt_boxes`` are quads: [B,K,4,2] or [B,K,8] and [sumG,4,2] or [sumG,8].
        ``gt_crowd`` / ``gt_area`` ([sumG], optional) are the ``iscrowd`` / ``area`` annotations (see ``ops.map_match``)."""
        dev = scores.device
        off = np.zeros(len(gt_counts) + 1, dtype=np.int32)
        off[1:] = np.cumsum(gt_counts)
        gt_offsets = torch.from_numpy(off).to(dev)
        match = ops.quad_map_match if self.iou_type == "quad" else ops.map_match
        res = match(boxes.float(), scores, classes, gt_boxes, gt_classes, gt_offsets, self.iou_thresholds,
                    self.area_ranges, gt_crowd=gt_crowd, gt_area=gt_area)
        order = res["det_order"].long()
        self._batches.append(dict(
            scores=torch.gather(scores.float(), 1, order), classes=torch.gather(classes, 1, order),   # by rank
            dt_match=res["dt_match"], dt_ignore=res["dt_ignore"], gt_ignore=res["gt_ignore"], gt_classes=gt_classes,
            gt_offsets=gt_offsets))

    # -- COCOeval.accumulate + summarize on the match tables ---------------------------------------------------------
    def _host_state(self):
        """Everything recorded so far as numpy arrays, images concatenated (and gathered over the ranks)."""
        per_image = []
        for b in self._batches:
            s, c = b["scores"].cpu().numpy(), b["classes"].cpu().numpy()
            dtm, dti = b["dt_match"].cpu().numpy(), b["dt_ignore"].cpu().numpy()
            gi, gcl, go = b["gt_ignore"].cpu().numpy(), b["gt_classes"].cpu().numpy(), b["gt_offsets"].cpu().numpy()
            for i in range(s.shape[0]):
                per_image.append((s[i], c[i], dtm[i] >= 0, dti[i] != 0, gcl[go[i]:go[i + 1]], gi[:, go[i]:go[i + 1]]))
        if self.sync_dist and torch.distributed.is_available() and torch.distributed.is_initialized() \
                and torch.distributed.get_world_size() > 1:
            gathered = [None] * torch.distributed.get_world_size()
            torch.distributed.all_gather_object(gathered, per_image)
            per_image = [im for part in gathered for im in part]
        return per_image

    def compute(self) -> Dict[str, Tensor]:
        images = self._host_state()
        T, R, NA, M = len(self.iou_thresholds), len(RECALL_THRESHOLDS), len(self.area_ranges), len(self.max_dets)
        cats = sorted(set(int(v) for im in images for v in np.unique(im[4])) | set(int(v) for im in images for v in np.unique(im[1])))
        precision = -np.ones((T, R, len(cats), NA, M))
        recall = -np.ones((T, len(cats), NA, M))
        if images:
            K = images[0][0].shape[0]
            scores = np.stack([im[0] for im in images]).astype(np.float64)                  # [I, K] by rank
            classes = np.stack([im[1] for im in images])
            matched = np.stack([im[2] for im in images])                                    # [I, NA, T, K]
            ignored = np.stack([im[3] for im in images])
            for k, cat in enumerate(cats):
                is_cat = classes == cat                                                     # [I, K]
                cat_rank = np.cumsum(is_cat, axis=1) - 1                                    # rank inside (image, category)
                # non-ignored ground truth of the category per area range, over all images
                npig = np.zeros(NA, dtype=np.int64)
                has_gt = np.zeros(len(images), dtype=bool)
                for i, im in enumerate(images):
                    g = im[4] == cat
                    has_gt[i] = g.any()
                    if has_gt[i]:
                        npig += (~(im[5][:, g] != 0)).sum(axis=1)
                for mi, max_det in enumerate(self.max_dets):
                    sel = is_cat & (cat_rank < max_det)
                    if not sel.any() and not has_gt.any():
                        continue
                    flat_scores = scores[sel]                                               # image-major, rank order inside
                    order = np.argsort(-flat_scores, kind="mergesort")
                    for a in range(NA):
                        if npig[a] == 0:
                            continue
                        m_a = matched[:, a].transpose(1, 0, 2)[:, sel][:, order]            # [T, n]
                        i_a = ignored[:, a].transpose(1, 0, 2)[:, sel][:, order]
                        tp = np.cumsum(m_a & ~i_a, axis=1).astype(np.float64)
                        fp = np.cumsum(~m_a & ~i_a, axis=1).astype(np.float64)
                        nd = tp.shape[1]
                        rc = tp / npig[a]
                        pr = tp / (fp + tp + np.spacing(1))
                        recall[:, k, a, mi] = rc[:, -1] if nd else 0.0
                        if nd:
                            pr = np.maximum.accumulate(pr[:, ::-1], axis=1)[:, ::-1]        # precision envelope
                        q = np.zeros((T, R))
                        for t in range(T):
                            idx = np.searchsorted(rc[t], RECALL_THRESHOLDS, side="left")
                            ok = idx < nd
                            q[t, ok] = pr[t, idx[ok]]
                        precision[:, :, k, a, mi] = q

        def mean_valid(x):
            x = x[x > -1]
            return float(x.mean()) if x.size else -1.0

        last = M - 1
        thr = np.asarray(self.iou_thresholds)
        out = {"map": mean_valid(precision[:, :, :, 0, last])}
        for name, iou in (("map_50", 0.5), ("map_75", 0.75)):
            pick = np.nonzero(np.abs(thr - iou) < 1e-9)[0]
            out[name] = mean_valid(precision[pick][:, :, :, 0, last]) if len(pick) else -1.0
        for name, a in (("map_small", 1), ("map_medium", 2), ("map_large", 3)):
            out[name] = mean_valid(precision[:, :, :, a, last])
        for mi, md in enumerate(self.max_dets):
            out[f"mar_{md}"] = mean_valid(recall[:, :, 0, mi])
        for name, a in (("mar_small", 1), ("mar_medium", 2), ("mar_large", 3)):
            out[name] = mean_valid(recall[:, :, a, last])
        result = {k: torch.tensor(v, dtype=torch.float32) for k, v in out.items()}
        result["classes"] = torch.tensor(cats, dtype=torch.int32)
        return result
