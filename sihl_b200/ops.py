"""Tensor-level entry points of the detection-head path.

Thin hand-off from ``torch.Tensor`` to the C ABI (``include/sihl_od.h``): check
device / dtype / contiguity, allocate outputs with torch, pass raw device
pointers and the current CUDA stream.  No arithmetic happens here and there is
no non-CUDA path: CPU tensors are rejected.

Reference lines (``/root/reference/src/sihl/heads/object_detection.py``) are cited
per function; the same citations are in the header next to each C entry point.
"""
from __future__ import annotations

import collections

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _native

NUM_SUMS = 8
MAX_TOPK = 16
DTYPE_CODES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}       # SIHL_OD_F32 / _F16 / _BF16 (sihl_od.h)


def _lib():
    return _native.load()


class _on:
    """``with _on(device):`` — make ``device`` current for the C call.  Unlike ``torch.cuda.device`` it does nothing
    when the device already is current (the usual case: ~1 us instead of ~15 us per call on the host path of the
    drop-in head, which makes a few dozen of these calls per training step)."""
    __slots__ = ("want", "prev")

    def __init__(self, device) -> None:
        self.want = torch.device(device).index

    def __enter__(self) -> None:
        self.prev = torch.cuda.current_device()
        if self.want is not None and self.want != self.prev:
            torch.cuda.set_device(self.want)

    def __exit__(self, *exc) -> None:
        if self.want is not None and self.want != self.prev:
            torch.cuda.set_device(self.prev)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(device) -> int:
    """Handle of torch's current stream on ``device``.  Through the raw accessor when this torch has it (~0.3 us): building a
    ``torch.cuda.Stream`` object per C call costs ~8 us, and the training step makes ~70 of these calls."""
    if _raw_stream is not None:
        idx = device.index if isinstance(device, torch.device) else torch.device(device).index
        return _raw_stream(torch.cuda.current_device() if idx is None else idx)
    return torch.cuda.current_stream(device).cuda_stream


def _p(t: Optional[Tensor]):
    return None if t is None else t.data_ptr()


def _req(t: Tensor, dtype, name: str, ndim: Optional[int] = None, pinned_ok: bool = False) -> Tensor:
    """``pinned_ok``: a page-locked host tensor is accepted as well — under unified addressing the kernels read it
    in place over PCIe (only for maps that a kernel *gathers* a few rows of; the compute is still on the GPU)."""
    if not isinstance(t, Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda and not (pinned_ok and t.is_pinned()):
        raise RuntimeError(f"{name}: sihl_b200 kernels run on CUDA tensors only (got {t.device}); there is no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise ValueError(f"{name}: expected {ndim} dims, got shape {tuple(t.shape)}")
    if t.is_contiguous():
        return t
    # a contiguous COPY: callers pass `_p(_req(...))` straight into a C call, so nothing else references the copy — keep
    # the last few alive here, or the allocator could hand its block to the next temporary before the kernel is enqueued
    t = t.contiguous()
    _KEEPALIVE.append(t)
    return t


_KEEPALIVE: "collections.deque" = collections.deque(maxlen=16)


def _req_map(t: Tensor, name: str, ndim: Optional[int] = None, pinned_ok: bool = False) -> Tuple[Tensor, int]:
    """A head-output map in any of the three supported element types -> (contiguous tensor, SIHL_OD_* dtype code);
    anything else (fp64, ...) is converted to fp32."""
    if isinstance(t, Tensor) and t.dtype not in DTYPE_CODES:
        t = t.float()
    t = _req(t, t.dtype if isinstance(t, Tensor) else torch.float32, name, ndim, pinned_ok)
    return t, DTYPE_CODES[t.dtype]


def _levels_array(levels: Sequence[Tuple[int, int]]) -> np.ndarray:
    arr = np.ascontiguousarray(np.asarray(levels, dtype=np.int32).reshape(-1, 2))
    return arr


# --------------------------------------------------------------------------- a1/a2
_anchor_cache: Dict[tuple, Tuple[Tensor, Tensor, Tensor, Tensor]] = {}


def anchor_tables(levels: Sequence[Tuple[int, int]], img_w: int, img_h: int, device,
                  cache: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
    """``(offsets, scales, anchors)``, each ``[A,4]`` fp32 — ref :83-97 and :134-140.

    The tables depend only on the feature-map shapes, so they are cached per
    (levels, image size, device) instead of being rebuilt by ~40 launches per call.
    """
    device = torch.device(device)
    key = (tuple(map(tuple, levels)), int(img_w), int(img_h), device.type, device.index)
    if cache and key in _anchor_cache:
        return _anchor_cache[key][:3]
    hw = _levels_array(levels)
    A = int((hw[:, 0].astype(np.int64) * hw[:, 1]).sum())
    with _on(device):
        out = tuple(torch.empty((A, 4), dtype=torch.float32, device=device) for _ in range(3))
        rc = _lib().sihl_od_anchors(hw.ctypes.data, len(hw), int(img_w), int(img_h), _p(out[0]), _p(out[1]), _p(out[2]),
                                    _stream(device))
        _native.check(rc, "sihl_od_anchors")
        terms = torch.empty((A, 4), dtype=torch.float32, device=device)
        rc = _lib().sihl_od_anchor_terms(_p(out[2]), A, _p(terms), _stream(device))
        _native.check(rc, "sihl_od_anchor_terms")
    if cache:
        _anchor_cache[key] = out + (terms,)
    return out


def anchor_terms(levels: Sequence[Tuple[int, int]], img_w: int, img_h: int, device) -> Tensor:
    """Per-anchor CIoU terms ``[A,4]`` = (area, cx, cy, atan(w/h)) of the cached grid (the per-anchor
    half of torchvision's ``complete_box_iou``, hoisted out of the pair loop)."""
    device = torch.device(device)
    anchor_tables(levels, img_w, img_h, device)
    key = (tuple(map(tuple, levels)), int(img_w), int(img_h), device.type, device.index)
    return _anchor_cache[key][3]


# --------------------------------------------------------------------------- ground truth
@dataclass
class GtBatch:
    """Ragged ground truth as CSR on the device (what the kernels consume)."""
    boxes: Tensor      # [sumG, 4] f32 xyxy px
    classes: Tensor    # [sumG] i64
    offsets: Tensor    # [B+1] i32
    counts: List[int]  # host copy of the per-image counts (from tensor shapes: no sync)

    @property
    def batch_size(self) -> int:
        return len(self.counts)

    @property
    def total(self) -> int:
        return int(sum(self.counts))

    @staticmethod
    def from_lists(boxes: Sequence[Tensor], classes: Optional[Sequence[Tensor]], device) -> "GtBatch":
        """ref :127-128 — per-image lists (possibly empty, possibly ``tv_tensors`` subclasses)."""
        device = torch.device(device)
        counts = [int(b.shape[0]) for b in boxes]
        plain = [b.as_subclass(Tensor).reshape(-1, 4) for b in boxes]
        if plain:
            cat = torch.cat(plain).to(device=device, dtype=torch.float32).contiguous()
        else:
            cat = torch.empty((0, 4), dtype=torch.float32, device=device)
        if classes is not None:
            cls = torch.cat([c.as_subclass(Tensor).reshape(-1) for c in classes]) if len(classes) else torch.empty(0)
            cls = cls.to(device=device, dtype=torch.int64).contiguous()
            if cls.numel() != cat.shape[0]:
                raise ValueError("classes and boxes disagree on the number of objects")
        else:
            cls = torch.zeros((cat.shape[0],), dtype=torch.int64, device=device)
        off = np.zeros(len(counts) + 1, dtype=np.int32)
        off[1:] = np.cumsum(counts)
        return GtBatch(cat, cls, torch.from_numpy(off).to(device), counts)


# --------------------------------------------------------------------------- a3/a4
def assign_select(anchors: Tensor, levels: Optional[Sequence[Tuple[int, int]]], img_w: int, img_h: int,
                  gt: GtBatch, topk: int = 9, sums: Optional[Tensor] = None, terms: Optional[Tensor] = None):
    """Stage 1 of ``bbox_matching`` for the whole batch (ref :263-268, :277).

    ``levels=None`` evaluates all ``A x G`` pairs (arbitrary anchors); otherwise
    ``anchors`` must be the grid of :func:`anchor_tables` for ``levels``.
    Returns ``(sel_anchor [sumG,k] i32, sel_val [sumG,k] f32, best_iou [sumG] f32)``.
    """
    anchors = _req(anchors, torch.float32, "anchors", 2)
    dev = anchors.device
    G = gt.total
    sel_anchor = torch.empty((G, topk), dtype=torch.int32, device=dev)
    sel_val = torch.empty((G, topk), dtype=torch.float32, device=dev)
    best = torch.empty((G,), dtype=torch.float32, device=dev)
    hw = None if levels is None else _levels_array(levels)
    with _on(dev):
        rc = _lib().sihl_od_assign_select(
            _p(anchors), _p(terms), anchors.shape[0], None if hw is None else hw.ctypes.data, 0 if hw is None else len(hw),
            int(img_w), int(img_h), _p(_req(gt.boxes, torch.float32, "gt.boxes", 2)),
            _p(_req(gt.offsets, torch.int32, "gt.offsets", 1)), gt.batch_size, G, int(topk),
            _p(sel_anchor), _p(sel_val), _p(best), _p(sums), _stream(dev))
    _native.check(rc, "sihl_od_assign_select")
    return sel_anchor, sel_val, best


def resolve_tiles(num_anchors: int) -> Tuple[int, int]:
    n_tiles, tile = C.c_int(0), C.c_int(0)
    _lib().sihl_od_resolve_tiles(int(num_anchors), C.byref(n_tiles), C.byref(tile))
    return n_tiles.value, tile.value


def assign_resolve(sel, gt: GtBatch, num_anchors: int, topk: int = 9, relative: bool = True,
                   loc_logits: Optional[Tensor] = None, iou_preds: Optional[Tensor] = None,
                   sums: Optional[Tensor] = None, fused: Optional[dict] = None):
    """Stage 2 (ref :270-282) with the dense losses (ref :157-163, :175-180) fused when
    ``loc_logits`` is given.  ``fused`` = dict(box_raw, cls_logits, offsets, scales, img_w, img_h)
    additionally runs the positive-row losses over dense maps from the per-tile lists.
    Returns dict(assignment, iou, tile_pos_count, tile_pos_rows)."""
    sel_anchor, sel_val, best = sel
    dev = sel_anchor.device
    B, A = gt.batch_size, int(num_anchors)
    assignment = torch.empty((B, A), dtype=torch.int64, device=dev)
    out_iou = torch.empty((B, A), dtype=torch.float32, device=dev)
    f = fused or {}
    tpc = tpr = chunks = aux = None
    if f:
        n_tiles, tile = resolve_tiles(A)
        tpc = torch.empty((B * n_tiles,), dtype=torch.int32, device=dev)
        tpr = torch.zeros((B * n_tiles * tile,), dtype=torch.int32, device=dev)
        chunks = torch.zeros((B * n_tiles * (tile // 32),), dtype=torch.int32, device=dev)
        aux = torch.zeros((B * n_tiles * tile, 2), dtype=torch.int32, device=dev)
    with _on(dev):
        rc = _lib().sihl_od_assign_resolve(
            _p(sel_anchor), _p(sel_val), _p(best), _p(gt.offsets), B, A, int(topk), int(bool(relative)),
            _p(None if loc_logits is None else _req(loc_logits, torch.float32, "loc_logits")),
            _p(None if iou_preds is None else _req(iou_preds, torch.float32, "iou_preds")),
            _p(assignment), _p(out_iou), _p(sums), _p(tpc), _p(tpr), _p(f.get("box_raw")), _p(f.get("cls_logits")),
            0 if f.get("cls_logits") is None else int(f["cls_logits"].shape[-1]), _p(chunks), _p(aux), _stream(dev))
        _native.check(rc, "sihl_od_assign_resolve")
        if f:
            pos_loss_tiles(chunks, tpr, aux, B, A, f["offsets"], f["scales"], f["img_w"], f["img_h"], gt,
                           f.get("box_raw"), f.get("cls_logits"), sums)
    return dict(assignment=assignment, iou=out_iou, tile_pos_count=tpc, tile_pos_rows=tpr)


def bbox_matching(anchors: Tensor, gt_boxes: Tensor, topk: int, relative: bool = False,
                  levels: Optional[Sequence[Tuple[int, int]]] = None, img_size: Optional[Tuple[int, int]] = None):
    """Drop-in for the static ``ObjectDetection.bbox_matching`` (ref :252-284), one image.

    Returns ``(assignment int64 [A], iou fp32 [A])`` in canonical form: ``assignment`` is -1
    wherever the returned iou is not > 0 (the reference leaves implementation-defined indices
    there; nothing downstream reads them — SURVEY.md §3.4).
    """
    anchors = _req(anchors, torch.float32, "anchors", 2)
    gt_boxes = gt_boxes.as_subclass(Tensor).to(device=anchors.device, dtype=torch.float32).reshape(-1, 4)
    gt = GtBatch.from_lists([gt_boxes], None, anchors.device)
    A = anchors.shape[0]
    if gt.total == 0:                                            # ref :258-261
        return (torch.full((A,), -1, dtype=torch.int64, device=anchors.device),
                torch.zeros((A,), dtype=torch.float32, device=anchors.device))
    w, h = img_size if img_size is not None else (0, 0)
    sel = assign_select(anchors, levels, w, h, gt, topk)
    out = assign_resolve(sel, gt, A, topk, relative)
    return out["assignment"][0], out["iou"][0]


# --------------------------------------------------------------------------- N1: un-clamped variant (QuadrilateralDetection)
def quad_bbox_matching(anchors: Tensor, gt: GtBatch, topk: int = 9) -> Dict[str, Tensor]:
    """``QuadrilateralDetection.bbox_matching`` (ref quadrilateral_detection.py:266-294) for a whole batch, i.e. the
    per-image loop + stacks of ref :165-172.  ``anchors`` fp32 [A,4] xyxy px (arbitrary), ``gt`` the per-image boxes
    (``quads_to_boxes`` of the quads).  Returns dict(assignment i64 [B,A] canonical, o2o_mask bool [B,A],
    iou f32 [B,A], rel_iou f32 [B,A], sel_anchor i32 [sumG,k], sel_val f32 [sumG,k])."""
    anchors = _req(anchors, torch.float32, "anchors", 2)
    dev = anchors.device
    B, A, G = gt.batch_size, anchors.shape[0], gt.total
    assignment = torch.empty((B, A), dtype=torch.int64, device=dev)
    o2o = torch.empty((B, A), dtype=torch.bool, device=dev)
    iou = torch.empty((B, A), dtype=torch.float32, device=dev)
    rel = torch.empty((B, A), dtype=torch.float32, device=dev)
    sel_anchor = torch.empty((G, topk), dtype=torch.int32, device=dev)
    sel_val = torch.empty((G, topk), dtype=torch.float32, device=dev)
    terms = torch.empty((A, 4), dtype=torch.float32, device=dev)
    with _on(dev):
        rc = _lib().sihl_od_quad_matching(
            _p(anchors), A, _p(_req(gt.boxes, torch.float32, "gt.boxes", 2)), _p(_req(gt.offsets, torch.int32, "gt.offsets", 1)),
            B, G, int(topk), _p(assignment), _p(o2o), _p(iou), _p(rel), _p(sel_anchor), _p(sel_val), _p(terms), _stream(dev))
    _native.check(rc, "sihl_od_quad_matching")
    return dict(assignment=assignment, o2o_mask=o2o, iou=iou, rel_iou=rel, sel_anchor=sel_anchor, sel_val=sel_val)


# --------------------------------------------------------------------------- a5-a10
def new_sums(device) -> Tensor:
    return torch.zeros((NUM_SUMS,), dtype=torch.float64, device=device)


def pos_loss_tiles(pos_chunks: Tensor, tile_pos_rows: Tensor, tile_pos_aux: Tensor, batch: int, num_anchors: int,
                   offsets: Tensor, scales: Tensor, img_w: int, img_h: int, gt: GtBatch,
                   box_raw: Optional[Tensor], cls_logits: Optional[Tensor], sums: Tensor,
                   losses: Optional[Tensor] = None, done_counter: Optional[Tensor] = None) -> Tensor:
    """ref :187-208 over dense maps, straight from the per-tile positive lists (no compaction);
    ``pos_chunks`` is the work list ``assign_resolve`` published (length in ``sums[7]``)."""
    dev = sums.device
    with _on(dev):
        rc = _lib().sihl_od_pos_loss_tiles(
            _p(pos_chunks), _p(tile_pos_rows), _p(tile_pos_aux), int(batch), int(num_anchors), _p(offsets),
            _p(scales), int(img_w), int(img_h), _p(gt.boxes), _p(gt.classes), _p(gt.offsets),
            _p(None if box_raw is None else _req(box_raw, torch.float32, "box_raw")),
            _p(None if cls_logits is None else _req(cls_logits, torch.float32, "cls_logits")),
            0 if cls_logits is None else int(cls_logits.shape[-1]), _p(sums), _p(losses), _p(done_counter), _stream(dev))
    _native.check(rc, "sihl_od_pos_loss_tiles")
    return sums


def loss_finalize(sums: Tensor) -> Tensor:
    """ref :163-172, :180, :197, :208, :210 -> fp32 [5] = [location, box, class, iou, total]."""
    out = torch.empty((5,), dtype=torch.float32, device=sums.device)
    with _on(sums.device):
        rc = _lib().sihl_od_loss_finalize(_p(sums), _p(out), _stream(sums.device))
    _native.check(rc, "sihl_od_loss_finalize")
    return out


# --------------------------------------------------------------------------- the drop-in head's training step (N2)
MAX_BATCH_BY_VALUE = 512                                                    # SIHL_OD_MAX_BATCH_BY_VALUE
_geom_cache: Dict[tuple, tuple] = {}
_ws_bytes_cache: Dict[tuple, int] = {}


def _geometry(levels, img_w: int, img_h: int, device):
    """Cached per (levels, image, device): anchor tables + terms + the host level array the C entry takes."""
    key = (tuple(map(tuple, levels)), int(img_w), int(img_h), device.type, device.index)
    g = _geom_cache.get(key)
    if g is None:
        offsets, scales, anchors = anchor_tables(levels, img_w, img_h, device)
        hw = _levels_array(levels)
        g = (offsets, scales, anchors, _anchor_cache[key][3], hw, hw.ctypes.data, len(hw), int(anchors.shape[0]))
        _geom_cache[key] = g
    return g


class TrainAssignment:
    """What ``sihl_od_train_assign`` leaves on the device for one training step (no host sync happened):
    ``assignment`` i64 [B,A], ``rel_iou`` f32 [B,A], ``pos_index`` i32 [capacity] (first P = ``pos_total`` entries
    real, the rest 0), plus the raw pointers ``sihl_od_train_loss`` / ``_bwd`` need."""
    __slots__ = ("assignment", "rel_iou", "pos_index", "capacity", "meta", "B", "A", "img_w", "img_h", "offsets", "scales",
                 "gt_boxes", "gt_classes", "device", "_p_sums", "_p_gt_offsets", "_p_pos_total", "grad_scale")

    @staticmethod
    def from_tensors(assignment: Tensor, rel_iou: Tensor, pos_index: Tensor, meta: Tensor, offsets: Tensor, scales: Tensor,
                     gt_boxes: Tensor, gt_classes: Optional[Tensor], img_w: int, img_h: int,
                     grad_scale: float = 1.0) -> "TrainAssignment":
        """Rebuild the state from the tensors ``train_assign`` returned (the torch.library ops pass tensors only)."""
        st = TrainAssignment()
        st.assignment, st.rel_iou, st.pos_index, st.meta = assignment, rel_iou, pos_index, meta
        st.B, st.A = int(rel_iou.shape[0]), int(rel_iou.shape[1])
        st.capacity, st.device, st.img_w, st.img_h = int(pos_index.numel()), rel_iou.device, int(img_w), int(img_h)
        st.offsets, st.scales, st.gt_boxes, st.gt_classes, st.grad_scale = offsets, scales, gt_boxes, gt_classes, grad_scale
        base = meta.data_ptr()
        st._p_sums, st._p_gt_offsets, st._p_pos_total = base, base + 64, base + 64 + 4 * (st.B + 1)
        return st

    @property
    def sums(self) -> Tensor:
        """fp64 [8] view of the step's partial sums (what crosses GPUs in ``loss_reduction="global"``)."""
        return self.meta[:16].view(torch.float64)

    @property
    def gt_offsets(self) -> Tensor:
        return self.meta[16:16 + self.B + 1]

    @property
    def pos_total(self) -> Tensor:
        return self.meta[16 + self.B + 1:16 + self.B + 2]


def train_assign(levels: Sequence[Tuple[int, int]], img_w: int, img_h: int, gt_boxes: Tensor, gt_classes: Optional[Tensor],
                 gt_counts: Optional[Sequence[int]], batch: int, topk: int = 9, gt_offsets: Optional[Tensor] = None,
                 pos_capacity: Optional[int] = None) -> TrainAssignment:
    """ref :134-148 + the positive compaction of :182-184 for the whole batch: ONE C call (select, resolve, compact),
    no host synchronisation.  ``gt_boxes`` fp32 [sumG,4] on the device; the per-image counts either as a host list
    ``gt_counts`` (they come from tensor shapes; passed to the kernel by value) or as ``gt_offsets`` int32 [B+1] on
    the device (then ``gt_boxes.shape[0]`` is only a capacity and the call is replayable from a CUDA graph on new
    ground truth)."""
    gt_boxes = _req(gt_boxes, torch.float32, "gt_boxes", 2)
    dev = gt_boxes.device
    offsets, scales, anchors, terms, hw, hw_ptr, n_levels, A = _geometry(levels, img_w, img_h, dev)
    B, G = int(batch), int(gt_boxes.shape[0])
    cap = int(pos_capacity) if pos_capacity is not None else max(1, min(int(topk) * G, B * A))
    key = (B, A, G, int(topk))
    ws_bytes = _ws_bytes_cache.get(key)
    if ws_bytes is None:
        ws_bytes = _ws_bytes_cache[key] = int(_lib().sihl_od_train_workspace_bytes(B, A, G, int(topk)))
    st = TrainAssignment()
    st.B, st.A, st.capacity, st.device, st.img_w, st.img_h = B, A, cap, dev, int(img_w), int(img_h)
    st.offsets, st.scales, st.gt_boxes, st.gt_classes, st.grad_scale = offsets, scales, gt_boxes, gt_classes, 1.0
    with _on(dev):
        st.assignment = torch.empty((B, A), dtype=torch.int64, device=dev)
        st.rel_iou = torch.empty((B, A), dtype=torch.float32, device=dev)
        st.pos_index = torch.empty((cap,), dtype=torch.int32, device=dev)
        # sums f64[8] | gt_offsets i32[B+1] | pos_total i32[1] in one small buffer (allocations are 512-byte aligned)
        st.meta = torch.empty((16 + B + 2,), dtype=torch.int32, device=dev)
        ws = torch.empty((max(ws_bytes, 16),), dtype=torch.uint8, device=dev)
        base = st.meta.data_ptr()
        st._p_sums, st._p_gt_offsets, st._p_pos_total = base, base + 64, base + 64 + 4 * (B + 1)
        counts_ptr = None
        if gt_offsets is not None:
            st.meta[16:16 + B + 1].copy_(_req(gt_offsets, torch.int32, "gt_offsets", 1))
        else:
            if len(gt_counts) != B:
                raise ValueError(f"{len(gt_counts)} gt counts for a batch of {B}")
            if B > MAX_BATCH_BY_VALUE:                      # too many images for the kernel-parameter table: upload
                off = np.zeros(B + 1, dtype=np.int32)
                off[1:] = np.cumsum(gt_counts)
                st.meta[16:16 + B + 1].copy_(torch.from_numpy(off))
            else:
                counts = np.asarray(gt_counts, dtype=np.int32)
                counts_ptr = counts.ctypes.data
        rc = _lib().sihl_od_train_assign(
            anchors.data_ptr(), terms.data_ptr(), A, hw_ptr, n_levels, int(img_w), int(img_h), gt_boxes.data_ptr() if G else None,
            counts_ptr, st._p_gt_offsets, B, G, int(topk), st.assignment.data_ptr(), st.rel_iou.data_ptr(),
            st.pos_index.data_ptr(), cap, st._p_pos_total, st._p_sums, ws.data_ptr(), ws.numel(), _stream(dev))
    _native.check(rc, "sihl_od_train_assign")
    return st


def _train_maps(st: TrainAssignment, loc_logits, iou_preds, box_rows, cls_rows):
    """Common dtype + contiguity of the four head outputs; mixed dtypes are upcast to fp32 (never seen under autocast:
    all four MLPs end in a Linear)."""
    maps = [loc_logits, iou_preds, box_rows, cls_rows]
    dt = loc_logits.dtype
    if dt not in DTYPE_CODES or any(m is not None and m.dtype != dt for m in maps):
        dt = torch.float32
        maps = [None if m is None else m.float() for m in maps]
    maps = [None if m is None else (m if m.is_contiguous() else m.contiguous()) for m in maps]
    if not maps[0].is_cuda:
        raise RuntimeError("sihl_b200 kernels run on CUDA tensors only; there is no CPU path")
    if maps[0].numel() != st.B * st.A or (maps[1] is not None and maps[1].numel() != st.B * st.A):
        raise ValueError("loc_logits / iou_preds must hold B*A elements")
    C = 0
    if maps[3] is not None:
        C = int(maps[3].shape[-1])
        if maps[3].numel() != st.capacity * C:
            raise ValueError(f"cls_rows must be [{st.capacity}, C], got {tuple(maps[3].shape)}")
    if maps[2] is not None and maps[2].numel() != st.capacity * 4:
        raise ValueError(f"box_rows must be [{st.capacity}, 4], got {tuple(maps[2].shape)}")
    return maps, DTYPE_CODES[dt], C


def _train_common_args(st: TrainAssignment, maps, code: int, C: int):
    return (_p(maps[0]), _p(maps[1]), _p(maps[2]), _p(maps[3]), code, st.B, st.A, C, st.rel_iou.data_ptr(),
            st.assignment.data_ptr(), st.pos_index.data_ptr(), st.capacity, st._p_pos_total, st.offsets.data_ptr(),
            st.scales.data_ptr(), st.img_w, st.img_h, _p(st.gt_boxes) if st.gt_boxes.numel() else None,
            _p(st.gt_classes) if (st.gt_classes is not None and st.gt_classes.numel()) else None, st._p_gt_offsets)


def train_loss(st: TrainAssignment, loc_logits: Tensor, iou_preds: Optional[Tensor], box_rows: Optional[Tensor],
               cls_rows: Optional[Tensor], finalize: bool = True):
    """ref :157-217 in one launch.  Returns ``(losses fp32 [5] or None, maps)`` — ``maps`` are the (contiguous, common
    dtype) tensors the kernel read, to be saved for :func:`train_loss_bwd`."""
    maps, code, C = _train_maps(st, loc_logits, iou_preds, box_rows, cls_rows)
    if cls_rows is not None and st.gt_classes is None:
        raise ValueError("the class loss needs gt classes")
    dev = st.device
    with _on(dev):
        losses = torch.empty((5,), dtype=torch.float32, device=dev) if finalize else None
        rc = _lib().sihl_od_train_loss(*_train_common_args(st, maps, code, C), st._p_sums, _p(losses), _stream(dev))
    _native.check(rc, "sihl_od_train_loss")
    return losses, maps


def train_loss_bwd(st: TrainAssignment, maps, grad_losses: Optional[Tensor], want=(True, True, True, True)):
    """SURVEY.md §7.4 in one launch; gradients come back in the dtype of ``maps``."""
    code = DTYPE_CODES[maps[0].dtype]
    C = 0 if maps[3] is None else int(maps[3].shape[-1])
    dev = st.device
    with _on(dev):
        grads = [torch.empty_like(m) if (m is not None and w) else None for m, w in zip(maps, want)]
        if grad_losses is not None:
            grad_losses = _req(grad_losses, torch.float32, "grad_losses", 1)
        rc = _lib().sihl_od_train_loss_bwd(*_train_common_args(st, maps, code, C), st._p_sums, _p(grad_losses),
                                           float(st.grad_scale), _p(grads[0]), _p(grads[1]), _p(grads[2]), _p(grads[3]),
                                           _stream(dev))
    _native.check(rc, "sihl_od_train_loss_bwd")
    return grads


# --------------------------------------------------------------------------- a11
def topk_locations(loc_logits: Tensor, k: int) -> Tuple[Tensor, Tensor]:
    """ref :109 — ``loc_logits.topk(k, dim=1)``: ``(values [B,k] f32, indices [B,k] i64)``,
    sorted descending, exact ties broken towards the lowest index."""
    loc, code = _req_map(loc_logits, "loc_logits", 2)
    B, A = loc.shape
    idx = torch.empty((B, k), dtype=torch.int64, device=loc.device)
    top = torch.empty((B, k), dtype=torch.float32, device=loc.device)       # half values are exact in fp32
    with _on(loc.device):
        rc = _lib().sihl_od_topk_t(_p(loc), code, B, A, int(k), _p(idx), _p(top), _stream(loc.device))
    _native.check(rc, "sihl_od_topk_t")
    return top, idx


def decode_rows(top_logits: Tensor, idx: Tensor, cls_rows: Tensor, box_rows: Tensor, offsets: Tensor, scales: Tensor,
                img_w: int, img_h: int):
    """ref :113-121 — ``(num_instances [B] i64, scores [B,K], classes [B,K] i64, boxes [B,K,4])``."""
    top = _req(top_logits, torch.float32, "top_logits", 2)
    B, K = top.shape
    dev = top.device
    if cls_rows.dtype != box_rows.dtype or cls_rows.dtype not in DTYPE_CODES:
        cls_rows, box_rows = cls_rows.float(), box_rows.float()
    cls_rows, code = _req_map(cls_rows, "cls_rows", 3)
    box_rows, _ = _req_map(box_rows, "box_rows", 3)
    num = torch.empty((B,), dtype=torch.int64, device=dev)
    scores = torch.empty((B, K), dtype=torch.float32, device=dev)
    classes = torch.empty((B, K), dtype=torch.int64, device=dev)
    boxes = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
    with _on(dev):
        rc = _lib().sihl_od_decode_rows_t(_p(top), _p(_req(idx, torch.int64, "idx", 2)), B, K, _p(cls_rows),
                                          int(cls_rows.shape[-1]), _p(box_rows), code,
                                          _p(offsets), _p(scales), int(img_w), int(img_h), _p(num), _p(scores),
                                          _p(classes), _p(boxes), _stream(dev))
    _native.check(rc, "sihl_od_decode_rows_t")
    return num, scores, classes, boxes


# --------------------------------------------------------------------------- a15 (extension)
@dataclass
class CandidateBuffers:
    count: Tensor      # [B] i32
    key: Tensor        # [B, cap] u64 (as int64 storage)
    box: Tensor        # [B, cap, 4] f32
    cls: Tensor        # [B, cap] i32
    capacity: int
    workspace: Optional[Tensor]

    @staticmethod
    def allocate(batch: int, capacity: int, device) -> "CandidateBuffers":
        ws_bytes = int(_lib().sihl_od_nms_workspace_bytes(int(batch), int(capacity)))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=device) if ws_bytes else None
        return CandidateBuffers(torch.zeros((batch,), dtype=torch.int32, device=device),
                                torch.empty((batch, capacity), dtype=torch.int64, device=device),
                                torch.empty((batch, capacity, 4), dtype=torch.float32, device=device),
                                torch.empty((batch, capacity), dtype=torch.int32, device=device), int(capacity), ws)


DECODE_MODES = ("dense", "candidate_first")


def dense_decode(loc_logits: Tensor, cls_logits: Tensor, box_raw: Tensor, offsets: Tensor, scales: Tensor,
                 img_w: int, img_h: int, score_thr: float, cand: CandidateBuffers, zero_counts: bool = True,
                 mode: str = "dense") -> None:
    """Fill the per-image candidate lists.  ``mode="dense"`` streams every class row (TMA ring, HBM bound);
    ``mode="candidate_first"`` streams only the location map and gathers the rows that pass the threshold
    (same lists up to order; far fewer bytes while candidates are sparse).  In that mode ``cls_logits`` and
    ``box_raw`` may be pinned host tensors: the candidates' rows are then read in place over PCIe (zero-copy)."""
    if mode not in DECODE_MODES:
        raise ValueError(f"mode={mode!r}: expected one of {DECODE_MODES}")
    host_ok = mode == "candidate_first"        # gathers rows: the class / box maps may stay in pinned host memory
    if loc_logits.dtype in (torch.float16, torch.bfloat16) and cls_logits.dtype == loc_logits.dtype \
            and box_raw.dtype == loc_logits.dtype and (mode == "candidate_first" or half_dense_scan_ok(cls_logits)):
        # half maps straight from the MLPs (autocast): loaded as they are, upcast in registers — half the bytes of the
        # dense scan (same TMA ring), or the candidates' rows only
        loc, code = _req_map(loc_logits, "loc_logits", 2)
        cls, _ = _req_map(cls_logits, "cls_logits", 3, pinned_ok=host_ok)
        box, _ = _req_map(box_raw, "box_raw", 3, pinned_ok=host_ok)
        B, A = loc.shape
        name = "sihl_od_dense_decode_t" if mode == "dense" else "sihl_od_candidate_decode_t"
        with _on(loc.device):
            rc = getattr(_lib(), name)(_p(loc), _p(cls), _p(box), code, B, A, int(cls.shape[-1]), _p(offsets),
                                       _p(scales), int(img_w), int(img_h), float(score_thr), _p(cand.count),
                                       cand.capacity, _p(cand.key), _p(cand.box), _p(cand.cls), int(zero_counts),
                                       _stream(loc.device))
        _native.check(rc, name)
        return
    loc = _req(loc_logits.float() if loc_logits.dtype != torch.float32 else loc_logits, torch.float32, "loc_logits", 2)
    cls = _req(cls_logits.float() if cls_logits.dtype != torch.float32 else cls_logits, torch.float32, "cls_logits", 3, pinned_ok=host_ok)
    box = _req(box_raw.float() if box_raw.dtype != torch.float32 else box_raw, torch.float32, "box_raw", 3, pinned_ok=host_ok)
    B, A = loc.shape
    name = "sihl_od_dense_decode" if mode == "dense" else "sihl_od_candidate_decode"
    with _on(loc.device):
        rc = getattr(_lib(), name)(_p(loc), _p(cls), _p(box), B, A, int(cls.shape[-1]), _p(offsets), _p(scales),
                                   int(img_w), int(img_h), float(score_thr), _p(cand.count), cand.capacity,
                                   _p(cand.key), _p(cand.box), _p(cand.cls), int(zero_counts), _stream(loc.device))
    _native.check(rc, name)


def half_dense_scan_ok(cls_logits: Tensor) -> bool:
    """Whether ``sihl_od_dense_decode_t`` takes these half class maps (C % 8 == 0, C <= 256, enough rows); otherwise
    the caller converts to fp32 or uses the candidate-first decode."""
    C = int(cls_logits.shape[-1])
    return C % 8 == 0 and C <= 256 and cls_logits.numel() // C >= 256


SPLIT_NMS_FROM = 16384     # list capacity (locations per image) from which the one-shot postprocess uses the class-split NMS

# The suppression test of the greedy NMS entries -> the infix of their C names: "iou" is torchvision's nms (IoU > thr),
# "diou" is DIoU-NMS (Zheng et al., AAAI 2020: IoU minus the normalised squared distance of the centres > thr).
NMS_OVERLAPS = {"iou": "", "diou": "diou_"}


def _overlap_infix(overlap: str) -> str:
    if overlap not in NMS_OVERLAPS:
        raise ValueError(f"overlap={overlap!r}: expected one of {tuple(NMS_OVERLAPS)}")
    return NMS_OVERLAPS[overlap]


def nms_topk(cand: CandidateBuffers, batch: int, iou_thr: float, k: int, out: Optional[tuple] = None,
             reset_counts: bool = False, split: bool = False, overlap: str = "iou"):
    """Class-aware NMS + top-k over the candidate lists.  ``split``: the class-split multi-CTA variant for long lists
    (same results; thousands of candidates per image).  ``overlap``: ``"iou"`` (greedy NMS) or ``"diou"`` (DIoU-NMS,
    ``iou_thr`` is the DIoU threshold; same order, outputs and workspace)."""
    infix = _overlap_infix(overlap)
    dev = cand.count.device
    if out is None:
        out = (torch.empty((batch,), dtype=torch.int64, device=dev), torch.empty((batch, k), dtype=torch.float32, device=dev),
               torch.empty((batch, k), dtype=torch.int64, device=dev), torch.empty((batch, k, 4), dtype=torch.float32, device=dev))
    if split:
        need = int(_lib().sihl_od_nms_split_workspace_bytes(int(batch), cand.capacity, int(k)))
        ws = getattr(cand, "_split_ws", None)
        if ws is None or ws.numel() < need:
            ws = torch.empty((need,), dtype=torch.uint8, device=dev)
            cand._split_ws = ws
        name = f"sihl_od_{infix}nms_topk_split"
        with _on(dev):
            rc = getattr(_lib(), name)(_p(cand.count), cand.capacity, _p(cand.key), _p(cand.box), _p(cand.cls), int(batch),
                                       float(iou_thr), int(k), _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]), _p(ws),
                                       int(reset_counts), _stream(dev))
        _native.check(rc, name)
        return out
    name = f"sihl_od_{infix}nms_topk"
    with _on(dev):
        rc = getattr(_lib(), name)(_p(cand.count), cand.capacity, _p(cand.key), _p(cand.box), _p(cand.cls), int(batch),
                                   float(iou_thr), int(k), _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]),
                                   _p(cand.workspace), int(reset_counts), _stream(dev))
    _native.check(rc, name)
    return out


def box_vote_topk(cand: CandidateBuffers, batch: int, iou_thr: float, out: tuple, overlap: str = "iou"):
    """Box voting (merge-NMS, YOLOv5's ``merge=True``) after :func:`nms_topk`: every kept box of ``out`` is replaced, in
    place, by the score-weighted mean of the boxes of its image's list and class that its suppression test claims
    (``overlap`` and ``iou_thr`` as in the NMS call, which must not have reset the counts).  Returns ``out``."""
    infix = _overlap_infix(overlap)
    num, _, classes, boxes = out
    k = int(boxes.shape[1])
    dev = cand.count.device
    name = f"sihl_od_{infix}box_vote_topk"
    with _on(dev):
        rc = getattr(_lib(), name)(_p(cand.count), cand.capacity, _p(cand.key), _p(cand.box), _p(cand.cls), int(batch),
                                   float(iou_thr), k, _p(num), _p(classes), _p(boxes), _stream(dev))
    _native.check(rc, name)
    return out


SOFT_NMS_METHODS = {"linear": 1, "gaussian": 2}          # SIHL_OD_SOFT_NMS_LINEAR / _GAUSSIAN (sihl_od.h)
NMS_KINDS = ("hard", "diou", "soft_linear", "soft_gaussian")


def _soft_method(method) -> int:
    if isinstance(method, str) and method in SOFT_NMS_METHODS:
        return SOFT_NMS_METHODS[method]
    if not isinstance(method, str) and method in SOFT_NMS_METHODS.values():
        return int(method)
    raise ValueError(f"method={method!r}: expected one of {tuple(SOFT_NMS_METHODS)}")


def soft_nms_topk(cand: CandidateBuffers, batch: int, method, iou_thr: float, sigma: float, score_thr: float, k: int,
                  out: Optional[tuple] = None, reset_counts: bool = False):
    """Class-aware Soft-NMS (Bodla et al. 2017) + top-k over the candidate lists, one launch; same outputs as
    :func:`nms_topk` with the decayed scores.  ``method``: ``"linear"`` (``iou_thr`` is Nt) or ``"gaussian"`` (``sigma``)."""
    code = _soft_method(method)
    dev = cand.count.device
    if out is None:
        out = (torch.empty((batch,), dtype=torch.int64, device=dev), torch.empty((batch, k), dtype=torch.float32, device=dev),
               torch.empty((batch, k), dtype=torch.int64, device=dev), torch.empty((batch, k, 4), dtype=torch.float32, device=dev))
    need = int(_lib().sihl_od_soft_nms_workspace_bytes(int(batch), cand.capacity))
    ws = None
    if need:
        ws = getattr(cand, "_soft_ws", None)
        if ws is None or ws.numel() < need:
            ws = torch.empty((need,), dtype=torch.uint8, device=dev)
            cand._soft_ws = ws
    with _on(dev):
        rc = _lib().sihl_od_soft_nms_topk(_p(cand.count), cand.capacity, _p(cand.key), _p(cand.box), _p(cand.cls), int(batch),
                                          code, float(iou_thr), float(sigma), float(score_thr), int(k), _p(out[0]), _p(out[1]),
                                          _p(out[2]), _p(out[3]), _p(ws), int(reset_counts), _stream(dev))
    _native.check(rc, "sihl_od_soft_nms_topk")
    return out


def dense_postprocess(loc_logits: Tensor, cls_logits: Tensor, box_raw: Tensor, levels, img_w: int, img_h: int,
                      score_thr: float = 0.05, iou_thr: float = 0.5, max_instances: int = 100,
                      cand: Optional[CandidateBuffers] = None, mode: str = "dense", split_nms: Optional[bool] = None,
                      nms: str = "hard", sigma: float = 0.5, box_voting: bool = False):
    """Extension (no reference counterpart): dense decode of every location + class-aware NMS.
    Output format of ``ObjectDetection.forward`` (ref :122), zero padded past ``num_instances``.
    ``mode``: see :func:`dense_decode` (identical results).  ``split_nms``: class-split NMS (default: whenever the
    lists can hold more than ``SPLIT_NMS_FROM`` candidates).  ``nms``: ``"hard"`` (greedy, torchvision's semantics),
    ``"diou"`` (greedy DIoU-NMS with ``iou_thr`` as the DIoU threshold), ``"soft_linear"`` (Soft-NMS with ``iou_thr`` as
    Nt) or ``"soft_gaussian"`` (Soft-NMS with ``sigma``); the soft methods keep decaying scores down to ``score_thr``
    and ignore ``split_nms``.  ``box_voting`` (``"hard"`` / ``"diou"`` only): each kept box becomes the score-weighted
    mean of the boxes of its class that its suppression test claims (:func:`box_vote_topk`); the kept set, scores and
    classes are those of the call without voting."""
    if nms not in NMS_KINDS:
        raise ValueError(f"nms={nms!r}: expected one of {NMS_KINDS}")
    if box_voting and nms.startswith("soft_"):
        raise ValueError(f"box_voting=True needs nms='hard' or 'diou', not {nms!r}")
    B, A = loc_logits.shape
    offsets, scales, _ = anchor_tables(levels, img_w, img_h, loc_logits.device)
    if cand is None:
        cand = CandidateBuffers.allocate(B, A, loc_logits.device)
    dense_decode(loc_logits, cls_logits, box_raw, offsets, scales, img_w, img_h, score_thr, cand, mode=mode)
    if nms.startswith("soft_"):
        return soft_nms_topk(cand, B, nms[len("soft_"):], iou_thr, sigma, score_thr, max_instances)
    if split_nms is None:
        # The list lengths are only known on the device, so the choice goes by what can happen: big images (>= 896^2)
        # can yield many thousands of candidates, which one CTA per image would serialise on a few SMs; with many
        # images the single-CTA kernel already fills the GPU, and for the few hundred candidates of a 640^2 image it is
        # 3x cheaper than three launches (measured: profiles/r01_postprocess_sweep.json)
        n_sub = min(32, max(2, -(-cand.capacity // 2048)))
        split_nms = cand.capacity >= SPLIT_NMS_FROM and B * n_sub <= 296
    overlap = "diou" if nms == "diou" else "iou"
    out = nms_topk(cand, B, iou_thr, max_instances, split=split_nms, overlap=overlap)
    if box_voting:
        box_vote_topk(cand, B, iou_thr, out, overlap=overlap)
    return out


def batched_nms(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float,
                seg_offsets: Optional[Tensor] = None, overlap: str = "iou"):
    """``torchvision.ops.batched_nms`` signature (exact per-class semantics, stable order).

    With ``seg_offsets`` (int32 ``[n_images+1]``) the call handles several images at once and
    returns ``(keep [N] i64, keep_count [n_images] i32)``; without it, the kept indices of the
    single segment (one deliberate sync to size the result, like torchvision).  ``overlap="diou"``: DIoU-NMS,
    ``iou_threshold`` is the DIoU threshold (same order and outputs)."""
    infix = _overlap_infix(overlap)
    boxes = _req(boxes, torch.float32, "boxes", 2)
    scores = _req(scores, torch.float32, "scores", 1)
    idxs = _req(idxs, torch.int64, "idxs", 1)
    dev = boxes.device
    N = scores.numel()
    single = seg_offsets is None
    if single:
        seg_offsets = torch.tensor([0, N], dtype=torch.int32, device=dev)
    n_images = seg_offsets.numel() - 1
    keep = torch.empty((max(N, 1),), dtype=torch.int64, device=dev)
    count = torch.zeros((n_images,), dtype=torch.int32, device=dev)
    ws_bytes = int(_lib().sihl_od_batched_nms_workspace_bytes(N))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
    name = f"sihl_od_batched_{infix}nms"
    with _on(dev):
        rc = getattr(_lib(), name)(_p(boxes), _p(scores), _p(idxs), _p(seg_offsets), n_images, N,
                                   float(iou_threshold), _p(keep), _p(count), _p(ws), _stream(dev))
    _native.check(rc, name)
    if single:
        return keep[: int(count.item())]
    return keep[:N], count


def batched_box_vote(boxes: Tensor, scores: Tensor, idxs: Tensor, keep: Tensor, iou_threshold: float,
                     keep_count: Optional[Tensor] = None, seg_offsets: Optional[Tensor] = None, overlap: str = "iou"):
    """Box voting (merge-NMS) after :func:`batched_nms` with the same inputs, threshold and ``overlap``: the voted box
    of every kept index, the score-weighted mean of the boxes of its segment and class that its suppression test
    claims.  Without ``seg_offsets``: ``keep`` is the single segment's result and the return value is ``[len(keep), 4]``.
    With ``seg_offsets``: ``keep`` and ``keep_count`` are :func:`batched_nms`'s and the return value is ``[N, 4]``,
    aligned with ``keep`` (zero past ``keep_count`` in every segment).  No host synchronisation."""
    infix = _overlap_infix(overlap)
    boxes = _req(boxes, torch.float32, "boxes", 2)
    scores = _req(scores, torch.float32, "scores", 1)
    idxs = _req(idxs, torch.int64, "idxs", 1)
    keep = _req(keep, torch.int64, "keep", 1)
    dev = boxes.device
    N = scores.numel()
    if seg_offsets is None:
        seg_offsets = torch.tensor([0, N], dtype=torch.int32, device=dev)
        rows = keep.numel()
        keep_count = torch.full((1,), rows, dtype=torch.int32, device=dev)
    else:
        if keep_count is None:
            raise ValueError("batched_box_vote with seg_offsets needs batched_nms's keep_count")
        seg_offsets = _req(seg_offsets, torch.int32, "seg_offsets", 1)
        keep_count = _req(keep_count, torch.int32, "keep_count", 1)
        rows = N
    n_images = seg_offsets.numel() - 1
    voted = torch.zeros((max(rows, 1), 4), dtype=torch.float32, device=dev)
    if rows == 0:
        return voted[:0]
    name = f"sihl_od_batched_{infix}box_vote"
    with _on(dev):
        rc = getattr(_lib(), name)(_p(boxes), _p(scores), _p(idxs), _p(seg_offsets), n_images, N, float(iou_threshold),
                                   _p(keep), _p(keep_count), _p(voted), _stream(dev))
    _native.check(rc, name)
    return voted[:rows]


def batched_soft_nms(boxes: Tensor, scores: Tensor, idxs: Tensor, max_output: int, method="gaussian",
                     iou_threshold: float = 0.3, sigma: float = 0.5, score_threshold: float = 0.001,
                     seg_offsets: Optional[Tensor] = None):
    """Class-aware Soft-NMS with :func:`batched_nms`'s inputs: the kept indices in selection order and their decayed
    scores, at most ``max_output`` per segment.  ``method``: ``"linear"`` (``iou_threshold`` is Nt) or ``"gaussian"``
    (``sigma``).  Boxes whose score is below ``score_threshold``, or decays below it, are dropped.

    With ``seg_offsets`` (int32 ``[n_images+1]``) returns ``(keep [N] i64, keep_scores [N] f32, keep_count [n_images]
    i32)``, segment s at ``[seg_offsets[s], seg_offsets[s] + keep_count[s])``; without it, ``(keep, keep_scores)`` of
    the single segment (one deliberate sync to size the result)."""
    code = _soft_method(method)
    if int(max_output) < 1:
        raise ValueError(f"max_output={max_output}: expected >= 1")
    boxes = _req(boxes, torch.float32, "boxes", 2)
    scores = _req(scores, torch.float32, "scores", 1)
    idxs = _req(idxs, torch.int64, "idxs", 1)
    dev = boxes.device
    N = scores.numel()
    single = seg_offsets is None
    if single:
        seg_offsets = torch.tensor([0, N], dtype=torch.int32, device=dev)
    else:
        seg_offsets = _req(seg_offsets, torch.int32, "seg_offsets", 1)
    n_images = seg_offsets.numel() - 1
    keep = torch.empty((max(N, 1),), dtype=torch.int64, device=dev)
    keep_scores = torch.empty((max(N, 1),), dtype=torch.float32, device=dev)
    count = torch.zeros((n_images,), dtype=torch.int32, device=dev)
    ws_bytes = int(_lib().sihl_od_batched_soft_nms_workspace_bytes(N))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
    with _on(dev):
        rc = _lib().sihl_od_batched_soft_nms(_p(boxes), _p(scores), _p(idxs), _p(seg_offsets), n_images, N, code,
                                             float(iou_threshold), float(sigma), float(score_threshold), int(max_output),
                                             _p(keep), _p(keep_scores), _p(count), _p(ws), _stream(dev))
    _native.check(rc, "sihl_od_batched_soft_nms")
    if single:
        m = int(count.item())
        return keep[:m], keep_scores[:m]
    return keep[:N], keep_scores[:N], count


QUAD_NMS_MAX = 90000            # quads per batched_quad_nms call (sihl_od.h)


def _req_quads(quads: Tensor, name: str) -> Tensor:
    """``[N, 4, 2]`` or ``[N, 8]`` fp32 CUDA quads -> contiguous ``[N, 8]``."""
    if isinstance(quads, Tensor) and not (quads.dim() == 2 and quads.shape[1] == 8) and \
            not (quads.dim() == 3 and tuple(quads.shape[1:]) == (4, 2)):
        raise ValueError(f"{name}: expected [N, 4, 2] or [N, 8], got shape {tuple(quads.shape)}")
    return _req(quads, torch.float32, name).reshape(-1, 8)


def batched_quad_nms(quads: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float,
                     seg_offsets: Optional[Tensor] = None):
    """Class-aware greedy NMS over quadrilaterals with :func:`batched_nms`'s contract: ``quads`` ``[N, 4, 2]`` or
    ``[N, 8]`` (four points (x, y) in pixels), and the overlap is the IoU of the convex hulls of the two vertex sets
    (``sihl_od.h``; see :func:`quad_iou`).  With ``seg_offsets`` (int32 ``[n_images+1]``) returns ``(keep [N] i64,
    keep_count [n_images] i32)`` without a host synchronisation; without it, the kept indices of the single segment (one
    deliberate sync to size the result).  At most ``QUAD_NMS_MAX`` quads per call."""
    if isinstance(quads, Tensor) and quads.shape[0] > QUAD_NMS_MAX:
        raise ValueError(f"batched_quad_nms takes at most {QUAD_NMS_MAX} quads per call, got {quads.shape[0]}")
    quads = _req_quads(quads, "quads")
    scores = _req(scores, torch.float32, "scores", 1)
    idxs = _req(idxs, torch.int64, "idxs", 1)
    dev = quads.device
    N = scores.numel()
    if quads.shape[0] != N or idxs.numel() != N:
        raise ValueError(f"quads, scores and idxs disagree on N: {quads.shape[0]}, {N}, {idxs.numel()}")
    single = seg_offsets is None
    if single:
        seg_offsets = torch.tensor([0, N], dtype=torch.int32, device=dev)
    else:
        seg_offsets = _req(seg_offsets, torch.int32, "seg_offsets", 1)
    n_images = seg_offsets.numel() - 1
    keep = torch.empty((max(N, 1),), dtype=torch.int64, device=dev)
    count = torch.zeros((n_images,), dtype=torch.int32, device=dev)
    ws_bytes = int(_lib().sihl_od_batched_quad_nms_workspace_bytes(N))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
    with _on(dev):
        rc = _lib().sihl_od_batched_quad_nms(_p(quads), _p(scores), _p(idxs), _p(seg_offsets), n_images, N,
                                             float(iou_threshold), _p(keep), _p(count), _p(ws), _stream(dev))
    _native.check(rc, "sihl_od_batched_quad_nms")
    if single:
        return keep[: int(count.item())]
    return keep[:N], count


def quad_iou(a: Tensor, b: Tensor) -> Tensor:
    """``[Na, Nb]`` fp32 IoU of the convex hulls of the quads ``a`` and ``b`` (``[N, 4, 2]`` or ``[N, 8]``): the polygon
    IoU for convex quads whatever their start vertex and orientation, 0 for a zero-area hull or AABBs that do not
    overlap, and the same bits for (a, b) and (b, a).  The overlap :func:`batched_quad_nms` compares with its threshold."""
    a = _req_quads(a, "a")
    b = _req_quads(b, "b")
    dev = a.device
    out = torch.empty((a.shape[0], b.shape[0]), dtype=torch.float32, device=dev)
    with _on(dev):
        rc = _lib().sihl_od_quad_iou(_p(a), a.shape[0], _p(b), b.shape[0], _p(out), _stream(dev))
    _native.check(rc, "sihl_od_quad_iou")
    return out


# --------------------------------------------------------------------------- N3: matching for the validation mAP
COCO_IOU_THRESHOLDS = tuple(0.5 + 0.05 * i for i in range(10))
COCO_AREA_RANGES = ((0.0, 1e5 ** 2), (0.0, 32.0 ** 2), (32.0 ** 2, 96.0 ** 2), (96.0 ** 2, 1e5 ** 2))    # all, small, medium, large


def _gt_annotations(gt_crowd: Optional[Tensor], gt_area: Optional[Tensor], G: int):
    """COCO's optional per-gt annotations for the ``_crowd`` matching entries: ``gt_crowd`` (bool or integer, nonzero
    marks a crowd region) -> uint8 0 / 1, ``gt_area`` (any real dtype) -> float64, both ``[G]`` CUDA tensors or None.
    Shapes and dtypes are checked before anything runs on the device."""
    for name, t in (("gt_crowd", gt_crowd), ("gt_area", gt_area)):
        if t is None:
            continue
        if not isinstance(t, Tensor):
            raise TypeError(f"{name}: expected a torch.Tensor or None, got {type(t).__name__}")
        if tuple(t.shape) != (G,):
            raise ValueError(f"{name}: expected shape [{G}] (one value per ground truth), got {tuple(t.shape)}")
        if t.is_complex() or (name == "gt_crowd" and t.is_floating_point()):
            raise TypeError(f"{name}: expected {'bool or integer' if name == 'gt_crowd' else 'real'} values, got {t.dtype}")
        if not t.is_cuda:
            raise RuntimeError(f"{name}: sihl_b200 kernels run on CUDA tensors only (got {t.device}); there is no CPU path")
    if gt_crowd is not None:
        gt_crowd = (gt_crowd != 0).to(torch.uint8).contiguous()
    if gt_area is not None:
        gt_area = gt_area.to(torch.float64).contiguous()
    return gt_crowd, gt_area


def map_match(det_boxes: Tensor, det_scores: Tensor, det_classes: Tensor, gt_boxes: Tensor, gt_classes: Tensor,
              gt_offsets: Tensor, iou_thresholds: Sequence[float] = COCO_IOU_THRESHOLDS,
              area_ranges: Sequence[Tuple[float, float]] = COCO_AREA_RANGES, gt_crowd: Optional[Tensor] = None,
              gt_area: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """COCOeval.evaluateImg for a whole batch on the GPU (ref object_detection.py:230-237 feeds this to torchmetrics,
    which matches on the CPU at epoch end).  ``det_*`` [B,K,...] as ``forward`` returns them, ground truth in CSR form.
    Returns dict(det_order i32 [B,K], dt_match i32 [B,NA,T,K], dt_ignore u8 [B,NA,T,K], gt_ignore u8 [NA,sumG]).

    ``gt_crowd`` / ``gt_area`` (``[sumG]`` CUDA tensors, optional) are COCO's ``iscrowd`` and ``area`` annotations
    (``sihl_od_map_match_crowd``): a crowd gt is ignored in every area range, overlaps a detection by intersection over
    the detection's area and may be matched by any number of detections, which are then ignored; an area > 0 replaces
    the box area in the area-range test.  Without either, the tables are those of the plain matching."""
    crowd, area = _gt_annotations(gt_crowd, gt_area, int(gt_boxes.shape[0]))
    det_boxes = _req(det_boxes, torch.float32, "det_boxes", 3)
    det_scores = _req(det_scores.float() if det_scores.dtype != torch.float32 else det_scores, torch.float32, "det_scores", 2)
    det_classes = _req(det_classes, torch.int64, "det_classes", 2)
    dev = det_boxes.device
    B, K = det_scores.shape
    G = int(gt_boxes.shape[0])
    thr = np.ascontiguousarray(np.asarray(iou_thresholds, dtype=np.float64))
    areas = np.ascontiguousarray(np.asarray(area_ranges, dtype=np.float64).reshape(-1, 2))
    T, NA = len(thr), len(areas)
    with _on(dev):
        order = torch.empty((B, K), dtype=torch.int32, device=dev)
        dtm = torch.empty((B, NA, T, K), dtype=torch.int32, device=dev)
        dti = torch.empty((B, NA, T, K), dtype=torch.uint8, device=dev)
        gti = torch.empty((NA, max(G, 1)), dtype=torch.uint8, device=dev)
        ws = torch.empty((int(_lib().sihl_od_map_workspace_bytes(G, T, NA)),), dtype=torch.uint8, device=dev)
        gt = (_p(_req(gt_boxes, torch.float32, "gt_boxes", 2)) if G else None,
              _p(_req(gt_classes, torch.int64, "gt_classes", 1)) if G else None,
              _p(_req(gt_offsets, torch.int32, "gt_offsets", 1)), G)
        rest = (thr.ctypes.data, T, areas.ctypes.data, NA, _p(order), _p(dtm), _p(dti), _p(gti), _p(ws), _stream(dev))
        if crowd is None and area is None:
            name = "sihl_od_map_match"
            rc = _lib().sihl_od_map_match(_p(det_boxes), _p(det_scores), _p(det_classes), B, K, *gt, *rest)
        else:
            name = "sihl_od_map_match_crowd"
            rc = _lib().sihl_od_map_match_crowd(_p(det_boxes), _p(det_scores), _p(det_classes), B, K, *gt,
                                                _p(crowd) if G else None, _p(area) if G else None, *rest)
    _native.check(rc, name)
    return dict(det_order=order, dt_match=dtm, dt_ignore=dti, gt_ignore=gti[:, :G])


MAP_MAX_K, MAP_MAX_THRESHOLDS, MAP_MAX_AREAS = 1024, 16, 8     # sihl_od_map_match / sihl_od_quad_map_match (sihl_od.h)


def quad_map_match(det_quads: Tensor, det_scores: Tensor, det_classes: Tensor, gt_quads: Tensor, gt_classes: Tensor,
                   gt_offsets: Tensor, iou_thresholds: Sequence[float] = COCO_IOU_THRESHOLDS,
                   area_ranges: Sequence[Tuple[float, float]] = COCO_AREA_RANGES, gt_crowd: Optional[Tensor] = None,
                   gt_area: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """:func:`map_match` for quadrilaterals: ``det_quads`` ``[B,K,4,2]`` or ``[B,K,8]``, ``gt_quads`` ``[sumG,4,2]`` or
    ``[sumG,8]`` (four points (x, y) in px).  The IoU is :func:`quad_iou`'s (convex hulls of the vertex sets) and the area
    that places a quad in an area range is its hull's polygon area.  Returns the same dict as :func:`map_match`.  Shapes
    and limits (K <= 1024, at most 16 thresholds and 8 area ranges) are checked before any CUDA call.  ``gt_crowd`` /
    ``gt_area`` as in :func:`map_match` (``sihl_od_quad_map_match_crowd``): a crowd quad ("don't care" region) overlaps
    a detection by the hulls' intersection over the detection's hull area, and an area > 0 replaces the hull area."""
    if isinstance(det_quads, Tensor) and not (det_quads.dim() == 3 and det_quads.shape[2] == 8) and \
            not (det_quads.dim() == 4 and tuple(det_quads.shape[2:]) == (4, 2)):
        raise ValueError(f"det_quads: expected [B, K, 4, 2] or [B, K, 8], got shape {tuple(det_quads.shape)}")
    if isinstance(det_scores, Tensor) and det_scores.dim() != 2:
        raise ValueError(f"det_scores: expected [B, K], got shape {tuple(det_scores.shape)}")
    B, K = (int(v) for v in det_scores.shape)
    if tuple(det_quads.shape[:2]) != (B, K) or tuple(det_classes.shape) != (B, K):
        raise ValueError(f"det_quads {tuple(det_quads.shape)}, det_scores {(B, K)} and det_classes "
                         f"{tuple(det_classes.shape)} disagree on [B, K]")
    if not 1 <= K <= MAP_MAX_K:
        raise ValueError(f"quad_map_match takes 1 to {MAP_MAX_K} detections per image, got K={K}")
    thr = np.ascontiguousarray(np.asarray(iou_thresholds, dtype=np.float64).reshape(-1))
    areas = np.ascontiguousarray(np.asarray(area_ranges, dtype=np.float64).reshape(-1, 2))
    T, NA = len(thr), len(areas)
    if not (1 <= T <= MAP_MAX_THRESHOLDS and 1 <= NA <= MAP_MAX_AREAS):
        raise ValueError(f"quad_map_match takes 1 to {MAP_MAX_THRESHOLDS} IoU thresholds and 1 to {MAP_MAX_AREAS} area "
                         f"ranges, got {T} and {NA}")
    crowd, area = _gt_annotations(gt_crowd, gt_area, int(gt_quads.shape[0]))
    det_quads = _req(det_quads, torch.float32, "det_quads").reshape(B, K, 8)
    det_scores = _req(det_scores.float() if det_scores.dtype != torch.float32 else det_scores, torch.float32, "det_scores", 2)
    det_classes = _req(det_classes, torch.int64, "det_classes", 2)
    gt_quads = _req_quads(gt_quads, "gt_quads")
    G = int(gt_quads.shape[0])
    gt_classes = _req(gt_classes, torch.int64, "gt_classes", 1)
    gt_offsets = _req(gt_offsets, torch.int32, "gt_offsets", 1)
    if gt_classes.numel() != G or gt_offsets.numel() != B + 1:
        raise ValueError(f"gt_quads [{G}], gt_classes [{gt_classes.numel()}] and gt_offsets [{gt_offsets.numel()}] "
                         f"do not describe {B} images")
    dev = det_quads.device
    ws_bytes = int(_lib().sihl_od_quad_map_workspace_bytes(B, K, G, T, NA))
    with _on(dev):
        order = torch.empty((B, K), dtype=torch.int32, device=dev)
        dtm = torch.empty((B, NA, T, K), dtype=torch.int32, device=dev)
        dti = torch.empty((B, NA, T, K), dtype=torch.uint8, device=dev)
        gti = torch.empty((NA, max(G, 1)), dtype=torch.uint8, device=dev)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        gt = (_p(gt_quads) if G else None, _p(gt_classes) if G else None, _p(gt_offsets), G)
        rest = (thr.ctypes.data, T, areas.ctypes.data, NA, _p(order), _p(dtm), _p(dti), _p(gti), _p(ws), ws_bytes,
                _stream(dev))
        if crowd is None and area is None:
            name = "sihl_od_quad_map_match"
            rc = _lib().sihl_od_quad_map_match(_p(det_quads), _p(det_scores), _p(det_classes), B, K, *gt, *rest)
        else:
            name = "sihl_od_quad_map_match_crowd"
            rc = _lib().sihl_od_quad_map_match_crowd(_p(det_quads), _p(det_scores), _p(det_classes), B, K, *gt,
                                                     _p(crowd) if G else None, _p(area) if G else None, *rest)
    _native.check(rc, name)
    return dict(det_order=order, dt_match=dtm, dt_ignore=dti, gt_ignore=gti[:, :G])


# ---- N4 (SURVEY.md §8f): the per-location MLP towers on the tensor cores -------------------------------------------------
MLP_CHANNELS = 256                      # the reference's num_channels default; the kernels are built for it
_MLP_OUT_PADS = (16, 32, 64, 96, 128, 256)


def mlp_out_pad(out_features: int) -> int:
    """Rows the output layer's weight is zero-padded to (tcgen05.mma needs N % 16 == 0)."""
    for n in _MLP_OUT_PADS:
        if out_features <= n:
            return n
    raise ValueError(f"out_features {out_features} > 256 is not supported by sihl_od_mlp_out")


def mlp_hidden(x: Tensor, weight: Tensor, bias: Tensor, gamma: Tensor, beta: Tensor, eps: float = 1e-5,
               out: Optional[Tensor] = None) -> Tensor:
    """One hidden layer of ``torchvision.ops.MLP(..., norm_layer=LayerNorm, activation_layer=SiLU)`` (ref
    object_detection.py:51, :56-60): ``SiLU(LayerNorm(x @ weight.T + bias))`` in ONE kernel.  x [M,256] bf16, weight
    [256,256] bf16, bias / gamma / beta fp32 [256]; returns bf16 [M,256].  Inference only."""
    x = _req(x, torch.bfloat16, "x", 2)
    weight = _req(weight, torch.bfloat16, "weight", 2)
    M, K = x.shape
    if K != MLP_CHANNELS or tuple(weight.shape) != (MLP_CHANNELS, MLP_CHANNELS):
        raise ValueError(f"mlp_hidden is built for {MLP_CHANNELS} channels, got x {tuple(x.shape)} weight {tuple(weight.shape)}")
    dev = x.device
    with _on(dev):
        y = out if out is not None else torch.empty((M, K), dtype=torch.bfloat16, device=dev)
        rc = _lib().sihl_od_mlp_hidden(_p(x), M, K, _p(weight), _p(_req(bias, torch.float32, "bias", 1)),
                                       _p(_req(gamma, torch.float32, "gamma", 1)), _p(_req(beta, torch.float32, "beta", 1)),
                                       float(eps), _p(_req(y, torch.bfloat16, "out", 2)), _stream(dev))
    _native.check(rc, "sihl_od_mlp_hidden")
    return y


def mlp_out(x: Tensor, weight_padded: Tensor, bias_padded: Tensor, out_features: int, out: Optional[Tensor] = None) -> Tensor:
    """The tower's last ``Linear(256, out_features)``: x [M,256] bf16, ``weight_padded`` [n_pad,256] bf16 with rows
    >= out_features zero (``mlp_out_pad``), ``bias_padded`` fp32 [n_pad]; returns fp32 [M,out_features]."""
    x = _req(x, torch.bfloat16, "x", 2)
    weight_padded = _req(weight_padded, torch.bfloat16, "weight_padded", 2)
    M, K = x.shape
    n_pad = int(weight_padded.shape[0])
    if K != MLP_CHANNELS or weight_padded.shape[1] != K or n_pad not in _MLP_OUT_PADS or not 1 <= out_features <= n_pad:
        raise ValueError(f"mlp_out: x {tuple(x.shape)}, weight_padded {tuple(weight_padded.shape)}, out_features {out_features}")
    dev = x.device
    with _on(dev):
        y = out if out is not None else torch.empty((M, out_features), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_mlp_out(_p(x), M, K, _p(weight_padded), _p(_req(bias_padded, torch.float32, "bias_padded", 1)),
                                    n_pad, int(out_features), _p(_req(y, torch.float32, "out", 2)), _stream(dev))
    _native.check(rc, "sihl_od_mlp_out")
    return y


def lateral_rows(x: Tensor, out: Optional[Tensor] = None) -> Tensor:
    """One NCHW fp32 pyramid level [B, C, H, W] -> its locations as bf16 rows [B*H*W, C] (C % 64 == 0): the layout the
    tensor-core layers read (ref object_detection.py:105 does ``rearrange(x, "b c h w -> b (h w) c")`` after the conv)."""
    x = _req(x, torch.float32, "x", 4)
    B, C, H, W = x.shape
    if C % 64:
        raise ValueError(f"lateral_rows needs channels % 64 == 0, got {C}")
    dev = x.device
    with _on(dev):
        y = out if out is not None else torch.empty((B * H * W, C), dtype=torch.bfloat16, device=dev)
        rc = _lib().sihl_od_lateral_rows(_p(x), B, C, H * W, _p(_req(y, torch.bfloat16, "out", 2)), _stream(dev))
    _native.check(rc, "sihl_od_lateral_rows")
    return y


def lateral_linear(rows: Tensor, weight: Tensor, bias: Tensor, rows_per_image: int, out: Tensor, out_row_offset: int) -> Tensor:
    """``rows @ weight.T + bias`` (bf16 [M,256] x bf16 [256,256], fp32 bias) written into ``out`` [B, A, 256] bf16 at
    ``out[b, out_row_offset + i]`` for row ``b * rows_per_image + i``: a lateral (1x1 conv with its BatchNorm folded in,
    ref object_detection.py:52-55) landing in its slice of the concatenated features (ref :105)."""
    rows = _req(rows, torch.bfloat16, "rows", 2)
    weight = _req(weight, torch.bfloat16, "weight", 2)
    out = _req(out, torch.bfloat16, "out", 3)
    M, K = rows.shape
    if K != MLP_CHANNELS or tuple(weight.shape) != (K, K) or out.shape[2] != K or M % rows_per_image or M // rows_per_image != out.shape[0]:
        raise ValueError(f"lateral_linear: rows {tuple(rows.shape)}, weight {tuple(weight.shape)}, out {tuple(out.shape)}, "
                         f"rows_per_image {rows_per_image}")
    dev = rows.device
    with _on(dev):
        rc = _lib().sihl_od_lateral_linear(_p(rows), M, K, _p(weight), _p(_req(bias, torch.float32, "bias", 1)), int(rows_per_image),
                                           int(out.shape[1]), int(out_row_offset), _p(out), _stream(dev))
    _native.check(rc, "sihl_od_lateral_linear")
    return out


_ZERO_BIAS: Dict[torch.device, Tensor] = {}


def zero_bias(device) -> Tensor:
    """A cached, read-only fp32 zero vector of ``MLP_CHANNELS`` entries on ``device`` (the bias of the gradient GEMMs)."""
    device = torch.device(device)
    z = _ZERO_BIAS.get(device)
    if z is None:
        z = _ZERO_BIAS[device] = torch.zeros((MLP_CHANNELS,), dtype=torch.float32, device=device)
    return z


def linear_bf16(x: Tensor, weight: Tensor, bias: Tensor) -> Tensor:
    """``x @ weight.T + bias`` for x [M,256] bf16, weight [256,256] bf16, bias fp32 -> bf16 [M,256] (the linear mode of the
    tensor-core layer kernel with the identity row map)."""
    M = int(x.shape[0])
    out = torch.empty((1, M, MLP_CHANNELS), dtype=torch.bfloat16, device=x.device)
    if M:
        lateral_linear(x, weight, bias, M, out, 0)
    return out[0]


def mlp_hidden_train(x: Tensor, weight: Tensor, bias: Tensor, gamma: Tensor, beta: Tensor, eps: float = 1e-5,
                     save_pre: bool = False):
    """:func:`mlp_hidden` that also returns every row's LayerNorm statistics [M,2] = (mean, rstd) for the backward and,
    with ``save_pre``, the pre-activation ``v = x W^T + b`` (bf16 [M,256], written by the same epilogue) as a third
    result, so that the backward does not recompute it."""
    x = _req(x, torch.bfloat16, "x", 2)
    weight = _req(weight, torch.bfloat16, "weight", 2)
    M, K = x.shape
    if K != MLP_CHANNELS or tuple(weight.shape) != (K, K):
        raise ValueError(f"mlp_hidden_train is built for {MLP_CHANNELS} channels, got x {tuple(x.shape)} weight {tuple(weight.shape)}")
    dev = x.device
    with _on(dev):
        y = torch.empty((M, K), dtype=torch.bfloat16, device=dev)
        stats = torch.empty((M, 2), dtype=torch.float32, device=dev)
        v = torch.empty((M, K), dtype=torch.bfloat16, device=dev) if save_pre else None
        rc = _lib().sihl_od_mlp_hidden_train(_p(x), M, K, _p(weight), _p(_req(bias, torch.float32, "bias", 1)),
                                             _p(_req(gamma, torch.float32, "gamma", 1)), _p(_req(beta, torch.float32, "beta", 1)),
                                             float(eps), _p(y), _p(stats), _p(v), _stream(dev))
    _native.check(rc, "sihl_od_mlp_hidden_train")
    return (y, stats, v) if save_pre else (y, stats)


def mlp_hidden_bwd(v: Tensor, dy: Tensor, row_stats: Tensor, gamma: Tensor, beta: Tensor) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Backward of LayerNorm + SiLU over rows: pre-activation ``v`` [M,256] bf16, upstream ``dy`` [M,256] bf16, the forward's
    ``row_stats`` -> (dv bf16 [M,256], d_gamma, d_beta, d_bias fp32 [256])."""
    v = _req(v, torch.bfloat16, "v", 2)
    dy = _req(dy, torch.bfloat16, "dy", 2)
    M, K = v.shape
    if K != MLP_CHANNELS or dy.shape != v.shape or tuple(row_stats.shape) != (M, 2):
        raise ValueError(f"mlp_hidden_bwd: v {tuple(v.shape)}, dy {tuple(dy.shape)}, row_stats {tuple(row_stats.shape)}")
    dev = v.device
    with _on(dev):
        n_part = int(_lib().sihl_od_mlp_hidden_bwd_partial_rows())
        dv = torch.empty((M, K), dtype=torch.bfloat16, device=dev)
        partials = torch.empty((n_part, 3, K), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_mlp_hidden_bwd(_p(v), _p(dy), _p(_req(row_stats, torch.float32, "row_stats", 2)),
                                           _p(_req(gamma, torch.float32, "gamma", 1)), _p(_req(beta, torch.float32, "beta", 1)),
                                           M, K, _p(dv), _p(partials), n_part, _stream(dev))
    _native.check(rc, "sihl_od_mlp_hidden_bwd")
    sums = partials.sum(0)
    return dv, sums[0], sums[1], sums[2]


def mlp_hidden_bwd_rank1(v: Tensor, dout: Tensor, w_out: Tensor, row_stats: Tensor, gamma: Tensor, beta: Tensor
                         ) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """:func:`mlp_hidden_bwd` for a tower's last hidden layer when the Linear behind it has ONE output: the upstream
    gradient ``bf16(dout)[:, None] * w_out[None, :]`` (``dout`` fp32 [M], ``w_out`` bf16 [256]) is formed in registers
    instead of being materialised by a K = 1 GEMM."""
    v = _req(v, torch.bfloat16, "v", 2)
    dout = _req(dout, torch.float32, "dout", 1)
    w_out = _req(w_out, torch.bfloat16, "w_out", 1)
    M, K = v.shape
    if K != MLP_CHANNELS or dout.shape[0] != M or w_out.shape[0] != K or tuple(row_stats.shape) != (M, 2):
        raise ValueError(f"mlp_hidden_bwd_rank1: v {tuple(v.shape)}, dout {tuple(dout.shape)}, w_out {tuple(w_out.shape)}, "
                         f"row_stats {tuple(row_stats.shape)}")
    dev = v.device
    with _on(dev):
        n_part = int(_lib().sihl_od_mlp_hidden_bwd_partial_rows())
        dv = torch.empty((M, K), dtype=torch.bfloat16, device=dev)
        partials = torch.empty((n_part, 3, K), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_mlp_hidden_bwd_rank1(_p(v), _p(dout), _p(w_out), _p(_req(row_stats, torch.float32, "row_stats", 2)),
                                                 _p(_req(gamma, torch.float32, "gamma", 1)), _p(_req(beta, torch.float32, "beta", 1)),
                                                 M, K, _p(dv), _p(partials), n_part, _stream(dev))
    _native.check(rc, "sihl_od_mlp_hidden_bwd_rank1")
    sums = partials.sum(0)
    return dv, sums[0], sums[1], sums[2]


def rows_colsum(rows: Tensor) -> Tensor:
    """fp32 column sums [256] of bf16 rows [M,256]: one HBM-bound pass (the first moment of a lateral's input)."""
    rows = _req(rows, torch.bfloat16, "rows", 2)
    M, K = rows.shape
    if K != MLP_CHANNELS:
        raise ValueError(f"rows_colsum is built for {MLP_CHANNELS} channels, got {tuple(rows.shape)}")
    dev = rows.device
    with _on(dev):
        n_part = int(_lib().sihl_od_mlp_bwd_partial_rows())
        partials = torch.empty((n_part, K), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_rows_colsum(_p(rows), M, K, _p(partials), n_part, _stream(dev))
    _native.check(rc, "sihl_od_rows_colsum")
    return partials.sum(0)


def bf16_to_f32(t: Tensor) -> Tensor:
    """fp32 copy of a contiguous bf16 tensor whose element count is a multiple of 8 (full-width loads and stores)."""
    t = _req(t, torch.bfloat16, "t")
    if t.numel() % 8:
        return t.float()
    dev = t.device
    with _on(dev):
        out = torch.empty(t.shape, dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_bf16_to_f32(_p(t), t.numel(), _p(out), _stream(dev))
    _native.check(rc, "sihl_od_bf16_to_f32")
    return out


def rows_to_nchw(rows: Tensor, batch: int, height: int, width: int) -> Tensor:
    """bf16 rows [B*H*W, C] -> fp32 NCHW [B, C, H, W] (inverse layout of :func:`lateral_rows`; C % 64 == 0)."""
    rows = _req(rows, torch.bfloat16, "rows", 2)
    C = int(rows.shape[1])
    if C % 64 or rows.shape[0] != batch * height * width:
        raise ValueError(f"rows_to_nchw: rows {tuple(rows.shape)} for batch {batch}, {height}x{width}")
    dev = rows.device
    with _on(dev):
        x = torch.empty((batch, C, height, width), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_rows_to_nchw(_p(rows), batch, C, height * width, _p(x), _stream(dev))
    _native.check(rc, "sihl_od_rows_to_nchw")
    return x


def bn_bwd_rows(dz: Tensor, n: Tensor, scale: Tensor, dz_rows_per_image: Optional[int] = None, dz_row_offset: int = 0,
                rows_per_image: Optional[int] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """Backward of a batch-statistics BatchNorm over rows: ``dz`` bf16 (gradient of the normalised + affine output),
    ``n`` [M,256] bf16 (normalised conv output), ``scale`` = gamma * invstd fp32 [256] -> (dy bf16 [M,256] = gradient of
    the conv output, d_gamma, d_beta fp32 [256]).

    ``dz`` is either [M,256], or — with ``rows_per_image`` / ``dz_rows_per_image`` / ``dz_row_offset`` — the whole
    contiguous [B, dz_rows_per_image, 256] gradient of the concatenated features, of which this level is the slice
    ``[:, dz_row_offset : dz_row_offset + rows_per_image]`` (read in place: no strided copy)."""
    n = _req(n, torch.bfloat16, "n", 2)
    M, K = n.shape
    if rows_per_image is None:
        dz = _req(dz, torch.bfloat16, "dz", 2)
        if dz.shape != n.shape:
            raise ValueError(f"bn_bwd_rows: dz {tuple(dz.shape)}, n {tuple(n.shape)}")
        rows_per_image, dz_rows_per_image, dz_row_offset = max(M, 1), max(M, 1), 0
    else:
        dz = _req(dz, torch.bfloat16, "dz", 3)
        if (dz.shape[2] != K or dz.shape[1] != dz_rows_per_image or dz.shape[0] * rows_per_image != M or dz_row_offset < 0
                or dz_row_offset + rows_per_image > dz_rows_per_image):
            raise ValueError(f"bn_bwd_rows: dz {tuple(dz.shape)}, n {tuple(n.shape)}, slice {dz_row_offset}+{rows_per_image}")
    if K != MLP_CHANNELS:
        raise ValueError(f"bn_bwd_rows is built for {MLP_CHANNELS} channels, got {K}")
    dev = n.device
    with _on(dev):
        n_part = int(_lib().sihl_od_mlp_bwd_partial_rows())
        partials = torch.empty((n_part, 2, K), dtype=torch.float32, device=dev)
        rc = _lib().sihl_od_bn_bwd_colsums_map(_p(dz), int(rows_per_image), int(dz_rows_per_image), int(dz_row_offset), _p(n), M, K,
                                               _p(partials), n_part, _stream(dev))
        _native.check(rc, "sihl_od_bn_bwd_colsums_map")
        sums = partials.sum(0)
        d_beta, d_gamma = sums[0], sums[1]
        dy = torch.empty((M, K), dtype=torch.bfloat16, device=dev)
        # named, so that they outlive the launch: a temporary inside the argument list is freed (and its block handed to the
        # next temporary) before the kernel is enqueued
        mean_dz, mean_dzn, scale = (d_beta / M).contiguous(), (d_gamma / M).contiguous(), _req(scale, torch.float32, "scale", 1)
        rc = _lib().sihl_od_bn_bwd_apply_map(_p(dz), int(rows_per_image), int(dz_rows_per_image), int(dz_row_offset), _p(n), _p(scale),
                                             _p(mean_dz), _p(mean_dzn), M, K, _p(dy), _stream(dev))
    _native.check(rc, "sihl_od_bn_bwd_apply_map")
    return dy, d_gamma, d_beta
