"""Steady-state pipeline over dense head outputs: assign + losses and dense decode + NMS
with every buffer preallocated, two CUDA streams and (optionally) one CUDA graph per step.

This is the whole-batch form of the hot path that ``bench.py`` measures
(BASELINE.json metric: det-head images/sec, assign + loss + NMS).  Per step and GPU:

  train chain  (stream A): k_assign_select -> k_assign_resolve (dense losses fused)
                           -> k_pos_loss_tiles (last CTA finalizes) [3 launches]
  infer chain  (stream B): k_dense_decode_tma (or k_candidate_decode, ``decode_mode``) -> k_nms  [2 launches]

The two chains share no data, so they run concurrently: the assignment is FP32-ALU/latency
bound, the dense decode is HBM bound (SURVEY.md §8d caveat).  Across GPUs the only exchange
is ``sums`` (8 doubles), all-reduced between resolve and finalize when ``world_size > 1``.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _native, ops

LAUNCHES_PER_STEP = 5     # select, resolve, pos_loss_tiles (+finalize) | dense_decode, nms


@dataclass
class StepInputs:
    """Inputs of one step (one batch shard), device resident — except that ``box_raw`` / ``cls_logits`` may be pinned
    host tensors when the pipeline runs ``decode_mode="candidate_first"``: both chains only gather rows of them
    (positives, candidates), which the kernels then read in place over PCIe instead of uploading the whole maps."""
    loc_logits: Tensor     # [B, A]      fp32, or fp16 / bf16 (all four maps alike: loaded as they are, upcast in registers)
    iou_preds: Tensor      # [B, A]
    box_raw: Tensor        # [B, A, 4]
    cls_logits: Tensor     # [B, A, C]
    gt: ops.GtBatch

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in
                   (self.loc_logits, self.iou_preds, self.box_raw, self.cls_logits, self.gt.boxes, self.gt.classes,
                    self.gt.offsets))


@dataclass
class StepOutputs:
    assignment: Tensor     # [B, A] i64
    rel_iou: Tensor        # [B, A] f32
    sums: Tensor           # [8] f64
    losses: Tensor         # [5] f32: location, box, class, iou, total
    num_instances: Tensor  # [B] i64
    scores: Tensor         # [B, K] f32
    classes: Tensor        # [B, K] i64
    boxes: Tensor          # [B, K, 4] f32


class DetectionHeadPipeline:
    def __init__(self, levels: Sequence[Tuple[int, int]], img_w: int, img_h: int, batch: int, num_classes: int,
                 max_gt_total: int, device, topk: int = 9, max_instances: int = 100, score_thr: float = 0.05,
                 iou_thr: float = 0.5, cand_capacity: Optional[int] = None, decode_mode: str = "dense"):
        if decode_mode not in ops.DECODE_MODES:
            raise ValueError(f"decode_mode={decode_mode!r}: expected one of {ops.DECODE_MODES}")
        self.decode_mode = decode_mode
        self.levels = [tuple(int(v) for v in l) for l in levels]
        self.img_w, self.img_h, self.B, self.C = int(img_w), int(img_h), int(batch), int(num_classes)
        self.device = torch.device(device)
        self.topk, self.K, self.score_thr, self.iou_thr = int(topk), int(max_instances), float(score_thr), float(iou_thr)
        self.offsets, self.scales, self.anchors = ops.anchor_tables(self.levels, img_w, img_h, self.device)
        self.terms = ops.anchor_terms(self.levels, img_w, img_h, self.device)
        self.A = int(self.anchors.shape[0])
        self._hw = ops._levels_array(self.levels)
        dev, B, A, K = self.device, self.B, self.A, self.K
        self.sel_anchor = torch.empty((max_gt_total, topk), dtype=torch.int32, device=dev)
        self.sel_val = torch.empty((max_gt_total, topk), dtype=torch.float32, device=dev)
        self.best_iou = torch.empty((max_gt_total,), dtype=torch.float32, device=dev)
        self.max_gt_total = int(max_gt_total)
        n_tiles, tile = ops.resolve_tiles(A)
        self.tile_pos_count = torch.zeros((B * n_tiles,), dtype=torch.int32, device=dev)
        self.tile_pos_rows = torch.zeros((B * n_tiles * tile,), dtype=torch.int32, device=dev)
        self.pos_chunks = torch.zeros((B * n_tiles * (tile // 32),), dtype=torch.int32, device=dev)
        self.tile_pos_aux = torch.zeros((B * n_tiles * tile, 2), dtype=torch.int32, device=dev)
        self.done_counter = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.cand = ops.CandidateBuffers.allocate(B, int(cand_capacity or A), dev)
        self.side = torch.cuda.Stream(device=dev)                 # the inference chain's stream
        self.lib = _native.load()
        self._exchange = None

    def new_outputs(self) -> StepOutputs:
        dev, B, A, K = self.device, self.B, self.A, self.K
        return StepOutputs(
            assignment=torch.empty((B, A), dtype=torch.int64, device=dev),
            rel_iou=torch.empty((B, A), dtype=torch.float32, device=dev),
            sums=torch.zeros((8,), dtype=torch.float64, device=dev),
            losses=torch.zeros((5,), dtype=torch.float32, device=dev),
            num_instances=torch.empty((B,), dtype=torch.int64, device=dev),
            scores=torch.empty((B, K), dtype=torch.float32, device=dev),
            classes=torch.empty((B, K), dtype=torch.int64, device=dev),
            boxes=torch.empty((B, K, 4), dtype=torch.float32, device=dev))

    # -- the two chains (enqueue only; no sync) --------------------------------------------
    def attach_exchange(self, exchange, region: int) -> None:
        """Multi-GPU: let the loss kernel all-reduce the 8 partial sums itself over peer memory
        (``dist.PeerExchange``, one region per pipeline / step in flight) instead of an NCCL node + a finalize launch."""
        self._exchange = (exchange.peer_array(region), exchange.world, exchange.rank)

    def train_chain(self, x: StepInputs, out: StepOutputs, finalize: bool = True) -> None:
        lib, st = self.lib, torch.cuda.current_stream(self.device).cuda_stream
        gt = x.gt
        assert gt.total <= self.max_gt_total and gt.batch_size == self.B
        p = ops._p
        # host-resident class / box maps (pinned): k_pos_loss_tiles gathers the positives' rows in place over PCIe;
        # the L2 prefetch hints of k_assign_resolve only make sense for device memory
        maps_on_device = x.cls_logits.is_cuda and x.box_raw.is_cuda
        assert maps_on_device or (x.cls_logits.is_pinned() and x.box_raw.is_pinned()), "host maps must be pinned"
        dt = x.loc_logits.dtype
        assert dt in ops.DTYPE_CODES and all(t.dtype == dt for t in (x.iou_preds, x.box_raw, x.cls_logits)), \
            "the four head-output maps must share one of fp32 / fp16 / bf16"
        code = ops.DTYPE_CODES[dt]
        _native.check(lib.sihl_od_assign_select(
            p(self.anchors), p(self.terms), self.A, self._hw.ctypes.data, len(self._hw), self.img_w, self.img_h, p(gt.boxes),
            p(gt.offsets), self.B, gt.total, self.topk, p(self.sel_anchor), p(self.sel_val), p(self.best_iou),
            p(out.sums), st), "sihl_od_assign_select")
        _native.check(lib.sihl_od_assign_resolve_t(
            p(self.sel_anchor), p(self.sel_val), p(self.best_iou), p(gt.offsets), self.B, self.A, self.topk, 1,
            p(x.loc_logits), p(x.iou_preds), code, p(out.assignment), p(out.rel_iou), p(out.sums), p(self.tile_pos_count),
            p(self.tile_pos_rows), p(x.box_raw) if maps_on_device else None, p(x.cls_logits) if maps_on_device else None,
            self.C, p(self.pos_chunks), p(self.tile_pos_aux), st),
            "sihl_od_assign_resolve_t")
        # single GPU: the last CTA of the positive-loss kernel also finalizes the five losses
        peers, world, rank = self._exchange if (finalize and self._exchange is not None) else (None, 1, 0)
        _native.check(lib.sihl_od_pos_loss_tiles_exchange_t(
            p(self.pos_chunks), p(self.tile_pos_rows), p(self.tile_pos_aux), self.B, self.A,
            p(self.offsets), p(self.scales), self.img_w, self.img_h, p(gt.boxes), p(gt.classes), p(gt.offsets),
            p(x.box_raw), p(x.cls_logits), code, self.C, p(out.sums), p(out.losses) if finalize else None,
            p(self.done_counter) if finalize else None, peers, world, rank, st), "sihl_od_pos_loss_tiles_exchange_t")

    def finalize(self, out: StepOutputs) -> None:
        st = torch.cuda.current_stream(self.device).cuda_stream
        _native.check(self.lib.sihl_od_loss_finalize(ops._p(out.sums), ops._p(out.losses), st), "sihl_od_loss_finalize")

    def infer_chain(self, x: StepInputs, out: StepOutputs) -> None:
        # the candidate counters start at zero and k_nms* re-zero them once consumed: no memset launch
        ops.dense_decode(x.loc_logits, x.cls_logits, x.box_raw, self.offsets, self.scales, self.img_w, self.img_h,
                         self.score_thr, self.cand, zero_counts=False, mode=self.decode_mode)
        ops.nms_topk(self.cand, self.B, self.iou_thr, self.K, (out.num_instances, out.scores, out.classes, out.boxes),
                     reset_counts=True)

    def step(self, x: StepInputs, out: StepOutputs, finalize: bool = True, after_train=None) -> None:
        """One pass of the hot path over one batch: both chains, concurrently, on two streams.
        ``after_train`` (optional callable) runs on the train stream right after the loss kernels — the
        multi-GPU all-reduce of ``out.sums`` + finalize go there, overlapping the inference chain."""
        main = torch.cuda.current_stream(self.device)
        self.side.wait_stream(main)
        with torch.cuda.stream(self.side):
            self.infer_chain(x, out)
        self.train_chain(x, out, finalize)
        if after_train is not None:
            after_train()
        main.wait_stream(self.side)

    def capture(self, x: StepInputs, out: StepOutputs, finalize: bool = True) -> torch.cuda.CUDAGraph:
        """Capture :meth:`step` for fixed buffers into a CUDA graph (one host launch per step)."""
        warm = torch.cuda.Stream(device=self.device)
        warm.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(warm):
            self.step(x, out, finalize)
        torch.cuda.current_stream(self.device).wait_stream(warm)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.step(x, out, finalize)
        return graph
