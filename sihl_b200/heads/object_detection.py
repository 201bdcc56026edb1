"""``ObjectDetection`` head — drop-in for ``sihl.heads.ObjectDetection`` with the dense,
non-learned tail running in ``libsihl_b200.so``.

Mirrors the reference class (``/root/reference/src/sihl/heads/object_detection.py``):
same constructor (:14-23), attributes, ``state_dict`` keys (``laterals.*``, ``loc_head.*``,
``cls_head.*``, ``box_head.*``, ``iou_head.*``), the ``Head`` protocol methods
(``src/sihl/heads/__init__.py:28-53``) with the same signatures, return types and error
behaviour, so ``SihlLightningModule`` (``src/sihl/lightning_module.py:95-98,145-148``),
``SihlModel`` and ``sihl.visualization`` keep working unchanged.

What stays PyTorch: the learned part (1x1 conv + BN laterals, four LayerNorm/SiLU MLPs —
dense contractions, out of scope here, SURVEY.md §2 row 2).  What moved to CUDA kernels behind
the C ABI: anchor tables (ref :83-97,:134-140), the per-image ``bbox_matching`` loop
(:143-148,:252-284), the four loss reductions and their backward (:157-210), the top-k decode
of ``forward`` (:108-121), plus the north-star extension ``postprocess`` (dense decode +
class-aware NMS; the reference has no NMS).

Differences a caller can observe, all documented in DESIGN.md:
  * tensors must live on a CUDA device (there is no CPU path);
  * ``assignment`` is canonical: -1 wherever ``rel_iou`` is not > 0 (SURVEY.md §3.4);
  * exact ties inside ``topk`` resolve to the lowest index (torch leaves them undefined);
  * ONNX export of ``forward`` is not available (custom kernels).
"""
from __future__ import annotations

from functools import partial
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor, nn
from torch.nn import functional
from torchvision import ops as tvops

from .. import ops

_TOTAL_WEIGHTS = (1.0, 10.0, 1.0, 1.0)          # loss = loc + 10*box + class + iou, ref :210


class _TrainLoss(torch.autograd.Function):
    """[location, box, class, iou, total] losses of ref :157-217 from the head outputs: one kernel launch forward
    (``sihl_od_train_loss``), one backward (``sihl_od_train_loss_bwd``, SURVEY.md §7.4), on fp32 / fp16 / bf16 maps as
    they come out of the MLPs (no fp32 copies).  The number of positives stays on the device: ``box_rows`` /
    ``cls_rows`` hold ``st.capacity`` rows of which the kernels use the first P.  ``assignment`` / ``rel_iou`` carry
    no gradient (functions of the anchors and the ground truth only)."""

    @staticmethod
    def forward(ctx, loc_logits, iou_preds, box_rows, cls_rows, st, reduce_sums):
        if reduce_sums is None:
            losses, maps = ops.train_loss(st, loc_logits, iou_preds, box_rows, cls_rows, finalize=True)
        else:                                   # global-batch normalisers: sums cross the ranks before the division
            _, maps = ops.train_loss(st, loc_logits, iou_preds, box_rows, cls_rows, finalize=False)
            reduce_sums(st.sums)
            losses = ops.loss_finalize(st.sums)
        ctx.st, ctx.maps = st, maps
        return losses

    @staticmethod
    def backward(ctx, grad_out):
        grads = ops.train_loss_bwd(ctx.st, ctx.maps, grad_out.float().contiguous() if grad_out.dtype != torch.float32
                                   or not grad_out.is_contiguous() else grad_out, ctx.needs_input_grad[:4])
        return grads[0], grads[1], grads[2], grads[3], None, None


def _cat_gt(boxes: List[Tensor], classes: Optional[List[Tensor]], device):
    """ref :127-128 — per-image lists (possibly empty, possibly ``tv_tensors`` subclasses) -> one [sumG,4] fp32 and one
    [sumG] int64 tensor on ``device`` + the host list of counts (from shapes: no sync)."""
    counts = [int(b.shape[0]) for b in boxes]
    plain = [b if type(b) is Tensor else b.as_subclass(Tensor) for b in boxes]
    plain = [b if b.dim() == 2 else b.reshape(-1, 4) for b in plain]
    cat = torch.cat(plain) if plain else torch.empty((0, 4))
    if cat.dtype != torch.float32 or cat.device != device:
        cat = cat.to(device=device, dtype=torch.float32)
    cls = None
    if classes is not None:
        plain_c = [c if type(c) is Tensor else c.as_subclass(Tensor) for c in classes]
        cls = torch.cat([c.reshape(-1) for c in plain_c]) if plain_c else torch.empty((0,), dtype=torch.int64)
        if cls.dtype != torch.int64 or cls.device != device:
            cls = cls.to(device=device, dtype=torch.int64)
        if cls.numel() != cat.shape[0]:
            raise ValueError("classes and boxes disagree on the number of objects")
    return cat.contiguous(), cls, counts


class ObjectDetection(nn.Module):
    def __init__(
        self,
        in_channels: List[int],
        num_classes: int,
        bottom_level: int = 3,
        top_level: int = 5,
        num_channels: int = 256,
        num_layers: int = 4,
        max_instances: int = 100,
    ) -> None:
        """Same arguments and checks as the reference constructor (ref :14-39)."""
        assert num_classes > 0, num_classes
        assert len(in_channels) > top_level, (len(in_channels), top_level)
        assert 0 < bottom_level <= top_level, (bottom_level, top_level)
        assert num_channels % 4 == 0, num_channels
        assert num_layers >= 0, num_layers
        assert max_instances > 0, max_instances
        super().__init__()

        self.in_channels = in_channels
        self.num_classes = num_classes
        self.bottom_level, self.top_level = bottom_level, top_level
        self.levels = range(bottom_level, top_level + 1)
        self.num_channels = num_channels
        self.num_layers = num_layers
        self.max_instances = max_instances
        self.topk = 9

        # learned part: identical modules => identical state_dict keys and initialisation (ref :51-61)
        mlp = partial(tvops.MLP, norm_layer=nn.LayerNorm, activation_layer=nn.SiLU)
        conv = partial(tvops.Conv2dNormActivation, activation_layer=None)
        self.laterals = nn.ModuleList([conv(in_channels[level], num_channels, 1) for level in self.levels])
        hidden = [num_channels] * num_layers
        self.loc_head = mlp(num_channels, hidden + [1])
        self.loc_head[-2].bias.data.fill_(-5.0)
        self.cls_head = mlp(num_channels, hidden + [num_classes])
        self.box_head = mlp(num_channels, hidden + [4])
        self.iou_head = mlp(num_channels, hidden + [1])

        self.output_shapes = {
            "num_instances": ("batch_size",),
            "scores": ("batch_size", max_instances),
            "classes": ("batch_size", max_instances),
            "boxes": ("batch_size", max_instances, 4),
        }
        # "local": normalise by this process's batch (what the reference does, also under DDP);
        # "global": all-reduce the 8 partial sums first: the losses equal one process over the global batch, the
        #   early-out of ref :165-172 is decided on the GLOBAL number of positives (every rank runs every head, so DDP
        #   sees gradients for every parameter on every rank), and the backward is scaled by the world size so that
        #   DDP's gradient *average* over the ranks equals the gradient of the global-batch loss.
        self.loss_reduction = "local"
        self.process_group = None
        # "torch": the towers run as the torchvision modules above (fp32 or autocast), in training and inference.
        # "tcgen05" (SURVEY.md §8f N4): wherever no gradient is being recorded (forward / postprocess / get_saliency under
        #   no_grad, i.e. validation and serving) the towers run through ``sihl_od_mlp_hidden`` / ``sihl_od_mlp_out`` —
        #   bf16 operands on the tensor cores, fp32 accumulation and LayerNorm, Linear + LayerNorm + SiLU in one kernel.
        #   Needs num_channels == 256; training steps keep the torch modules.
        # "tcgen05+train": additionally the towers of ``training_step`` run in bf16 mixed precision (what Lightning's
        #   precision="bf16-mixed" gives the torch towers): forward on the tensor cores, recomputing backward
        #   (``mlp_tower._HiddenLayerFn``); parameter gradients and LayerNorm statistics stay fp32.
        self.mlp_backend = "torch"
        self._packed_towers: Dict[str, object] = {}

    # ------------------------------------------------------------------ helpers
    def _level_sizes(self, inputs: List[Tensor]) -> List[Tuple[int, int]]:
        return [tuple(int(v) for v in inputs[level].shape[2:]) for level in self.levels]

    def _use_tcgen05(self, x: Tensor) -> bool:
        if self.mlp_backend == "torch":
            return False
        if self.mlp_backend not in ("tcgen05", "tcgen05+train"):
            raise ValueError(f"mlp_backend must be 'torch', 'tcgen05' or 'tcgen05+train', got {self.mlp_backend!r}")
        return x.is_cuda and not torch.is_grad_enabled() and not torch.compiler.is_compiling()

    def _use_tcgen05_training(self, x: Tensor) -> bool:
        return (self.mlp_backend == "tcgen05+train" and x.is_cuda and torch.is_grad_enabled() and x.shape[0] > 0
                and not torch.compiler.is_compiling())

    def _tower(self, name: str, x: Tensor) -> Tensor:
        """One of the four per-location MLPs (ref :108, :116, :121, :175) on ``x`` [..., C]."""
        mlp = getattr(self, name)
        if self._use_tcgen05_training(x):
            from ..mlp_tower import PackedTower, run_tower_train
            if not PackedTower.supported(mlp):
                raise ValueError(f"mlp_backend='tcgen05+train' needs num_channels == 256 and the reference's tower structure ({name})")
            return run_tower_train(mlp, x)
        if not self._use_tcgen05(x):
            return mlp(x)
        from ..mlp_tower import PackedTower, run_tower
        packed = self._packed_towers.get(name)
        if packed is None or packed.mlp is not mlp:
            if not PackedTower.supported(mlp):
                raise ValueError(f"mlp_backend='tcgen05' needs num_channels == 256 and the reference's tower structure ({name})")
            packed = self._packed_towers[name] = PackedTower(mlp)
        return run_tower(packed, x)

    def _tower_input(self, flat_feats: Tensor) -> Tensor:
        """The towers' common input: converted to bf16 ONCE when they run on the tensor cores."""
        return flat_feats.to(torch.bfloat16) if self._use_tcgen05(flat_feats) else flat_feats

    def _folded_laterals(self):
        """Per level (W', b') with the BatchNorm of ``Conv2dNormActivation`` folded into the 1x1 conv (eval semantics:
        running statistics), W' bf16 [256, C_in], b' fp32; re-folded when a parameter or buffer changes.  None when the
        laterals cannot run on the tensor-core path (training-mode BatchNorm, other widths, a conv with bias / stride)."""
        if self.training or self.num_channels != ops.MLP_CHANNELS:
            return None
        tensors = []
        for lateral in self.laterals:
            conv, bn = lateral[0], lateral[1]
            if not (isinstance(conv, nn.Conv2d) and isinstance(bn, nn.BatchNorm2d) and len(lateral) == 2 and conv.bias is None
                    and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.in_channels == ops.MLP_CHANNELS
                    and bn.track_running_stats and bn.affine and conv.groups == 1):
                return None
            tensors += [conv.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var]
        key = tuple((t.data_ptr(), t._version, t.device) for t in tensors)
        if getattr(self, "_folded_key", None) != key:
            with torch.no_grad():
                folded = []
                for lateral in self.laterals:
                    conv, bn = lateral[0], lateral[1]
                    scale = bn.weight.float() / torch.sqrt(bn.running_var.float() + bn.eps)
                    w = (conv.weight.float()[:, :, 0, 0] * scale[:, None]).to(torch.bfloat16).contiguous()
                    b = (bn.bias.float() - bn.running_mean.float() * scale).contiguous()
                    folded.append((w, b))
            self._folded, self._folded_key = folded, key
        return self._folded

    def _flat_feats_tensor_cores(self, inputs: List[Tensor]) -> Optional[Tensor]:
        """ref :102-105 for the tcgen05 backend: every level's lateral as one GEMM writing bf16 straight into its slice of
        the concatenated [B, A, 256] features (no fp32 feature maps, no cat, no cast pass).  None if not applicable."""
        folded = self._folded_laterals()
        if folded is None or any(inputs[level].dtype != torch.float32 for level in self.levels):
            return None
        sizes = self._level_sizes(inputs)
        batch, device = inputs[self.bottom_level].shape[0], inputs[self.bottom_level].device
        flat = torch.empty((batch, sum(h * w for h, w in sizes), ops.MLP_CHANNELS), dtype=torch.bfloat16, device=device)
        offset = 0
        for level, (h, w), (wt, bias) in zip(self.levels, sizes, folded):
            rows = ops.lateral_rows(inputs[level].contiguous())
            ops.lateral_linear(rows, wt, bias, h * w, flat, offset)
            offset += h * w
        return flat

    def _flat_feats_training(self, inputs: List[Tensor]) -> Tensor:
        """ref :151-154 inside ``training_step``.  Backend "tcgen05+train": one bf16 [B, A, 256] tensor feeds all four
        towers (their input gradients are accumulated in bf16); when the laterals have the reference's structure at 256
        channels and are in training mode, they run on the tensor-core path too (``mlp_tower._LateralsTrainFn``: batch
        statistics from the input's moments, conv + BatchNorm as one folded GEMM per level) and the modules' running
        statistics are updated here exactly as ``nn.BatchNorm2d`` does."""
        probe = inputs[self.bottom_level]
        if not self._use_tcgen05_training(probe):
            return self._flat_feats(inputs)
        from ..mlp_tower import _LateralsTrainFn, _ToBf16Fn
        fusable = self.training and self.num_channels == ops.MLP_CHANNELS and all(
            isinstance(lat[0], nn.Conv2d) and isinstance(lat[1], nn.BatchNorm2d) and len(lat) == 2 and lat[0].bias is None
            and lat[0].kernel_size == (1, 1) and lat[0].stride == (1, 1) and lat[0].groups == 1
            and lat[0].in_channels == ops.MLP_CHANNELS and lat[1].affine and lat[1].track_running_stats
            and lat[1].momentum is not None and inputs[level].dtype == torch.float32
            for lat, level in zip(self.laterals, self.levels))
        if not fusable:
            return _ToBf16Fn.apply(self._flat_feats(inputs))
        args = []
        for lat, level in zip(self.laterals, self.levels):
            args += [inputs[level], lat[0].weight, lat[1].weight, lat[1].bias]
        out = _LateralsTrainFn.apply(tuple(float(lat[1].eps) for lat in self.laterals), *args)
        with torch.no_grad():
            for i, (lat, level) in enumerate(zip(self.laterals, self.levels)):
                bn, mean, var = lat[1], out[1 + 2 * i], out[2 + 2 * i]
                count = inputs[level].shape[0] * inputs[level].shape[2] * inputs[level].shape[3]
                bn.running_mean.mul_(1 - bn.momentum).add_(mean.to(bn.running_mean.dtype), alpha=bn.momentum)
                bn.running_var.mul_(1 - bn.momentum).add_((var * (count / max(count - 1, 1))).to(bn.running_var.dtype), alpha=bn.momentum)
                bn.num_batches_tracked += 1
        return out[0]

    def _tower_feats(self, inputs: List[Tensor]) -> Tensor:
        """The towers' common input [B, A, C] (ref :102-105), bf16 when they run on the tensor cores."""
        if self._use_tcgen05(inputs[self.bottom_level]):
            flat = self._flat_feats_tensor_cores(inputs)
            if flat is not None:
                return flat
        return self._tower_input(self._flat_feats(inputs))

    def _flat_feats(self, inputs: List[Tensor]) -> Tensor:
        feats = [lateral(inputs[level]) for level, lateral in zip(self.levels, self.laterals)]     # ref :102-105
        return torch.cat([x.flatten(2).transpose(1, 2) for x in feats], 1)

    def get_offsets_and_scales(self, inputs: List[Tensor]) -> Tuple[Tensor, Tensor]:
        """ref :83-97 — one cached kernel launch instead of ~40 ATen launches per call."""
        device = inputs[0].device
        height, width = inputs[0].shape[2:]
        offsets, scales, _ = ops.anchor_tables(self._level_sizes(inputs), int(width), int(height), device)
        return offsets.clone(), scales.clone()      # the cached tables stay private: callers may edit what they get

    def get_saliency(self, inputs: List[Tensor]) -> Tensor:
        """ref :70-81 (visualisation only; learned part, stays PyTorch)."""
        device = inputs[self.bottom_level].device
        batch_size, _, full_height, full_width = inputs[self.bottom_level].shape
        output = torch.zeros((batch_size, full_height, full_width), device=device)
        for lateral, level in zip(self.laterals, self.levels):
            height, width = inputs[level].shape[2:]
            feats = lateral(inputs[level]).flatten(2).transpose(1, 2)
            scores = self._tower("loc_head", feats).sigmoid().transpose(1, 2).reshape(batch_size, 1, height, width)
            scores = functional.interpolate(scores, size=(full_height, full_width))
            output = torch.maximum(output, scores.squeeze(1))
        return output

    # ------------------------------------------------------------------ inference
    def forward(self, inputs: List[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        """ref :99-122 -> (num_instances i64 [B], scores [B,K], classes i64 [B,K], boxes [B,K,4] px).

        The MLP outputs go to the kernels in the dtype they have (fp32, or fp16 / bf16 under autocast: upcast in
        registers, no fp32 copies); ``scores`` come back in the dtype of the location logits like the reference's
        ``loc_logits.sigmoid()``.  Traceable: under ``torch.compile`` the same kernels run as ``sihl_b200::*`` custom ops
        (``sihl_b200/torch_ops.py``) with fake implementations."""
        (batch_size, _, height, width), device = inputs[0].shape, inputs[0].device
        flat_feats = self._tower_feats(inputs)
        levels = self._level_sizes(inputs)
        loc_logits = self._tower("loc_head", flat_feats).squeeze(2)                         # ref :108
        compiling = torch.compiler.is_compiling()
        if compiling:
            from .. import torch_ops
            level_hw = torch_ops.flat_levels(levels)
            top_logits, loc_idxs = torch_ops.topk_locations(loc_logits.detach(), self.max_instances)
        else:
            top_logits, loc_idxs = ops.topk_locations(loc_logits.detach(), self.max_instances)   # ref :109
        rows = torch.arange(batch_size, device=device).view(batch_size, 1)
        top_feats = flat_feats[rows, loc_idxs]                                              # ref :112
        class_logits = self._tower("cls_head", top_feats)                                   # ref :116
        box_raw = self._tower("box_head", top_feats)                                        # ref :121
        if compiling:
            num, scores, classes, boxes = torch_ops.decode_rows(top_logits, loc_idxs, class_logits.detach(), box_raw.detach(),
                                                                level_hw, int(width), int(height))
        else:
            offsets, scales, _ = ops.anchor_tables(levels, int(width), int(height), device)
            num, scores, classes, boxes = ops.decode_rows(top_logits, loc_idxs, class_logits.detach(), box_raw.detach(),
                                                          offsets, scales, int(width), int(height))
        if loc_logits.dtype != torch.float32:
            scores = scores.to(loc_logits.dtype)
        return num, scores, classes, boxes

    @torch.no_grad()
    def postprocess(self, inputs: List[Tensor], score_threshold: float = 0.05, iou_threshold: float = 0.5,
                    mode: Optional[str] = None, nms: str = "hard", sigma: float = 0.5,
                    box_voting: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
        """North-star extension (the reference has no NMS): every location is decoded with the
        score/class semantics of ``forward`` (score = sigmoid(location logit), class = argmax),
        thresholded, and de-duplicated by class-aware NMS; same output format as ``forward``.

        ``mode``: ``"dense"`` streams the whole class map (TMA ring), ``"candidate_first"`` reads the class row and raw
        box of the locations that pass the threshold only — identical results; default: ``"dense"`` for fp32 maps,
        ``"candidate_first"`` for half maps (autocast), which are then read as they are (no fp32 copies).

        ``nms``: ``"hard"`` (greedy NMS), ``"diou"`` (greedy DIoU-NMS, ``iou_threshold`` is the DIoU threshold: a box
        survives an overlapping box of its class when their centres lie far enough apart), ``"soft_linear"`` (Soft-NMS,
        ``iou_threshold`` is Nt) or ``"soft_gaussian"`` (Soft-NMS with ``sigma``): overlapping boxes of a class have
        their scores decayed instead of being dropped, which keeps real objects in crowds; the returned scores are the
        decayed ones.

        ``box_voting`` (with ``"hard"`` or ``"diou"``): box voting / merge-NMS (YOLOv5's ``merge=True``): every kept box
        becomes the score-weighted mean of the boxes of its class that its suppression test claims; the detections,
        scores and classes are those of the call without it."""
        if nms not in ops.NMS_KINDS:
            raise ValueError(f"nms={nms!r}: expected one of {ops.NMS_KINDS}")
        if box_voting and nms.startswith("soft_"):
            raise ValueError(f"box_voting=True needs nms='hard' or 'diou', not {nms!r}")
        (_, _, height, width) = inputs[0].shape
        flat_feats = self._tower_feats(inputs)
        loc_logits = self._tower("loc_head", flat_feats).squeeze(2)
        cls_logits = self._tower("cls_head", flat_feats)
        box_raw = self._tower("box_head", flat_feats)
        if mode is None:
            mode = "dense" if loc_logits.dtype == torch.float32 else "candidate_first"
        return ops.dense_postprocess(loc_logits, cls_logits, box_raw, self._level_sizes(inputs), int(width), int(height),
                                     score_threshold, iou_threshold, self.max_instances, mode=mode, nms=nms, sigma=sigma,
                                     box_voting=box_voting)

    # ------------------------------------------------------------------ training
    def _reduce_sums(self) -> Optional[callable]:
        if self.loss_reduction != "global":
            return None
        from .. import dist
        return partial(dist.all_reduce_sums, group=self.process_group)

    def _world_size(self) -> int:
        import torch.distributed as tdist
        return tdist.get_world_size(self.process_group) if (tdist.is_available() and tdist.is_initialized()) else 1

    def training_step(
        self,
        inputs: List[Tensor],
        classes: List[Tensor],
        boxes: List[Tensor],
        is_validating: bool = False,
    ) -> Tuple[Tensor, Dict[str, float]]:
        """ref :124-217 -> (loss, {"location_loss", "box_loss", "class_loss", "iou_loss"}).

        Three C calls and no host synchronisation (the reference syncs ~7x per image): ``sihl_od_train_assign`` before
        the MLPs, ``sihl_od_train_loss`` after them, ``sihl_od_train_loss_bwd`` in backward.  The number of positives P
        stays on the device, so ``box_head`` / ``cls_head`` run on a static ``min(9 * sumG, B * A)`` rows
        (``flat_feats[o2m_mask]`` followed by repeats of row 0 whose gradient is zero) and the early-out of ref :165-172
        is taken inside the kernels: with no positive in the batch the loss is the location loss alone and the other
        three heads receive zero gradients (the reference leaves them without any)."""
        assert len(inputs) > self.top_level, "too few input levels"
        device = inputs[0].device
        batch_size, _, full_height, full_width = inputs[0].shape
        levels = self._level_sizes(inputs)
        width, height = int(full_width), int(full_height)

        # anchors + assignment: functions of shapes and gt only (ref :139-148) -> before the MLPs
        gt_boxes, gt_classes, counts = _cat_gt(boxes, classes, device)
        assert len(counts) == batch_size, (len(counts), batch_size)
        if torch.compiler.is_compiling():
            return self._training_step_traced(inputs, levels, width, height, gt_boxes, gt_classes, counts)
        st = ops.train_assign(levels, width, height, gt_boxes, gt_classes, counts, batch_size, self.topk)
        reduce_sums = self._reduce_sums()
        if reduce_sums is not None:
            st.grad_scale = float(self._world_size())      # DDP averages the gradients of W ranks (see loss_reduction)

        flat_feats = self._flat_feats_training(inputs)                                      # ref :151-154
        if self._use_tcgen05_training(flat_feats) and flat_feats.requires_grad:
            # one autograd node for the three consumers of the features: its backward is one add + one in-place index_add
            from ..mlp_tower import _FanOutFn
            loc_in, iou_in, o2m_feats = _FanOutFn.apply(flat_feats.reshape(batch_size * st.A, -1), st.pos_index)
            loc_logits = self._tower("loc_head", loc_in).reshape(batch_size, st.A)          # ref :157
            iou_preds = self._tower("iou_head", iou_in).reshape(batch_size, st.A)           # ref :175
        else:
            loc_logits = self._tower("loc_head", flat_feats).squeeze(2)                     # ref :157
            iou_preds = self._tower("iou_head", flat_feats).squeeze(2)                      # ref :175
            o2m_feats = flat_feats.reshape(batch_size * st.A, -1).index_select(0, st.pos_index)  # ref :184 (+ padding rows)
        box_raw = self._tower("box_head", o2m_feats)                                        # ref :189
        class_logits = self._tower("cls_head", o2m_feats)                                   # ref :200
        out = _TrainLoss.apply(loc_logits, iou_preds, box_raw, class_logits, st, reduce_sums)
        self.last_assignment, self.last_rel_iou, self.last_train_state = st.assignment, st.rel_iou, st
        metrics = {"location_loss": out[0], "box_loss": out[1], "class_loss": out[2], "iou_loss": out[3]}
        return out[4], metrics

    def _training_step_traced(self, inputs, levels, width, height, gt_boxes, gt_classes, counts):
        """The same step through the ``sihl_b200::*`` custom ops (fake implementations + registered autograd): what
        ``torch.compile`` / ``torch.export`` trace.  ``loss_reduction="global"`` is an eager-only feature."""
        from .. import torch_ops
        assert self.loss_reduction == "local", "loss_reduction='global' is not traceable; call the eager module"
        batch_size, device = len(counts), gt_boxes.device
        level_hw = torch_ops.flat_levels(levels)
        num_anchors = sum(h * w for h, w in levels)
        prefix = [0]
        for c in counts:
            prefix.append(prefix[-1] + c)
        gt_offsets = torch.tensor(prefix, dtype=torch.int32, device=device)
        capacity = max(1, min(self.topk * prefix[-1], batch_size * num_anchors))
        assignment, rel_iou, pos_index, meta = torch_ops.train_assign(gt_boxes, gt_offsets, level_hw, width, height,
                                                                      self.topk, capacity)
        flat_feats = self._flat_feats(inputs)
        loc_logits = self.loc_head(flat_feats).squeeze(2)
        iou_preds = self.iou_head(flat_feats).squeeze(2)
        o2m_feats = flat_feats.reshape(batch_size * num_anchors, -1).index_select(0, pos_index)
        box_raw = self.box_head(o2m_feats)
        class_logits = self.cls_head(o2m_feats)
        out, _ = torch_ops.train_loss(loc_logits, iou_preds, box_raw, class_logits, assignment, rel_iou, pos_index, meta,
                                      gt_boxes, gt_classes, level_hw, width, height)
        metrics = {"location_loss": out[0], "box_loss": out[1], "class_loss": out[2], "iou_loss": out[3]}
        return out[4], metrics

    training_loss = training_step          # north-star name for the same entry point

    # ------------------------------------------------------------------ validation
    def on_validation_start(self) -> None:
        """ref :219-225.  ``self.map_backend``: "auto" (default) uses torchmetrics' MeanAveragePrecision exactly like the
        reference when torchmetrics is importable and the GPU matcher ``sihl_b200.metrics.DetectionMAP`` (SURVEY.md §8f
        N3: COCO matching per batch on the GPU, same metric keys) otherwise; "gpu" always uses the GPU matcher."""
        thresholds = [1, min(self.max_instances, 10), self.max_instances]
        use_tm = getattr(self, "map_backend", "auto") != "gpu"
        if use_tm:
            try:
                from torchmetrics import MeanMetric
                from torchmetrics.detection.mean_ap import MeanAveragePrecision
                self.loss_computer = MeanMetric(nan_strategy="ignore")
                self.map_computer = MeanAveragePrecision(max_detection_thresholds=thresholds, backend="faster_coco_eval")
                return
            except Exception:
                pass
        from ..metrics import DetectionMAP
        self.loss_computer = _RunningMean()
        self.map_computer = DetectionMAP(max_detection_thresholds=thresholds)

    def validation_step(self, inputs: List[Tensor], classes: List[Tensor], boxes: List[Tensor]
                        ) -> Tuple[Tensor, Dict[str, float]]:
        """ref :227-240."""
        from ..metrics import DetectionMAP
        num_instances, scores, pred_classes, pred_boxes = self.forward(inputs)
        if isinstance(getattr(self, "map_computer", None), DetectionMAP):
            gt_boxes, gt_classes, counts = _cat_gt(boxes, classes, scores.device)
            self.map_computer.update_batch(scores, pred_classes, pred_boxes, gt_boxes, gt_classes, counts)   # one kernel, no sync
        elif hasattr(self, "map_computer"):
            self.map_computer.to(scores.device).update(
                [{"scores": s, "labels": c, "boxes": b} for s, c, b in zip(scores, pred_classes, pred_boxes)],
                [{"labels": c, "boxes": b} for c, b in zip(classes, boxes)],
            )
        loss, metrics = self.training_step(inputs, classes, boxes, is_validating=True)
        self.loss_computer.to(loss.device).update(loss)
        return loss, metrics

    def on_validation_end(self) -> Dict[str, float]:
        """ref :242-250."""
        metrics = {}
        if hasattr(self, "map_computer"):
            metrics = self.map_computer.compute()
            for key in list(metrics.keys()):
                if "per_class" in key or key in {"classes", "ious"}:
                    del metrics[key]
        metrics["loss"] = self.loss_computer.compute()
        return metrics

    # ------------------------------------------------------------------ assigner (also used by sibling heads)
    @staticmethod
    def bbox_matching(anchors: Tensor, gt_boxes: Tensor, topk: int, relative: bool = False) -> Tuple[Tensor, Tensor]:
        """ref :252-284 — ``(assignment i64 [A], iou f32 [A])`` for one image, arbitrary anchors
        (``InstanceSegmentation`` / ``KeypointDetection`` call this verbatim)."""
        return ops.bbox_matching(anchors, gt_boxes, topk, relative)


class _RunningMean:
    """Stand-in for ``torchmetrics.MeanMetric(nan_strategy="ignore")`` when torchmetrics is absent."""

    def __init__(self) -> None:
        self.total, self.count = 0.0, 0

    def to(self, device):
        return self

    def update(self, value: Tensor) -> None:
        v = float(value.detach()) if hasattr(value, "detach") else float(value)
        if v == v:                       # ignore NaN
            self.total, self.count = self.total + v, self.count + 1

    def compute(self) -> Tensor:
        return torch.tensor(self.total / self.count if self.count else float("nan"))
