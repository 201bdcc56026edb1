"""Half-precision head outputs through the steady-state pipeline (SURVEY.md §5 "accept fp16/bf16 logits and upcast on
load"): the maps are read as they are — TMA ring with 2-byte elements for the dense scan, 16-byte row loads for the
positive-row losses — and the results follow what the reference's operators compute on half tensors under autocast
(``.sigmoid()`` / ``.exp()`` in the map dtype, BCE with the half log-sigmoid, everything else after an upcast)."""
import numpy as np
import pytest
import torch
from torch.nn import functional as F

from oracle import torch_restatement as tr
from sihl_b200 import ops, synth
from sihl_b200.pipeline import DetectionHeadPipeline, StepInputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _expected_detections(levels, W, H, loc, box, cls, thr, iou_thr, K):
    """The reference's operator sequence on HALF maps (ref :113-121 semantics over all locations + per-class NMS)."""
    offsets, scales = tr.offsets_and_scales(levels, DEV)
    size = tr.full_size(W, H, DEV)
    out = []
    for b in range(loc.shape[0]):
        s = loc[b].sigmoid()                                           # half
        cand = (s > thr).nonzero().squeeze(1)
        cb = (offsets[cand] + scales[cand] * box[b, cand].exp()) * size    # half exp, fp32 product
        cc = cls[b, cand].max(dim=1).indices
        sf = s[cand].float()
        keep = tr.nms_per_class(cb, sf, cc, iou_thr)[:K]
        out.append((sf[keep], cc[keep], cb[keep]))
    return out


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("mode", ops.DECODE_MODES)
@pytest.mark.parametrize("size,B,C", [(256, 3, 16), (640, 40, 16)])          # 32-row ring / 64-row ring of the dense scan
def test_pipeline_on_half_maps(dtype, mode, size, B, C):
    G, K = 12, 50
    levels = synth.level_sizes(size, size)
    gt = synth.gt_batch_np(31, B, size, size, C, G, ragged=False)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(32, B, A, C, loc_mean=-3.0, loc_std=1.5)
    loc, iou, box, cls = (_t(m).to(dtype) for m in (maps.loc_logits, maps.iou_preds, maps.box_raw, maps.cls_logits))
    gtb = ops.GtBatch(_t(gt.boxes), _t(gt.classes), _t(gt.offsets), [G] * B)
    pipe = DetectionHeadPipeline(levels, size, size, B, C, B * G, DEV, max_instances=K, decode_mode=mode)
    out = pipe.new_outputs()
    pipe.step(StepInputs(loc, iou, box, cls, gtb), out)
    # the same pipeline on the upcast maps: assignment is prediction independent; box / class / iou losses see the same
    # fp32 values (half -> fp32 is exact)
    ref = DetectionHeadPipeline(levels, size, size, B, C, B * G, DEV, max_instances=K, decode_mode=mode)
    r_out = ref.new_outputs()
    ref.step(StepInputs(loc.float(), iou.float(), box.float(), cls.float(), gtb), r_out)
    torch.cuda.synchronize()
    assert torch.equal(out.assignment, r_out.assignment) and torch.equal(out.rel_iou, r_out.rel_iou)
    torch.testing.assert_close(out.losses[1:4], r_out.losses[1:4], rtol=2e-5, atol=1e-7)
    # location loss: ATen's BCE-with-logits on the HALF logits (ref :160-161)
    target = (out.rel_iou == 1.0).float()
    want_loc = F.binary_cross_entropy_with_logits(loc, target, reduction="none").sum() / target.sum()
    assert out.losses[0].item() == pytest.approx(want_loc.item(), rel=1e-5)
    assert out.losses[4].item() == pytest.approx((out.losses[0] + 10 * out.losses[1] + out.losses[2] + out.losses[3]).item(), rel=1e-6)
    # detections: the reference's half semantics
    want = _expected_detections(levels, size, size, loc, box, cls, 0.05, 0.5, K)
    assert int(out.num_instances.sum()) > 0
    for b, (ws, wc, wb) in enumerate(want):
        n = int(out.num_instances[b])
        assert n == ws.numel(), b
        assert torch.equal(out.scores[b, :n], ws) and torch.equal(out.classes[b, :n], wc)
        torch.testing.assert_close(out.boxes[b, :n], wb, rtol=1e-6, atol=1e-4)


def _dense_and_candidate_first_lists_agree(dtype, C):
    size, B = 320, 4
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(5, B, A, C, loc_mean=-3.0, loc_std=2.0)
    loc, box, cls = (_t(m).to(dtype) for m in (maps.loc_logits, maps.box_raw, maps.cls_logits))
    res = [ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, 100, mode=m) for m in ops.DECODE_MODES]
    for a, b in zip(*res):
        assert torch.equal(a, b)
    assert int(res[0][0].sum()) > 0


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_dense_and_candidate_first_lists_agree_on_half_maps(dtype):
    _dense_and_candidate_first_lists_agree(dtype, 80)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_dense_scan_of_half_rows_not_a_multiple_of_its_vectors_per_lane(dtype):
    """C = 160: rows of 20 16-byte vectors, 5 per lane; the scan takes its 8-vector kernel, which must stop at the row end."""
    _dense_and_candidate_first_lists_agree(dtype, 160)
