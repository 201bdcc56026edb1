"""Soft-NMS without a GPU: the numpy oracle (oracle/soft_nms_oracle.py) on hand-computed cases, and the host-side
argument checks of the two C entry points (sihl_od_soft_nms_topk, sihl_od_batched_soft_nms)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import soft_nms_oracle as sno
from sihl_b200 import _native, ops

f32 = np.float32
A = [0, 0, 10, 10]
B = [5, 0, 15, 10]                     # overlaps A by half its width: inter 50, union 150, IoU 1/3


def test_two_boxes_with_known_iou_both_methods():
    iou = sno.box_iou(np.array(A, f32), np.array([B], f32))[0]
    assert iou == f32(50) / f32(150) and abs(float(iou) - 1 / 3) < 1e-7
    # linear, Nt = 0.3 < 1/3: the second box keeps 1 - IoU of its score
    keep, s = sno.soft_nms([A, B], [0.9, 0.8], [0, 0], "linear", iou_thr=0.3)
    assert keep.tolist() == [0, 1]
    assert s[0] == f32(0.9) and s[1] == f32(0.8) * (f32(1) - iou)
    assert abs(float(s[1]) - 0.8 * 2 / 3) < 1e-6
    # linear, Nt = 0.5 > 1/3: no decay at all
    keep, s = sno.soft_nms([A, B], [0.9, 0.8], [0, 0], "linear", iou_thr=0.5)
    assert keep.tolist() == [0, 1] and s[1] == f32(0.8)
    # gaussian, sigma 0.5: w = exp(-(1/3)^2 / 0.5) = exp(-2/9)
    keep, s = sno.soft_nms([A, B], [0.9, 0.8], [0, 0], "gaussian", sigma=0.5)
    assert keep.tolist() == [0, 1]
    assert s[1] == f32(0.8) * f32(np.exp(-(np.float64(iou) ** 2) / 0.5))
    assert abs(float(s[1]) - 0.8 * np.exp(-2 / 9)) < 1e-6


def test_decay_can_reorder_the_output():
    """A box that overlaps the winner falls behind a weaker box that does not overlap it."""
    C = [40, 40, 50, 50]
    keep, s = sno.soft_nms([A, B, C], [0.9, 0.8, 0.6], [0, 0, 0], "linear", iou_thr=0.3)
    assert keep.tolist() == [0, 2, 1] and s.tolist() == sorted(s.tolist(), reverse=True)


def test_identical_boxes():
    # linear: IoU 1 > Nt gives weight 0, the score drops below the threshold and the box is pruned
    keep, s = sno.soft_nms([A, A], [0.9, 0.8], [3, 3], "linear", iou_thr=0.3, score_thr=0.001)
    assert keep.tolist() == [0] and s.tolist() == [f32(0.9)]
    # gaussian: weight exp(-2), the box survives with the decayed score
    keep, s = sno.soft_nms([A, A], [0.9, 0.8], [3, 3], "gaussian", sigma=0.5)
    assert keep.tolist() == [0, 1] and s[1] == f32(0.8) * f32(np.exp(-2.0))


def test_zero_area_boxes_give_no_nan():
    Z = [5, 5, 5, 5]
    for method in sno.METHODS:
        keep, s = sno.soft_nms([Z, Z, A], [0.9, 0.8, 0.7], [1, 1, 1], method, iou_thr=0.3, sigma=0.5)
        assert not np.isnan(s).any()
        assert keep.tolist() == [0, 1, 2]
        assert s.tolist() == [f32(0.9), f32(0.8), f32(0.7)]          # IoU 0 (0/0 -> 0 for the pair of empty boxes)


def test_classes_never_decay_each_other():
    for method in sno.METHODS:
        keep, s = sno.soft_nms([A, A, B], [0.9, 0.8, 0.7], [0, 1, 2], method, iou_thr=0.3, sigma=0.5)
        assert keep.tolist() == [0, 1, 2] and s.tolist() == [f32(0.9), f32(0.8), f32(0.7)]


def test_ties_threshold_and_max_out():
    # equal scores: the lower index first; a score below the threshold is never emitted; max_out stops early
    keep, s = sno.soft_nms([A, [100, 100, 110, 110], B], [0.5, 0.5, 0.0005], [0, 0, 0], "gaussian", score_thr=0.001)
    assert keep.tolist() == [0, 1]
    keep, _ = sno.soft_nms([A, [100, 100, 110, 110], B], [0.5, 0.5, 0.4], [0, 0, 0], "gaussian", max_out=1)
    assert keep.tolist() == [0]


def test_candidate_form_breaks_ties_by_location():
    """The candidate-list form orders equal scores by location (the key's low word is ~location), not list position."""
    score_bits = np.array([0.5, 0.5], f32).view(np.uint32).astype(np.uint64)
    locs = np.array([9, 4], np.uint64)
    key = (score_bits << np.uint64(32)) | (~locs & np.uint64(0xFFFFFFFF))
    box = np.array([A, [100, 100, 110, 110]], f32)
    num, sc, cl, bx = sno.soft_nms_candidates(key, box, np.array([2, 2], np.int32), "linear", 0.3, 0.5, 0.05, 3)
    assert num == 2 and bx[0].tolist() == [100, 100, 110, 110] and bx[2].tolist() == [0, 0, 0, 0] and cl.tolist() == [2, 2, 0]


def test_python_entry_points_validate_the_method():
    with pytest.raises(ValueError, match="method"):
        ops.batched_soft_nms(torch.zeros(2, 4), torch.zeros(2), torch.zeros(2, dtype=torch.int64), 10, method="hard")
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.batched_soft_nms(torch.zeros(2, 4), torch.zeros(2), torch.zeros(2, dtype=torch.int64), 10)
    with pytest.raises(ValueError, match="nms"):
        ops.dense_postprocess(torch.zeros(1, 4), torch.zeros(1, 4, 3), torch.zeros(1, 4, 4), [(2, 2)], 8, 8, nms="soft")


def test_head_postprocess_rejects_an_unknown_nms():
    from sihl_b200.heads import ObjectDetection
    model = ObjectDetection(in_channels=[3] + [8] * 5, num_classes=3, num_channels=16, num_layers=1)
    with pytest.raises(ValueError, match="nms"):
        model.postprocess([torch.zeros(1, 3, 32, 32)], nms="matrix")


def test_cabi_rejects_bad_arguments_before_touching_the_device():
    lib = _native.load()
    buf = (ctypes.c_char * 256)()
    p = ctypes.addressof(buf)
    # candidate form: cand_count, cap, key, box, cls, batch, method, iou_thr, sigma, score_thr, k, num, scores, classes,
    # boxes, workspace, reset_counts, stream
    topk = lambda **kw: lib.sihl_od_soft_nms_topk(*[kw.get(n, d) for n, d in (
        ("count", p), ("cap", 100), ("key", p), ("box", p), ("cls", p), ("batch", 2), ("method", 2), ("iou", 0.3),
        ("sigma", 0.5), ("thr", 0.05), ("k", 100), ("num", p), ("scores", p), ("classes", p), ("boxes", p), ("ws", None),
        ("reset", 0), ("stream", None))])
    assert topk(method=0) == 1 and b"method" in lib.sihl_od_last_error_string()
    assert topk(method=3) == 1
    assert topk(sigma=0.0) == 1 and b"sigma" in lib.sihl_od_last_error_string()
    assert topk(sigma=-1.0) == 1
    assert topk(sigma=float("nan")) == 1
    assert topk(method=1, sigma=0.0, k=0) == 1 and b"bad sizes" in lib.sihl_od_last_error_string()   # sigma unused by linear
    assert topk(k=0) == 1
    assert topk(cap=0) == 1 and topk(cap=1 << 30) == 1
    assert topk(batch=-1) == 1
    assert topk(key=None) == 1 and b"NULL" in lib.sihl_od_last_error_string()
    assert topk(boxes=None) == 1
    assert topk(cap=40000) == 1 and b"workspace" in lib.sihl_od_last_error_string()
    assert topk(batch=0) == 0                                              # nothing to do
    # segment form: boxes, scores, classes, seg_offsets, n_images, n, method, iou_thr, sigma, score_thr, max_out, keep,
    # keep_scores, keep_count, workspace, stream
    seg = lambda **kw: lib.sihl_od_batched_soft_nms(*[kw.get(n, d) for n, d in (
        ("boxes", p), ("scores", p), ("classes", p), ("seg", p), ("n_images", 1), ("n", 10), ("method", 1), ("iou", 0.3),
        ("sigma", 0.5), ("thr", 0.001), ("max_out", 10), ("keep", p), ("keep_scores", p), ("count", p), ("ws", None),
        ("stream", None))])
    assert seg(method=-1) == 1 and b"method" in lib.sihl_od_last_error_string()
    assert seg(method=2, sigma=0.0) == 1 and b"sigma" in lib.sihl_od_last_error_string()
    assert seg(max_out=0) == 1 and seg(n=-1) == 1 and seg(n=1 << 30) == 1 and seg(n_images=-1) == 1
    assert seg(keep_scores=None) == 1 and seg(seg=None) == 1 and seg(count=None) == 1
    assert seg(n=40000) == 1 and b"workspace" in lib.sihl_od_last_error_string()
    assert seg(n_images=0) == 0
    # workspace: none while every list fits the cluster's shared memory (8 x 4096 candidates)
    assert lib.sihl_od_soft_nms_workspace_bytes(64, 8525) == 0 and lib.sihl_od_soft_nms_workspace_bytes(8, 32768) == 0
    assert lib.sihl_od_soft_nms_workspace_bytes(2, 40000) == 2 * 40000 * 28
    assert lib.sihl_od_batched_soft_nms_workspace_bytes(30000) == 0 and lib.sihl_od_batched_soft_nms_workspace_bytes(40000) == 40000 * 28
    assert lib.sihl_od_version() == 102
