"""Box voting without a GPU: the numpy oracle (oracle/box_vote_oracle.py) against a restatement of YOLOv5's merge-NMS
formula and against torchvision's pair arithmetic, hand-computed cases and edge cases, the argument checks of the four
C entries and of the Python entries, and the footprint of the voting kernels on the built library."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from torchvision import ops as tvops

from oracle import box_vote_oracle as bvo
from oracle import od_oracle as orc
from sihl_b200 import _native, build, ops

f32 = np.float32


def _ulps(got, want):
    """Distance in fp32 units in the last place (same-sign values)."""
    g = np.asarray(got, f32).view(np.int32).astype(np.int64)
    w = np.asarray(want, f32).view(np.int32).astype(np.int64)
    return np.abs(g - w)


def _crowd(seed, n, n_classes, scale=100.0):
    rng = np.random.RandomState(seed)
    xy = rng.uniform(0, scale, (n, 2))
    wh = rng.uniform(2.0, scale / 3, (n, 2))
    boxes = np.concatenate([xy, xy + wh], 1).astype(f32)
    boxes[n // 2:] = boxes[: n - n // 2] + rng.normal(0, 2.0, (n - n // 2, 4)).astype(f32)    # near-duplicates
    boxes[:, 2:] = np.maximum(boxes[:, 2:], boxes[:, :2] + f32(0.5))
    scores = rng.uniform(0.05, 1.0, n).astype(f32)
    classes = rng.randint(0, n_classes, n).astype(np.int64)
    return boxes, scores, classes


def _yolov5_merge(boxes, scores, classes, keep, thr, kind):
    """YOLOv5's non_max_suppression(merge=True) restated in fp64 torch: class-offset boxes, an overlap > thr mask times
    the scores, one matrix product, the offset taken off again."""
    max_wh = 7680.0
    b = torch.from_numpy(boxes).double()
    off = b + torch.from_numpy(classes).double()[:, None] * max_wh
    k = torch.from_numpy(keep)
    ov = tvops.box_iou(off[k], off) if kind == "iou" else tvops.distance_box_iou(off[k], off)
    weights = (ov > float(f32(thr))).double() * torch.from_numpy(scores).double()[None]
    merged = torch.mm(weights, off) / weights.sum(1, keepdim=True)
    return (merged - torch.from_numpy(classes[keep]).double()[:, None] * max_wh).numpy().astype(f32)


@pytest.mark.parametrize("kind", bvo.OVERLAPS)
@pytest.mark.parametrize("n,n_classes,thr", [(1, 1, 0.5), (200, 1, 0.5), (400, 3, 0.45), (300, 1, 0.7), (500, 8, 0.3)])
def test_oracle_equals_yolov5_merge_formula(kind, n, n_classes, thr):
    boxes, scores, classes = _crowd(n * 13 + n_classes, n, n_classes)
    keep, voted = bvo.batched_nms_vote(boxes, scores, classes, thr, kind)
    want = _yolov5_merge(boxes, scores, classes, keep, thr, kind)
    assert _ulps(voted, want).max() <= 1
    assert not np.array_equal(voted, boxes[keep]) or n == 1                 # voting moved some boxes


def test_numpy_overlaps_equal_torchvision_bit_for_bit():
    """The oracle's fp32 IoU / DIoU is torchvision's box_iou / distance_box_iou, i.e. the kernels' operator order
    (diou_pair is checked against distance_box_iou in test_diou_nms_oracle.py)."""
    boxes, _, _ = _crowd(5, 400, 1)
    boxes[10] = [5, 5, 5, 5]                                                # zero area
    tb = torch.from_numpy(boxes)
    for kind, fn in (("iou", tvops.box_iou), ("diou", tvops.distance_box_iou)):
        want = fn(tb, tb).numpy()
        got = np.stack([bvo.overlap(kind, boxes[i], boxes) for i in range(len(boxes))])
        np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
        ok = ~np.isnan(want)
        np.testing.assert_array_equal(got[ok].view(np.uint32), want[ok].view(np.uint32))


A = [0, 0, 10, 10]
B = [2, 0, 12, 10]          # IoU with A: 80 / 120
FAR = [20, 0, 30, 10]       # disjoint from A: DIoU -400 / 1000


def test_hand_case_moves_the_kept_box_by_the_weighted_mean():
    boxes = np.array([A, B, B, [0, 0, 9, 10], [40, 40, 50, 50]], f32)
    scores = np.array([0.75, 0.25, 0.5, 0.125, 0.9], f32)
    classes = np.array([0, 0, 1, 0, 0], np.int64)                          # box 2: same place, other class
    keep, voted = bvo.batched_nms_vote(boxes, scores, classes, 0.5)
    assert keep.tolist() == [4, 0, 2]
    # cluster of box 0: itself, box 1 (IoU 0.67) and box 3 (IoU 0.9); weights 0.75, 0.25, 0.125 (sum 1.125)
    np.testing.assert_array_equal(voted[1], np.array([(0.25 * 2) / 1.125, 0, (0.75 * 10 + 0.25 * 12 + 0.125 * 9) / 1.125, 10],
                                                     f32))
    np.testing.assert_array_equal(voted[0], boxes[4])                      # alone in its cluster
    np.testing.assert_array_equal(voted[2], boxes[2])                      # the other class does not vote
    # with a threshold above IoU(A, B) only box 3 joins
    _, v = bvo.batched_nms_vote(boxes, scores, classes, 0.7)
    np.testing.assert_array_equal(v[1], np.array([0, 0, (0.75 * 10 + 0.125 * 9) / 0.875, 10], f32))


@pytest.mark.parametrize("kind", bvo.OVERLAPS)
@pytest.mark.parametrize("thr", [1.0, 1.5])
def test_threshold_of_one_or_more_leaves_boxes_unchanged(kind, thr):
    boxes, scores, classes = _crowd(3, 300, 2)
    boxes[7] = boxes[3]                                                     # a duplicate: overlap exactly 1
    classes[7] = classes[3]
    keep, voted = bvo.batched_nms_vote(boxes, scores, classes, thr, kind)
    assert len(keep) == len(boxes)
    np.testing.assert_array_equal(voted, boxes[keep])


def test_zero_area_nan_and_negative_diou_threshold():
    pt = [5, 5, 5, 5]
    boxes = np.array([pt, pt, A], f32)
    scores = np.array([0.9, 0.8, 0.7], f32)
    classes = np.zeros(3, np.int64)
    # a zero-area kept box: NaN against itself and its duplicate, IoU 0 against A -> unchanged
    for kind in bvo.OVERLAPS:
        np.testing.assert_array_equal(bvo.vote(boxes[0], 0, boxes, scores, classes, 0.5, kind), boxes[0])
    # scores that sum to zero leave the box as it is
    np.testing.assert_array_equal(bvo.vote(np.array(A, f32), 0, np.array([A], f32), np.zeros(1, f32), classes[:1], 0.5, "iou"),
                                  np.array(A, f32))
    # a negative DIoU threshold admits a disjoint box of the class (DIoU -0.4 > -0.5), not one of another class
    boxes = np.array([A, FAR, FAR], f32)
    scores = np.array([0.75, 0.25, 0.5], f32)
    classes = np.array([0, 0, 1], np.int64)
    keep, voted = bvo.batched_nms_vote(boxes, scores, classes, -0.5, "diou")
    assert keep.tolist() == [0, 2]
    np.testing.assert_array_equal(voted[0], np.array([5, 0, 15, 10], f32))
    np.testing.assert_array_equal(voted[1], boxes[2])
    _, voted = bvo.batched_nms_vote(boxes, scores, classes, -0.3, "diou")
    np.testing.assert_array_equal(voted[0], boxes[0])


def test_topk_form_on_candidate_lists():
    """topk_vote on hand-made lists: the keys give the visit order and the scores, counts beyond the capacity clip."""
    boxes, scores, classes = _crowd(11, 60, 2)
    key = (scores.view(np.uint32).astype(np.uint64) << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.arange(60, dtype=np.uint64))
    num, sc, cl, voted, plain = bvo.topk_vote(key[None], boxes[None], classes[None].astype(np.int32), [99], 0.5, 10)
    keep, want = bvo.batched_nms_vote(boxes, scores, classes, 0.5)
    assert num[0] == min(10, len(keep))
    np.testing.assert_array_equal(voted[0, :num[0]], want[:10])
    np.testing.assert_array_equal(plain[0, :num[0]], boxes[keep[:10]])
    np.testing.assert_array_equal(sc[0, :num[0]], scores[keep[:10]])
    assert orc.batched_nms(boxes, scores, classes, 0.5).tolist() == keep.tolist()


def test_python_entries_reject_bad_options_before_any_cuda_call():
    z = torch.zeros
    for nms in ("soft_linear", "soft_gaussian"):
        with pytest.raises(ValueError, match="box_voting"):
            ops.dense_postprocess(z(1, 4), z(1, 4, 3), z(1, 4, 4), [(2, 2)], 8, 8, nms=nms, box_voting=True)
    with pytest.raises(ValueError, match="overlap"):
        ops.batched_box_vote(z(2, 4), z(2), z(2, dtype=torch.int64), z(1, dtype=torch.int64), 0.5, overlap="giou")
    cand = ops.CandidateBuffers(z(1, dtype=torch.int32), z(1, 4, dtype=torch.int64), z(1, 4, 4), z(1, 4, dtype=torch.int32), 4, None)
    with pytest.raises(ValueError, match="overlap"):
        ops.box_vote_topk(cand, 1, 0.5, (z(1), z(1, 10), z(1, 10), z(1, 10, 4)), overlap="DIoU")
    with pytest.raises(RuntimeError, match="CUDA tensors only"):           # valid options get as far as the tensor checks
        ops.batched_box_vote(z(2, 4), z(2), z(2, dtype=torch.int64), z(1, dtype=torch.int64), 0.5, overlap="diou")
    from sihl_b200.heads import ObjectDetection
    model = ObjectDetection(in_channels=[3] + [8] * 5, num_classes=3, num_channels=16, num_layers=1)
    with pytest.raises(ValueError, match="box_voting"):
        model.postprocess([torch.zeros(1, 3, 32, 32)], nms="soft_gaussian", box_voting=True)


def test_cabi_argument_checks():
    """The four entries refuse NULL pointers and bad sizes on the host with the messages of their NMS counterparts, and
    accept an empty batch."""
    lib = _native.load()
    buf = (C.c_char * 256)()
    p = C.addressof(buf)
    topk = (("count", p), ("cap", 100), ("key", p), ("box", p), ("cls", p), ("batch", 2), ("thr", 0.5), ("k", 100),
            ("num", p), ("classes", p), ("boxes", p), ("stream", None))
    seg = (("boxes", p), ("scores", p), ("classes", p), ("seg", p), ("n_images", 1), ("n", 10), ("thr", 0.5),
           ("keep", p), ("count", p), ("voted", p), ("stream", None))

    def call(fn, spec, **kw):
        rc = fn(*[kw.get(n, d) for n, d in spec])
        return rc, lib.sihl_od_last_error_string() if rc else None

    for name in ("sihl_od_box_vote_topk", "sihl_od_diou_box_vote_topk"):
        fn = getattr(lib, name)
        for kw, msg in ((dict(key=None), b"NULL input"), (dict(cls=None), b"NULL input"), (dict(boxes=None), b"NULL output"),
                        (dict(num=None), b"NULL output"), (dict(k=0), b"bad sizes"), (dict(cap=0), b"bad sizes"),
                        (dict(cap=1 << 30), b"bad sizes")):
            assert call(fn, topk, **kw) == (1, msg), (name, kw)
        assert call(fn, topk, batch=0) == (0, None)
        assert call(fn, topk, batch=-3) == (0, None)
    for name in ("sihl_od_batched_box_vote", "sihl_od_batched_diou_box_vote"):
        fn = getattr(lib, name)
        for kw in (dict(seg=None), dict(count=None), dict(keep=None), dict(voted=None), dict(scores=None)):
            assert call(fn, seg, **kw) == (1, b"NULL argument"), (name, kw)
        for kw in (dict(n=-1), dict(n=1 << 30), dict(n_images=-1)):
            assert call(fn, seg, **kw) == (1, b"bad sizes"), (name, kw)
        assert call(fn, seg, n_images=0) == (0, None)
        assert call(fn, seg, n=0, keep=None, voted=None, boxes=None, scores=None, classes=None, n_images=0) == (0, None)
    # the same conditions give the same messages in the NMS entries
    assert lib.sihl_od_nms_topk(p, 100, None, p, p, 2, 0.5, 100, p, p, p, p, None, 0, None) == 1
    assert lib.sihl_od_last_error_string() == b"NULL input"
    assert lib.sihl_od_batched_nms(p, p, p, p, 1, -1, 0.5, p, p, None, None) == 1
    assert lib.sihl_od_last_error_string() == b"bad sizes"


VOTE_KERNELS = tuple(f"_ZN4sihl10k_box_voteILi{kind}ELi{layout}EEEvNS_10VoteParamsE" for kind in (0, 1) for layout in (0, 1))


def test_vote_kernels_spill_nothing():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    _native.load()
    out = subprocess.run([exe, "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage = {name: dict(REG=int(r), STACK=int(s), SHARED=int(sh), LOCAL=int(lo)) for name, r, s, sh, lo in
             re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out)}
    for name in VOTE_KERNELS:
        u = usage[name]
        assert u["STACK"] == 0 and u["LOCAL"] == 0 and u["SHARED"] == 0, (name, u)
        assert u["REG"] <= 64, (name, u)                                    # 256 threads x 64 registers: 4 CTAs per SM
