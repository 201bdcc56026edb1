"""DIoU-NMS without a GPU: the DIoU arithmetic every DIoU kernel calls (od_math.h diou_pair, compiled for the host)
against torchvision, the C oracle (oracle/diou_nms_oracle.c) against a plain greedy loop over
torchvision.ops.distance_box_iou, hand-computed cases, the argument checks of the Python and C entries, and the
footprint of the DIoU kernels on the built library."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from torchvision import ops as tvops

from oracle import diou_nms_oracle as dno
from oracle import od_oracle as orc
from sihl_b200 import _native, build, ops

HERE = os.path.dirname(os.path.abspath(__file__))
f32 = np.float32


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = tmp_path_factory.mktemp("diou_shim") / "libdiou_shim.so"
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                           os.path.join(HERE, "host_diou_shim.cpp"), "-o", str(out)])
    return C.CDLL(str(out))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _diou_matrix(shim, a, b):
    a, b = np.ascontiguousarray(a, f32), np.ascontiguousarray(b, f32)
    out = np.empty((len(a), len(b)), f32)
    shim.shim_diou_matrix(_ptr(a), len(a), _ptr(b), len(b), _ptr(out))
    return out


def _assert_bits_equal(got, want):
    got, want = np.asarray(got, f32), np.asarray(want, f32)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _random_boxes(rng, n, scale=100.0):
    xy = rng.uniform(0, scale, (n, 2))
    wh = rng.uniform(0.5, scale / 3, (n, 2))
    return np.concatenate([xy, xy + wh], 1).astype(f32)


def _pair_cases(rng):
    """Random, identical, nested, disjoint, edge-touching and zero-area pairs (a [n,4], b [n,4])."""
    a = _random_boxes(rng, 3000)
    b = _random_boxes(rng, 3000)
    near = a + rng.normal(0, 2.0, a.shape).astype(f32)                 # near-duplicates
    near[:, 2:] = np.maximum(near[:, 2:], near[:, :2])
    inner = a.copy()
    inner[:, :2] += (a[:, 2:] - a[:, :2]) * f32(0.25)
    inner[:, 2:] -= (a[:, 2:] - a[:, :2]) * f32(0.3)                  # nested inside a
    far = a + f32(500.0)                                               # disjoint
    touch = a.copy()
    touch[:, 0], touch[:, 2] = a[:, 2], a[:, 2] + (a[:, 2] - a[:, 0])   # shares the right edge of a
    pt = np.concatenate([a[:, :2], a[:, :2]], 1)                      # zero area (a point), inside or on a
    line = a.copy()
    line[:, 3] = line[:, 1]                                            # zero area (a segment)
    left = np.concatenate([a, a, a, a, a, a, a, pt, pt, line])
    right = np.concatenate([b, a, near, inner, far, touch, pt, a, pt, line])
    return left, right


def test_diou_pair_equals_torchvision_bit_for_bit_and_is_symmetric(shim):
    a, b = _pair_cases(np.random.RandomState(0))
    ta, tb = torch.from_numpy(a), torch.from_numpy(b)
    want = np.concatenate([np.diagonal(tvops.distance_box_iou(ta[s:s + 500], tb[s:s + 500]).numpy())
                           for s in range(0, len(a), 500)])
    got = np.concatenate([np.diagonal(_diou_matrix(shim, a[s:s + 500], b[s:s + 500])) for s in range(0, len(a), 500)])
    _assert_bits_equal(got, want)
    back = np.concatenate([np.diagonal(_diou_matrix(shim, b[s:s + 500], a[s:s + 500])) for s in range(0, len(a), 500)])
    _assert_bits_equal(back, got)
    assert np.isnan(got).sum() == 3000 + 3000          # exactly the pairs of two zero-area boxes (point/point, line/line)
    # a whole matrix, as the kernels evaluate it, and the C oracle's restatement of the same pair
    m = _random_boxes(np.random.RandomState(1), 300)
    full = _diou_matrix(shim, m, m)
    _assert_bits_equal(full, tvops.distance_box_iou(torch.from_numpy(m), torch.from_numpy(m)).numpy())
    _assert_bits_equal(full, full.T)
    assert all(dno.diou_pair(a[i], b[i]).view(np.uint32) == got[i].view(np.uint32) for i in range(0, 3000, 37))


def _greedy_diou_nms(boxes, scores, classes, thr):
    """The definition: visit by (score desc, index asc); a kept box suppresses later same-class boxes with DIoU > thr."""
    d = tvops.distance_box_iou(torch.from_numpy(boxes), torch.from_numpy(boxes)).numpy()
    order = np.lexsort((np.arange(len(scores)), -scores.astype(np.float64)))
    dead = np.zeros(len(scores), bool)
    keep = []
    for oi, i in enumerate(order):
        if dead[i]:
            continue
        keep.append(i)
        for j in order[oi + 1:]:
            if not dead[j] and classes[j] == classes[i] and d[i, j] > f32(thr):
                dead[j] = True
    return np.array(keep, np.int64)


@pytest.mark.parametrize("n,n_classes,thr", [(1, 1, 0.5), (60, 1, 0.5), (400, 3, 0.5), (400, 1, 0.3), (300, 5, 0.7),
                                             (250, 2, -0.2), (200, 1, 0.0)])
def test_oracle_equals_a_greedy_loop_over_distance_box_iou(n, n_classes, thr):
    rng = np.random.RandomState(n * 7 + n_classes)
    boxes = _random_boxes(rng, n)
    boxes[n // 2:] = boxes[: n - n // 2] + rng.normal(0, 3.0, (n - n // 2, 4)).astype(f32)   # crowded: near-duplicates
    boxes[:, 2:] = np.maximum(boxes[:, 2:], boxes[:, :2] + f32(0.5))
    scores = rng.choice(np.linspace(0.05, 1.0, 40), n).astype(f32)                          # many tied scores
    classes = rng.randint(0, n_classes, n).astype(np.int64)
    np.testing.assert_array_equal(dno.batched_diou_nms(boxes, scores, classes, thr),
                                  _greedy_diou_nms(boxes, scores, classes, thr))


A = [0, 0, 10, 10]
B = [4, 0, 14, 10]          # IoU 60 / 140 = 0.4286; centres 4 apart, enclosing box 14 x 10: DIoU = 0.4286 - 16 / 296


def test_diou_keeps_a_neighbour_that_hard_nms_drops():
    d = dno.diou_pair(A, B)
    assert abs(float(d) - (60 / 140 - 16 / 296)) < 1e-6
    boxes, scores, classes = np.array([A, B], f32), np.array([0.9, 0.8], f32), np.array([0, 0], np.int64)
    assert orc.batched_nms(boxes, scores, classes, 0.4).tolist() == [0]            # IoU 0.43 > 0.4: dropped
    assert dno.batched_diou_nms(boxes, scores, classes, 0.4).tolist() == [0, 1]    # DIoU 0.37 <= 0.4: kept
    assert dno.batched_diou_nms(boxes, scores, classes, 0.35).tolist() == [0]
    # same centres (nested boxes): no distance penalty, DIoU = IoU
    inner = [2.5, 2.5, 7.5, 7.5]
    assert dno.diou_pair(A, inner) == f32(25) / f32(100)


def test_negative_threshold_suppresses_disjoint_boxes_of_the_same_class_only():
    far = [20, 0, 30, 10]   # disjoint: IoU 0, centres 20 apart, enclosing box 30 x 10: DIoU = -400 / 1000
    assert abs(float(dno.diou_pair(A, far)) + 0.4) < 1e-6
    boxes, scores = np.array([A, far, far], f32), np.array([0.9, 0.8, 0.7], f32)
    same = np.array([0, 0, 1], np.int64)
    assert dno.batched_diou_nms(boxes, scores, same, -0.5).tolist() == [0, 2]   # -0.4 > -0.5: box 1 suppressed by box 0
    assert dno.batched_diou_nms(boxes, scores, same, -0.3).tolist() == [0, 1, 2]
    assert orc.batched_nms(boxes, scores, same, -0.5).tolist() == [0, 2]        # hard NMS: IoU 0 > -0.5 as well
    zero = [5, 5, 5, 5]                                                         # two zero-area boxes: NaN, never suppresses
    assert dno.batched_diou_nms(np.array([zero, zero], f32), scores[:2], same[:2], -1.0).tolist() == [0, 1]


def test_python_entries_reject_an_unknown_overlap_before_any_cuda_call():
    z = torch.zeros
    with pytest.raises(ValueError, match="overlap"):
        ops.batched_nms(z(2, 4), z(2), z(2, dtype=torch.int64), 0.5, overlap="giou")
    cand = ops.CandidateBuffers(z(1, dtype=torch.int32), z(1, 4, dtype=torch.int64), z(1, 4, 4), z(1, 4, dtype=torch.int32), 4, None)
    with pytest.raises(ValueError, match="overlap"):
        ops.nms_topk(cand, 1, 0.5, 10, overlap="DIoU")
    with pytest.raises(ValueError, match="nms"):
        ops.dense_postprocess(z(1, 4), z(1, 4, 3), z(1, 4, 4), [(2, 2)], 8, 8, nms="diou_soft")
    with pytest.raises(RuntimeError, match="CUDA tensors only"):      # a valid overlap gets as far as the tensor checks
        ops.batched_nms(z(2, 4), z(2), z(2, dtype=torch.int64), 0.5, overlap="diou")
    assert "diou" in ops.NMS_KINDS


def test_head_postprocess_rejects_an_unknown_nms():
    from sihl_b200.heads import ObjectDetection
    model = ObjectDetection(in_channels=[3] + [8] * 5, num_classes=3, num_channels=16, num_layers=1)
    with pytest.raises(ValueError, match="nms"):
        model.postprocess([torch.zeros(1, 3, 32, 32)], nms="DIoU")


def test_cabi_checks_match_the_greedy_entries():
    """The DIoU entries refuse exactly what their greedy counterparts refuse, before touching the device."""
    lib = _native.load()
    buf = (C.c_char * 256)()
    p = C.addressof(buf)
    topk_args = (("count", p), ("cap", 100), ("key", p), ("box", p), ("cls", p), ("batch", 2), ("thr", 0.5), ("k", 100),
                 ("num", p), ("scores", p), ("classes", p), ("boxes", p), ("ws", None), ("reset", 0), ("stream", None))
    seg_args = (("boxes", p), ("scores", p), ("classes", p), ("seg", p), ("n_images", 1), ("n", 10), ("thr", 0.5),
                ("keep", p), ("count", p), ("ws", None), ("stream", None))

    def call(fn, spec, **kw):
        rc = fn(*[kw.get(n, d) for n, d in spec])
        return rc, lib.sihl_od_last_error_string()

    bad_topk = [dict(k=0), dict(cap=0), dict(cap=1 << 30), dict(key=None), dict(boxes=None), dict(cap=300), dict(batch=0)]
    for kw in bad_topk:
        assert call(lib.sihl_od_diou_nms_topk, topk_args, **kw) == call(lib.sihl_od_nms_topk, topk_args, **kw), kw
    assert call(lib.sihl_od_diou_nms_topk, topk_args, cap=300)[0] == 1      # a long list needs the workspace
    bad_split = [dict(k=0), dict(k=5000), dict(ws=None), dict(key=None), dict(batch=0)]
    for kw in bad_split:
        assert call(lib.sihl_od_diou_nms_topk_split, topk_args, **kw) == call(lib.sihl_od_nms_topk_split, topk_args, **kw), kw
    bad_seg = [dict(n=-1), dict(n=1 << 30), dict(n_images=-1), dict(seg=None), dict(count=None), dict(keep=None),
               dict(n=5000), dict(n=30000), dict(n_images=0)]
    for kw in bad_seg:
        assert call(lib.sihl_od_batched_diou_nms, seg_args, **kw) == call(lib.sihl_od_batched_nms, seg_args, **kw), kw
    assert call(lib.sihl_od_batched_diou_nms, seg_args, n=30000)[0] == 1    # the wide path's mask workspace


# ---- footprint of the DIoU kernels (cuobjdump on the built library, as tests/test_kernel_footprint.py) ----------------
REGS_PER_SM = 65536
REG_ALLOC_UNIT = 256
SCAN_CTAS_PER_SM = 2
SCAN_THREADS = 256
NMS_SHARED_BUDGET = 64 * 1024
CFG1_SCAN = "_ZN4sihl18k_dense_decode_tmaILi5ELb1ELi64EfEEvNS_17DenseDecodeParamsEii"
DIOU_KERNELS = ("_ZN4sihl10k_nms_diouILi512EEEvNS_9NmsParamsE", "_ZN4sihl10k_nms_diouILi1024EEEvNS_9NmsParamsE",
                "_ZN4sihl16k_wide_mask_diouENS_11WideBuffersEif")


def _res_usage():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    _native.load()
    out = subprocess.run([exe, "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    return {name: dict(REG=int(r), STACK=int(s), SHARED=int(sh), LOCAL=int(lo)) for name, r, s, sh, lo in
            re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+) LOCAL:(\d+)", out)}


def _cta_registers(regs_per_thread, threads):
    return -(-regs_per_thread * 32 // REG_ALLOC_UNIT) * REG_ALLOC_UNIT * (threads // 32)


def test_diou_top_k_kernel_fits_beside_two_scan_ctas_and_spills_nothing():
    usage = _res_usage()
    nms = usage[DIOU_KERNELS[0]]                                             # k_nms_diou<512>: the top-K entry
    scan_regs = _cta_registers(usage[CFG1_SCAN]["REG"], SCAN_THREADS)
    assert _cta_registers(nms["REG"], 512) <= REGS_PER_SM - SCAN_CTAS_PER_SM * scan_regs, (nms, usage[CFG1_SCAN])
    assert nms["SHARED"] <= NMS_SHARED_BUDGET, nms
    hard = usage["_ZN4sihl5k_nmsILi512EEEvNS_9NmsParamsE"]
    assert nms["SHARED"] == hard["SHARED"]
    for name in DIOU_KERNELS:
        assert usage[name]["STACK"] == 0 and usage[name]["LOCAL"] == 0, (name, usage[name])   # no spills
