"""Quadrilateral NMS without a GPU: the quad overlap every quad kernel calls (od_math.h, compiled for the host by
tests/host_quad_shim.cpp) against an exact rational restatement, its symmetry and vertex-order invariance, hand cases,
the greedy host oracle, the argument checks of the C and Python entries, and the footprint of the new kernels."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch
from torchvision import ops as tvops

import quad_reference as qr
from sihl_b200 import _native, build, ops, synth

f32 = np.float32


def _quads(rng, n, small_far=False):
    """Seeded rotated rectangles with vertex jitter, coordinates in [0, 4096], sides >= 2 px, aspect <= 100."""
    if small_far:
        cx, cy = rng.uniform(3900, 4090, n), rng.uniform(3900, 4090, n)
        w, h = rng.uniform(2, 6, n), rng.uniform(2, 6, n)
    else:
        cx, cy = rng.uniform(200, 3900, n), rng.uniform(200, 3900, n)
        w = np.exp(rng.uniform(np.log(2), np.log(300), n))
        h = np.clip(w * np.exp(rng.uniform(np.log(0.01), np.log(1), n)), 2, None)
    th = rng.uniform(-np.pi, np.pi, n)
    q = np.stack([qr.rotated_rect(*p) for p in zip(cx, cy, w, h, th)])
    q += rng.normal(0, 0.05, (n, 4, 2)) * np.minimum(w, h)[:, None, None]
    return q, np.minimum(w, h)


def _pairs(seed, n, small_far=False):
    rng = np.random.RandomState(seed)
    a, side = _quads(rng, n, small_far)
    b = a + rng.normal(0, 0.5, (n, 1, 2)) * side[:, None, None] + rng.normal(0, 0.05, (n, 4, 2)) * side[:, None, None]
    return a.astype(f32), b.astype(f32)


@pytest.mark.parametrize("small_far", [False, True])
def test_host_quad_iou_within_1e5_of_the_exact_iou(small_far):
    a, b = _pairs(11 + small_far, 1500, small_far)
    got = qr.quad_iou_pairs(a, b)
    want = np.array([qr.exact_iou(x, y) for x, y in zip(a, b)])
    assert np.abs(got - want).max() <= 1e-5, np.abs(got - want).max()
    assert (want > 0.1).sum() > 500                                  # most pairs overlap substantially


def test_bitwise_symmetric_and_invariant_to_vertex_order():
    """quad_iou(a, b) and quad_iou(b, a) are the same bits.  The hull is built from the sorted point set, so any
    permutation of either quad's vertices (other start vertex, reversed orientation, bow-tie order) gives the same bits
    as well."""
    a, b = _pairs(5, 2000)
    got = qr.quad_iou_pairs(a, b)
    assert np.array_equal(got.view(np.uint32), qr.quad_iou_pairs(b, a).view(np.uint32))
    rng = np.random.RandomState(6)
    for perm_a, perm_b in [([1, 2, 3, 0], [3, 2, 1, 0]), ([0, 2, 1, 3], [2, 3, 0, 1])] + \
            [(list(rng.permutation(4)), list(rng.permutation(4))) for _ in range(4)]:
        p = qr.quad_iou_pairs(a[:, perm_a], b[:, perm_b])
        assert np.array_equal(p.view(np.uint32), got.view(np.uint32)), (perm_a, perm_b)


def _one(a, b):
    return float(qr.quad_iou_pairs(np.array([a], f32), np.array([b], f32))[0])


SQ = [[0, 0], [10, 0], [10, 10], [0, 10]]


def test_hand_cases():
    assert abs(_one(SQ, SQ) - 1.0) <= 1e-6                                           # identical
    rot = qr.rotated_rect(500.0, 700.0, 40.0, 8.0, 0.6)
    assert abs(_one(rot, rot) - 1.0) <= 1e-6
    inner = [[2, 2], [8, 2], [8, 8], [2, 8]]                                         # containment: 36 / 100
    assert _one(SQ, inner) == f32(36) / f32(100)
    assert _one(SQ, [[20, 0], [30, 0], [30, 10], [20, 10]]) == 0.0                  # disjoint
    assert _one(SQ, [[10, 0], [20, 0], [20, 10], [10, 10]]) == 0.0                  # touching along an axis-aligned edge
    diamond = [[0, 0], [10, 10], [0, 20], [-10, 10]]                                 # touching along a slanted edge
    assert abs(_one(diamond, [[0, 0], [10, 10], [20, 0], [10, -10]])) <= 1e-6
    assert _one(SQ, [[0, 0], [10, 0], [10, 5], [0, 5]]) == f32(0.5)                 # a shared collinear edge: 50 / 100
    tri = [[0, 0], [10, 0], [10, 10], [10, 10]]                                      # a triangle (repeated vertex)
    assert _one(SQ, tri) == f32(0.5)
    bowtie = [[0, 0], [10, 10], [10, 0], [0, 10]]                                    # self-intersecting order: its hull
    assert _one(SQ, bowtie) == 1.0
    for degenerate in ([[0, 0], [5, 5], [10, 10], [2, 2]], [[3, 3]] * 4, [[0, 5], [10, 5], [10, 5], [0, 5]]):
        assert _one(SQ, degenerate) == 0.0 and _one(degenerate, degenerate) == 0.0
        assert qr.exact_iou(SQ, degenerate) == 0.0
    for a, b in [(SQ, inner), (SQ, tri), (diamond, SQ), (rot, qr.rotated_rect(505.0, 702.0, 40.0, 8.0, 0.7))]:
        assert abs(_one(a, b) - qr.exact_iou(a, b)) <= 1e-6


def test_axis_aligned_quads_match_box_iou():
    boxes, _, _ = synth.nms_candidates_np(3, 400, 1024, 1)
    x1, y1, x2, y2 = boxes.T
    quads = np.stack([np.stack([x1, y1], 1), np.stack([x2, y1], 1), np.stack([x2, y2], 1), np.stack([x1, y2], 1)], 1)
    got = qr.quad_iou_matrix(quads, quads)
    want = tvops.box_iou(torch.from_numpy(boxes), torch.from_numpy(boxes)).numpy()
    assert np.abs(got - want).max() <= 1e-5
    assert np.array_equal(got == 0, want == 0)


def test_slanted_parallel_lines_overlap_as_boxes_but_not_as_quads():
    """Two parallel 30-degree text lines one line height apart: the AABB workaround would drop one of them."""
    a = qr.rotated_rect(400.0, 300.0, 300.0, 20.0, np.pi / 6).astype(f32)
    b = qr.rotated_rect(400.0 - 20.0 * np.sin(np.pi / 6) * 1.2, 300.0 + 20.0 * np.cos(np.pi / 6) * 1.2, 300.0, 20.0,
                        np.pi / 6).astype(f32)
    bb = lambda q: [q[:, 0].min(), q[:, 1].min(), q[:, 0].max(), q[:, 1].max()]
    aabb = float(tvops.box_iou(torch.tensor([bb(a)]), torch.tensor([bb(b)]))[0, 0])
    assert aabb > 0.5 and _one(a, b) == 0.0 and qr.exact_iou(a, b) == 0.0
    keep = qr.batched_quad_nms(np.stack([a, b]), np.array([0.9, 0.8], f32), np.zeros(2, np.int64), 0.5)
    assert keep.tolist() == [0, 1]


def _greedy_exact(quads, scores, classes, thr):
    order = np.lexsort((np.arange(len(scores)), -scores.astype(np.float64)))
    keep, dead = [], np.zeros(len(scores), bool)
    iou = qr.quad_iou_matrix(quads, quads)
    for oi, i in enumerate(order):
        if dead[i]:
            continue
        keep.append(i)
        for j in order[oi + 1:]:
            if classes[j] == classes[i] and iou[i, j] > f32(thr):
                dead[j] = True
    return np.array(keep, np.int64)


@pytest.mark.parametrize("n,n_cls,thr", [(1, 1, 0.5), (300, 1, 0.5), (300, 4, 0.3), (200, 2, -0.3), (250, 3, 0.0),
                                         (300, 1, 0.9)])
def test_host_oracle_equals_a_plain_greedy_loop(n, n_cls, thr):
    """The shim's AABB pre-reject changes nothing: it equals the definition over the full IoU matrix."""
    quads, scores, classes = synth.quad_candidates_np(n + n_cls, n, 1024, n_cls)
    scores[::7] = scores[0]                                                         # ties: index order decides
    np.testing.assert_array_equal(qr.batched_quad_nms(quads, scores, classes, thr),
                                  _greedy_exact(quads, scores, classes, thr))


def test_synthetic_quads_have_clusters_and_parallel_neighbours():
    quads, scores, classes = synth.quad_candidates_np(1, 2000, 1024, 5)
    assert quads.shape == (2000, 4, 2) and quads.dtype == f32 and scores.dtype == f32 and classes.dtype == np.int64
    assert quads.min() >= 0 and quads.max() <= 1024
    keep = qr.batched_quad_nms(quads, scores, classes, 0.5)
    assert 300 < keep.size < 1500
    again = synth.quad_candidates_np(1, 2000, 1024, 5)
    assert all(np.array_equal(x, y) for x, y in zip((quads, scores, classes), again))


# ---- argument checks ------------------------------------------------------------------------------------------------
def test_cabi_argument_checks_and_workspace_query():
    lib = _native.load()
    assert lib.sihl_od_batched_quad_nms_workspace_bytes(0) == 0
    small, big = lib.sihl_od_batched_quad_nms_workspace_bytes(1), lib.sihl_od_batched_quad_nms_workspace_bytes(90000)
    assert 0 < small < big and big > 90000 * 90000 // 8 + 90000 * 32
    assert lib.sihl_od_batched_quad_nms_workspace_bytes(90001) == 0 and lib.sihl_od_batched_quad_nms_workspace_bytes(-1) == 0
    # the box path's buffers plus 32 bytes of hull vertices per quad, rounded to 256
    assert lib.sihl_od_batched_quad_nms_workspace_bytes(30000) == lib.sihl_od_batched_nms_workspace_bytes(30000) + 30000 * 32
    buf = (C.c_char * 256)()
    p = C.addressof(buf)
    spec = (("quads", p), ("scores", p), ("classes", p), ("seg", p), ("n_images", 1), ("n", 10), ("thr", 0.5),
            ("keep", p), ("count", p), ("ws", p), ("stream", None))

    def call(**kw):
        rc = lib.sihl_od_batched_quad_nms(*[kw.get(n, d) for n, d in spec])
        return rc, lib.sihl_od_last_error_string()

    for kw in [dict(n=-1), dict(n_images=-1), dict(seg=None), dict(count=None), dict(keep=None), dict(quads=None),
               dict(scores=None), dict(classes=None), dict(ws=None)]:
        assert call(**kw)[0] == 1, kw
    rc, msg = call(n=90001)
    assert rc == 1 and b"90000" in msg
    assert call(n_images=0)[0] == 0                                                 # nothing to do: no CUDA call
    assert call(n=0, quads=None, scores=None, classes=None, keep=None, ws=None, n_images=0)[0] == 0
    assert lib.sihl_od_quad_iou(None, 0, None, 5, None, None) == 0                 # empty: no CUDA call
    assert lib.sihl_od_quad_iou(None, 3, p, 5, p, None) == 1
    assert lib.sihl_od_quad_iou(p, -1, p, 5, p, None) == 1
    assert lib.sihl_od_quad_iou(p, 1 << 20, p, 1 << 20, p, None) == 1               # 2^40 pairs
    assert b"2^38" in lib.sihl_od_last_error_string()


def test_python_entries_check_their_arguments_before_any_cuda_call():
    z = torch.zeros
    with pytest.raises(ValueError, match="90000"):
        ops.batched_quad_nms(z(90001, 4, 2), z(90001), z(90001, dtype=torch.int64), 0.5)
    with pytest.raises(ValueError, match=r"\[N, 4, 2\]"):
        ops.batched_quad_nms(z(10, 4), z(10), z(10, dtype=torch.int64), 0.5)
    with pytest.raises(ValueError, match=r"\[N, 4, 2\]"):
        ops.quad_iou(z(3, 3, 2), z(3, 8))
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.batched_quad_nms(z(10, 4, 2), z(10), z(10, dtype=torch.int64), 0.5)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.quad_iou(z(3, 8), z(3, 4, 2))


# ---- footprint of the quad kernels (cuobjdump on the built library) --------------------------------------------------
QUAD_KERNELS = ("_ZN4sihl19k_wide_scatter_quadEPKfPKiS3_iNS_11WideBuffersEP6float4",
                "_ZN4sihl16k_wide_mask_quadENS_11WideBuffersEPK6float4if", "_ZN4sihl10k_quad_iouEPKflS1_lPf")


def test_quad_kernels_are_built_for_sm100a_with_a_small_stack():
    """The clip keeps its two 8-vertex polygons in a per-thread stack frame (dynamic indices); nothing else is local."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    _native.load()
    out = subprocess.run([exe, "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage = {name: dict(REG=int(r), STACK=int(s), SHARED=int(sh)) for name, r, s, sh in
             re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:(\d+)", out)}
    for name in QUAD_KERNELS:
        assert name in usage, name
        assert usage[name]["STACK"] <= 256 and usage[name]["REG"] <= 128, (name, usage[name])
    assert usage[QUAD_KERNELS[0]]["STACK"] == 0
