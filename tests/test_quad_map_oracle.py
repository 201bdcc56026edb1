"""Polygon-IoU COCO matching without a GPU: the quad oracle (tests/quad_map_reference.py: the COCOeval loop of
oracle/map_oracle.py on the host build of od_math.h's hull IoU and hull area) against the box oracle, its invariances,
the cases where polygons and AABBs disagree, the argument checks of ops.quad_map_match and sihl_od_quad_map_match, the
workspace query and the footprint of the new kernels."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import quad_map_reference as qm
import quad_reference as qr
from oracle import map_oracle as mo
from sihl_b200 import _native, build, ops, synth

f32 = np.float32
THR, AREAS = mo.IOU_THRESHOLDS, mo.AREA_RANGES


def _images_entry(w, scores, classes, gt_classes):
    return dict(scores=np.asarray(scores)[w["order"]], classes=np.asarray(classes)[w["order"]], dt_match=w["dt_match"],
                dt_ignore=w["dt_ignore"], gt_classes=np.asarray(gt_classes), gt_ignore=w["gt_ignore"])


def _summary(images, max_dets=(1, 10, 100)):
    cats = sorted(set(int(c) for im in images for c in im["classes"]) | set(int(c) for im in images for c in im["gt_classes"]))
    return mo.summarize(*mo.accumulate(images, cats, max_dets=max_dets), max_dets=max_dets)


def _quad_summary(det_quads, det_scores, det_classes, gt_quads, gt_classes):
    w = qm.match_image_quads(det_quads, det_scores, det_classes, gt_quads, gt_classes, THR, AREAS)
    return _summary([_images_entry(w, det_scores, det_classes, gt_classes)])


def _box_summary(det_boxes, det_scores, det_classes, gt_boxes, gt_classes):
    w = mo.match_image(det_boxes, det_scores, det_classes, gt_boxes, gt_classes)
    return _summary([_images_entry(w, det_scores, det_classes, gt_classes)])


def _box_quads(boxes):
    """xyxy -> the four corners (x1,y1), (x2,y1), (x2,y2), (x1,y2)."""
    b = np.asarray(boxes, f32).reshape(-1, 4)
    return np.stack([b[:, [0, 1]], b[:, [2, 1]], b[:, [2, 3]], b[:, [0, 3]]], 1)


def _aabb(quads):
    q = np.asarray(quads, f32).reshape(-1, 4, 2)
    return np.concatenate([q.min(1), q.max(1)], 1)


def _rotate(quads, theta, cx, cy):
    q = np.asarray(quads, np.float64)
    c, s = np.cos(theta), np.sin(theta)
    x, y = q[..., 0] - cx, q[..., 1] - cy
    return np.stack([cx + c * x - s * y, cy + s * x + c * y], -1).astype(f32)


def _tables_equal(a, b):
    for k in ("order", "dt_match", "dt_ignore", "gt_ignore"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)


# ---- the quad oracle's COCOeval loop is map_oracle's ------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_match_loop_equals_the_box_oracle_given_box_ious_and_areas(seed):
    rng = np.random.RandomState(seed)
    K, G = 30, 12
    gt = rng.uniform(0, 200, (G, 2)).astype(f32)
    gt = np.concatenate([gt, gt + rng.uniform(4, 120, (G, 2)).astype(f32)], 1)
    pick = rng.randint(0, G, K)
    det = (gt[pick] + rng.uniform(-10, 10, (K, 4))).astype(f32)
    det[:, 2:] = np.maximum(det[:, 2:], det[:, :2] + 1)
    gt[3] = gt[2]                                                                   # duplicate gts: the later one wins
    scores = np.round(rng.uniform(0, 1, K), 1).astype(f32)                          # ties
    dc, gc = rng.randint(0, 3, K).astype(np.int64), rng.randint(0, 3, G).astype(np.int64)
    gc[3] = gc[2]
    thr = np.concatenate([[0.0], THR])
    areas = AREAS + ((50.0 ** 2, 70.0 ** 2),)
    want = mo.match_image(det, scores, dc, gt, gc, thr, areas)
    got = qm.match_image(scores, dc, gc, mo.box_iou(det, gt), mo.box_area(det), mo.box_area(gt), thr, areas)
    _tables_equal(got, want)
    assert (want["dt_match"] >= 0).any() and (want["dt_ignore"] != 0).any()


# ---- known answers --------------------------------------------------------------------------------------------------
def _doc_example_quads():
    e = mo.TORCHMETRICS_DOC_EXAMPLE
    return (_box_quads(e["det_boxes"]), np.asarray(e["det_scores"], f32), np.asarray(e["det_classes"], np.int64),
            _box_quads(e["gt_boxes"]), np.asarray(e["gt_classes"], np.int64), e["want"])


def test_published_torchmetrics_example_as_axis_aligned_quads():
    dq, ds, dc, gq, gc, want = _doc_example_quads()
    got = _quad_summary(dq, ds, dc, gq, gc)
    for k, v in want.items():
        assert got[k] == pytest.approx(v, abs=1e-12), k


def test_published_example_rotated_by_30_degrees_gives_the_same_summary():
    """Polygon IoU, areas and therefore area ranges do not change under a rotation."""
    dq, ds, dc, gq, gc, want = _doc_example_quads()
    rot = lambda q: _rotate(q, np.pi / 6, 400.0, 160.0)
    got = _quad_summary(rot(dq), ds, dc, rot(gq), gc)
    for k, v in want.items():
        assert got[k] == pytest.approx(v, abs=1e-12), k
    iou = qm.quad_iou_grid(rot(dq), rot(gq))[0, 0]
    assert iou == pytest.approx(304 / 392, abs=1e-5)


def test_detection_on_the_parallel_neighbour_line_scores_zero_with_quads():
    """A 30-degree text line and its neighbour one line height further: the AABB match is a hit, the polygon one is not."""
    gt = qr.rotated_rect(400.0, 300.0, 300.0, 20.0, np.pi / 6).astype(f32)[None]
    det = qr.rotated_rect(400.0 - 20.0 * np.sin(np.pi / 6) * 1.2, 300.0 + 20.0 * np.cos(np.pi / 6) * 1.2, 300.0, 20.0,
                          np.pi / 6).astype(f32)[None]
    ds, dc, gc = np.array([0.9], f32), np.zeros(1, np.int64), np.zeros(1, np.int64)
    q = _quad_summary(det, ds, dc, gt, gc)
    b = _box_summary(_aabb(det), ds, dc, _aabb(gt), gc)
    assert q["map"] == 0.0 and q["map_50"] == 0.0 and q["mar_100"] == 0.0
    assert b["map"] > 0.0 and b["map_50"] == pytest.approx(1.0)


def test_thin_slanted_quad_counts_in_the_area_range_of_its_polygon():
    """A 45-degree 136.4 x 5 px line: AABB 100 x 100 (large as a box), polygon area ~682 < 32^2 (small as a quad)."""
    L, W = 100.0 * np.sqrt(2) - 5.0, 5.0
    q = qr.rotated_rect(300.0, 300.0, L, W, np.pi / 4).astype(f32)
    box = _aabb(q[None])[0]
    assert (box[2] - box[0]) == pytest.approx(100.0, abs=1e-3) and (box[3] - box[1]) == pytest.approx(100.0, abs=1e-3)
    area = float(qm.quad_hull_areas(q[None])[0])
    assert area == pytest.approx(L * W, rel=1e-4) and area < 32.0 ** 2
    w = qm.match_image_quads(q[None], np.array([0.8], f32), np.zeros(1, np.int64), q[None], np.zeros(1, np.int64), THR, AREAS)
    assert w["gt_ignore"][:, 0].tolist() == [0, 0, 1, 1]                            # all, small | not medium, large
    assert (w["dt_match"][1] == 0).all()
    wb = mo.match_image(box[None], np.array([0.8], f32), np.zeros(1, np.int64), box[None], np.zeros(1, np.int64))
    assert wb["gt_ignore"][:, 0].tolist() == [0, 1, 1, 0]
    # and unmatched: a lone thin detection is not ignored at "small", ignored at "medium" and "large"
    far = q[None] + f32(1000.0)
    w = qm.match_image_quads(far, np.array([0.8], f32), np.zeros(1, np.int64), q[None], np.zeros(1, np.int64), THR, AREAS)
    assert (w["dt_match"] == -1).all() and w["dt_ignore"][:, :, 0].tolist() == [[0] * 10, [0] * 10, [1] * 10, [1] * 10]


@pytest.mark.parametrize("seed", [3, 4])
def test_vertex_permutations_and_reversals_give_identical_tables(seed):
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(seed, 2, 40, 15, 3)
    rng = np.random.RandomState(seed)
    thr, areas = np.concatenate([[0.0], THR]), AREAS
    for b in range(2):
        g0, g1 = go[b], go[b + 1]
        base = qm.match_image_quads(dq[b], ds[b], dc[b], gq[g0:g1], gc[g0:g1], thr, areas)
        assert (base["dt_match"] >= 0).any()
        for trial in range(3):
            perm = lambda q: np.stack([x[rng.permutation(4) if trial else np.arange(4)[::-1]] for x in q])
            _tables_equal(qm.match_image_quads(perm(dq[b]), ds[b], dc[b], perm(gq[g0:g1]), gc[g0:g1], thr, areas), base)


def test_axis_aligned_integer_quads_agree_with_the_box_oracle_away_from_ties():
    rng = np.random.RandomState(7)
    G, K = 10, 40
    gt = rng.randint(0, 300, (G, 2))
    gt = np.concatenate([gt, gt + rng.randint(5, 150, (G, 2))], 1).astype(f32)
    det = (gt[rng.randint(0, G, K)] + rng.randint(-12, 13, (K, 4))).astype(f32)
    det[:, 2:] = np.maximum(det[:, 2:], det[:, :2] + 2)
    ious = mo.box_iou(det, gt)
    near = np.abs(ious[..., None] - THR).min(-1) < 1e-6
    det = det[~near.any(1)]
    assert len(det) >= 30
    ds, dc, gc = rng.uniform(0, 1, len(det)).astype(f32), np.zeros(len(det), np.int64), np.zeros(G, np.int64)
    q = _quad_summary(_box_quads(det), ds, dc, _box_quads(gt), gc)
    b = _box_summary(det, ds, dc, gt, gc)
    for k in b:
        assert q[k] == pytest.approx(b[k], abs=1e-6), k


# ---- argument checks ------------------------------------------------------------------------------------------------
def _ws_formula(B, K, G, T, NA):
    up = lambda v: (v + 255) // 256 * 256
    return up((B * K + G) * 52) + up(K * G * 4) + max(G, 1) * T * NA * 4


def test_workspace_query():
    lib = _native.load()
    for args in [(1, 1, 0, 1, 1), (6, 100, 37, 10, 4), (16, 1024, 8000, 16, 8), (0, 5, 0, 10, 4)]:
        assert lib.sihl_od_quad_map_workspace_bytes(*args) == _ws_formula(*args), args
    for bad in [(-1, 10, 5, 10, 4), (1, 0, 5, 10, 4), (1, 1025, 5, 10, 4), (1, 10, -1, 10, 4), (1, 10, 5, 0, 4),
                (1, 10, 5, 17, 4), (1, 10, 5, 10, 0), (1, 10, 5, 10, 9)]:
        assert lib.sihl_od_quad_map_workspace_bytes(*bad) == 0, bad


def test_cabi_argument_checks_before_any_cuda_call():
    lib = _native.load()
    buf = (C.c_char * 256)()
    p = C.addressof(buf)
    thr = (C.c_double * 16)(*([0.5] * 16))
    areas = (C.c_double * 18)(*([0.0, 1e10] * 9))
    spec = [("dq", p), ("ds", p), ("dc", p), ("B", 2), ("K", 10), ("gq", p), ("gc", p), ("go", p), ("G", 5),
            ("thr", C.addressof(thr)), ("T", 10), ("areas", C.addressof(areas)), ("NA", 4), ("order", p), ("dtm", p),
            ("dti", p), ("gti", p), ("ws", p), ("ws_bytes", None), ("stream", None)]

    def call(**kw):
        args = dict(spec)
        args.update(kw)
        if args["ws_bytes"] is None:
            args["ws_bytes"] = _ws_formula(args["B"], args["K"], args["G"], args["T"], args["NA"])
        rc = lib.sihl_od_quad_map_match(*[args[n] for n, _ in spec])
        return rc, lib.sihl_od_last_error_string()

    for name in ("dq", "ds", "dc", "go", "thr", "areas", "order", "dtm", "dti", "ws", "gq", "gc", "gti"):
        assert call(**{name: None})[0] == 1, name
    assert call(gq=None, gc=None, gti=None, G=0, B=0)[0] == 0                       # no ground truth, no images: no CUDA call
    for kw, text in [(dict(K=1025), b"1024"), (dict(K=0), b"1024"), (dict(B=-1), b"bad sizes"), (dict(G=-1), b"bad sizes"),
                     (dict(T=17), b"16"), (dict(T=0), b"16"), (dict(NA=9), b"8"), (dict(NA=0), b"8")]:
        rc, msg = call(**kw)
        assert rc == 1 and text in msg, (kw, msg)
    need = _ws_formula(2, 10, 5, 10, 4)
    rc, msg = call(ws_bytes=need - 1)
    assert rc == 1 and b"workspace" in msg and str(need).encode() in msg
    assert call(B=0)[0] == 0                                                        # batch 0: checked, nothing launched
    assert call(B=0, dq=None, ds=None, dc=None, order=None, dtm=None, dti=None, ws=None, ws_bytes=0)[0] == 0
    assert call(B=0, K=1025)[0] == 1 and call(B=0, thr=None)[0] == 1


def test_python_entry_checks_its_arguments_before_any_cuda_call():
    z = torch.zeros
    i64 = dict(dtype=torch.int64)
    off = torch.tensor([0, 3, 5], dtype=torch.int32)
    good = lambda K=10: (z(2, K, 4, 2), z(2, K), z(2, K, **i64), z(5, 8), z(5, **i64), off)
    with pytest.raises(ValueError, match=r"\[B, K, 4, 2\]"):
        ops.quad_map_match(z(2, 10, 4), *good()[1:])
    with pytest.raises(ValueError, match=r"\[B, K, 4, 2\]"):
        ops.quad_map_match(z(20, 8), *good()[1:])
    with pytest.raises(ValueError, match="disagree"):
        ops.quad_map_match(z(2, 9, 8), *good()[1:])
    with pytest.raises(ValueError, match="1024"):
        ops.quad_map_match(*good(1025))
    with pytest.raises(ValueError, match="16 IoU thresholds"):
        ops.quad_map_match(*good(), iou_thresholds=[0.5] * 17)
    with pytest.raises(ValueError, match="8 area"):
        ops.quad_map_match(*good(), area_ranges=[(0.0, 1.0)] * 9)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.quad_map_match(*good())


def test_detection_map_iou_type():
    from sihl_b200 import metrics
    assert metrics.DetectionMAP().iou_type == "bbox"
    assert metrics.DetectionMAP(iou_type="quad").iou_type == "quad"
    with pytest.raises(ValueError, match="iou_type"):
        metrics.DetectionMAP(iou_type="segm")


# ---- footprint of the new kernels (cuobjdump on the built library) ---------------------------------------------------
QUAD_MAP_KERNELS = ("_ZN4sihl16k_quad_map_hullsEPKflS1_lPNS_8QuadHullE",
                    "_ZN4sihl14k_quad_map_iouEPKNS_8QuadHullEPKlS4_PKiiiiPf",
                    "_ZN4sihl16k_quad_map_matchENS_9MapParamsEPKfPKNS_8QuadHullE")


def test_quad_map_kernels_are_built_for_sm100a_with_a_small_stack():
    """The clip's two 8-vertex polygons live in k_quad_map_iou's stack frame; the hull kernel has none."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    _native.load()
    out = subprocess.run([exe, "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage = {name: dict(REG=int(r), STACK=int(s)) for name, r, s in
             re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)}
    for name in QUAD_MAP_KERNELS:
        assert name in usage, name
        assert usage[name]["STACK"] <= 256 and usage[name]["REG"] <= 128, (name, usage[name])
    assert usage[QUAD_MAP_KERNELS[0]]["STACK"] == 0
