"""COCO crowd regions and annotated areas without a GPU: closed-form cases of the crowd oracle
(tests/crowd_map_reference.py: match_image_boxes, match_image_quads with gt_crowd / gt_area) through map_oracle's
accumulate / summarize; its agreement with the plain oracles without annotations; the host IoA of od_math.h; the
argument checks of the ops, of DetectionMAP and of the two C entries; the new kernels' footprint."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import crowd_map_reference as cr
import quad_map_reference as qm
from oracle import map_oracle as mo
from sihl_b200 import _native, build, metrics, ops

f32 = np.float32
THR, AREAS = mo.IOU_THRESHOLDS, mo.AREA_RANGES


def _summary(w, scores, classes, gt_classes):
    im = dict(scores=np.asarray(scores, f32)[w["order"]], classes=np.asarray(classes)[w["order"]], dt_match=w["dt_match"],
              dt_ignore=w["dt_ignore"], gt_classes=np.asarray(gt_classes), gt_ignore=w["gt_ignore"])
    cats = sorted(set(int(c) for c in classes) | set(int(c) for c in gt_classes))
    return mo.summarize(*mo.accumulate([im], cats))


def _box_quads(boxes):
    b = np.asarray(boxes, f32).reshape(-1, 4)
    return np.stack([b[:, [0, 1]], b[:, [2, 1]], b[:, [2, 3]], b[:, [0, 3]]], 1)


def _rotate(quads, theta=np.pi / 6, cx=300.0, cy=300.0):
    q = np.asarray(quads, np.float64)
    c, s = np.cos(theta), np.sin(theta)
    x, y = q[..., 0] - cx, q[..., 1] - cy
    return np.stack([cx + c * x - s * y, cy + s * x + c * y], -1).astype(f32)


def _match(geometry, det, scores, dc, gt, gc, **kw):
    """The box oracle on xyxy boxes, or the quad oracle on their corners rotated by 30 degrees."""
    if geometry == "box":
        return cr.match_image_boxes(det, scores, dc, gt, gc, **kw)
    thr, areas = kw.pop("iou_thresholds", THR), kw.pop("area_ranges", AREAS)
    return cr.match_image_quads(_rotate(_box_quads(det)), scores, dc, _rotate(_box_quads(gt)), gc, thr, areas, **kw)


GEOMETRIES = ("box", "quad")
# one regular object, a crowd region far from it, a good detection of the object and a detection inside the region
OBJ, CROWD = [100.0, 100.0, 200.0, 200.0], [400.0, 400.0, 600.0, 600.0]
HIT, INSIDE = [102.0, 101.0, 201.0, 199.0], [450.0, 450.0, 490.0, 480.0]


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_detection_inside_a_crowd_region_is_ignored(geometry):
    gt, gc = np.array([OBJ, CROWD], f32), np.zeros(2, np.int64)
    det, dc = np.array([INSIDE, HIT], f32), np.zeros(2, np.int64)
    scores = np.array([0.9, 0.8], f32)                                              # the one inside ranks first
    crowd = np.array([0, 1], np.uint8)
    w = _match(geometry, det, scores, dc, gt, gc, gt_crowd=crowd)
    assert (w["dt_match"][0, :, 0] == 1).all() and (w["dt_ignore"][0, :, 0] == 1).all()
    assert w["gt_ignore"][:, 1].tolist() == [1, 1, 1, 1]
    with_crowd = _summary(w, scores, dc, gc)
    alone = _summary(_match(geometry, det[1:], scores[1:], dc[1:], gt[:1], gc[:1]), scores[1:], dc[1:], gc[:1])
    for k in alone:                                 # mar_1: the ignored detection still fills the one maxDets slot
        assert with_crowd[k] == pytest.approx(0.0 if k == "mar_1" else alone[k], abs=1e-12), k
    # without the flag: the region is a missed object and the detection a false positive ranked above the hit
    plain = _summary(_match(geometry, det, scores, dc, gt, gc), scores, dc, gc)
    assert (_match(geometry, det, scores, dc, gt, gc)["dt_match"][0, :, 0] == -1).all()
    # precision at recall <= 0.5 is 1/2 (the hit comes second); recall never passes 0.5: 51 of 101 points, each 0.5
    assert plain["map_50"] == pytest.approx(51 * 0.5 / 101, abs=1e-12)
    assert plain["mar_100"] == pytest.approx(0.5, abs=1e-12) and with_crowd["mar_100"] == pytest.approx(1.0, abs=1e-12)
    assert with_crowd["map_50"] == pytest.approx(1.0, abs=1e-12)


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_several_detections_on_one_crowd_region_are_all_ignored(geometry):
    gt, gc = np.array([CROWD], f32), np.zeros(1, np.int64)
    det = np.array([[410, 410, 450, 440], [500, 420, 560, 470], [430, 500, 520, 590], [405, 405, 595, 595]], f32)
    dc, scores = np.zeros(4, np.int64), np.array([0.9, 0.8, 0.7, 0.6], f32)
    w = _match(geometry, det, scores, dc, gt, gc, gt_crowd=np.ones(1, np.uint8))
    assert (w["dt_match"][0] == 0).all() and (w["dt_ignore"] == 1).all()            # every range, threshold and rank
    s = _summary(w, scores, dc, gc)
    assert s["map"] == -1.0 and s["mar_100"] == -1.0                                # nothing left to evaluate
    w = _match(geometry, det, scores, dc, gt, gc)                                   # regular: one match per threshold
    assert ((w["dt_match"][0] == 0).sum(axis=1) <= 1).all()


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_small_detection_in_a_large_crowd_region_matches_at_every_threshold(geometry):
    gt, gc = np.array([CROWD], f32), np.zeros(1, np.int64)
    det, dc, scores = np.array([INSIDE], f32), np.zeros(1, np.int64), np.array([0.5], f32)
    if geometry == "box":
        assert mo.box_iou(det, gt)[0, 0] == pytest.approx(1200 / 40000)
        assert cr.box_ioa(det, gt)[0, 0] == 1.0
    else:
        dq, gq = _rotate(_box_quads(det)), _rotate(_box_quads(gt))
        assert qm.quad_iou_grid(dq, gq)[0, 0] == pytest.approx(1200 / 40000, rel=1e-4)
        assert cr.quad_ioa_grid(dq, gq)[0, 0] == pytest.approx(1.0, abs=1e-6)
    w = _match(geometry, det, scores, dc, gt, gc, gt_crowd=[1])
    assert (w["dt_match"] == 0).all() and (w["dt_ignore"] == 1).all()
    assert (_match(geometry, det, scores, dc, gt, gc)["dt_match"] == -1).all()


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_a_regular_gt_wins_over_an_overlapping_crowd_gt(geometry):
    # the object lies inside the crowd region; a detection on it has IoU 2400 / 2596 with the object, IoA 1 with the region
    gt, gc = np.array([[400, 400, 600, 600], [450, 450, 500, 500]], f32), np.zeros(2, np.int64)
    det, dc, scores = np.array([[452, 450, 500, 502]], f32), np.zeros(1, np.int64), np.array([0.7], f32)
    w = _match(geometry, det, scores, dc, gt, gc, gt_crowd=[1, 0])
    assert (w["dt_match"][0, :9, 0] == 1).all() and (w["dt_ignore"][0, :9, 0] == 0).all()
    # at 0.95 the object is out of reach (IoU < 0.95) and the crowd region takes the detection, ignored
    assert w["dt_match"][0, 9, 0] == 0 and w["dt_ignore"][0, 9, 0] == 1


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_area_annotations_move_gts_between_ranges(geometry):
    gt = np.array([[0, 0, 20, 20], [100, 100, 140, 140], [300, 300, 420, 420], [600, 600, 620, 620]], f32)
    gc = np.zeros(4, np.int64)
    det, dc, scores = gt.copy(), np.zeros(4, np.int64), np.array([0.9, 0.8, 0.7, 0.6], f32)
    want_plain = [[0, 0, 0, 0], [0, 1, 1, 0], [1, 0, 1, 1], [1, 1, 0, 1]]           # [all, small, medium, large][g]
    assert _match(geometry, det, scores, dc, gt, gc)["gt_ignore"].tolist() == want_plain
    # 400 px^2 annotated as large; 1600 -> small; 14400 -> medium; the last one: 0 keeps its computed (small) area
    area = np.array([200.0 ** 2, 20.0 ** 2, 50.0 ** 2, 0.0])
    w = _match(geometry, det, scores, dc, gt, gc, gt_area=area)
    assert w["gt_ignore"].tolist() == [[0, 0, 0, 0], [1, 0, 1, 0], [1, 1, 0, 1], [0, 1, 1, 1]]
    for bad in (-5.0, np.nan):                                                      # <= 0 and NaN fall back as well
        assert _match(geometry, det, scores, dc, gt, gc, gt_area=np.full(4, bad))["gt_ignore"].tolist() == want_plain
    # detections keep their own area: unmatched detections far away are placed by it
    far = det + f32(2000.0)
    w = _match(geometry, far, scores, dc, gt, gc, gt_area=area)
    assert (w["dt_match"] == -1).all() and w["dt_ignore"][:, 0, :].tolist() == want_plain


def test_quad_ioa_is_the_hull_intersection_over_the_detection_hull():
    a = _rotate(_box_quads([[0, 0, 10, 10]]), 0.3, 0, 0)
    b = _box_quads([[-100, -100, 100, 100]])
    assert cr.quad_ioa_grid(a, b)[0, 0] == 1.0
    half = _box_quads([[5, 0, 15, 10]])
    assert cr.quad_ioa_grid(_box_quads([[0, 0, 10, 10]]), half)[0, 0] == pytest.approx(0.5, abs=1e-6)
    assert cr.quad_ioa_grid(_box_quads([[0, 0, 10, 10]]), _box_quads([[20, 20, 30, 30]]))[0, 0] == 0.0
    flat = np.array([[[0, 0], [5, 0], [10, 0], [2, 0]]], f32)                       # zero-area hull
    assert cr.quad_ioa_grid(flat, b)[0, 0] == 0.0 and cr.quad_ioa_grid(b, flat)[0, 0] == 0.0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_without_annotations_the_crowd_oracle_is_the_plain_one(seed):
    """No annotations, all-zero flags and areas <= 0 give map_oracle's (boxes) and quad_map_reference's (quads) tables."""
    rng = np.random.RandomState(seed)
    K, G = 30, 12
    gt = rng.uniform(0, 200, (G, 2)).astype(f32)
    gt = np.concatenate([gt, gt + rng.uniform(4, 120, (G, 2)).astype(f32)], 1)
    det = (gt[rng.randint(0, G, K)] + rng.uniform(-10, 10, (K, 4))).astype(f32)
    det[:, 2:] = np.maximum(det[:, 2:], det[:, :2] + 1)
    gt[3] = gt[2]
    scores = np.round(rng.uniform(0, 1, K), 1).astype(f32)
    dc, gc = rng.randint(0, 3, K).astype(np.int64), rng.randint(0, 3, G).astype(np.int64)
    thr, areas = np.concatenate([[0.0], THR]), AREAS + ((50.0 ** 2, 70.0 ** 2),)
    dq, gq = _rotate(_box_quads(det)), _rotate(_box_quads(gt))
    want_box = mo.match_image(det, scores, dc, gt, gc, thr, areas)
    want_quad = qm.match_image_quads(dq, scores, dc, gq, gc, thr, areas)
    assert (want_box["dt_match"] >= 0).any() and (want_quad["dt_match"] >= 0).any()
    for kw in (dict(), dict(gt_crowd=np.zeros(G)), dict(gt_area=np.zeros(G)),
               dict(gt_crowd=np.zeros(G, bool), gt_area=np.where(np.arange(G) % 2, -1.0, np.nan))):
        got_box = cr.match_image_boxes(det, scores, dc, gt, gc, thr, areas, **kw)
        got_quad = cr.match_image_quads(dq, scores, dc, gq, gc, thr, areas, **kw)
        for k in want_box:
            np.testing.assert_array_equal(got_box[k], want_box[k], err_msg=f"box {kw.keys()} {k}")
            np.testing.assert_array_equal(got_quad[k], want_quad[k], err_msg=f"quad {kw.keys()} {k}")


# ---- argument checks ------------------------------------------------------------------------------------------------
def test_python_entries_check_the_annotations_before_any_cuda_call():
    z, i64 = torch.zeros, dict(dtype=torch.int64)
    off = torch.tensor([0, 3, 5], dtype=torch.int32)
    boxes = (z(2, 10, 4), z(2, 10), z(2, 10, **i64), z(5, 4), z(5, **i64), off)
    quads = (z(2, 10, 8), z(2, 10), z(2, 10, **i64), z(5, 8), z(5, **i64), off)
    for fn, args in ((ops.map_match, boxes), (ops.quad_map_match, quads)):
        with pytest.raises(ValueError, match=r"gt_crowd: expected shape \[5\]"):
            fn(*args, gt_crowd=z(4, dtype=torch.bool))
        with pytest.raises(ValueError, match=r"gt_area: expected shape \[5\]"):
            fn(*args, gt_area=z(5, 1))
        with pytest.raises(TypeError, match="gt_crowd"):
            fn(*args, gt_crowd=[0] * 5)
        with pytest.raises(TypeError, match="bool or integer"):
            fn(*args, gt_crowd=z(5))
        with pytest.raises(TypeError, match="real"):
            fn(*args, gt_area=z(5, dtype=torch.complex64))
        with pytest.raises(RuntimeError, match="gt_crowd: sihl_b200 kernels run on CUDA tensors only"):
            fn(*args, gt_crowd=z(5, dtype=torch.bool))


def test_detection_map_rejects_annotations_that_disagree_with_labels():
    tgt = dict(labels=torch.zeros(2, dtype=torch.int64), boxes=torch.zeros(2, 4))
    for key, bad in (("iscrowd", torch.zeros(3)), ("area", torch.zeros(2, 1))):
        with pytest.raises(ValueError, match=key):
            metrics.DetectionMAP._annotations([tgt, dict(tgt, **{key: bad})], "cpu")
    out = metrics.DetectionMAP._annotations([tgt, dict(tgt, iscrowd=torch.tensor([True, False]))], "cpu")
    assert out["gt_area"] is None and out["gt_crowd"].tolist() == [0, 0, 1, 0] and out["gt_crowd"].dtype == torch.uint8
    out = metrics.DetectionMAP._annotations([dict(tgt, area=torch.tensor([5.0, 7.0])), tgt], "cpu")
    assert out["gt_crowd"] is None and out["gt_area"].tolist() == [5.0, 7.0, 0.0, 0.0]
    assert out["gt_area"].dtype == torch.float64
    assert metrics.DetectionMAP._annotations([tgt], "cpu") == dict(gt_crowd=None, gt_area=None)


def _ws_quad(B, K, G, T, NA):
    up = lambda v: (v + 255) // 256 * 256
    return up((B * K + G) * 52) + up(K * G * 4) + max(G, 1) * T * NA * 4


@pytest.mark.parametrize("entry", ["sihl_od_map_match_crowd", "sihl_od_quad_map_match_crowd"])
def test_cabi_argument_checks_before_any_cuda_call(entry):
    lib = _native.load()
    fn = getattr(lib, entry)
    quad = "quad" in entry
    buf = (C.c_char * 256)()
    p = C.addressof(buf)
    thr = (C.c_double * 16)(*([0.5] * 16))
    areas = (C.c_double * 18)(*([0.0, 1e10] * 9))
    spec = [("det", p), ("ds", p), ("dc", p), ("B", 2), ("K", 10), ("gt", p), ("gc", p), ("go", p), ("G", 5),
            ("crowd", p), ("area", p), ("thr", C.addressof(thr)), ("T", 10), ("areas", C.addressof(areas)), ("NA", 4),
            ("order", p), ("dtm", p), ("dti", p), ("gti", p), ("ws", p)] + ([("ws_bytes", None)] if quad else []) + \
           [("stream", None)]

    def call(**kw):
        args = dict(spec)
        args.update(kw)
        if quad and args["ws_bytes"] is None:
            args["ws_bytes"] = _ws_quad(args["B"], args["K"], args["G"], args["T"], args["NA"])
        rc = fn(*[args[n] for n, _ in spec])
        return rc, lib.sihl_od_last_error_string()

    for name in ("det", "ds", "dc", "go", "thr", "areas", "order", "dtm", "dti", "ws", "gt", "gc", "gti"):
        assert call(**{name: None})[0] == 1, name
    for kw, text in [(dict(K=1025), b"1024"), (dict(K=0), b"1024"), (dict(B=-1), b"bad sizes"), (dict(G=-1), b"bad sizes"),
                     (dict(T=17), b"16"), (dict(T=0), b"16"), (dict(NA=9), b"8"), (dict(NA=0), b"8")]:
        rc, msg = call(**kw)
        assert rc == 1 and text in msg, (kw, msg)
    if quad:
        rc, msg = call(ws_bytes=_ws_quad(2, 10, 5, 10, 4) - 1)
        assert rc == 1 and b"workspace" in msg
    # no images: checked, nothing launched, with or without annotations; the empty arrays may be NULL
    for kw in (dict(), dict(crowd=None), dict(area=None), dict(crowd=None, area=None)):
        assert call(B=0, **kw)[0] == 0, kw
    assert call(B=0, det=None, ds=None, dc=None, order=None, dtm=None, dti=None, ws=None, gt=None, gc=None, gti=None,
                G=0, **(dict(ws_bytes=0) if quad else {}))[0] == 0
    assert call(B=0, K=1025)[0] == 1 and call(B=0, thr=None)[0] == 1 and call(B=0, T=0)[0] == 1


def test_crowd_entries_are_in_the_header_and_the_bindings():
    header = open(os.path.join(os.path.dirname(build.HERE), "include", "sihl_od.h")).read()
    for name in ("sihl_od_map_match_crowd", "sihl_od_quad_map_match_crowd"):
        assert re.search(rf"SIHL_OD_API int {name}\(", header), name
        assert name in _native._SIGNATURES


# ---- footprint of the new kernels (cuobjdump on the built library) ---------------------------------------------------
CROWD_KERNELS = ("_ZN4sihl17k_map_match_crowdENS_9MapParamsENS_14MapAnnotationsE",
                 "_ZN4sihl20k_quad_map_iou_crowdEPKNS_8QuadHullEPKlS4_PKiiiiPKhPf",
                 "_ZN4sihl22k_quad_map_match_crowdENS_9MapParamsEPKfPKNS_8QuadHullENS_14MapAnnotationsE")


def test_crowd_kernels_are_built_for_sm100a_with_a_small_stack():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not found")
    _native.load()
    out = subprocess.run([exe, "-res-usage", build.LIB_PATH], capture_output=True, text=True, check=True).stdout
    usage = {name: dict(REG=int(r), STACK=int(s)) for name, r, s in
             re.findall(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)}
    for name in CROWD_KERNELS:
        assert name in usage, name
        assert usage[name]["STACK"] <= 256 and usage[name]["REG"] <= 128, (name, usage[name])
    assert usage[CROWD_KERNELS[0]]["STACK"] == 0
