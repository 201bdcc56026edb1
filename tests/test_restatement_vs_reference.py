"""oracle/torch_restatement.py against outputs of the REAL reference functions, stored under tests/golden/ by
oracle/make_golden.py (same seeded inputs, torch CPU).  This is the link that lets the gpu tests use the restatement as
"the reference on the same device"."""
import numpy as np
import pytest
import torch

from oracle import golden_cases as gc
from oracle import ref_loader
from oracle import torch_restatement as tr


@pytest.mark.parametrize("name", sorted(gc.GEOMETRIES))
def test_offsets_scales_anchors(name):
    g = gc.GEOMETRIES[name]
    levels = gc.geom_levels(g)
    gold = gc.load("geom_" + name)
    off_t, sc_t = tr.offsets_and_scales(levels, "cpu")
    assert torch.equal(off_t, torch.from_numpy(gold["offsets"])) and torch.equal(sc_t, torch.from_numpy(gold["scales"]))
    assert torch.equal(tr.anchors_px(levels, g["width"], g["height"], "cpu"), torch.from_numpy(gold["anchors"]))


@pytest.mark.parametrize("name", sorted(gc.ASSIGN_CASES))
@pytest.mark.parametrize("relative", [True, False])
def test_match_one_is_the_reference_bbox_matching(name, relative):
    """tr.match_one == ObjectDetection.bbox_matching (ref :252-284) in the stored form: positives (flat index, value,
    assignment) bit-equal, and the number of anchors the raw output assigns per image."""
    case = gc.ASSIGN_CASES[name]
    gold, tag = gc.load(name), "rel" if relative else "abs"
    anchors = torch.from_numpy(gc.load("geom_" + case["geom"])["anchors"])
    flat, vals, asg, n_valid_raw = [], [], [], []
    for b, (bx, _) in enumerate(gc.case_gt(case).per_image()):
        a, v = tr.match_one(anchors, torch.from_numpy(bx), 9, relative)
        a, v = a.numpy(), v.numpy()
        n_valid_raw.append(int((a >= 0).sum()))
        pos = np.nonzero(v > 0)[0]
        flat.append(pos + b * len(a)); vals.append(v[pos]); asg.append(a[pos])
    np.testing.assert_array_equal(np.concatenate(flat), gold[f"{tag}_pos_flat"])
    np.testing.assert_array_equal(np.concatenate(vals), gold[f"{tag}_pos_val"])
    np.testing.assert_array_equal(np.concatenate(asg), gold[f"{tag}_pos_assign"])
    np.testing.assert_array_equal(n_valid_raw, gold[f"{tag}_n_valid_raw"])


@pytest.mark.parametrize("name", ["train_cfg0", "train_test128", "train_cfg1", "train_empty"])
def test_train_losses_equal_the_reference_training_step(name):
    case = gc.TRAIN_CASES[name]
    g = gc.GEOMETRIES[case["geom"]]
    levels = gc.geom_levels(g)
    gold = gc.load(name)
    gt, maps = gc.case_gt(case), gc.train_maps(case)
    boxes = [torch.from_numpy(b) for b, _ in gt.per_image()]
    classes = [torch.from_numpy(c) for _, c in gt.per_image()]
    t = torch.from_numpy
    loss, metrics, _, _ = tr.train_losses(levels, g["width"], g["height"], boxes, classes, t(maps.loc_logits),
                                          t(maps.iou_preds), t(maps.box_raw), t(maps.cls_logits))
    for key in ("location_loss", "box_loss", "class_loss", "iou_loss"):
        want = float(gold[key])
        got = float(metrics[key])
        assert got == want or (got != got and want != want) or abs(got - want) <= 1e-6 * abs(want), (key, got, want)
    want = float(gold["loss"])
    assert float(loss) == want or abs(float(loss) - want) <= 1e-6 * abs(want) or (want != want)


@pytest.mark.parametrize("name", sorted(gc.FORWARD_CASES))
def test_forward_tail_equals_the_reference_forward(name):
    case = gc.FORWARD_CASES[name]
    g = gc.GEOMETRIES[case["geom"]]
    levels = gc.geom_levels(g)
    gold = gc.load(name)
    maps = gc.forward_maps(case)
    t = torch.from_numpy
    num, scores, cls, boxes, idx = tr.forward_tail(levels, g["width"], g["height"], t(maps.loc_logits), t(maps.box_raw),
                                                   t(maps.cls_logits), case["k"])
    assert torch.equal(num, t(gold["num_instances"])) and torch.equal(cls, t(gold["classes"]).long())
    assert torch.equal(scores, t(gold["scores"])) and torch.equal(boxes, t(gold["boxes"]))
    assert torch.equal(idx, t(gold["idx"]).long())


@pytest.mark.parametrize("name", sorted(gc.QUAD_CASES))
def test_quad_match_one_is_the_reference_quad_bbox_matching(name):
    """N1: tr.quad_match_one == QuadrilateralDetection.bbox_matching (ref quadrilateral_detection.py:266-294) in the
    stored canonical form, bit-equal, and the sihl_b200 anchor helper == the reference's inline anchor construction
    (ref :156-161)."""
    case, gold = gc.QUAD_CASES[name], gc.load(name)
    anchors = torch.from_numpy(gold["anchors"])
    for b, (bx, _) in enumerate(gc.quad_gt(case).per_image()):
        t = torch.from_numpy(bx).reshape(-1, 4)
        got = tr.quad_canonical(*tr.quad_match_one(anchors, t, int(gold["topk"])))
        for key, g in zip(("assignment", "o2o", "iou", "rel"), got):
            np.testing.assert_array_equal(g.numpy(), gold[key][b], err_msg=key)
    from sihl_b200.heads.quadrilateral_detection import quad_anchors
    sizes = [tuple(int(v) for v in s) for s in gold["level_sizes"]]
    mine = quad_anchors(sizes, range(case["bottom"], case["top"] + 1), case["top"], case["width"], case["height"], "cpu")
    assert torch.equal(mine, anchors)


@pytest.mark.skipif(not ref_loader.available(), reason="needs the reference's source (SIHL_REFERENCE_ROOT); no stored outputs")
def test_quads_to_boxes_equals_the_reference():
    """sihl_b200.heads.quadrilateral_detection.quads_to_boxes == QuadrilateralDetection.quads_to_boxes (ref :318-324)."""
    from sihl_b200.heads.quadrilateral_detection import quads_to_boxes
    Q = ref_loader.QuadrilateralDetection()
    g = torch.Generator().manual_seed(3)
    quads = torch.rand((17, 4, 2), generator=g) * 300
    assert torch.equal(quads_to_boxes(quads), Q.quads_to_boxes(quads))
    assert quads_to_boxes(quads[:0]).shape == (0, 4)
