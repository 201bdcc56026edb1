"""GPU parity tests proper: every kernel is called through the C ABI (sihl_b200.ops ->
libsihl_b200.so) and compared with

  * the committed golden fixtures (outputs of the unmodified reference, CPU torch),
  * the CPU oracle (oracle/od_oracle.c) on the same seeded inputs,
  * oracle/torch_restatement.py run on cuda:0 — the reference's computation with the
    reference's own torch/torchvision operators on the same device, where bit equality is
    well defined (SURVEY.md §7.1).

Contract (BASELINE.json north_star): assignment indices / keep lists / top-k indices exact;
decoded boxes and losses within 1e-5 relative in fp32.
"""
import numpy as np
import pytest
import torch

from oracle import golden_cases as gc
from oracle import od_oracle as orc
from oracle import torch_restatement as tr
from sihl_b200 import _native, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _geom(name):
    g = gc.load("geom_" + name)
    return g, [tuple(int(v) for v in x) for x in g["levels"]], int(g["img_wh"][0]), int(g["img_wh"][1])


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


def _gt_dev(gt: synth.GtBatch) -> ops.GtBatch:
    counts = [int(gt.offsets[i + 1] - gt.offsets[i]) for i in range(gt.batch_size)]
    return ops.GtBatch(_t(gt.boxes).reshape(-1, 4), _t(gt.classes), _t(gt.offsets), counts)


def _assign(anchors, levels, W, H, gt, relative=True, brute=False):
    sel = ops.assign_select(anchors, None if brute else levels, W, H, gt, 9)
    out = ops.assign_resolve(sel, gt, anchors.shape[0], 9, relative)
    return out["assignment"], out["iou"], sel


# --------------------------------------------------------------------------- a1/a2
@pytest.mark.parametrize("name", sorted(gc.GEOMETRIES))
def test_anchor_tables(name):
    g, levels, W, H = _geom(name)
    off, sc, an = ops.anchor_tables(levels, W, H, DEV, cache=False)
    # same device, same operators as the reference: bit equality
    off_t, sc_t = tr.offsets_and_scales(levels, DEV)
    an_t = (off_t + sc_t) * tr.full_size(W, H, DEV)
    assert torch.equal(off, off_t) and torch.equal(sc, sc_t) and torch.equal(an, an_t)
    # reference run on CPU (golden): linspace differs in the last bit across devices
    np.testing.assert_allclose(off.cpu().numpy(), g["offsets"], rtol=1e-6)
    np.testing.assert_array_equal(sc.cpu().numpy(), g["scales"])
    np.testing.assert_allclose(an.cpu().numpy(), g["anchors"], rtol=1e-6, atol=1e-4)


# --------------------------------------------------------------------------- a3/a4
def _dense(flat, vals, n, dtype, fill):
    out = np.full(n, fill, dtype)
    out[flat] = vals
    return out


@pytest.mark.parametrize("name", sorted(gc.ASSIGN_CASES))
@pytest.mark.parametrize("relative", [True, False])
def test_assign_vs_golden_and_oracle(name, relative):
    case = gc.ASSIGN_CASES[name]
    g, levels, W, H = _geom(case["geom"])
    gold = gc.load(name)
    gt_np = gc.case_gt(case)
    gt = _gt_dev(gt_np)
    anchors = _t(g["anchors"])            # the reference's own table: isolates the assignment arithmetic
    tag = "rel" if relative else "abs"
    B, A = gt.batch_size, anchors.shape[0]
    want_v = _dense(gold[f"{tag}_pos_flat"], gold[f"{tag}_pos_val"], B * A, np.float32, 0).reshape(B, A)
    want_a = _dense(gold[f"{tag}_pos_flat"], gold[f"{tag}_pos_assign"], B * A, np.int64, -1).reshape(B, A)
    for brute in (False, True):
        a, v, _ = _assign(anchors, levels, W, H, gt, relative, brute)
        a, v = a.cpu().numpy(), v.cpu().numpy()
        orc_a, orc_v, _ = orc.assign_batch(g["anchors"], gt_np.boxes, gt_np.offsets, 9, relative)
        if case.get("integer_coords"):
            # lattice ties: torch.topk's winner is implementation-defined; ours is the oracle's rule
            np.testing.assert_array_equal(a, orc_a)
            np.testing.assert_allclose(v, orc_v, rtol=1e-5, atol=1e-7)
            continue
        np.testing.assert_array_equal(v > 0, want_v > 0)
        if relative:
            np.testing.assert_array_equal(v == 1, want_v == 1)
        np.testing.assert_array_equal(a, want_a)
        np.testing.assert_allclose(v, want_v, rtol=1e-5, atol=1e-7)
        np.testing.assert_array_equal(a, orc_a)
        np.testing.assert_allclose(v, orc_v, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", ["assign_cfg0", "assign_test128", "assign_cfg1", "assign_nonsq", "assign_flipped"])
def test_assign_bit_exact_vs_torch_cuda(name):
    """The reference's operators on the same GPU: indices AND values bit-equal."""
    case = gc.ASSIGN_CASES[name]
    g, levels, W, H = _geom(case["geom"])
    gt_np = gc.case_gt(case)
    gt = _gt_dev(gt_np)
    off, sc, anchors = ops.anchor_tables(levels, W, H, DEV)
    for relative in (True, False):
        a, v, _ = _assign(anchors, levels, W, H, gt, relative)
        for b, (bx, _) in enumerate(gt_np.per_image()):
            ra, rv = tr.match_one(anchors, _t(bx).reshape(-1, 4), 9, relative)
            ra, rv = tr.canonical(ra, rv)
            assert torch.equal(a[b], ra), (name, relative, b)
            assert torch.equal(v[b], rv), (name, relative, b, (v[b] - rv).abs().max().item())


def test_bbox_matching_static_api():
    g, levels, W, H = _geom("cfg0_320")
    anchors = _t(g["anchors"])
    gt_np = gc.case_gt(gc.ASSIGN_CASES["assign_cfg0"])
    bx = _t(gt_np.boxes[:20])
    a, v = ops.bbox_matching(anchors, bx, 9, relative=True)
    ra, rv = tr.canonical(*tr.match_one(anchors, bx, 9, True))
    assert torch.equal(a, ra) and torch.equal(v, rv)
    a0, v0 = ops.bbox_matching(anchors, bx[:0], 9, relative=True)      # ref :258-261
    assert (a0 == -1).all() and (v0 == 0).all()


def test_assign_errors_mirror_reference():
    anchors = torch.rand((5, 4), device=DEV)
    gt = ops.GtBatch.from_lists([torch.tensor([[1.0, 1.0, 5.0, 5.0]])], None, DEV)
    with pytest.raises(ops._native.NativeError):           # torch.topk(k=9) over 5 anchors raises in the reference
        ops.assign_select(anchors, None, 0, 0, gt, 9)
    with pytest.raises(ops._native.NativeError):
        ops.assign_select(torch.rand((50, 4), device=DEV), None, 0, 0, gt, 0)
    with pytest.raises(RuntimeError):                      # no CPU path
        ops.assign_select(torch.rand((50, 4)), None, 0, 0, gt, 9)


# --------------------------------------------------------------------------- a5-a10
def _train_inputs(case):
    gt_np, maps = gc.case_gt(case), gc.train_maps(case)
    return gt_np, maps, [_t(m) for m in (maps.loc_logits, maps.iou_preds, maps.box_raw, maps.cls_logits)]


def _pipeline_losses(case, g, levels, W, H):
    """assign_select + assign_resolve with the fused dense and positive-row losses + loss_finalize, on the golden tables."""
    gt_np, maps, (loc, iou, box, cls) = _train_inputs(case)
    gt = _gt_dev(gt_np)
    A = maps.loc_logits.shape[1]
    off, sc, anchors = _t(g["offsets"]), _t(g["scales"]), _t(g["anchors"])
    sums = ops.new_sums(DEV)
    sums.fill_(123.0)                                  # select must zero it
    sel = ops.assign_select(anchors, levels, W, H, gt, 9, sums=sums)
    res = ops.assign_resolve(sel, gt, A, 9, True, loc, iou, sums,
                             fused=dict(box_raw=box, cls_logits=cls, offsets=off, scales=sc, img_w=W, img_h=H))
    losses = ops.loss_finalize(sums)
    # the per-tile positive lists, concatenated in tile order, are the compact positive index
    _, tile = ops.resolve_tiles(A)
    counts = res["tile_pos_count"].cpu().numpy()
    lists = res["tile_pos_rows"].cpu().numpy().reshape(-1, tile)
    pos_index = np.concatenate([np.zeros(0, np.int32)] + [lists[s, :n] for s, n in enumerate(counts)])
    return dict(tables=(g["anchors"], g["offsets"], g["scales"]), assignment=res["assignment"], pos_index=pos_index,
                sums=sums, losses=losses)


def _train_losses(case, levels, W, H):
    """train_assign + train_loss on the compact rows gathered by pos_index (what the drop-in head runs).  train_assign
    builds its own anchor tables on the device; they are returned for the oracle."""
    gt_np, maps, (loc, iou, box, cls) = _train_inputs(case)
    B, A = maps.loc_logits.shape
    st = ops.train_assign(levels, W, H, _t(gt_np.boxes).reshape(-1, 4), _t(gt_np.classes), np.diff(gt_np.offsets).tolist(),
                          B, 9)
    rows = st.pos_index.long()
    losses, maps_used = ops.train_loss(st, loc, iou, box.reshape(B * A, 4)[rows], cls.reshape(B * A, -1)[rows])
    P = int(st.pos_total.item())
    off, sc, anchors = ops.anchor_tables(levels, W, H, DEV)
    return dict(tables=(anchors.cpu().numpy(), off.cpu().numpy(), sc.cpu().numpy()), assignment=st.assignment,
                pos_index=st.pos_index[:P].cpu().numpy(), sums=st.sums, losses=losses, st=st, maps=maps_used)


@pytest.mark.parametrize("name", sorted(gc.TRAIN_CASES))
@pytest.mark.parametrize("path", ["pipeline", "train"])
def test_train_losses(name, path):
    case = gc.TRAIN_CASES[name]
    g, levels, W, H = _geom(case["geom"])
    gold = gc.load(name)
    r = _pipeline_losses(case, g, levels, W, H) if path == "pipeline" else _train_losses(case, levels, W, H)
    gt_np, maps = gc.case_gt(case), gc.train_maps(case)
    B, A = maps.loc_logits.shape
    anchors, off, sc = r["tables"]
    want = orc.train_losses(anchors, off, sc, W, H, gt_np.boxes, gt_np.classes, gt_np.offsets,
                            maps.loc_logits, maps.iou_preds, maps.box_raw, maps.cls_logits, dense_rows=True)
    np.testing.assert_array_equal(r["assignment"].cpu().numpy(), want["assignment"])
    pos_index = r["pos_index"]
    np.testing.assert_array_equal(pos_index, want["pos_index"])     # row order of flat_feats[o2m_mask]
    got_sums = r["sums"].cpu().numpy()
    np.testing.assert_allclose(got_sums[:7], want["sums"][:7], rtol=1e-5, atol=1e-9)
    assert got_sums[6] == len(pos_index)
    got = r["losses"].cpu().numpy()
    gold_l = [gold["location_loss"], gold["box_loss"], gold["class_loss"], gold["iou_loss"], gold["loss"]]
    for gv, wv, ov in zip(got, gold_l, want["losses"]):
        if np.isfinite(wv):
            assert gv == pytest.approx(float(wv), rel=1e-5)
            assert gv == pytest.approx(float(ov), rel=1e-5)
        else:
            assert not np.isfinite(gv)
    per_img = (want["rel_iou"] > 0).sum(1)
    np.testing.assert_array_equal(np.bincount(pos_index // A, minlength=B), per_img)


@pytest.mark.parametrize("name", ["train_cfg0", "train_test128", "train_cfg1"])
def test_loss_backward_vs_reference_autograd(name):
    case = gc.TRAIN_CASES[name]
    g, levels, W, H = _geom(case["geom"])
    gold = gc.load(name)
    if not np.isfinite(gold["loss"]) or "dloc" not in gold:
        pytest.skip("reference loss is not finite for this fixture (no anchor with rel==1)")
    r = _train_losses(case, levels, W, H)
    dloc, diou, dbox, dcls = (t.cpu().numpy() for t in ops.train_loss_bwd(r["st"], r["maps"], None))
    np.testing.assert_allclose(dloc.reshape(-1), gold["dloc"].reshape(-1), rtol=2e-5, atol=1e-9)
    # rel_iou of the CPU-run reference differs by ~1e-7 absolute (atan last bit); 2*(p-rel)/R inherits it
    np.testing.assert_allclose(diou.reshape(-1), gold["diou"].reshape(-1), rtol=2e-5, atol=2e-8)
    np.testing.assert_array_equal(r["pos_index"], gold["grad_rows"])
    P = len(r["pos_index"])
    np.testing.assert_allclose(dbox[:P], gold["dbox"], rtol=2e-4, atol=2e-7)
    np.testing.assert_allclose(dcls[:P], gold["dcls"], rtol=2e-5, atol=1e-9)
    np.testing.assert_array_equal(dbox[P:], 0)                       # padding rows: zero gradient (sihl_od.h)
    np.testing.assert_array_equal(dcls[P:], 0)


# --------------------------------------------------------------------------- a11
@pytest.mark.parametrize("name", sorted(gc.FORWARD_CASES))
def test_forward_tail(name):
    case = gc.FORWARD_CASES[name]
    g, levels, W, H = _geom(case["geom"])
    gold = gc.load(name)
    maps = gc.forward_maps(case)
    K = case["k"]
    loc, box, cls = _t(maps.loc_logits), _t(maps.box_raw), _t(maps.cls_logits)
    top, idx = ops.topk_locations(loc, K)
    np.testing.assert_array_equal(idx.cpu().numpy(), gold["idx"])
    want_top, want_idx = loc.topk(K, dim=1)
    assert torch.equal(top, want_top) and torch.equal(idx, want_idx)
    B = loc.shape[0]
    rows = torch.arange(B, device=DEV).view(B, 1)
    off, sc, _ = ops.anchor_tables(levels, W, H, DEV)
    num, scores, classes, boxes = ops.decode_rows(top, idx, cls[rows, idx].contiguous(), box[rows, idx].contiguous(), off, sc, W, H)
    np.testing.assert_array_equal(num.cpu().numpy(), gold["num_instances"])
    np.testing.assert_array_equal(classes.cpu().numpy(), gold["classes"])
    np.testing.assert_allclose(scores.cpu().numpy(), gold["scores"], rtol=1e-6)
    np.testing.assert_allclose(boxes.cpu().numpy(), gold["boxes"], rtol=1e-5, atol=1e-4)
    # same device, same operators: bit equality
    t_num, t_scores, t_cls, t_boxes, _ = tr.forward_tail(levels, W, H, loc, box, cls, K)
    assert torch.equal(num, t_num) and torch.equal(classes, t_cls)
    assert torch.equal(scores, t_scores)
    assert torch.equal(boxes, t_boxes)


def test_topk_ties_lowest_index_first():
    loc = torch.zeros((3, 500), device=DEV)
    loc[1, 100:400] = 1.0
    loc[2] = torch.arange(500, device=DEV).float().remainder(7)
    top, idx = ops.topk_locations(loc, 100)
    assert idx[0].tolist() == list(range(100))
    assert idx[1].tolist() == list(range(100, 200))
    want = sorted(range(500), key=lambda i: (-(i % 7), i))[:100]
    assert idx[2].tolist() == want


# --------------------------------------------------------------------------- a15 (extension)
@pytest.mark.parametrize("name", sorted(gc.NMS_CASES))
def test_batched_nms_vs_torchvision_golden(name):
    case = gc.NMS_CASES[name]
    boxes, scores, classes = gc.nms_inputs(case)
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), case["thr"]).cpu().numpy()
    want = gc.load(name)["keep"].astype(np.int64)
    order = np.lexsort((want, -scores[want].astype(np.float64)))     # torchvision's last sort is unstable on ties
    np.testing.assert_array_equal(keep, want[order])
    np.testing.assert_array_equal(keep, orc.batched_nms(boxes, scores, classes, case["thr"]))


def test_batched_nms_segments_and_crowd():
    """config[3]-style stress: many candidates per image, several images in one call (spills to the workspace)."""
    sizes = [0, 1, 30, 5000, 12000]
    parts = [synth.nms_candidates_np(900 + i, n, 1024, 80) for i, n in enumerate(sizes)]
    boxes = np.concatenate([p[0] for p in parts]); scores = np.concatenate([p[1] for p in parts])
    classes = np.concatenate([p[2] for p in parts])
    seg = np.zeros(len(sizes) + 1, np.int32); seg[1:] = np.cumsum(sizes)
    keep, count = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5, seg_offsets=_t(seg))
    keep, count = keep.cpu().numpy(), count.cpu().numpy()
    for i, n in enumerate(sizes):
        s, e = seg[i], seg[i + 1]
        want = orc.batched_nms(boxes[s:e], scores[s:e], classes[s:e], 0.5) + s
        assert count[i] == len(want)
        np.testing.assert_array_equal(keep[s:s + count[i]], want)


def test_nms_idempotent_and_one_class():
    boxes, scores, classes = synth.nms_candidates_np(77, 6000, 640, 1)      # one class: the CTA-wide sweep
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5)
    np.testing.assert_array_equal(keep.cpu().numpy(), orc.batched_nms(boxes, scores, classes, 0.5))
    k = keep.cpu().numpy()
    again = ops.batched_nms(_t(boxes[k]), _t(scores[k]), _t(classes[k]), 0.5)
    assert again.cpu().numpy().tolist() == list(range(len(k)))              # survivors suppress nothing


@pytest.mark.parametrize("geom,C,B,loc_mean,loc_std", [("test_128", 16, 5, -2.0, 2.0), ("cfg0_320", 10, 3, -2.0, 2.0),
                                                        ("cfg1_640", 80, 4, -5.0, 1.0), ("cfg1_640", 80, 2, -4.0, 2.0)])
@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("mode", ops.DECODE_MODES)
def test_dense_postprocess(geom, C, B, loc_mean, loc_std, mode, split):
    g, levels, W, H = _geom(geom)
    A = len(g["anchors"])
    maps = synth.dense_maps_np(4242, B, A, C, loc_mean, loc_std)
    loc, box, cls = _t(maps.loc_logits), _t(maps.box_raw), _t(maps.cls_logits)
    num, scores, classes, boxes = ops.dense_postprocess(loc, cls, box, levels, W, H, 0.05, 0.5, 100, mode=mode, split_nms=split)
    o_num, o_scores, o_cls, o_boxes, ncand = orc.dense_postprocess(maps.loc_logits, maps.cls_logits, maps.box_raw,
                                                                    g["offsets"], g["scales"], W, H, 0.05, 0.5, 100)
    np.testing.assert_array_equal(num.cpu().numpy(), o_num)
    np.testing.assert_array_equal(classes.cpu().numpy(), o_cls)
    np.testing.assert_allclose(scores.cpu().numpy(), o_scores, rtol=1e-6)
    np.testing.assert_allclose(boxes.cpu().numpy(), o_boxes, rtol=1e-5, atol=1e-4)
    t_num, t_scores, t_cls, t_boxes = tr.dense_postprocess(levels, W, H, loc, box, cls, 0.05, 0.5, 100)
    assert torch.equal(num, t_num) and torch.equal(classes, t_cls)
    assert torch.equal(scores, t_scores) and torch.equal(boxes, t_boxes)


def _candidate_sets(cand: ops.CandidateBuffers, B):
    n = cand.count.cpu().numpy()
    key, box, cls = cand.key.cpu().numpy(), cand.box.cpu().numpy(), cand.cls.cpu().numpy()
    out = []
    for b in range(B):
        order = np.argsort(key[b, :n[b]].view(np.uint64))
        out.append((key[b, :n[b]][order], box[b, :n[b]][order], cls[b, :n[b]][order]))
    return n, out


@pytest.mark.parametrize("C,thr,loc_mean", [(80, 0.05, -5.0), (80, 0.05, -1.0), (10, 0.3, 0.0), (7, 0.05, -2.0), (3, 0.0, 0.0),
                                            (132, 0.05, -2.0), (80, 1.0, 0.0)])
def test_candidate_first_lists_equal_dense_lists(C, thr, loc_mean):
    """Both decode variants fill the same candidate lists (as sets: slot order comes from atomics) — every class count
    path (16-byte rows, scalar rows, C > 128), duplicated row maxima (first index wins), thresholds 0 and 1."""
    levels = synth.level_sizes(256, 320)
    W, H, B = 320, 256, 3
    off, sc, anchors = ops.anchor_tables(levels, W, H, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(99 + C, B, A, C, loc_mean, 2.0)
    cls_np = maps.cls_logits.copy()
    cls_np[:, ::3, C // 2] = cls_np[:, ::3].max(axis=-1)                  # exact ties between two classes on every third row
    cls_np[0, 5] = -np.inf                                                # all -inf row: class 0
    loc, box, cls = _t(maps.loc_logits), _t(maps.box_raw), _t(cls_np)
    lists = {}
    for mode in ops.DECODE_MODES:
        cand = ops.CandidateBuffers.allocate(B, A, DEV)
        ops.dense_decode(loc, cls, box, off, sc, W, H, thr, cand, mode=mode)
        lists[mode] = _candidate_sets(cand, B)
    n_d, l_d = lists["dense"]
    n_c, l_c = lists["candidate_first"]
    np.testing.assert_array_equal(n_d, n_c)
    want_n = (torch.sigmoid(loc) > thr).sum(dim=1).cpu().numpy()
    np.testing.assert_array_equal(n_c, want_n)
    for b in range(B):
        for x, y in zip(l_d[b], l_c[b]):
            np.testing.assert_array_equal(x, y)
        rows = (0xFFFFFFFF - (l_c[b][0].view(np.uint64) & np.uint64(0xFFFFFFFF))).astype(np.int64)
        first_max = np.argmax(cls_np[b, rows], axis=-1)                   # numpy argmax: first maximum
        np.testing.assert_array_equal(l_c[b][2], first_max)


# --------------------------------------------------------------------------- full size (config[1]) properties
def test_full_size_properties():
    """B=64, A=8525, G=100, C=80: size-independent properties + oracle spot checks."""
    levels = synth.level_sizes(640, 640)
    W = H = 640
    B, G, C = 64, 100, 80
    off, sc, anchors = ops.anchor_tables(levels, W, H, DEV)
    A = anchors.shape[0]
    gt_np = synth.gt_batch_np(2024, B, H, W, C, G, ragged=False)
    gt = _gt_dev(gt_np)
    a1, v1, sel1 = _assign(anchors, levels, W, H, gt, True, brute=False)
    a2, v2, sel2 = _assign(anchors, levels, W, H, gt, True, brute=True)
    assert torch.equal(a1, a2) and torch.equal(v1, v2)                       # pruning never changes the result
    for s1, s2 in zip(sel1, sel2):
        assert torch.equal(s1, s2)
    assert ((v1 > 0) == (a1 >= 0)).all() and (v1 <= 1).all() and (v1 >= 0).all()
    per_gt = torch.zeros(B * G, device=DEV)
    flat_g = (a1 + torch.arange(B, device=DEV).view(B, 1) * G)[a1 >= 0]
    per_gt.index_add_(0, flat_g, torch.ones_like(flat_g, dtype=torch.float32))
    assert per_gt.max() <= 9                                                 # at most top-k anchors per gt
    an_np = anchors.cpu().numpy()
    for b in (0, 17, 63):
        oa, ov, _ = orc.bbox_matching(an_np, gt_np.boxes[b * G:(b + 1) * G], 9, True)
        np.testing.assert_array_equal(a1[b].cpu().numpy(), oa)
        np.testing.assert_allclose(v1[b].cpu().numpy(), ov, rtol=1e-5, atol=1e-7)


# --------------------------------------------------------------------------- configs[3] / configs[4]
def test_crowd_config_assign_parity():
    """configs[3]: 1024x1024, 500 gt / image — pruned select == all-pairs select == C oracle."""
    W = H = 1024
    levels = synth.level_sizes(H, W)
    off, sc, anchors = ops.anchor_tables(levels, W, H, DEV)
    assert anchors.shape[0] == 21824
    gt_np = synth.gt_batch_np(31, 3, H, W, 80, 500, counts=[500, 0, 377])
    gt = _gt_dev(gt_np)
    a1, v1, s1 = _assign(anchors, levels, W, H, gt, True, brute=False)
    a2, v2, s2 = _assign(anchors, levels, W, H, gt, True, brute=True)
    assert torch.equal(a1, a2) and torch.equal(v1, v2) and all(torch.equal(x, y) for x, y in zip(s1, s2))
    oa, ov, _ = orc.assign_batch(anchors.cpu().numpy(), gt_np.boxes, gt_np.offsets, 9, True)
    np.testing.assert_array_equal(a1.cpu().numpy(), oa)
    np.testing.assert_allclose(v1.cpu().numpy(), ov, rtol=1e-5, atol=1e-7)
    for b, (bx, _) in enumerate(gt_np.per_image()):
        ra, rv = tr.canonical(*tr.match_one(anchors, _t(bx).reshape(-1, 4), 9, True))
        assert torch.equal(a1[b], ra) and torch.equal(v1[b], rv)


def test_crowd_config_nms_30k_candidates():
    """configs[3]: NMS over 30 000 pre-NMS candidates of one image, 80 classes (workspace path)."""
    boxes, scores, classes = synth.nms_candidates_np(555, 30000, 1024, 80)
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5).cpu().numpy()
    np.testing.assert_array_equal(keep, orc.batched_nms(boxes, scores, classes, 0.5))


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("mode", ops.DECODE_MODES)
@pytest.mark.parametrize("size,batch", [(640, 3), (1280, 2)])
def test_inference_sweep_postprocess(size, batch, mode, split):
    """configs[4]: decode + NMS at 640-1280 px with loc ~ N(-4, 2^2) (about 30 % of the locations pass 0.05)."""
    levels = synth.level_sizes(size, size)
    off, sc, an = orc.anchors(levels, size, size)
    A, C = len(an), 80
    maps = synth.dense_maps_np(900 + size, batch, A, C, loc_mean=-4.0, loc_std=2.0)
    loc, box, cls = _t(maps.loc_logits), _t(maps.box_raw), _t(maps.cls_logits)
    num, scores, classes, boxes = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, 100, mode=mode,
                                                        split_nms=split)
    o_num, o_scores, o_cls, o_boxes, ncand = orc.dense_postprocess(maps.loc_logits, maps.cls_logits, maps.box_raw, off, sc,
                                                                    size, size, 0.05, 0.5, 100)
    assert ncand.min() > 0.2 * A
    np.testing.assert_array_equal(num.cpu().numpy(), o_num)
    np.testing.assert_array_equal(classes.cpu().numpy(), o_cls)
    np.testing.assert_allclose(scores.cpu().numpy(), o_scores, rtol=1e-6)
    np.testing.assert_allclose(boxes.cpu().numpy(), o_boxes, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("mode", ops.DECODE_MODES)
def test_pipeline_matches_unfused_ops_and_is_replayable(mode):
    """The bench pipeline (graphs, two streams, fused finalize, counter recycling) gives the same numbers as the
    step-by-step ops, and the same numbers again on every replay."""
    from sihl_b200.pipeline import DetectionHeadPipeline, StepInputs
    W = H = 320
    B, C, G = 4, 80, 30
    levels = synth.level_sizes(H, W)
    pipe = DetectionHeadPipeline(levels, W, H, B, C, B * G, DEV, decode_mode=mode)
    gt_np = synth.gt_batch_np(12, B, H, W, C, G, ragged=False)
    maps = synth.dense_maps_np(13, B, pipe.A, C, loc_mean=-3.0, loc_std=2.0)
    gt = _gt_dev(gt_np)
    x = StepInputs(_t(maps.loc_logits), _t(maps.iou_preds), _t(maps.box_raw), _t(maps.cls_logits), gt)
    out = pipe.new_outputs()
    graph = pipe.capture(x, out)
    results = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        results.append([t.clone() for t in (out.losses, out.assignment, out.rel_iou, out.num_instances, out.scores, out.classes, out.boxes)])
    for r in results[1:]:
        assert all(torch.equal(a, b) for a, b in zip(results[0][1:], r[1:]))           # everything but the float sums is deterministic
        torch.testing.assert_close(results[0][0], r[0], rtol=1e-6, atol=0)
    off, sc, an = orc.anchors(levels, W, H)
    want = orc.train_losses(an, off, sc, W, H, gt_np.boxes, gt_np.classes, gt_np.offsets, maps.loc_logits, maps.iou_preds,
                            maps.box_raw, maps.cls_logits, dense_rows=True)
    np.testing.assert_array_equal(results[0][1].cpu().numpy(), want["assignment"])
    np.testing.assert_allclose(results[0][0].cpu().numpy(), want["losses"], rtol=1e-5)
    o_num, o_scores, o_cls, o_boxes, _ = orc.dense_postprocess(maps.loc_logits, maps.cls_logits, maps.box_raw, off, sc, W, H, 0.05, 0.5, 100)
    np.testing.assert_array_equal(results[0][3].cpu().numpy(), o_num)
    np.testing.assert_array_equal(results[0][5].cpu().numpy(), o_cls)
    np.testing.assert_allclose(results[0][6].cpu().numpy(), o_boxes, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("dtype,C", [(torch.float32, 80), (torch.bfloat16, 80), (torch.float16, 24), (torch.float32, 132),
                                     (torch.float32, 7)])
def test_pipeline_reads_pinned_host_maps_in_place(dtype, C):
    """candidate-first pipeline with the class / box maps left in pinned host memory (the kernels gather the rows of the
    positives and of the candidates over PCIe): bit-identical to the run on device-resident maps.  The class counts cover
    the whole-row-per-warp reads (rows of at most 32 16-byte vectors: 80 fp32 / bf16, 24 fp16), the 8-lane reads (132 fp32 =
    33 vectors) and the element reads (7)."""
    from sihl_b200.pipeline import DetectionHeadPipeline, StepInputs
    W = H = 320
    B, G = 3, 25
    levels = synth.level_sizes(H, W)
    pipe = DetectionHeadPipeline(levels, W, H, B, C, B * G, DEV, decode_mode="candidate_first")
    gt = _gt_dev(synth.gt_batch_np(21, B, H, W, C, G, ragged=True))
    maps = synth.dense_maps_np(22, B, pipe.A, C, loc_mean=-3.0, loc_std=2.0)
    loc, iou = _t(maps.loc_logits).to(dtype), _t(maps.iou_preds).to(dtype)
    outs = []
    for on_host in (False, True):
        box = torch.from_numpy(maps.box_raw).to(dtype).pin_memory() if on_host else _t(maps.box_raw).to(dtype)
        cls = torch.from_numpy(maps.cls_logits).to(dtype).pin_memory() if on_host else _t(maps.cls_logits).to(dtype)
        out = pipe.new_outputs()
        pipe.step(StepInputs(loc, iou, box, cls, gt), out)
        torch.cuda.synchronize()
        outs.append(out)
    a, b = outs
    for name in ("assignment", "rel_iou", "num_instances", "scores", "classes", "boxes"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    torch.testing.assert_close(a.losses, b.losses, rtol=3e-6, atol=0)     # the row sums associate differently per lane layout
    if dtype != torch.float32 or C != 80:
        return
    with pytest.raises(RuntimeError, match="CUDA tensors only"):          # the dense scan streams everything: device only
        ops.dense_decode(loc, torch.from_numpy(maps.cls_logits).pin_memory(), _t(maps.box_raw), pipe.offsets, pipe.scales,
                         W, H, 0.05, pipe.cand, mode="dense")


def test_c_entries_refuse_pageable_host_maps():
    """A C-ABI caller that hands a PAGEABLE host pointer for the class / box map gets EINVAL from the entry, not a faulting
    kernel (the Python layer already refuses unpinned host tensors; device and pinned pointers keep working, see above)."""
    from sihl_b200 import _native
    lib = _native.load()
    W = H = 320
    B, C = 2, 80
    levels = synth.level_sizes(H, W)
    off, sc, _ = ops.anchor_tables(levels, W, H, DEV)
    A = int(off.shape[0])
    maps = synth.dense_maps_np(5, B, A, C, loc_mean=-3.0, loc_std=2.0)
    loc, box = _t(maps.loc_logits), _t(maps.box_raw)
    cls_pageable = np.ascontiguousarray(maps.cls_logits)              # plain numpy memory: neither device nor pinned
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    st = torch.cuda.current_stream().cuda_stream
    rc = lib.sihl_od_candidate_decode_t(loc.data_ptr(), cls_pageable.ctypes.data, box.data_ptr(), ops.DTYPE_CODES[torch.float32],
                                        B, A, C, off.data_ptr(), sc.data_ptr(), W, H, 0.05, cand.count.data_ptr(), cand.capacity,
                                        cand.key.data_ptr(), cand.box.data_ptr(), cand.cls.data_ptr(), 1, st)
    with pytest.raises(_native.NativeError, match="PINNED host memory"):
        _native.check(rc, "sihl_od_candidate_decode_t")
    torch.cuda.synchronize()                                           # nothing was launched on bad memory: the context is alive
    assert float(loc.sum().item()) == float(torch.from_numpy(maps.loc_logits).to(DEV).sum().item())


# --------------------------------------------------------------------------- N1: QuadrilateralDetection.bbox_matching
def _quad_check_vs_restatement(anchors_dev, boxes_np_list, topk=9):
    from sihl_b200.heads import quadrilateral_detection as qd
    boxes = [_t(b).reshape(-1, 4) for b in boxes_np_list]
    a, o, i, r = qd.batched_bbox_matching(anchors_dev, boxes, topk)
    for b, bx in enumerate(boxes):
        ra, ro, ri, rr = tr.quad_canonical(*tr.quad_match_one(anchors_dev, bx, topk))     # the reference's operators on this GPU
        assert torch.equal(a[b], ra), b
        assert torch.equal(o[b], ro), b
        assert torch.equal(i[b], ri) and torch.equal(r[b], rr), b                           # bit-exact values
    return a, o, i, r


@pytest.mark.parametrize("name", sorted(gc.QUAD_CASES))
def test_quad_matching(name):
    """Un-clamped four-output assignment (ref quadrilateral_detection.py:266-294) vs the golden outputs of the reference
    (CPU), the C oracle, and the reference's operator sequence on the same GPU (bit-exact)."""
    case, g = gc.QUAD_CASES[name], gc.load(name)
    gt = gc.quad_gt(case)
    anchors = _t(g["anchors"])
    per_image = [bx for bx, _ in gt.per_image()]
    a, o, i, r = _quad_check_vs_restatement(anchors, per_image, int(g["topk"]))
    np.testing.assert_array_equal(a.cpu().numpy(), g["assignment"])
    np.testing.assert_array_equal(o.cpu().numpy(), g["o2o"])
    np.testing.assert_allclose(i.cpu().numpy(), g["iou"], rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose(r.cpu().numpy(), g["rel"], rtol=1e-5, atol=1e-7)
    for b, bx in enumerate(per_image):
        oa, oo, oi, orr = orc.quad_matching(g["anchors"], bx, int(g["topk"]))
        np.testing.assert_array_equal(a[b].cpu().numpy(), oa)
        np.testing.assert_array_equal(o[b].cpu().numpy(), oo)
        np.testing.assert_allclose(i[b].cpu().numpy(), oi, rtol=1e-5, atol=1e-7)


def test_quad_matching_corner_cases_and_full_size():
    from sihl_b200.heads import quadrilateral_detection as qd
    # (i) one distant gt: every candidate is negative, its 9 selections get rel = v / best >= 1 (the reference's rule)
    sizes = [(16, 16), (8, 8), (4, 4)]
    anchors = qd.quad_anchors(sizes, range(3, 6), 5, 128, 128, DEV)
    far = np.array([[900.0, 900.0, 903.0, 904.0]], np.float32)
    a, o, i, r = _quad_check_vs_restatement(anchors, [far])
    assert int((r > 0).sum()) == 9 and bool((i[r > 0] < 0).all()) and int(o.sum()) == 1 and float(r.max()) > 1
    # (ii) A == topk: every gt selects every anchor, no zero entry takes part in the max
    few = anchors[:9].contiguous()
    gts = np.array([[200, 200, 204, 203], [2, 2, 38, 41], [60, 60, 100, 90]], np.float32)
    _quad_check_vs_restatement(few, [gts, gts[:1], gts[:0]])
    with pytest.raises(ops._native.NativeError, match="selected index k out of range"):
        qd.bbox_matching(anchors[:5].contiguous(), _t(gts), 9)
    # (iii) config[1]-sized: 640^2, levels 3..7 (A = 8525 anchors), 64 images x <= 100 gts; spot-check images vs the restatement
    levels = synth.level_sizes(640, 640)
    big = qd.quad_anchors(levels, range(3, 8), 7, 640, 640, DEV)
    gt_np = synth.gt_batch_np(77, 64, 640, 640, 80, 100, ragged=True)
    per_image = [bx for bx, _ in gt_np.per_image()]
    a, o, i, r = qd.batched_bbox_matching(big, [_t(b).reshape(-1, 4) for b in per_image], 9)
    assert a.shape == (64, 8525) and ((r > 0) == (a >= 0)).all()
    counts = torch.tensor([len(b) for b in per_image], device=DEV)
    assert torch.equal(o.sum(dim=1), torch.minimum(counts, o.sum(dim=1))) and (o.sum(dim=1) <= counts).all()
    for b in (0, 31, 63):
        ra, ro, ri, rr = tr.quad_canonical(*tr.quad_match_one(big, _t(per_image[b]).reshape(-1, 4), 9))
        assert torch.equal(a[b], ra) and torch.equal(o[b], ro) and torch.equal(i[b], ri) and torch.equal(r[b], rr)


def test_fused_loss_sum_exchange_against_a_scripted_peer():
    """The in-kernel all-reduce of the 8 loss sums (sihl_od_pos_loss_tiles_exchange, world = 2) on ONE GPU: the peer's
    pushes are written into this rank's region from the host before each launch, so no kernel ever waits on another
    kernel.  Checks the sums / losses of two consecutive steps (both parities), what this rank pushed to the peer, and
    that a peer that never shows up ends in NaN after the bounded wait instead of hanging."""
    from sihl_b200 import dist as sdist
    from sihl_b200.pipeline import DetectionHeadPipeline, StepInputs
    W = H = 256
    B, C, G, world = 2, 16, 12, 2
    levels = synth.level_sizes(H, W)
    pipe = DetectionHeadPipeline(levels, W, H, B, C, B * G, DEV)
    gt = _gt_dev(synth.gt_batch_np(31, B, H, W, C, G, ragged=False))
    maps = synth.dense_maps_np(32, B, pipe.A, C)
    x = StepInputs(_t(maps.loc_logits), _t(maps.iou_preds), _t(maps.box_raw), _t(maps.cls_logits), gt)
    plain = pipe.new_outputs()
    pipe.train_chain(x, plain)
    torch.cuda.synchronize()
    local = plain.sums.clone()

    words = 18 * world + 3
    assert words * 8 <= _native.load().sihl_od_exchange_region_bytes(world)
    mine = torch.zeros(words, dtype=torch.float64, device=DEV)        # rank 0's region (this GPU)
    theirs = torch.zeros(words, dtype=torch.float64, device=DEV)      # stands in for rank 1's region
    table = torch.tensor([mine.data_ptr(), theirs.data_ptr()], dtype=torch.int64, device=DEV)
    pipe._exchange = (table.data_ptr(), world, 0)
    out = pipe.new_outputs()
    for step in (1, 2, 3):
        parity = step & 1
        fake = torch.arange(8, dtype=torch.float64, device=DEV) * 0.5 + step
        fake[7] = 0.0
        mine[(parity * world + 1) * 8:(parity * world + 1) * 8 + 8] = fake          # the peer's push ...
        mine.view(torch.int64)[16 * world + parity * world + 1] = step              # ... and its release flag
        torch.cuda.synchronize()
        pipe.train_chain(x, out)
        torch.cuda.synchronize()
        want = local + fake
        torch.testing.assert_close(out.sums[:7], want[:7], rtol=1e-12, atol=0)
        torch.testing.assert_close(out.losses.double(), sdist.losses_from_sums(want), rtol=1e-6, atol=0)
        pushed = theirs[(parity * world + 0) * 8:(parity * world + 0) * 8 + 7]
        torch.testing.assert_close(pushed, local[:7], rtol=1e-12, atol=0)           # what the peer would have received
        assert int(theirs.view(torch.int64)[16 * world + parity * world + 0]) == step
        assert int(mine.view(torch.int64)[18 * world]) == step                      # own step counter
    import ctypes as C
    import time
    lib = _native.load()
    bad, done = C.c_uint64(7), C.c_uint64(0)
    _native.check(lib.sihl_od_exchange_status(mine.data_ptr(), world, C.byref(bad), C.byref(done)), "status")
    assert bad.value == 0 and done.value == 3                                       # nothing timed out so far
    _native.check(lib.sihl_od_exchange_set_timeout(mine.data_ptr(), world, int(2e9)), "set_timeout")   # default: 120 s
    t0 = time.perf_counter()
    pipe.train_chain(x, out)                                                        # step 4: the peer never arrives
    torch.cuda.synchronize()
    assert 1.5 < time.perf_counter() - t0 < 10.0
    assert torch.isnan(out.losses).all()
    _native.check(lib.sihl_od_exchange_status(mine.data_ptr(), world, C.byref(bad), C.byref(done)), "status")
    assert bad.value == 4 and done.value == 4                                       # the host can see WHICH step gave up


@pytest.mark.parametrize("C,K,loc_mean", [(80, 100, -4.0), (1, 100, -4.0), (3, 300, 0.0), (80, 1000, -7.0)])
def test_class_split_nms_equals_single_cta_nms(C, K, loc_mean):
    """sihl_od_nms_topk_split (candidates dealt to per-class-group sub-lists, one CTA each, merged) == sihl_od_nms_topk:
    many classes, ONE class (everything lands in one sub-list, beyond shared memory), few classes with more outputs
    than one sub-list yields, and almost no candidates (empty sub-lists, K larger than what survives)."""
    size, B = 1024, 3
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(700 + C, B, A, C, loc_mean, 2.0)
    loc, box, cls = _t(maps.loc_logits), _t(maps.box_raw), _t(maps.cls_logits)
    outs = []
    for split in (False, True):
        cand = ops.CandidateBuffers.allocate(B, A, DEV)
        ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, mode="candidate_first")
        n_cand = cand.count.clone()
        outs.append(ops.nms_topk(cand, B, 0.5, K, reset_counts=True, split=split))
        assert int(cand.count.abs().sum()) == 0                     # consumed and re-zeroed in both variants
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert int(n_cand.max()) > (4096 if loc_mean > -5 else 0)


# ---------------------------------------------------------------------------------------------------------------------
# long lists on the whole GPU (od_nms_wide.cu) and the lazy top-K prefix of k_nms
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,n_cls", [(30000, 1), (30000, 80), (8192, 3), (20000, 5000)])
def test_wide_batched_nms_one_long_list(n, n_cls):
    """8192..90000 boxes take the multi-CTA bitmask path: keep lists equal to the C oracle (torchvision's per-class
    semantics, (score desc, index asc) order) — incl. 30 000 boxes of ONE class, the case one CTA handled worst."""
    boxes, scores, classes = synth.nms_candidates_np(4242 + n_cls, n, 1024, n_cls)
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5).cpu().numpy()
    np.testing.assert_array_equal(keep, orc.batched_nms(boxes, scores, classes, 0.5))
    import torchvision
    tv = torchvision.ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5).cpu().numpy()
    assert set(keep.tolist()) == set(tv.tolist())                                  # the library this path extends


def test_wide_batched_nms_segments_ties_and_threshold_edge():
    """Several segments in one wide call (a 256-item tile straddles segment borders), tied scores (index order decides),
    duplicate boxes (IoU == 1) and a threshold that equals an IoU exactly (strict '>')."""
    sizes = [3000, 0, 7000, 1, 2500]
    parts = [synth.nms_candidates_np(77 + i, n, 800, 7) for i, n in enumerate(sizes)]
    boxes = np.concatenate([p[0] for p in parts]); scores = np.concatenate([p[1] for p in parts])
    classes = np.concatenate([p[2] for p in parts])
    scores[::3] = np.round(scores[::3], 2)                                          # many exact score ties
    boxes[100:200] = boxes[0:100]; classes[100:200] = classes[0:100]                # duplicates of earlier boxes
    boxes[5000] = [0, 0, 10, 10]; boxes[5001] = [0, 0, 10, 5]; classes[5000] = classes[5001] = 3   # IoU = 0.5 exactly
    scores[5000], scores[5001] = 0.99, 0.98
    seg = np.zeros(len(sizes) + 1, np.int32); seg[1:] = np.cumsum(sizes)
    assert seg[-1] >= 8192
    keep, count = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5, seg_offsets=_t(seg))
    keep, count = keep.cpu().numpy(), count.cpu().numpy()
    for i, n in enumerate(sizes):
        s, e = seg[i], seg[i + 1]
        want = orc.batched_nms(boxes[s:e], scores[s:e], classes[s:e], 0.5) + s
        assert count[i] == len(want), i
        np.testing.assert_array_equal(keep[s:s + count[i]], want)
    kept = set(keep[seg[2]:seg[2] + count[2]].tolist())
    assert 5000 in kept and 5001 in kept                                            # IoU == thr does not suppress


@pytest.mark.parametrize("C,loc_mean,K,what", [(80, 0.0, 100, "prefix holds K survivors"), (1, 3.0, 100, "one class: prefix exhausted, full list decides"),
                                              (80, 0.0, 128, "largest K of the lazy path"), (3, 1.0, 20, "few classes")])
def test_lazy_topk_prefix_equals_full_nms(C, loc_mean, K, what):
    """k_nms, top-K entry, long lists: the ~200 highest-ranked candidates decide when K of them survive; otherwise the
    full list is processed.  Both outcomes must equal the oracle's full NMS."""
    size, B = 640, 3
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(91, B, A, C, loc_mean=loc_mean, loc_std=2.0)
    maps.loc_logits[:, ::5] = np.round(maps.loc_logits[:, ::5], 1)                  # tied scores inside the prefix
    if what == "few classes":
        maps.loc_logits[1, :] = 1.5                                                 # one image where EVERY score ties: the prefix cannot be cut, the full list runs
    num, scores, classes, boxes = ops.dense_postprocess(_t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw), levels,
                                                        size, size, 0.05, 0.5, K, mode="candidate_first", split_nms=False)
    o_off, o_sc, _ = orc.anchors(levels, size, size)
    w_num, w_scores, w_cls, w_boxes, _ = orc.dense_postprocess(maps.loc_logits, maps.cls_logits, maps.box_raw, o_off, o_sc,
                                                               size, size, 0.05, 0.5, K)
    np.testing.assert_array_equal(num.cpu().numpy(), w_num)
    np.testing.assert_array_equal(classes.cpu().numpy(), w_cls)
    np.testing.assert_allclose(scores.cpu().numpy(), w_scores, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(boxes.cpu().numpy(), w_boxes, rtol=1e-5, atol=1e-4)
