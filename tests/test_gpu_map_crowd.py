"""COCO crowd regions and annotated areas in the GPU matching (sihl_od_map_match_crowd, sihl_od_quad_map_match_crowd,
DetectionMAP with "iscrowd" / "area" targets) against the crowd oracle of tests/crowd_map_reference.py
(match_image_boxes, match_image_quads with gt_crowd / gt_area).  The tables must be equal, not
close."""
import numpy as np
import pytest
import torch

import crowd_map_reference as cr
from oracle import map_oracle as mo
from sihl_b200 import _native, metrics, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
THR, AREAS = ops.COCO_IOU_THRESHOLDS, ops.COCO_AREA_RANGES
GEOMETRIES = ("box", "quad")


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _oracle(geometry, det, ds, dc, gt, gc, go, crowd, area, thr=THR, areas=AREAS):
    out = []
    for b in range(len(ds)):
        g0, g1 = go[b], go[b + 1]
        if geometry == "box":
            out.append(cr.match_image_boxes(det[b], ds[b], dc[b], gt[g0:g1], gc[g0:g1], thr, areas,
                                            gt_crowd=None if crowd is None else crowd[g0:g1],
                                            gt_area=None if area is None else area[g0:g1]))
        else:
            out.append(cr.match_image_quads(det[b], ds[b], dc[b], gt[g0:g1], gc[g0:g1], thr, areas,
                                            gt_crowd=None if crowd is None else crowd[g0:g1],
                                            gt_area=None if area is None else area[g0:g1]))
    return out


def _check(res, want, go):
    order, dtm, dti, gti = (res[k].cpu().numpy() for k in ("det_order", "dt_match", "dt_ignore", "gt_ignore"))
    assert gti.shape[1] == go[-1]
    for b, w in enumerate(want):
        g0, g1 = go[b], go[b + 1]
        np.testing.assert_array_equal(order[b], w["order"], err_msg=f"image {b}")
        np.testing.assert_array_equal(np.where(dtm[b] >= 0, dtm[b] - g0, -1), w["dt_match"], err_msg=f"image {b}")
        np.testing.assert_array_equal(dti[b], w["dt_ignore"], err_msg=f"image {b}")
        np.testing.assert_array_equal(gti[:, g0:g1], w["gt_ignore"], err_msg=f"image {b}")
    return dtm, dti


def _run(geometry, det, ds, dc, gt, gc, go, crowd=None, area=None, **kw):
    match = ops.map_match if geometry == "box" else ops.quad_map_match
    return match(_t(det), _t(ds), _t(dc), _t(gt), _t(gc), _t(go), gt_crowd=None if crowd is None else _t(crowd),
                 gt_area=None if area is None else _t(area), **kw)


def _crowd_matches(dtm, crowd):
    """How many (image, range, threshold, rank) entries matched a crowd gt, and how many gts were matched twice or more
    in one chain."""
    hits = dtm[dtm >= 0]
    on_crowd = int(crowd[hits].sum()) if hits.size else 0
    multi = 0
    for chain in dtm.reshape(-1, dtm.shape[-1]):
        m = chain[chain >= 0]
        multi += int((np.bincount(m, minlength=len(crowd)) > 1).sum()) if m.size else 0
    return on_crowd, multi


@pytest.mark.parametrize("geometry", GEOMETRIES)
@pytest.mark.parametrize("seed,B,K,G,C", [(1, 6, 40, 14, 5), (2, 6, 1, 6, 1), (3, 6, 1024, 30, 80), (4, 6, 300, 40, 1),
                                          (5, 64, 100, 12, 80), (6, 64, 37, 5, 1)])
def test_tables_equal_the_oracle(geometry, seed, B, K, G, C):
    rng = np.random.RandomState(seed)
    counts = rng.randint(0, 2 * G + 1, B)
    counts[0] = 0                                                                   # an image without ground truth
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(seed, B, K, G, C, geometry=geometry, counts=counts,
                                                                    crowd_frac=0.15)
    dtm, dti = _check(_run(geometry, det, ds, dc, gt, gc, go, crowd, area),
                      _oracle(geometry, det, ds, dc, gt, gc, go, crowd, area), go)
    if K > 1 and crowd.any():
        on_crowd, multi = _crowd_matches(dtm, crowd)
        assert on_crowd > 0 and multi > 0, (on_crowd, multi)


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_duplicate_crowd_gts_ties_threshold_zero_and_custom_ranges(geometry):
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(8, 4, 60, 10, 2, geometry=geometry, crowd_frac=0.3)
    for b in range(3):                                                              # duplicate crowd gts
        g = go[b] + 1
        crowd[g] = crowd[g + 1] = 1
        gt[g + 1] = gt[g]; gc[g + 1] = gc[g]; area[g + 1] = area[g]
    ds[:, ::3] = 0.5                                                                # tied scores: input order decides
    thr = (0.0, 0.1, 0.5, 0.99, 1.0)
    areas = ((0.0, 1e10), (0.0, 400.0), (400.0, 4000.0), (4000.0, 1e10), (1e3, 1e3), (0.0, 0.0))
    want = _oracle(geometry, det, ds, dc, gt, gc, go, crowd, area, thr, areas)
    _check(_run(geometry, det, ds, dc, gt, gc, go, crowd, area, iou_thresholds=thr, area_ranges=areas), want, go)


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_empty_images_and_empty_batch(geometry):
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(10, 3, 20, 0, 4, geometry=geometry)
    go = np.zeros(4, np.int32)
    _check(_run(geometry, det, ds, dc, gt, gc, go, crowd, area), _oracle(geometry, det, ds, dc, gt, gc, go, crowd, area), go)
    shape = (0, 5, 4) if geometry == "box" else (0, 5, 8)
    res = _run(geometry, np.zeros(shape, np.float32), np.zeros((0, 5), np.float32), np.zeros((0, 5), np.int64),
               np.zeros((0,) + shape[2:], np.float32), np.zeros(0, np.int64), np.zeros(1, np.int32),
               np.zeros(0, np.uint8), np.zeros(0, np.float64))
    assert res["dt_match"].shape == (0, 4, 10, 5) and res["gt_ignore"].shape == (4, 0)


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_zero_annotations_give_the_plain_tables_bit_for_bit(geometry):
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(17, 8, 90, 15, 3, geometry=geometry)
    plain = _run(geometry, det, ds, dc, gt, gc, go)
    G = int(go[-1])
    for kw in (dict(crowd=np.zeros(G, np.uint8)), dict(area=np.zeros(G)), dict(crowd=np.zeros(G, bool), area=-np.ones(G))):
        got = _run(geometry, det, ds, dc, gt, gc, go, **kw)
        for k in plain:
            assert torch.equal(got[k], plain[k]), (kw.keys(), k)


# ---- the metric --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_detection_map_with_iscrowd_and_area_equals_the_oracle_pipeline(geometry):
    max_dets = (1, 10, 50)
    m = metrics.DetectionMAP(max_detection_thresholds=list(max_dets), sync_dist=False,
                             iou_type="bbox" if geometry == "box" else "quad")
    key = "boxes" if geometry == "box" else "quads"
    batches = [synth.map_crowd_batch_np(s, 5, 50, 12, 4, geometry=geometry, counts=[12, 0, 5, 20, 9], crowd_frac=0.2)
               for s in (11, 12)]
    det, ds, dc, gt, gc, go, crowd, area = batches[0]
    m.update_batch(_t(ds), _t(dc), _t(det), _t(gt), _t(gc), np.diff(go).tolist(), gt_crowd=_t(crowd != 0),
                   gt_area=_t(area))
    det, ds, dc, gt, gc, go, crowd, area = batches[1]                               # the per-image dict form
    targets = []
    for b in range(5):
        t = {"labels": _t(gc[go[b]:go[b + 1]]), key: _t(gt[go[b]:go[b + 1]])}
        if b != 2:
            t["iscrowd"] = _t(crowd[go[b]:go[b + 1]].astype(np.int64))
        if b != 3:
            t["area"] = _t(area[go[b]:go[b + 1]].astype(np.float32))
        targets.append(t)
    m.update([{"scores": _t(ds[b]), "labels": _t(dc[b]), key: _t(det[b])} for b in range(5)], targets)
    crowd1, area1 = crowd.copy(), area.astype(np.float32).astype(np.float64)
    crowd1[go[2]:go[3]] = 0                                                         # missing keys mean zeros
    area1[go[3]:go[4]] = 0.0
    batches[1] = batches[1][:6] + (crowd1, area1)
    images = []
    for det, ds, dc, gt, gc, go, crowd, area in batches:
        for b, w in enumerate(_oracle(geometry, det, ds, dc, gt, gc, go, crowd, area)):
            images.append(dict(scores=ds[b][w["order"]], classes=dc[b][w["order"]], dt_match=w["dt_match"],
                               dt_ignore=w["dt_ignore"], gt_classes=gc[go[b]:go[b + 1]], gt_ignore=w["gt_ignore"]))
    cats = sorted(set(int(c) for im in images for c in im["classes"]) | set(int(c) for im in images for c in im["gt_classes"]))
    want = mo.summarize(*mo.accumulate(images, cats, max_dets=max_dets), max_dets=max_dets)
    got = m.compute()
    for k, v in want.items():
        assert float(got[k]) == pytest.approx(v, abs=1e-6), k
    assert 0.0 < float(got["map"]) < 1.0


def test_detection_map_rejects_annotations_that_disagree_with_labels():
    m = metrics.DetectionMAP(sync_dist=False)
    pred = [{"scores": _t(np.ones(3, np.float32)), "labels": _t(np.zeros(3, np.int64)),
             "boxes": _t(np.tile(np.array([0, 0, 10, 10], np.float32), (3, 1)))}]
    tgt = {"labels": _t(np.zeros(2, np.int64)), "boxes": _t(np.tile(np.array([0, 0, 10, 10], np.float32), (2, 1)))}
    for key in ("iscrowd", "area"):
        with pytest.raises(ValueError, match=key):
            m.update(pred, [dict(tgt, **{key: _t(np.zeros(3, np.int64))})])


# ---- memory safety and graph capture ------------------------------------------------------------------------------------
@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_guard_bands_around_outputs_and_workspace(geometry):
    lib = _native.load()
    PAD, S = 2048, 0x5A
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(14, 5, 70, 9, 3, geometry=geometry,
                                                                    counts=[9, 0, 4, 17, 1], crowd_frac=0.3)
    B, K = ds.shape
    G, T, NA = int(go[-1]), len(THR), len(AREAS)
    ws_bytes = int(lib.sihl_od_map_workspace_bytes(G, T, NA) if geometry == "box" else
                   lib.sihl_od_quad_map_workspace_bytes(B, K, G, T, NA))
    sizes = dict(order=B * K * 4, dtm=B * NA * T * K * 4, dti=B * NA * T * K, gti=NA * G, ws=ws_bytes)
    bufs = {k: torch.full((n + 2 * PAD,), S, dtype=torch.uint8, device=DEV) for k, n in sizes.items()}
    thr = np.asarray(THR, np.float64)
    areas = np.asarray(AREAS, np.float64).reshape(-1)
    t = [_t(x) for x in (det, ds, dc, gt, gc, go, crowd, area)]
    args = [t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), B, K, t[3].data_ptr(), t[4].data_ptr(), t[5].data_ptr(),
            G, t[6].data_ptr(), t[7].data_ptr(), thr.ctypes.data, T, areas.ctypes.data, NA,
            *[bufs[k].data_ptr() + PAD for k in ("order", "dtm", "dti", "gti", "ws")]]
    stream = torch.cuda.current_stream().cuda_stream
    if geometry == "box":
        rc = lib.sihl_od_map_match_crowd(*args, stream)
    else:
        rc = lib.sihl_od_quad_map_match_crowd(*args, ws_bytes, stream)
    assert rc == 0
    torch.cuda.synchronize()
    for k, buf in bufs.items():
        assert bool((buf[:PAD] == S).all()) and bool((buf[-PAD:] == S).all()), k
    res = dict(det_order=bufs["order"][PAD:PAD + sizes["order"]].view(torch.int32).view(B, K),
               dt_match=bufs["dtm"][PAD:PAD + sizes["dtm"]].view(torch.int32).view(B, NA, T, K),
               dt_ignore=bufs["dti"][PAD:PAD + sizes["dti"]].view(B, NA, T, K),
               gt_ignore=bufs["gti"][PAD:PAD + sizes["gti"]].view(NA, G))
    _check(res, _oracle(geometry, det, ds, dc, gt, gc, go, crowd, area), go)


@pytest.mark.parametrize("geometry", GEOMETRIES)
def test_cuda_graph_replay_on_fresh_inputs_equals_eager(geometry):
    B, K = 6, 120
    counts = [10, 0, 30, 5, 22, 1]
    inputs = [synth.map_crowd_batch_np(s, B, K, 0, 4, geometry=geometry, counts=counts, crowd_frac=0.2) for s in (15, 16)]
    match = ops.map_match if geometry == "box" else ops.quad_map_match
    static = [_t(x) for x in inputs[0]]
    call = lambda s: match(*s[:6], gt_crowd=s[6], gt_area=s[7])
    call(static)                                                                     # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = call(static)
    for arrays in inputs[::-1]:
        for dst, src in zip(static, arrays):
            dst.copy_(_t(src))
        for v in out.values():
            v.fill_(0x7f) if v.dtype == torch.uint8 else v.fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        eager = call([_t(x) for x in arrays])
        for k in eager:
            assert torch.equal(out[k], eager[k]), k
