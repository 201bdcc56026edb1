"""Polygon-IoU COCO matching on the GPU (sihl_od_quad_map_match, DetectionMAP(iou_type="quad")) against the quad oracle
of tests/quad_map_reference.py: the COCOeval loop of oracle/map_oracle.py on the host build of the same hull IoU and hull
area.  The tables must be equal, not close: the kernel and the host shim compute the same fp32 bits."""
import numpy as np
import pytest
import torch

import quad_map_reference as qm
from oracle import map_oracle as mo
from sihl_b200 import _native, metrics, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
THR, AREAS = ops.COCO_IOU_THRESHOLDS, ops.COCO_AREA_RANGES


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _oracle(dq, ds, dc, gq, gc, go, thr=THR, areas=AREAS):
    return [qm.match_image_quads(dq[b], ds[b], dc[b], gq[go[b]:go[b + 1]], gc[go[b]:go[b + 1]], thr, areas)
            for b in range(len(ds))]


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


def _run(dq, ds, dc, gq, gc, go, **kw):
    return ops.quad_map_match(_t(dq), _t(ds), _t(dc), _t(gq), _t(gc), _t(go), **kw)


@pytest.mark.parametrize("seed,B,K,G,C", [(1, 6, 40, 14, 5), (2, 6, 1, 6, 1), (3, 6, 1024, 30, 80), (4, 6, 300, 40, 1),
                                          (5, 64, 100, 12, 80), (6, 64, 37, 5, 1)])
def test_tables_equal_the_quad_oracle(seed, B, K, G, C):
    rng = np.random.RandomState(seed)
    counts = rng.randint(0, 2 * G + 1, B)
    counts[0] = 0                                                                   # an image without ground truth
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(seed, B, K, G, C, counts=counts)
    dtm, dti = _check(_run(dq, ds, dc, gq, gc, go), _oracle(dq, ds, dc, gq, gc, go), go)
    assert (dtm >= 0).any() and (dti != 0).any()


def test_duplicates_ties_threshold_zero_and_custom_area_ranges():
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(8, 4, 60, 10, 2)
    gq[go[1] + 1] = gq[go[1]]; gc[go[1] + 1] = gc[go[1]]                            # duplicate gts: the later one wins
    gq[go[2] + 3] = gq[go[2] + 2][::-1]; gc[go[2] + 3] = gc[go[2] + 2]               # ... also with reversed vertices
    ds[:, ::3] = 0.5                                                                 # tied scores: input order decides
    thr = (0.0, 0.1, 0.5, 0.99, 1.0)
    areas = ((0.0, 1e10), (0.0, 400.0), (400.0, 4000.0), (4000.0, 1e10), (1e3, 1e3), (0.0, 0.0))
    want = _oracle(dq, ds, dc, gq, gc, go, thr, areas)
    dtm, _ = _check(_run(dq, ds, dc, gq, gc, go, iou_thresholds=thr, area_ranges=areas), want, go)
    # threshold 0 matches a same-class gt whose polygon does not touch the detection (IoU exactly 0)
    far = [(b, r) for b, w in enumerate(want) for r in range(dq.shape[1]) if w["dt_match"][0, 0, r] >= 0 and
           qm.quad_iou_grid(dq[b][w["order"][r]][None], gq[go[b] + w["dt_match"][0, 0, r]][None])[0, 0] == 0]
    assert far, "no IoU-0 match at threshold 0 was exercised"
    assert (dtm[:, 0, 1] == go[1] + 1).any()


def test_vertex_permutations_give_identical_tables():
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(9, 6, 80, 15, 3)
    base = {k: v.cpu() for k, v in _run(dq, ds, dc, gq, gc, go).items()}
    rng = np.random.RandomState(9)
    for trial in range(3):
        pd = np.take_along_axis(dq, rng.permutation(4)[None, None, :, None] if trial else np.arange(4)[::-1][None, None, :, None], 2)
        pg = np.stack([q[rng.permutation(4)] for q in gq])
        got = _run(pd, ds, dc, pg, gc, go)
        for k in base:
            assert torch.equal(got[k].cpu(), base[k]), (trial, k)


def test_empty_batch_and_no_ground_truth_at_all():
    dq, ds, dc, gq, gc, _ = synth.quad_map_batch_np(10, 3, 20, 0, 4)
    go = np.zeros(4, np.int32)
    _check(_run(dq, ds, dc, gq, gc, go), _oracle(dq, ds, dc, gq, gc, go), go)
    res = _run(np.zeros((0, 5, 8), np.float32), np.zeros((0, 5), np.float32), np.zeros((0, 5), np.int64),
               np.zeros((0, 8), np.float32), np.zeros(0, np.int64), np.zeros(1, np.int32))
    assert res["dt_match"].shape == (0, 4, 10, 5) and res["gt_ignore"].shape == (4, 0)


# ---- the metric --------------------------------------------------------------------------------------------------------
def _oracle_summary(batches, max_dets):
    images = []
    for dq, ds, dc, gq, gc, go in batches:
        for b, w in enumerate(_oracle(dq, ds, dc, gq, gc, go)):
            images.append(dict(scores=ds[b][w["order"]], classes=dc[b][w["order"]], dt_match=w["dt_match"],
                               dt_ignore=w["dt_ignore"], gt_classes=gc[go[b]:go[b + 1]], gt_ignore=w["gt_ignore"]))
    cats = sorted(set(int(c) for im in images for c in im["classes"]) | set(int(c) for im in images for c in im["gt_classes"]))
    return mo.summarize(*mo.accumulate(images, cats, max_dets=max_dets), max_dets=max_dets)


def test_detection_map_quad_equals_the_oracle_pipeline():
    max_dets = (1, 10, 50)
    m = metrics.DetectionMAP(max_detection_thresholds=list(max_dets), sync_dist=False, iou_type="quad")
    batches = [synth.quad_map_batch_np(s, 5, 50, 12, 4, counts=[12, 0, 5, 20, 9]) for s in (11, 12)]
    dq, ds, dc, gq, gc, go = batches[0]
    m.update_batch(_t(ds), _t(dc), _t(dq), _t(gq), _t(gc), np.diff(go).tolist())
    dq, ds, dc, gq, gc, go = batches[1]                                             # the per-image dict form, [n, 8] quads
    m.update([{"scores": _t(ds[b]), "labels": _t(dc[b]), "quads": _t(dq[b].reshape(-1, 8))} for b in range(5)],
             [{"labels": _t(gc[go[b]:go[b + 1]]), "quads": _t(gq[go[b]:go[b + 1]])} for b in range(5)])
    want = _oracle_summary(batches, max_dets)
    got = m.compute()
    for k, v in want.items():                                                       # compute() returns fp32 scalars
        assert float(got[k]) == pytest.approx(float(np.float32(v)), abs=1e-12), k
    assert 0.0 < float(got["map"]) < 1.0


def _box_quads(b):
    return np.stack([b[..., [0, 1]], b[..., [2, 1]], b[..., [2, 3]], b[..., [0, 3]]], -2)


def test_quad_and_box_metrics_agree_on_axis_aligned_integer_quads():
    rng = np.random.RandomState(13)
    B, K, C = 8, 60, 3
    counts = rng.randint(3, 15, B)
    go = np.zeros(B + 1, np.int32); go[1:] = np.cumsum(counts)
    G = int(go[-1])
    gxy = rng.randint(0, 400, (G, 2))
    gb = np.concatenate([gxy, gxy + rng.randint(4, 160, (G, 2))], 1).astype(np.float32)
    gc = rng.randint(0, C, G).astype(np.int64)
    db = np.zeros((B, K, 4), np.float32); dc = np.zeros((B, K), np.int64)
    for b in range(B):
        pick = go[b] + rng.randint(0, counts[b], K)
        db[b] = gb[pick] + rng.randint(-10, 11, (K, 4))
        dc[b] = np.where(rng.uniform(0, 1, K) < 0.85, gc[pick], rng.randint(0, C, K))
    db[..., 2:] = np.maximum(db[..., 2:], db[..., :2] + 2)
    ds = rng.uniform(0, 1, (B, K)).astype(np.float32)
    # drop detections whose box IoU with a same-class gt is within 1e-6 of a threshold or of another gt's IoU: there the
    # fp32 polygon IoU and the fp64 box IoU may decide differently
    kept, total = 0, 0
    for b in range(B):
        ious = mo.box_iou(db[b], gb[go[b]:go[b + 1]])
        same = dc[b][:, None] == gc[go[b]:go[b + 1]][None]
        for k in range(K):
            v = ious[k][same[k] & (ious[k] > 0)]
            total += 1
            bad = (np.abs(v[:, None] - np.asarray(THR)[None]) < 1e-6).any() or \
                  (np.abs(v[:, None] - v[None]) + np.eye(len(v)) * 1 < 1e-6).any()
            if bad:
                db[b, k] = [5000, 5000, 5004, 5004]                                   # far away: no overlap with anything
            else:
                kept += v.size > 0
    assert kept >= 0.8 * total, (kept, total)
    mb = metrics.DetectionMAP(sync_dist=False)
    mq = metrics.DetectionMAP(sync_dist=False, iou_type="quad")
    mb.update_batch(_t(ds), _t(dc), _t(db), _t(gb), _t(gc), counts.tolist())
    mq.update_batch(_t(ds), _t(dc), _t(_box_quads(db)), _t(_box_quads(gb)), _t(gc), counts.tolist())
    rb, rq = mb.compute(), mq.compute()
    for k in rb:
        if k != "classes":
            assert float(rq[k]) == pytest.approx(float(rb[k]), abs=1e-6), k
    assert float(rb["map"]) > 0.2


# ---- memory safety and graph capture ------------------------------------------------------------------------------------
def test_guard_bands_around_outputs_and_workspace():
    lib = _native.load()
    PAD, S = 2048, 0x5A
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(14, 5, 70, 9, 3, counts=[9, 0, 4, 17, 1])
    B, K = ds.shape
    G, T, NA = int(go[-1]), len(THR), len(AREAS)
    ws_bytes = int(lib.sihl_od_quad_map_workspace_bytes(B, K, G, T, NA))
    sizes = dict(order=B * K * 4, dtm=B * NA * T * K * 4, dti=B * NA * T * K, gti=NA * G, ws=ws_bytes)
    bufs = {k: torch.full((n + 2 * PAD,), S, dtype=torch.uint8, device=DEV) for k, n in sizes.items()}
    thr = np.asarray(THR, np.float64)
    areas = np.asarray(AREAS, np.float64).reshape(-1)
    t = [_t(x) for x in (dq, ds, dc, gq, gc, go)]
    rc = lib.sihl_od_quad_map_match(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), B, K, t[3].data_ptr(),
                                    t[4].data_ptr(), t[5].data_ptr(), G, thr.ctypes.data, T, areas.ctypes.data, NA,
                                    *[bufs[k].data_ptr() + PAD for k in ("order", "dtm", "dti", "gti", "ws")], ws_bytes,
                                    torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    for k, buf in bufs.items():
        assert bool((buf[:PAD] == S).all()) and bool((buf[-PAD:] == S).all()), k
    res = dict(det_order=bufs["order"][PAD:PAD + sizes["order"]].view(torch.int32).view(B, K),
               dt_match=bufs["dtm"][PAD:PAD + sizes["dtm"]].view(torch.int32).view(B, NA, T, K),
               dt_ignore=bufs["dti"][PAD:PAD + sizes["dti"]].view(B, NA, T, K),
               gt_ignore=bufs["gti"][PAD:PAD + sizes["gti"]].view(NA, G))
    _check(res, _oracle(dq, ds, dc, gq, gc, go), go)


def test_cuda_graph_replay_on_fresh_inputs_equals_eager():
    B, K = 6, 120
    counts = [10, 0, 30, 5, 22, 1]
    inputs = [synth.quad_map_batch_np(s, B, K, 0, 4, counts=counts) for s in (15, 16)]
    static = [_t(x) for x in inputs[0]]
    ops.quad_map_match(*static)                                                      # warm-up outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ops.quad_map_match(*static)
    for arrays in inputs[::-1]:
        for dst, src in zip(static, arrays):
            dst.copy_(_t(src))
        for v in out.values():
            v.fill_(0x7f) if v.dtype == torch.uint8 else v.fill_(-7)
        g.replay()
        torch.cuda.synchronize()
        eager = ops.quad_map_match(*[_t(x) for x in arrays])
        for k in eager:
            assert torch.equal(out[k], eager[k]), k
