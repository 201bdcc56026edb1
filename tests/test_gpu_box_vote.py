"""Box voting on the GPU (sihl_od_box_vote_topk, sihl_od_diou_box_vote_topk, sihl_od_batched_box_vote,
sihl_od_batched_diou_box_vote) against the numpy oracle (oracle/box_vote_oracle.py): every voted coordinate within one
fp32 ulp of the oracle (fp64 sums in another order can round differently in the last bit), everything else equal to
the oracle and bit for bit to the same call without voting."""
import numpy as np
import pytest
import torch

from oracle import box_vote_oracle as bvo
from sihl_b200 import _native, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OVERLAPS = bvo.OVERLAPS
NMS_OF = {"iou": "hard", "diou": "diou"}


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


def _eq(got, want, what=""):
    np.testing.assert_array_equal(np.asarray(got), np.asarray(want), err_msg=what)


def _near(got, want, what=""):
    """Within one fp32 ulp per coordinate (and the same sign)."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, what
    d = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert d.size == 0 or d.max() <= 1, (what, np.argwhere(d > 1)[:5], got[d > 1][:5], want[d > 1][:5])


# ---- the segment form ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("n", [0, 1, 256, 4097, 10000, 30000])
@pytest.mark.parametrize("n_cls", [1, 80])
def test_batched_box_vote_vs_oracle(overlap, n, n_cls):
    boxes, scores, classes = synth.nms_candidates_np(4000 + n + n_cls, max(n, 1), 1024, n_cls)
    boxes, scores, classes = boxes[:n], scores[:n], classes[:n]
    b, s, c = _t(boxes), _t(scores), _t(classes)
    keep = ops.batched_nms(b, s, c, 0.5, overlap=overlap)
    voted = ops.batched_box_vote(b, s, c, keep, 0.5, overlap=overlap)
    want_keep, want = bvo.batched_nms_vote(boxes, scores, classes, 0.5, overlap)
    _eq(keep.cpu().numpy(), want_keep)
    _near(voted.cpu().numpy(), want)
    if n > 256:
        assert not np.array_equal(voted.cpu().numpy(), boxes[want_keep])


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("sizes", [[300, 0, 57, 1, 0, 4000], [3000, 0, 7000, 1, 2500, 0]])
def test_segments_with_empty_segments(overlap, sizes):
    parts = [synth.nms_candidates_np(91 + i, max(m, 1), 800, 7) for i, m in enumerate(sizes)]
    boxes = np.concatenate([p[0][:m] for p, m in zip(parts, sizes)])
    scores = np.concatenate([p[1][:m] for p, m in zip(parts, sizes)])
    classes = np.concatenate([p[2][:m] for p, m in zip(parts, sizes)])
    seg = np.zeros(len(sizes) + 1, np.int32)
    seg[1:] = np.cumsum(sizes)
    b, s, c, st = _t(boxes), _t(scores), _t(classes), _t(seg)
    keep, count = ops.batched_nms(b, s, c, 0.4, seg_offsets=st, overlap=overlap)
    voted = ops.batched_box_vote(b, s, c, keep, 0.4, keep_count=count, seg_offsets=st, overlap=overlap).cpu().numpy()
    keep, count = keep.cpu().numpy(), count.cpu().numpy()
    for i in range(len(sizes)):
        lo, hi = seg[i], seg[i + 1]
        want_keep, want = bvo.batched_nms_vote(boxes[lo:hi], scores[lo:hi], classes[lo:hi], 0.4, overlap)
        _eq(keep[lo:lo + count[i]], want_keep + lo, f"segment {i}")
        _near(voted[lo:lo + count[i]], want, f"segment {i}")
        assert (voted[lo + count[i]:hi] == 0).all()


@pytest.mark.parametrize("overlap", OVERLAPS)
def test_ties_and_duplicate_boxes(overlap):
    n = 3000
    boxes, scores, classes = synth.nms_candidates_np(17, n, 640, 3)
    scores = np.round(scores, 1).astype(np.float32)                        # many exact ties
    boxes[n // 2:n // 2 + 50] = boxes[:50]
    classes[n // 2:n // 2 + 50] = classes[:50]                             # duplicates of earlier boxes
    b, s, c = _t(boxes), _t(scores), _t(classes)
    keep = ops.batched_nms(b, s, c, 0.5, overlap=overlap)
    want_keep, want = bvo.batched_nms_vote(boxes, scores, classes, 0.5, overlap)
    _eq(keep.cpu().numpy(), want_keep)
    _near(ops.batched_box_vote(b, s, c, keep, 0.5, overlap=overlap).cpu().numpy(), want)


def test_equals_a_torch_cuda_restatement_of_yolov5_merge():
    """YOLOv5's merge: an IoU > thr mask (torchvision's box_iou, same class) times the scores, one fp64 matrix product
    over class-offset boxes, on the GPU."""
    import torchvision
    for n, n_cls in [(4000, 80), (3000, 1)]:
        boxes, scores, classes = synth.nms_candidates_np(n + n_cls, n, 1024, n_cls)
        b, s, c = _t(boxes), _t(scores), _t(classes)
        keep = ops.batched_nms(b, s, c, 0.5)
        mask = (torchvision.ops.box_iou(b[keep], b) > 0.5) & (c[keep][:, None] == c[None, :])
        weights = mask.double() * s.double()[None]
        off = c.double()[:, None] * 7680.0
        merged = (weights @ (b.double() + off)) / weights.sum(1, keepdim=True) - off[keep]
        np.testing.assert_allclose(ops.batched_box_vote(b, s, c, keep, 0.5).cpu().numpy(), merged.float().cpu().numpy(),
                                   rtol=1e-6, atol=1e-5)          # the offset costs fp64 bits near zero


# ---- the top-K form on decoded candidate lists -------------------------------------------------------------------------
def _decode(size, B, C, loc_mean, seed, mode="candidate_first", dtype=torch.float32):
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(seed, B, A, C, loc_mean, 2.0)
    loc, cls, box = (_t(m, dtype) for m in (maps.loc_logits, maps.cls_logits, maps.box_raw))
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, mode=mode)
    return cand, (loc, cls, box, levels)


def _oracle(cand, B, thr, K, overlap):
    return bvo.topk_vote(cand.key.cpu().numpy(), cand.box.cpu().numpy(), cand.cls.cpu().numpy(), cand.count.cpu().numpy(),
                         thr, K, overlap)


def _check(voted_out, plain_out, want):
    num, scores, classes, boxes, plain = want
    for got, w, what in zip(plain_out, (num, scores, classes, plain), ("num", "scores", "classes", "boxes")):
        _eq(got.cpu().numpy(), w, what)                                     # the NMS alone equals the oracle
    for got, ref, what in zip(voted_out[:3], plain_out[:3], ("num", "scores", "classes")):
        assert torch.equal(got, ref), what                                  # voting leaves these bit for bit
    _near(voted_out[3].cpu().numpy(), boxes, "voted boxes")
    v = voted_out[3].cpu().numpy()
    for b in range(len(num)):
        assert (v[b, num[b]:] == 0).all()                                   # padding stays zero


def _topk_both(cand, B, thr, K, overlap, split=False):
    plain = [x.clone() for x in ops.nms_topk(cand, B, thr, K, split=split, overlap=overlap)]
    out = ops.nms_topk(cand, B, thr, K, split=split, overlap=overlap)
    ops.box_vote_topk(cand, B, thr, out, overlap=overlap)
    return out, plain


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("size,B,C,loc_mean,K,what", [
    (640, 64, 80, -6.0, 100, "cfg1: short lists (<= 256)"),
    (640, 3, 80, 0.0, 100, "lazy prefix holds K survivors"),
    (640, 3, 1, 3.0, 100, "one class: the prefix is exhausted, the full list decides"),
    (640, 2, 80, 0.0, 300, "K > 128: medium body in the workspace"),
    (1024, 2, 80, 1.0, 100, "crowd: thousands of candidates"),
    (640, 2, 600, 0.0, 50, "more than 512 classes: the two-sort body"),
])
def test_box_vote_topk_vs_oracle(overlap, size, B, C, loc_mean, K, what):
    cand, _ = _decode(size, B, C, loc_mean, 500 + size + C + K)
    want = _oracle(cand, B, 0.5, K, overlap)
    out, plain = _topk_both(cand, B, 0.5, K, overlap)
    _check(out, plain, want)
    n = cand.count.cpu().numpy()
    assert n.max() > 0 if "short" in what else n.min() > 256


def test_empty_lists():
    cand, _ = _decode(320, 4, 80, -30.0, 3)
    assert int(cand.count.abs().sum()) == 0
    for overlap in OVERLAPS:
        out, plain = _topk_both(cand, 4, 0.5, 100, overlap)
        _check(out, plain, _oracle(cand, 4, 0.5, 100, overlap))


@pytest.mark.parametrize("overlap", OVERLAPS)
def test_cluster_member_beyond_the_lazy_prefix(overlap):
    """The selection of a long list runs on its ~200 best candidates; a cluster member ranked last still votes."""
    B, K = 2, 100
    cand, _ = _decode(640, B, 80, 0.0, 77)
    num, _, classes, _, plain = _oracle(cand, B, 0.5, K, overlap)
    n = int(cand.count[0])
    assert n > 1000 and num[0] == K
    key = cand.key[0, :n].cpu().numpy().view(np.uint64)
    loc = np.uint64(0xFFFFFFFF) - (key & np.uint64(0xFFFFFFFF))
    score = (key >> np.uint64(32)).astype(np.uint32).view(np.float32)
    last = int(np.lexsort((loc, -score.astype(np.float64)))[-1])          # ranked last: (score desc, location asc)
    kept = plain[0, 0]
    w, h = kept[2] - kept[0], kept[3] - kept[1]
    cand.box[0, last] = torch.tensor(kept + np.float32([0.05, -0.04, 0.06, 0.03]) * np.float32([w, h, w, h]),
                                     device=DEV)                            # IoU with the best box ~0.85
    cand.cls[0, last] = int(classes[0, 0])
    want = _oracle(cand, B, 0.5, K, overlap)
    out, plain_out = _topk_both(cand, B, 0.5, K, overlap)
    _check(out, plain_out, want)
    # without the last-ranked member (moved to another class) the best box would vote differently
    cls_alt = cand.cls.cpu().numpy()
    cls_alt[0, last] += 1000
    alt = bvo.topk_vote(cand.key.cpu().numpy(), cand.box.cpu().numpy(), cls_alt, cand.count.cpu().numpy(), 0.5, K, overlap)
    assert not np.array_equal(alt[3][0, 0], want[3][0, 0])


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("C,K,loc_mean", [(80, 100, -2.0), (1, 100, -2.0), (3, 300, 0.0)])
def test_class_split_entry_vs_oracle(overlap, C, K, loc_mean):
    B = 3
    cand, _ = _decode(1024, B, C, loc_mean, 900 + C)
    want = _oracle(cand, B, 0.5, K, overlap)
    out, plain = _topk_both(cand, B, 0.5, K, overlap, split=True)
    _check(out, plain, want)


@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("mode", ops.DECODE_MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_dense_postprocess_box_voting(overlap, mode, dtype):
    size, B, C, K = 640, 4, 80, 100
    cand, (loc, cls, box, levels) = _decode(size, B, C, -3.0, 23, mode=mode, dtype=dtype)
    want = _oracle(cand, B, 0.45, K, overlap)
    nms = NMS_OF[overlap]
    plain = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.45, K, mode=mode, nms=nms)
    out = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.45, K, mode=mode, nms=nms, box_voting=True)
    _check(out, plain, want)
    big = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.45, K, mode=mode, nms=nms, split_nms=True,
                                box_voting=True)
    for a, b in zip(big[:3], out[:3]):
        assert torch.equal(a, b)
    _near(big[3].cpu().numpy(), out[3].cpu().numpy())                      # each call decodes its own lists (below)


def test_head_postprocess_box_voting():
    from sihl_b200.heads import ObjectDetection
    torch.manual_seed(0)
    CH, SIZE, TOP = 32, 128, 7
    model = ObjectDetection(in_channels=[3] + [CH] * TOP, num_classes=16, bottom_level=3, top_level=TOP, num_channels=CH,
                            num_layers=2).to(DEV).eval()
    g = torch.Generator().manual_seed(1)
    inputs = [torch.randn((4, 3, SIZE, SIZE), generator=g).to(DEV)] + [
        torch.randn((4, CH, SIZE // 2 ** l, SIZE // 2 ** l), generator=g).to(DEV) for l in range(1, TOP + 1)]
    with torch.no_grad():
        model.loc_head[-2].bias.data.fill_(-1.0)
        flat = model._tower_feats(inputs)
        loc = model._tower("loc_head", flat).squeeze(2)
        cls = model._tower("cls_head", flat)
        box = model._tower("box_head", flat)
        off, sc, _ = ops.anchor_tables(model._level_sizes(inputs), SIZE, SIZE, DEV)
        for overlap in OVERLAPS:
            cand = ops.CandidateBuffers.allocate(4, loc.shape[1], DEV)
            ops.dense_decode(loc, cls, box, off, sc, SIZE, SIZE, 0.05, cand)
            want = _oracle(cand, 4, 0.5, model.max_instances, overlap)
            plain = model.postprocess(inputs, 0.05, 0.5, nms=NMS_OF[overlap])
            out = model.postprocess(inputs, 0.05, 0.5, nms=NMS_OF[overlap], box_voting=True)
            _check(out, plain, want)
            assert int(out[0].min()) > 0


def test_guard_bands():
    """Nothing is written past num_instances, past the output arrays, or past keep_count inside a segment."""
    B, K, G = 4, 50, 64
    cand, _ = _decode(640, B, 80, 0.0, 5)
    for overlap in OVERLAPS:
        for split in (False, True):
            flat_b = torch.full((B * K * 4 + G,), -7.0, device=DEV)
            out = ops.nms_topk(cand, B, 0.5, K, split=split, overlap=overlap)
            boxes = flat_b[:B * K * 4].view(B, K, 4)
            boxes.copy_(out[3])
            boxes[:, 40:] = -5.0                                            # rows past num_instances (set to 40 below)
            num = torch.full((B,), 40, dtype=torch.int64, device=DEV)
            ops.box_vote_topk(cand, B, 0.5, (num, out[1], out[2], boxes), overlap=overlap)
            torch.cuda.synchronize()
            assert (flat_b[B * K * 4:] == -7).all() and (boxes[:, 40:] == -5).all()
    lib = _native.load()
    for n in (3000, 9000):
        boxes, scores, classes = synth.nms_candidates_np(4, n, 512, 1)
        cuts = np.array([0, n // 3, n // 3, n], np.int32)
        bt, st, ct, seg = _t(boxes), _t(scores), _t(classes), _t(cuts)
        keep, count = ops.batched_nms(bt, st, ct, 0.5, seg_offsets=seg)
        voted = torch.full(((n + G) * 4,), -7.0, device=DEV)
        rc = lib.sihl_od_batched_box_vote(bt.data_ptr(), st.data_ptr(), ct.data_ptr(), seg.data_ptr(), 3, n, 0.5,
                                          keep.data_ptr(), count.data_ptr(), voted.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        v = voted.view(-1, 4)
        c = count.tolist()
        assert c[1] == 0 and (v[n:] == -7).all()
        for s, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
            assert (v[a + c[s]:b] == -7).all()
            _near(v[a:a + c[s]].cpu().numpy(), bvo.vote_boxes(boxes[a:b], scores[a:b], classes[a:b],
                                                              keep[a:a + c[s]].cpu().numpy() - a, 0.5))


@pytest.mark.parametrize("nms", ["hard", "diou"])
def test_cuda_graph_replay_of_postprocess_equals_eager(nms):
    size, B, C, K = 640, 16, 80, 100
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(55, B, A, C, -4.0, 2.0)
    loc, cls, box = _t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw)
    run = lambda: ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, nms=nms, box_voting=True)
    eager = [x.clone() for x in run()]
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        run()                                                               # warm-up
        with torch.cuda.graph(graph, stream=stream):
            out = run()
    torch.cuda.current_stream().wait_stream(stream)
    for _ in range(3):
        for x in out:
            x.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        for a, b in zip(eager[:3], out[:3]):
            assert torch.equal(a, b)
        # the decode appends candidates in the order its CTAs finish, and the fp64 sums follow the list order
        _near(out[3].cpu().numpy(), eager[3].cpu().numpy())
        assert torch.equal(out[3][:, :, 0] == 0, eager[3][:, :, 0] == 0)
