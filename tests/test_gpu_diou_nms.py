"""Class-aware DIoU-NMS on the GPU (sihl_od_diou_nms_topk, sihl_od_diou_nms_topk_split, sihl_od_batched_diou_nms)
against the C oracle (oracle/diou_nms_oracle.c): kept indices, and the scores, classes and boxes of the top-K entries,
must be EQUAL in every regime of the kernels, no tolerance."""
import numpy as np
import pytest
import torch

from oracle import diou_nms_oracle as dno
from oracle import od_oracle as orc
from sihl_b200 import _native, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


def _eq(got, want, what=""):
    np.testing.assert_array_equal(np.asarray(got), np.asarray(want), err_msg=what)


# ---- the segment form: every regime of the one-CTA kernel, the wide path, and the big (> 512 classes) body -----------
@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 4096, 4097, 8191, 8192, 30000])
@pytest.mark.parametrize("n_cls", [1, 80])
def test_batched_diou_nms_vs_oracle(n, n_cls):
    """<= 256: short-list body; <= 4096: medium body on chip; 4097..8191: medium body in the workspace; 8192..90000:
    the whole-GPU bitmask path (k_wide_mask_diou)."""
    boxes, scores, classes = synth.nms_candidates_np(2000 + n + n_cls, max(n, 1), 1024, n_cls)
    boxes, scores, classes = boxes[:n], scores[:n], classes[:n]
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.5, overlap="diou").cpu().numpy()
    want = dno.batched_diou_nms(boxes, scores, classes, 0.5)
    _eq(keep, want)


@pytest.mark.parametrize("n,n_cls", [(5000, 700), (30000, 3000)])
def test_batched_diou_nms_many_classes(n, n_cls):
    """More than 512 distinct classes: the two-sort body (one CTA) and the wide path."""
    boxes, scores, classes = synth.nms_candidates_np(n_cls, n, 1024, n_cls)
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.3, overlap="diou").cpu().numpy()
    _eq(keep, dno.batched_diou_nms(boxes, scores, classes, 0.3))


@pytest.mark.parametrize("n", [200, 3000, 12000])
@pytest.mark.parametrize("thr", [-0.3, 0.0, 0.7])
def test_thresholds_including_negative(n, thr):
    """A negative threshold suppresses same-class boxes that do not overlap at all: no body may skip a disjoint pair."""
    boxes, scores, classes = synth.nms_candidates_np(31 + n, n, 2048, 4)
    boxes[0], boxes[1] = [0, 0, 10, 10], [12, 0, 22, 10]        # disjoint, visited first: DIoU = -144 / 584 = -0.247
    scores[0], scores[1] = 2.0, 1.9
    classes[0] = classes[1] = 0
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), thr, overlap="diou").cpu().numpy()
    want = dno.batched_diou_nms(boxes, scores, classes, thr)
    _eq(keep, want)
    assert (1 in want) == (thr >= 0)


@pytest.mark.parametrize("sizes", [[300, 0, 57, 1, 0, 4000], [3000, 0, 7000, 1, 2500, 0]])
def test_segments_with_empty_segments(sizes):
    """Several images in one call, the one-CTA kernel (first) and the wide path (second: 12 501 boxes in all)."""
    parts = [synth.nms_candidates_np(77 + i, max(m, 1), 800, 7) for i, m in enumerate(sizes)]
    boxes = np.concatenate([p[0][:m] for p, m in zip(parts, sizes)])
    scores = np.concatenate([p[1][:m] for p, m in zip(parts, sizes)])
    classes = np.concatenate([p[2][:m] for p, m in zip(parts, sizes)])
    seg = np.zeros(len(sizes) + 1, np.int32)
    seg[1:] = np.cumsum(sizes)
    keep, count = ops.batched_nms(_t(boxes), _t(scores), _t(classes), 0.4, seg_offsets=_t(seg), overlap="diou")
    keep, count = keep.cpu().numpy(), count.cpu().numpy()
    for i in range(len(sizes)):
        s, e = seg[i], seg[i + 1]
        want = dno.batched_diou_nms(boxes[s:e], scores[s:e], classes[s:e], 0.4) + s
        assert count[i] == len(want), i
        _eq(keep[s:s + count[i]], want, f"segment {i}")


@pytest.mark.parametrize("n", [200, 3000, 9000])
def test_ties_duplicates_and_the_threshold_itself(n):
    """Tied scores (index order decides), duplicate boxes (DIoU 1), and pairs whose DIoU EQUALS the threshold: strict '>'
    keeps them."""
    boxes, scores, classes = synth.nms_candidates_np(5 + n, n, 640, 3)
    scores = np.round(scores, 1).astype(np.float32)                                 # many exact ties
    boxes[n // 2:n // 2 + 50] = boxes[:50]
    classes[n // 2:n // 2 + 50] = classes[:50]                                      # duplicates of earlier boxes
    a, b = np.array([0, 0, 10, 10], np.float32), np.array([4, 0, 14, 10], np.float32)
    thr = float(dno.diou_pair(a, b))                                                # 0.3745..., an fp32 value
    boxes[7], boxes[8] = a, b
    scores[7], scores[8] = 2.0, 1.5                                                 # visited first among their class
    classes[7] = classes[8] = 2
    keep = ops.batched_nms(_t(boxes), _t(scores), _t(classes), thr, overlap="diou").cpu().numpy()
    want = dno.batched_diou_nms(boxes, scores, classes, thr)
    _eq(keep, want)
    assert 7 in want and 8 in want                                                  # DIoU == thr does not suppress
    nudged = dno.batched_diou_nms(boxes, scores, classes, np.nextafter(np.float32(thr), np.float32(0)))
    assert 8 not in nudged
    _eq(ops.batched_nms(_t(boxes), _t(scores), _t(classes), float(np.nextafter(np.float32(thr), np.float32(0))),
                        overlap="diou").cpu().numpy(), nudged)


def test_keep_sets_equal_a_torch_cuda_greedy_loop():
    """distance_box_iou on the GPU plus a greedy loop (what a user of torchvision writes today) keeps the same boxes."""
    import torchvision
    for n, n_cls, seed in [(1500, 1, 3), (4000, 5, 4)]:
        boxes, scores, classes = synth.nms_candidates_np(seed, n, 1024, n_cls)
        b, s, c = _t(boxes), _t(scores), _t(classes)
        d = torchvision.ops.distance_box_iou(b, b).cpu().numpy()
        same = classes[:, None] == classes[None, :]
        order = np.lexsort((np.arange(n), -scores.astype(np.float64)))
        alive = np.ones(n, bool)
        kept = []
        for i in order:
            if alive[i]:
                kept.append(i)
                alive &= ~(same[i] & (d[i] > np.float32(0.5)))
        keep = ops.batched_nms(b, s, c, 0.5, overlap="diou").cpu().numpy()
        assert set(keep.tolist()) == set(kept)
        _eq(keep, kept)                                                             # and in the same order


# ---- the top-K form on decoded candidate lists -------------------------------------------------------------------------
def _oracle_topk(cand, B, thr, K):
    """The oracle on the device's candidate lists: visit order (score desc, location asc) from the keys."""
    n = cand.count.cpu().numpy()
    keys = cand.key.cpu().numpy().view(np.uint64)
    box_all, cls_all = cand.box.cpu().numpy(), cand.cls.cpu().numpy()
    num = np.zeros(B, np.int64)
    scores, classes, boxes = np.zeros((B, K), np.float32), np.zeros((B, K), np.int64), np.zeros((B, K, 4), np.float32)
    for b in range(B):
        key, box, cls = keys[b, :n[b]], box_all[b, :n[b]], cls_all[b, :n[b]]
        loc = np.uint64(0xFFFFFFFF) - (key & np.uint64(0xFFFFFFFF))
        perm = np.argsort(loc, kind="stable")                                       # index order = location order
        sc = (key >> np.uint64(32)).astype(np.uint32).view(np.float32)
        keep = perm[dno.batched_diou_nms(box[perm], sc[perm], cls[perm].astype(np.int64), thr)][:K]
        num[b] = keep.size
        scores[b, :keep.size], classes[b, :keep.size], boxes[b, :keep.size] = sc[keep], cls[keep], box[keep]
    return num, scores, classes, boxes, n


def _check(out, want):
    for got, w, what in zip(out, want, ("num_instances", "scores", "classes", "boxes")):
        _eq(got.cpu().numpy(), w, what)


def _decode(size, B, C, loc_mean, seed, cap=None, mode="candidate_first", dtype=torch.float32):
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(seed, B, A, C, loc_mean, 2.0)
    loc, cls, box = (_t(m, dtype) for m in (maps.loc_logits, maps.cls_logits, maps.box_raw))
    cand = ops.CandidateBuffers.allocate(B, cap or A, DEV)
    ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, mode=mode)
    return cand, (loc, cls, box, levels)


@pytest.mark.parametrize("size,B,C,loc_mean,K,what", [
    (640, 64, 80, -6.0, 100, "cfg1: short lists (<= 256)"),
    (640, 3, 80, 0.0, 100, "lazy prefix holds K survivors"),
    (640, 3, 80, 0.0, 128, "lazy prefix, largest K"),
    (640, 3, 1, 3.0, 100, "one class: the prefix is exhausted, the full list decides"),
    (640, 3, 1, 3.0, 128, "one class, K = 128: prefix exhausted"),
    (640, 2, 80, 0.0, 300, "K > 128: medium body in the workspace"),
    (1024, 2, 80, 1.0, 100, "crowd: thousands of candidates"),
    (640, 2, 600, 0.0, 50, "more than 512 classes: the two-sort body"),
])
def test_diou_nms_topk_vs_oracle(size, B, C, loc_mean, K, what):
    cand, _ = _decode(size, B, C, loc_mean, 300 + size + C + K)
    want = _oracle_topk(cand, B, 0.5, K)
    out = ops.nms_topk(cand, B, 0.5, K, reset_counts=True, overlap="diou")
    assert int(cand.count.abs().sum()) == 0
    _check(out, want[:4])
    n = want[4]
    assert n.max() > 0 if "short" in what else n.min() > 256


@pytest.mark.parametrize("C,K,loc_mean", [(80, 100, -2.0), (1, 100, -2.0), (3, 300, 0.0), (80, 1000, -7.0)])
def test_class_split_entry_vs_oracle(C, K, loc_mean):
    """sihl_od_diou_nms_topk_split == the oracle == the single-CTA entry: many classes, one class (one sub-list beyond
    shared memory), few classes with K larger than a sub-list yields, and almost no candidates."""
    size, B = 1024, 3
    cand, _ = _decode(size, B, C, loc_mean, 700 + C)
    want = _oracle_topk(cand, B, 0.5, K)
    n_cand = cand.count.clone()
    out = ops.nms_topk(cand, B, 0.5, K, split=True, overlap="diou")
    _check(out, want[:4])
    _check(ops.nms_topk(cand, B, 0.5, K, reset_counts=True, overlap="diou"), want[:4])
    assert int(n_cand.max()) > (4096 if loc_mean > -5 else 0)


@pytest.mark.parametrize("mode", ops.DECODE_MODES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_dense_postprocess_diou_vs_oracle(mode, dtype):
    """ops.dense_postprocess(nms="diou") in both decode modes and on half maps, against the oracle on the same lists."""
    size, B, C, K = 640, 4, 80, 100
    cand, (loc, cls, box, levels) = _decode(size, B, C, -3.0, 17, mode=mode, dtype=dtype)
    want = _oracle_topk(cand, B, 0.45, K)
    out = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.45, K, mode=mode, nms="diou")
    _check(out, want[:4])


def test_dense_postprocess_diou_equals_the_end_to_end_oracle():
    """Decode + DIoU-NMS against the CPU restatement of the whole postprocess (decode on the CPU too)."""
    size, B, C, K = 320, 2, 80, 100
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(9, B, A, C, loc_mean=-3.0, loc_std=2.0)
    num, scores, classes, boxes = ops.dense_postprocess(_t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw), levels,
                                                        size, size, 0.05, 0.5, K, nms="diou")
    o_off, o_sc, _ = orc.anchors(levels, size, size)
    w_num, w_scores, w_cls, w_boxes = dno.dense_postprocess_diou(maps.loc_logits, maps.cls_logits, maps.box_raw, o_off, o_sc,
                                                                 size, size, 0.05, 0.5, K)
    _eq(num.cpu().numpy(), w_num)
    _eq(classes.cpu().numpy(), w_cls)
    np.testing.assert_allclose(scores.cpu().numpy(), w_scores, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(boxes.cpu().numpy(), w_boxes, rtol=1e-5, atol=1e-4)


def test_head_postprocess_diou():
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
        for mode in ops.DECODE_MODES:
            out = model.postprocess(inputs, 0.05, 0.5, mode=mode, nms="diou")
            cand = ops.CandidateBuffers.allocate(4, loc.shape[1], DEV)
            ops.dense_decode(loc, cls, box, off, sc, SIZE, SIZE, 0.05, cand, mode=mode)
            want = _oracle_topk(cand, 4, 0.5, model.max_instances)
            _check(out, want[:4])
            assert int(out[0].min()) > 0


def test_guard_bands():
    """Nothing is written past K per image, past the output arrays, or past keep_count inside a segment."""
    B, K, G = 4, 50, 64
    cand, _ = _decode(640, B, 80, 0.0, 5)
    flat = [torch.full((B * K + G,), -7, dtype=d, device=DEV) for d in (torch.float32, torch.int64)]
    flat_b = torch.full((B * K * 4 + G,), -7.0, device=DEV)
    num = torch.full((B + G,), -7, dtype=torch.int64, device=DEV)
    for split in (False, True):
        out = (num[:B], flat[0][:B * K].view(B, K), flat[1][:B * K].view(B, K), flat_b[:B * K * 4].view(B, K, 4))
        ops.nms_topk(cand, B, 0.5, K, out=out, split=split, overlap="diou")
        torch.cuda.synchronize()
        assert (num[B:] == -7).all() and (flat[0][B * K:] == -7).all() and (flat[1][B * K:] == -7).all()
        assert (flat_b[B * K * 4:] == -7).all() and (num[:B] == K).all()
    # segment form, one-CTA and wide: sentinels past keep_count in every segment and past the arrays
    lib = _native.load()
    for n in (3000, 9000):
        boxes, scores, classes = synth.nms_candidates_np(4, n, 512, 1)
        cuts = np.array([0, n // 3, n // 3, n], np.int32)
        keep = torch.full((n + G,), -7, dtype=torch.int64, device=DEV)
        count = torch.full((3 + G,), -7, dtype=torch.int32, device=DEV)
        bt, st, ct, seg = _t(boxes), _t(scores), _t(classes), _t(cuts)
        ws_bytes = int(lib.sihl_od_batched_nms_workspace_bytes(n))
        ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=DEV)
        rc = lib.sihl_od_batched_diou_nms(bt.data_ptr(), st.data_ptr(), ct.data_ptr(), seg.data_ptr(), 3, n, 0.5,
                                          keep.data_ptr(), count.data_ptr(), ws.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        c = count[:3].tolist()
        assert c[1] == 0 and (count[3:] == -7).all()
        for s, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
            assert (keep[a + c[s]:b] == -7).all()
            _eq(keep[a:a + c[s]].cpu().numpy(), dno.batched_diou_nms(boxes[a:b], scores[a:b], classes[a:b], 0.5) + a)
        assert (keep[n:] == -7).all()


def test_cuda_graph_replay_of_postprocess_equals_eager():
    size, B, C, K = 640, 16, 80, 100
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    maps = synth.dense_maps_np(55, B, A, C, -4.0, 2.0)
    loc, cls, box = _t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw)
    eager = [x.clone() for x in ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, nms="diou")]
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, nms="diou")          # warm-up
        with torch.cuda.graph(graph, stream=stream):
            out = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, nms="diou")
    torch.cuda.current_stream().wait_stream(stream)
    for _ in range(3):
        for x in out:
            x.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        for a, b in zip(eager, out):
            assert torch.equal(a, b)
