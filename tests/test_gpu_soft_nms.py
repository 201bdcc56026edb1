"""Class-aware Soft-NMS on the GPU (sihl_od_soft_nms_topk, sihl_od_batched_soft_nms) against the numpy oracle
(oracle/soft_nms_oracle.py): kept indices, classes, boxes and decayed scores must be EQUAL, no tolerance."""
import numpy as np
import pytest
import torch

from oracle import soft_nms_oracle as sno
from sihl_b200 import _native, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PARAMS = [("linear", 0.3, 0.5), ("linear", 0.5, 0.5), ("gaussian", 0.3, 0.5), ("gaussian", 0.3, 0.1)]   # method, Nt, sigma


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


def _eq(got, want, what):
    np.testing.assert_array_equal(np.asarray(got), np.asarray(want), err_msg=what)


@pytest.mark.parametrize("n", [0, 1, 2, 255, 256, 257, 4096, 4097, 30000])
@pytest.mark.parametrize("n_cls", [1, 3, 80])
@pytest.mark.parametrize("method,nt,sigma", PARAMS)
def test_batched_soft_nms_vs_oracle(n, n_cls, method, nt, sigma):
    """Every list-length regime: one CTA (up to 4096), the cluster (4097, 30000 over 8 CTAs' shared memory)."""
    boxes, scores, classes = synth.nms_candidates_np(1000 + n + n_cls, max(n, 1), 1024, n_cls)
    boxes, scores, classes = boxes[:n], scores[:n], classes[:n]
    max_out = n if n <= 4097 else 1000
    keep, ks = ops.batched_soft_nms(_t(boxes), _t(scores), _t(classes), max(max_out, 1), method, nt, sigma, 0.001)
    want_keep, want_s = sno.soft_nms(boxes, scores, classes, method, nt, sigma, 0.001, max_out)
    _eq(keep.cpu().numpy(), want_keep, "indices")
    _eq(ks.cpu().numpy(), want_s, "scores")
    if n:
        assert keep.numel() > 0


def test_batched_soft_nms_beyond_shared_memory():
    """40 000 boxes of one class: more than the cluster's shared memory holds, the lists go to the workspace."""
    boxes, scores, classes = synth.nms_candidates_np(77, 40000, 1024, 1)
    assert ops._lib().sihl_od_batched_soft_nms_workspace_bytes(40000) > 0
    for method in sno.METHODS:
        keep, ks = ops.batched_soft_nms(_t(boxes), _t(scores), _t(classes), 300, method, 0.3, 0.5, 0.001)
        want_keep, want_s = sno.soft_nms(boxes, scores, classes, method, 0.3, 0.5, 0.001, 300)
        _eq(keep.cpu().numpy(), want_keep, method)
        _eq(ks.cpu().numpy(), want_s, method)


@pytest.mark.parametrize("method", sno.METHODS)
def test_segments_with_empty_segments(method):
    boxes, scores, classes = synth.nms_candidates_np(5, 9000, 1024, 3)
    cuts = [0, 0, 300, 300, 301, 5000, 5000, 9000, 9000]
    keep, ks, count = ops.batched_soft_nms(_t(boxes), _t(scores), _t(classes), 200, method, 0.3, 0.5, 0.001,
                                           seg_offsets=_t(np.array(cuts, np.int32)))
    keep, ks, count = keep.cpu().numpy(), ks.cpu().numpy(), count.cpu().numpy()
    for s in range(len(cuts) - 1):
        a, b = cuts[s], cuts[s + 1]
        wk, ws = sno.soft_nms(boxes[a:b], scores[a:b], classes[a:b], method, 0.3, 0.5, 0.001, 200)
        assert count[s] == wk.size
        _eq(keep[a:a + count[s]], wk + a, f"segment {s}")
        _eq(ks[a:a + count[s]], ws, f"segment {s}")


@pytest.mark.parametrize("n", [200, 6000])
@pytest.mark.parametrize("method,nt,sigma", PARAMS)
def test_duplicated_scores_and_boxes(n, method, nt, sigma):
    """Ties: scores on a coarse grid (many equal), every box twice, some boxes empty."""
    boxes, scores, classes = synth.nms_candidates_np(31 + n, n // 2, 512, 2)
    boxes = np.concatenate([boxes, boxes])
    boxes[::17, 2] = boxes[::17, 0]                                          # zero width
    scores = np.round(np.concatenate([scores, scores[::-1]]), 1).astype(np.float32)
    classes = np.concatenate([classes, classes])
    keep, ks = ops.batched_soft_nms(_t(boxes), _t(scores), _t(classes), n, method, nt, sigma, 0.001)
    want_keep, want_s = sno.soft_nms(boxes, scores, classes, method, nt, sigma, 0.001, n)
    _eq(keep.cpu().numpy(), want_keep, "indices")
    _eq(ks.cpu().numpy(), want_s, "scores")


def _lists(cand, B):
    n = cand.count.cpu().numpy()
    key, box, cls = cand.key.cpu().numpy(), cand.box.cpu().numpy(), cand.cls.cpu().numpy()
    return n, [(key[b, :n[b]], box[b, :n[b]], cls[b, :n[b]]) for b in range(B)]


def _check_topk_vs_oracle(out, lists, method, nt, sigma, thr, K):
    num, scores, classes, boxes = (x.cpu().numpy() for x in out)
    for b, (key, box, cls) in enumerate(lists):
        w_num, w_s, w_c, w_b = sno.soft_nms_candidates(key, box, cls, method, nt, sigma, thr, K)
        assert num[b] == w_num, b
        _eq(scores[b], w_s, f"scores {b}")
        _eq(classes[b], w_c, f"classes {b}")
        _eq(boxes[b], w_b, f"boxes {b}")


# cfg1 (640^2, B=64, 80 classes, a few hundred candidates), the crowd (1024^2, thousands of candidates over the
# cluster), and the crowd with one class
@pytest.mark.parametrize("size,B,C,loc_mean", [(640, 64, 80, -6.0), (1024, 8, 80, -2.0), (1024, 8, 1, -2.0)])
@pytest.mark.parametrize("method,nt,sigma", [PARAMS[0], PARAMS[3]])
def test_soft_nms_topk_on_decoded_candidates(size, B, C, loc_mean, method, nt, sigma):
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(400 + size + C, B, A, C, loc_mean, 2.0)
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    ops.dense_decode(_t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw), off, sc, size, size, 0.05, cand,
                     mode="candidate_first")
    n, lists = _lists(cand, B)
    K = 100
    out = ops.soft_nms_topk(cand, B, method, nt, sigma, 0.05, K, reset_counts=True)
    assert int(cand.count.abs().sum()) == 0
    _check_topk_vs_oracle(out, lists, method, nt, sigma, 0.05, K)
    if size == 1024:
        assert n.min() > 4096                                               # the cluster path
    else:
        assert 0 < n.max() <= 4096


def test_postprocess_soft_gaussian_equals_the_oracle():
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
        hard = model.postprocess(inputs, 0.05, 0.5)
        out = model.postprocess(inputs, 0.05, 0.5, nms="soft_gaussian", sigma=0.5)
        flat = model._tower_feats(inputs)
        loc = model._tower("loc_head", flat).squeeze(2)
        cls = model._tower("cls_head", flat)
        box = model._tower("box_head", flat)
        levels = model._level_sizes(inputs)
        off, sc, _ = ops.anchor_tables(levels, SIZE, SIZE, DEV)
        cand = ops.CandidateBuffers.allocate(4, loc.shape[1], DEV)
        ops.dense_decode(loc, cls, box, off, sc, SIZE, SIZE, 0.05, cand, mode="dense")
        _, lists = _lists(cand, 4)
    _check_topk_vs_oracle(out, lists, "gaussian", 0.5, 0.5, 0.05, model.max_instances)
    assert int(out[0].min()) > 0 and int(hard[0].min()) > 0


@pytest.mark.parametrize("method", sno.METHODS)
def test_properties_order_bounds_and_permutation(method):
    rng = np.random.RandomState(3)
    boxes, _, classes = synth.nms_candidates_np(8, 5000, 1024, 4)
    scores = (rng.permutation(5000).astype(np.float32) + 1) / 5001          # distinct: the order does not depend on indices
    thr, max_out = 0.01, 700
    keep, ks = ops.batched_soft_nms(_t(boxes), _t(scores), _t(classes), max_out, method, 0.3, 0.5, thr)
    keep, ks = keep.cpu().numpy(), ks.cpu().numpy()
    assert 0 < keep.size <= max_out and (ks >= np.float32(thr)).all() and (ks[:-1] >= ks[1:]).all()
    assert np.unique(keep).size == keep.size
    perm = rng.permutation(5000)
    keep_p, ks_p = ops.batched_soft_nms(_t(boxes[perm]), _t(scores[perm]), _t(classes[perm]), max_out, method, 0.3, 0.5, thr)
    _eq(perm[keep_p.cpu().numpy()], keep, "permuted indices")
    _eq(ks_p.cpu().numpy(), ks, "permuted scores")


def _grid_candidates(B, cap, per_image, C, seed):
    """Candidate lists whose boxes overlap only across classes: same-class boxes sit on disjoint cells of a grid."""
    rng = np.random.RandomState(seed)
    cand = ops.CandidateBuffers.allocate(B, cap, DEV)
    count = np.zeros(B, np.int32)
    key = np.zeros((B, cap), np.uint64)
    box = np.zeros((B, cap, 4), np.float32)
    cls = np.zeros((B, cap), np.int32)
    for b in range(B):
        m = per_image[b]
        cells = rng.permutation(128 * 128)[:m]
        c = rng.randint(0, C, m)
        x, y = (cells % 128) * 8.0, (cells // 128) * 8.0
        jitter = (c % 4) * 1.5                                              # other classes overlap the cell
        box[b, :m] = np.stack([x + jitter, y, x + 6 + jitter, y + 6], 1)
        s = rng.uniform(0.06, 1.0, m).astype(np.float32)
        loc = rng.permutation(cap)[:m].astype(np.uint64)
        key[b, :m] = (s.view(np.uint32).astype(np.uint64) << np.uint64(32)) | (~loc & np.uint64(0xFFFFFFFF))
        cls[b, :m] = c
        count[b] = m
    cand.count.copy_(_t(count))
    cand.key.copy_(_t(key.view(np.int64)))
    cand.box.copy_(_t(box))
    cand.cls.copy_(_t(cls))
    return cand, count


@pytest.mark.parametrize("per_image", [[300, 0, 57, 1], [6000, 4500]])
def test_without_same_class_overlaps_soft_equals_hard(per_image):
    """No two boxes of a class overlap: nothing decays, so both soft methods return exactly what nms_topk returns."""
    B, K = len(per_image), 200
    cand, count = _grid_candidates(B, 8192, per_image, 5, sum(per_image))
    hard = ops.nms_topk(cand, B, 0.5, K)
    for method in sno.METHODS:
        soft = ops.soft_nms_topk(cand, B, method, 0.3, 0.5, 0.05, K)
        for a, b in zip(hard, soft):
            assert torch.equal(a, b), method
    assert torch.equal(cand.count.cpu(), torch.from_numpy(count))          # reset_counts=False leaves the counts


def test_guard_bands():
    """Nothing is written past K per image, past the output arrays, or past keep_count inside a segment."""
    B, K, G = 4, 50, 64
    cand, _ = _grid_candidates(B, 8192, [700, 3, 0, 4000], 2, 9)
    flat = [torch.full((B * K + G,), -7, dtype=d, device=DEV) for d in (torch.float32, torch.int64)]
    flat_b = torch.full((B * K * 4 + G,), -7.0, device=DEV)
    num = torch.full((B + G,), -7, dtype=torch.int64, device=DEV)
    out = (num[:B], flat[0][:B * K].view(B, K), flat[1][:B * K].view(B, K), flat_b[:B * K * 4].view(B, K, 4))
    ops.soft_nms_topk(cand, B, "gaussian", 0.3, 0.5, 0.05, K, out=out)
    assert (num[B:] == -7).all() and (flat[0][B * K:] == -7).all() and (flat[1][B * K:] == -7).all()
    assert (flat_b[B * K * 4:] == -7).all()
    assert out[0].tolist() == [K, 3, 0, K] and (out[1][1, 3:] == 0).all()
    # segment form: sentinels past keep_count in every segment, and past the arrays
    boxes, scores, classes = synth.nms_candidates_np(4, 3000, 512, 1)
    cuts = np.array([0, 1000, 1000, 3000], np.int32)
    keep = torch.full((3000 + G,), -7, dtype=torch.int64, device=DEV)
    ks = torch.full((3000 + G,), -7.0, device=DEV)
    count = torch.full((3 + G,), -7, dtype=torch.int32, device=DEV)
    bt, st, ct, seg = _t(boxes), _t(scores), _t(classes), _t(cuts)
    lib = _native.load()
    rc = lib.sihl_od_batched_soft_nms(bt.data_ptr(), st.data_ptr(), ct.data_ptr(), seg.data_ptr(), 3, 3000, 1, 0.3, 0.5, 0.001,
                                      40, keep.data_ptr(), ks.data_ptr(), count.data_ptr(), None,
                                      torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    c = count[:3].tolist()
    assert c == [40, 0, 40] and (count[3:] == -7).all()
    for s, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        assert (keep[a + c[s]:b] == -7).all() and (ks[a + c[s]:b] == -7).all()
        assert ((keep[a:a + c[s]] >= a) & (keep[a:a + c[s]] < b)).all()
    assert (keep[3000:] == -7).all() and (ks[3000:] == -7).all()


def test_cuda_graph_replay_equals_eager():
    """decode + soft_nms_topk(reset_counts=True) captured once: every replay consumes and re-zeroes the counters."""
    size, B, C, K = 640, 16, 80, 100
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(55, B, A, C, -4.0, 2.0)
    loc, cls, box = _t(maps.loc_logits), _t(maps.cls_logits), _t(maps.box_raw)
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand)
    eager = [x.clone() for x in ops.soft_nms_topk(cand, B, "gaussian", 0.3, 0.5, 0.05, K, reset_counts=True)]
    out = tuple(torch.empty_like(x) for x in eager)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, zero_counts=False)      # warm-up outside the graph
        ops.soft_nms_topk(cand, B, "gaussian", 0.3, 0.5, 0.05, K, out=out, reset_counts=True)
        with torch.cuda.graph(graph, stream=stream):
            ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, zero_counts=False)
            ops.soft_nms_topk(cand, B, "gaussian", 0.3, 0.5, 0.05, K, out=out, reset_counts=True)
    torch.cuda.current_stream().wait_stream(stream)
    for _ in range(3):
        for x in out:
            x.fill_(-1)
        graph.replay()
        torch.cuda.synchronize()
        for a, b in zip(eager, out):
            assert torch.equal(a, b)
        assert int(cand.count.abs().sum()) == 0
