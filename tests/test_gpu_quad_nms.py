"""Quadrilateral NMS on the GPU (sihl_od_batched_quad_nms, sihl_od_quad_iou) against the host build of the same
arithmetic (tests/host_quad_shim.cpp): IoU values bit for bit, keep lists EQUAL, in every regime of the wide path."""
import numpy as np
import pytest
import torch

import quad_reference as qr
from sihl_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _eq(got, want, what=""):
    np.testing.assert_array_equal(np.asarray(got), np.asarray(want), err_msg=what)


def _size(n):
    return 1024 if n <= 8192 else 4096


def test_quad_iou_bit_equal_to_the_host():
    quads, _, _ = synth.quad_candidates_np(4, 700, 512, 1)
    quads[::5] = quads[::5, ::-1]                                        # some clockwise
    quads[1::9] = quads[1::9][:, [0, 2, 1, 3]]                          # some bow-tie orders
    quads[2::11, 3] = quads[2::11, 2]                                   # some triangles
    quads[3::13] = quads[3::13, :1]                                     # some points (zero area)
    got = ops.quad_iou(_t(quads), _t(quads[:300].reshape(-1, 8))).cpu().numpy()
    want = qr.quad_iou_matrix(quads, quads[:300])
    _eq(got.view(np.uint32), want.view(np.uint32))
    assert (want > 0).sum() > 1000
    assert ops.quad_iou(_t(quads[:0]), _t(quads)).shape == (0, 700)


@pytest.mark.parametrize("n", [0, 1, 63, 64, 65, 4097, 8192, 30000, 90000])
@pytest.mark.parametrize("n_cls", [1, 80])
def test_batched_quad_nms_vs_oracle(n, n_cls):
    quads, scores, classes = synth.quad_candidates_np(100 + n + n_cls, max(n, 1), _size(n), n_cls)
    quads, scores, classes = quads[:n], scores[:n], classes[:n]
    keep = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), 0.5).cpu().numpy()
    _eq(keep, qr.batched_quad_nms(quads, scores, classes, 0.5))


def test_many_classes():
    quads, scores, classes = synth.quad_candidates_np(3000, 30000, 4096, 3000)
    keep = ops.batched_quad_nms(_t(quads.reshape(-1, 8)), _t(scores), _t(classes), 0.3).cpu().numpy()
    _eq(keep, qr.batched_quad_nms(quads, scores, classes, 0.3))


@pytest.mark.parametrize("n", [200, 5000])
@pytest.mark.parametrize("thr", [-0.3, 0.0, 0.5, 0.9])
def test_thresholds(n, thr):
    """A negative threshold suppresses same-class quads whose AABBs are apart: the pre-reject must not skip them."""
    quads, scores, classes = synth.quad_candidates_np(31 + n, n, 1024, 4)
    keep = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), thr).cpu().numpy()
    want = qr.batched_quad_nms(quads, scores, classes, thr)
    _eq(keep, want)
    if thr < 0:
        assert want.size == len(np.unique(classes))


@pytest.mark.parametrize("sizes", [[300, 0, 57, 1, 0, 4000], [0, 0], [3000, 0, 7000, 1, 2500, 0], [100] * 64])
def test_segments_with_empty_segments(sizes):
    parts = [synth.quad_candidates_np(77 + i, max(m, 1), 800, 7) for i, m in enumerate(sizes)]
    quads = np.concatenate([p[0][:m] for p, m in zip(parts, sizes)])
    scores = np.concatenate([p[1][:m] for p, m in zip(parts, sizes)])
    classes = np.concatenate([p[2][:m] for p, m in zip(parts, sizes)])
    seg = np.zeros(len(sizes) + 1, np.int32)
    seg[1:] = np.cumsum(sizes)
    keep, count = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), 0.4, seg_offsets=_t(seg))
    keep, count = keep.cpu().numpy(), count.cpu().numpy()
    for i in range(len(sizes)):
        s, e = seg[i], seg[i + 1]
        want = qr.batched_quad_nms(quads[s:e], scores[s:e], classes[s:e], 0.4) + s
        assert count[i] == len(want), i
        _eq(keep[s:s + count[i]], want, f"segment {i}")


@pytest.mark.parametrize("n", [200, 9000])
def test_ties_and_duplicates(n):
    quads, scores, classes = synth.quad_candidates_np(5 + n, n, 1024, 3)
    scores = np.round(scores * 20).astype(np.float32) / 20                   # many tied scores: index order decides
    quads[1::4] = quads[0::4][: len(quads[1::4])]                            # duplicate quads (IoU 1)
    keep = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), 0.5).cpu().numpy()
    _eq(keep, qr.batched_quad_nms(quads, scores, classes, 0.5))
    one = np.repeat(quads[:1], 500, 0)                                       # one quad repeated: the first survives
    for s in (np.full(500, 0.5, np.float32), np.resize(scores, 500)):
        keep = ops.batched_quad_nms(_t(one), _t(s), _t(np.zeros(500, np.int64)), 0.5).cpu().numpy()
        _eq(keep, qr.batched_quad_nms(one, s, np.zeros(500, np.int64), 0.5))
        assert keep.size == 1


def _margin_ok(quads, thr):
    """True when no pair's overlap lies within 1e-5 of the threshold."""
    iou = qr.quad_iou_matrix(quads, quads)
    return not (np.abs(iou - thr) <= 1e-5).any()


def test_vertex_permutation_gives_the_same_keep():
    quads, scores, classes = synth.quad_candidates_np(9, 1500, 1024, 2)
    thr = next(t for t in (0.5, 0.45, 0.55, 0.6) if _margin_ok(quads, t))
    rng = np.random.RandomState(1)
    perm = np.stack([rng.permutation(4) for _ in range(len(quads))])
    shuffled = np.take_along_axis(quads, perm[:, :, None], 1)
    a = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), thr).cpu().numpy()
    b = ops.batched_quad_nms(_t(shuffled), _t(scores), _t(classes), thr).cpu().numpy()
    _eq(a, b)


def test_axis_aligned_quads_match_batched_nms():
    """Same keep as the box NMS on the same boxes, at thresholds no pair's IoU lies within 1e-5 of."""
    from torchvision import ops as tvops
    boxes, scores, classes = synth.nms_candidates_np(12, 2000, 1024, 3)
    x1, y1, x2, y2 = boxes.T
    quads = np.stack([np.stack([x1, y1], 1), np.stack([x2, y1], 1), np.stack([x2, y2], 1), np.stack([x1, y2], 1)], 1)
    iou = tvops.box_iou(torch.from_numpy(boxes), torch.from_numpy(boxes)).numpy()
    thresholds = [t for t in (0.3, 0.4, 0.5, 0.6, 0.7) if not (np.abs(iou - t) <= 1e-5).any()]
    assert len(thresholds) >= 2
    for thr in thresholds:
        a = ops.batched_quad_nms(_t(quads), _t(scores), _t(classes), thr).cpu().numpy()
        b = ops.batched_nms(_t(boxes), _t(scores), _t(classes), thr).cpu().numpy()
        _eq(a, b, f"thr {thr}")


def test_guard_bands_around_outputs_and_workspace():
    from sihl_b200 import _native
    lib = _native.load()
    G = 2048
    quads, scores, classes = synth.quad_candidates_np(21, 5000, 1024, 5)
    N, n_img = len(quads), 3
    seg = np.array([0, 1000, 1000, N], np.int32)
    ws_bytes = int(lib.sihl_od_batched_quad_nms_workspace_bytes(N))
    keep_buf = torch.full((N * 8 + 2 * G,), 0x5A, dtype=torch.uint8, device=DEV)
    cnt_buf = torch.full((n_img * 4 + 2 * G,), 0x5A, dtype=torch.uint8, device=DEV)
    ws_buf = torch.full((ws_bytes + 2 * G,), 0x5A, dtype=torch.uint8, device=DEV)
    tq, ts, tc, tseg = _t(quads), _t(scores), _t(classes), _t(seg)
    rc = lib.sihl_od_batched_quad_nms(tq.data_ptr(), ts.data_ptr(), tc.data_ptr(), tseg.data_ptr(), n_img, N, 0.5,
                                      keep_buf.data_ptr() + G, cnt_buf.data_ptr() + G, ws_buf.data_ptr() + G,
                                      torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    for buf in (keep_buf, cnt_buf, ws_buf):
        assert bool((buf[:G] == 0x5A).all()) and bool((buf[-G:] == 0x5A).all())
    count = cnt_buf[G:G + 4 * n_img].view(torch.int32).cpu().numpy()
    keep = keep_buf[G:G + 8 * N].view(torch.int64).cpu().numpy()
    for i in range(n_img):
        s, e = seg[i], seg[i + 1]
        want = qr.batched_quad_nms(quads[s:e], scores[s:e], classes[s:e], 0.5) + s
        _eq(keep[s:s + count[i]], want, f"segment {i}")


def test_cuda_graph_replay_of_the_segment_form_equals_eager():
    sizes = [400, 0, 3000, 600]
    quads, scores, classes = synth.quad_candidates_np(33, sum(sizes), 1024, 6)
    seg = np.zeros(len(sizes) + 1, np.int32)
    seg[1:] = np.cumsum(sizes)
    tq, ts, tc, tseg = _t(quads), _t(scores), _t(classes), _t(seg)
    eager = ops.batched_quad_nms(tq, ts, tc, 0.5, seg_offsets=tseg)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.batched_quad_nms(tq, ts, tc, 0.5, seg_offsets=tseg)                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        keep, count = ops.batched_quad_nms(tq, ts, tc, 0.5, seg_offsets=tseg)
    for _ in range(2):
        keep.fill_(-1)
        count.fill_(-1)
        g.replay()
        torch.cuda.synchronize()
        _eq(count.cpu().numpy(), eager[1].cpu().numpy())
        c = count.cpu().numpy()
        k, ke = keep.cpu().numpy(), eager[0].cpu().numpy()
        for i in range(len(sizes)):
            _eq(k[seg[i]:seg[i] + c[i]], ke[seg[i]:seg[i] + c[i]])
