"""Memory-safety net for the kernels (``compute-sanitizer`` is closed on this GPU pool: the call is refused).

Every tensor that ``sihl_b200.ops`` / ``sihl_b200.pipeline`` allocate — outputs, candidate lists, NMS / train workspaces,
tile lists — is carved out of a larger allocation whose 2 KiB before and after are filled with a sentinel byte; after
the kernels ran the sentinels must be intact.  Covers the hand-rolled shared/global carving of the NMS kernels in all
their regimes (<= 256 candidates, <= 4096 in shared memory, spill to the global workspace, > 512 classes, the class-split
variant, stand-alone batched NMS), ``cap``-limited candidate lists, capacity-limited positive lists and the training
entry points with padding rows.  Results are checked elsewhere (test_gpu_parity.py); here only the bytes next to every
buffer are.
"""
import numpy as np
import pytest
import torch

from sihl_b200 import ops, pipeline, synth

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
PAD, SENTINEL = 2048, 0xA5


class GuardedTorch:
    """Drop-in for the ``torch`` module inside ops / pipeline: device allocations get guard bands."""

    def __init__(self):
        self.guards = []

    def __getattr__(self, name):
        return getattr(torch, name)

    def _alloc(self, shape, dtype, device, fill=None):
        if isinstance(shape, int):
            shape = (shape,)
        shape = tuple(int(s) for s in shape)
        dtype = dtype or torch.float32
        n = int(np.prod(shape, dtype=np.int64)) * torch.empty((), dtype=dtype).element_size()
        base = torch.full((n + 2 * PAD,), SENTINEL, dtype=torch.uint8, device=device)
        view = base[PAD:PAD + n].view(dtype).view(shape)
        if fill is not None:
            view.fill_(fill)
        self.guards.append((base, n, shape, dtype))
        return view

    def _on_device(self, device):
        return device is not None and torch.device(device).type == "cuda"

    def empty(self, *size, dtype=None, device=None, **kw):
        shape = size[0] if len(size) == 1 else size
        if not self._on_device(device):
            return torch.empty(*size, dtype=dtype, device=device, **kw)
        return self._alloc(shape, dtype, device)

    def zeros(self, *size, dtype=None, device=None, **kw):
        shape = size[0] if len(size) == 1 else size
        if not self._on_device(device):
            return torch.zeros(*size, dtype=dtype, device=device, **kw)
        return self._alloc(shape, dtype, device, fill=0)

    def full(self, size, value, dtype=None, device=None, **kw):
        if not self._on_device(device):
            return torch.full(size, value, dtype=dtype, device=device, **kw)
        return self._alloc(size, dtype if dtype is not None else (torch.int64 if isinstance(value, int) else torch.float32),
                           device, fill=value)

    def empty_like(self, t, dtype=None, **kw):
        return self._alloc(t.shape, dtype or t.dtype, t.device) if t.is_cuda else torch.empty_like(t, dtype=dtype, **kw)

    def zeros_like(self, t, dtype=None, **kw):
        return self._alloc(t.shape, dtype or t.dtype, t.device, fill=0) if t.is_cuda else torch.zeros_like(t, dtype=dtype, **kw)

    def check(self):
        torch.cuda.synchronize()
        assert self.guards, "nothing was allocated through the guarded allocator"
        for base, n, shape, dtype in self.guards:
            lo, hi = base[:PAD], base[PAD + n:]
            ok = bool((lo == SENTINEL).all()) and bool((hi == SENTINEL).all())
            assert ok, f"guard band of a {dtype} tensor of shape {shape} was overwritten " \
                       f"(before: {int((lo != SENTINEL).sum())} bytes, after: {int((hi != SENTINEL).sum())} bytes)"
        return len(self.guards)


@pytest.fixture
def guarded(monkeypatch):
    g = GuardedTorch()
    monkeypatch.setattr(ops, "torch", g)
    monkeypatch.setattr(pipeline, "torch", g)
    ops._anchor_cache.clear(); ops._geom_cache.clear()          # tables are re-created through the guarded allocator
    yield g
    ops._anchor_cache.clear(); ops._geom_cache.clear()


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _maps(seed, B, A, C, loc_mean, loc_std=2.0):
    m = synth.dense_maps_np(seed, B, A, C, loc_mean=loc_mean, loc_std=loc_std)
    return _t(m.loc_logits), _t(m.iou_preds), _t(m.box_raw), _t(m.cls_logits)


@pytest.mark.parametrize("size,B,C,loc_mean,cap,K,what", [
    (128, 3, 16, -3.0, None, 100, "short lists (<= 256 candidates)"),
    (320, 2, 80, 0.0, None, 100, "lists in shared memory (~1000 candidates)"),
    (1024, 2, 80, 1.0, None, 100, "lists beyond 4096: global workspace"),
    (640, 2, 600, 0.0, None, 50, "more than 512 distinct classes: sort fallback"),
    (640, 3, 80, 0.0, 64, 100, "cap-limited lists (capacity 64 << candidates)"),
    (640, 2, 1, 2.0, 1000, 300, "one class, K = 300, capacity 1000 < candidates"),
])
@pytest.mark.parametrize("mode", ops.DECODE_MODES)
def test_decode_and_nms_stay_inside_their_buffers(guarded, size, B, C, loc_mean, cap, K, what, mode):
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    loc, _, box, cls = _maps(11, B, A, C, loc_mean)
    cand = ops.CandidateBuffers.allocate(B, cap or A, DEV)
    num, scores, classes, boxes = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, cand=cand, mode=mode,
                                                        split_nms=False)
    assert int(num.max()) <= K
    guarded.check()
    if cap is None:
        num2, *_ = ops.dense_postprocess(loc, cls, box, levels, size, size, 0.05, 0.5, K, mode=mode, split_nms=True)
        assert torch.equal(num, num2)
        guarded.check()


@pytest.mark.parametrize("n,n_cls,segments", [(200, 3, 1), (3000, 80, 2), (12000, 1, 1), (30000, 80, 3), (5000, 700, 1)])
def test_batched_nms_stays_inside_its_buffers(guarded, n, n_cls, segments):
    rng = np.random.RandomState(n)
    xy = rng.uniform(0, 900, (n, 2)).astype(np.float32)
    wh = rng.uniform(4, 300, (n, 2)).astype(np.float32)
    boxes = _t(np.concatenate([xy, xy + wh], 1))
    scores = _t(rng.uniform(0.05, 1, n).astype(np.float32))
    idxs = _t(rng.randint(0, n_cls, n).astype(np.int64))
    cuts = np.linspace(0, n, segments + 1).astype(np.int32)
    keep, count = ops.batched_nms(boxes, scores, idxs, 0.5, seg_offsets=_t(cuts))
    assert int(count.sum()) > 0
    guarded.check()


def test_training_and_assignment_entries_stay_inside_their_buffers(guarded):
    size, B, C, G = 320, 3, 10, 20
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    gt = synth.gt_batch_np(5, B, size, size, C, G, counts=[20, 0, 7])
    loc, iou, box, cls = _maps(6, B, A, C, -3.0)
    gt_boxes, gt_classes = _t(gt.boxes), _t(gt.classes)
    for capacity in (None, 40):                       # None: 9 * sumG rows; 40: fewer rows than positives
        st = ops.train_assign(levels, size, size, gt_boxes, gt_classes, [20, 0, 7], B, 9, pos_capacity=capacity)
        P = int(st.pos_total.item())
        assert P > 40 and (capacity is None or st.capacity == 40)
        bx = box.view(-1, 4).index_select(0, st.pos_index.long())
        cl = cls.view(-1, C).index_select(0, st.pos_index.long())
        for dtype in (torch.float32, torch.bfloat16, torch.float16):
            maps_in = [t.to(dtype) for t in (loc, iou, bx, cl)]
            losses, maps = ops.train_loss(st, *maps_in)
            grads = ops.train_loss_bwd(st, maps, None)
            assert all(g.dtype == dtype for g in grads)
            st = ops.train_assign(levels, size, size, gt_boxes, gt_classes, [20, 0, 7], B, 9, pos_capacity=capacity)
    # device-resident offsets (the CUDA-graph form) + the unfused building blocks with their tile lists
    ops.train_assign(levels, size, size, gt_boxes, gt_classes, None, B, 9, gt_offsets=_t(gt.offsets))
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    g = ops.GtBatch(gt_boxes, gt_classes, _t(gt.offsets), [20, 0, 7])
    sums = ops.new_sums(DEV)
    sel = ops.assign_select(anchors, levels, size, size, g, 9, sums=sums)
    ops.assign_resolve(sel, g, A, 9, True, loc, iou, sums,
                       fused=dict(box_raw=box, cls_logits=cls, offsets=off, scales=sc, img_w=size, img_h=size))
    ops.loss_finalize(sums)
    ops.bbox_matching(anchors, gt_boxes[:20], 9, True)
    ops.quad_bbox_matching(anchors, g, 9)
    top, idx = ops.topk_locations(loc, 100)
    rows = torch.arange(B, device=DEV).view(B, 1)
    ops.decode_rows(top, idx, cls[rows, idx], box[rows, idx], off, sc, size, size)
    assert guarded.check() > 40


@pytest.mark.parametrize("mode", ops.DECODE_MODES)
def test_pipeline_buffers_are_not_overrun(guarded, mode):
    size, B, C, G = 256, 3, 16, 12
    levels = synth.level_sizes(size, size)
    pipe = pipeline.DetectionHeadPipeline(levels, size, size, B, C, B * G, DEV, decode_mode=mode)
    gt = synth.gt_batch_np(31, B, size, size, C, G, ragged=False)
    loc, iou, box, cls = _maps(32, B, pipe.A, C, -2.0)
    x = pipeline.StepInputs(loc, iou, box, cls, ops.GtBatch(_t(gt.boxes), _t(gt.classes), _t(gt.offsets), [G] * B))
    out = pipe.new_outputs()
    for _ in range(3):
        pipe.step(x, out)
    assert torch.isfinite(out.losses).all()
    guarded.check()


def test_map_match_stays_inside_its_buffers(guarded):
    rng = np.random.RandomState(3)
    B, K, G = 4, 33, 9
    xy = rng.uniform(0, 300, (B, K, 2)).astype(np.float32)
    det = np.concatenate([xy, xy + rng.uniform(5, 120, (B, K, 2)).astype(np.float32)], -1)
    gxy = rng.uniform(0, 300, (3 * G, 2)).astype(np.float32)
    gtb = np.concatenate([gxy, gxy + rng.uniform(5, 120, (3 * G, 2)).astype(np.float32)], -1)
    off = np.array([0, G, G, 2 * G, 3 * G], np.int32)                  # image 1 has no ground truth
    res = ops.map_match(_t(det), _t(rng.uniform(0, 1, (B, K)).astype(np.float32)), _t(rng.randint(0, 3, (B, K)).astype(np.int64)),
                        _t(gtb), _t(rng.randint(0, 3, 3 * G).astype(np.int64)), _t(off))
    assert res["dt_match"].shape == (B, 4, 10, K)
    guarded.check()


@pytest.mark.parametrize("loc_mean,what", [(-5.0, "short lists"), (-2.0, "lists beyond 256: lazy prefix, then the full-list body")])
def test_nms_survives_lists_with_repeated_entries(guarded, loc_mean, what):
    """Not a valid input (sihl_od.h: keys must be distinct) but a plausible mistake — the decode called twice without
    zeroing the counters appends every candidate twice.  The ranks stay a permutation, so nothing is read or written
    out of bounds and the call completes; (an earlier version took stale shared-memory indices and faulted)."""
    size, B, C, K = 640, 2, 80, 100
    levels = synth.level_sizes(size, size)
    A = synth.num_anchors(levels)
    loc, _, box, cls = _maps(21, B, A, C, loc_mean, 1.0)
    off, sc, _ = ops.anchor_tables(levels, size, size, DEV)
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    for _ in range(3):
        ops.dense_decode(loc, cls, box, off, sc, size, size, 0.05, cand, zero_counts=False)
    num, scores, classes, boxes = ops.nms_topk(cand, B, 0.5, K, reset_counts=True)
    torch.cuda.synchronize()
    assert int(num.max()) <= K and int(cand.count.sum()) == 0 and torch.isfinite(boxes).all()
    guarded.check()
