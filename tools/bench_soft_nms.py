"""Soft-NMS timings (CUDA events, after warm-up) on the same candidate lists as the hard NMS, with two baselines in the
same run: a torch-on-GPU loop of the same algorithm (argmax + decay per selected detection, all images at once) and the
numpy oracle on the host (one thread).

    python tools/bench_soft_nms.py [--iters 20] [--out result.json]

Workloads: cfg1 (640^2, B=64, C=80), crowd (1024^2, B=8, C=80, thousands of candidates per image), the crowd with one
class, and 30 000 stand-alone boxes of one class (sihl_od_batched_soft_nms vs sihl_od_batched_nms).  The candidate
maps are seeded synthetic head outputs; the list lengths are printed with the times.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import soft_nms_oracle as sno  # noqa: E402
from sihl_b200 import ops, synth  # noqa: E402

DEV = "cuda:0"
SOFT = (("soft_linear", "linear", 0.3, 0.5), ("soft_gaussian", "gaussian", 0.3, 0.5))   # name, method, Nt, sigma


def cuda_ms(fn, iters: int, warmup: int = 3) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def torch_loop(scores, boxes, classes, method, nt, sigma, thr, K):
    """The same algorithm in eager torch on the GPU, all images at once: [B, n] padded lists sorted by location (so that
    argmax's first maximum is the lowest location), dead entries at -inf."""
    s = scores.clone()
    B = s.shape[0]
    rows = torch.arange(B, device=s.device)
    area = (boxes[..., 2] - boxes[..., 0]) * (boxes[..., 3] - boxes[..., 1])
    out_s = torch.zeros((B, K), device=s.device)
    out_i = torch.zeros((B, K), dtype=torch.int64, device=s.device)
    for k in range(K):
        m = s.argmax(dim=1)
        sm = s[rows, m]
        out_s[:, k] = torch.where(torch.isfinite(sm), sm, torch.zeros_like(sm))
        out_i[:, k] = m
        s[rows, m] = float("-inf")
        bm, cm, am = boxes[rows, m], classes[rows, m], area[rows, m]
        w_ = (torch.minimum(bm[:, None, 2], boxes[..., 2]) - torch.maximum(bm[:, None, 0], boxes[..., 0])).clamp_min(0)
        h_ = (torch.minimum(bm[:, None, 3], boxes[..., 3]) - torch.maximum(bm[:, None, 1], boxes[..., 1])).clamp_min(0)
        inter = w_ * h_
        iou = torch.nan_to_num(inter / ((am[:, None] + area) - inter), nan=0.0)
        if method == "linear":
            w = torch.where(iou > nt, 1 - iou, torch.ones_like(iou))
        else:
            w = torch.exp(-(iou.double() ** 2) / sigma).float()
        same = (classes == cm[:, None]) & torch.isfinite(s) & torch.isfinite(sm)[:, None]
        s = torch.where(same, s * w, s)
        s = torch.where(s >= thr, s, torch.full_like(s, float("-inf")))
    return out_s, out_i


def padded_lists(cand, B):
    """Candidate lists read back, sorted by location, padded to the longest with dead (-inf) entries."""
    n = cand.count.cpu().numpy()
    key, box, cls = cand.key.cpu().numpy().view(np.uint64), cand.box.cpu().numpy(), cand.cls.cpu().numpy()
    L = max(int(n.max()), 1)
    S = np.full((B, L), -np.inf, np.float32)
    Bx = np.zeros((B, L, 4), np.float32)
    Cl = np.full((B, L), -1, np.int64)
    per = []
    for b in range(B):
        k = key[b, :n[b]]
        loc = (~k & np.uint64(0xFFFFFFFF)).astype(np.int64)
        o = np.argsort(loc)
        sc = (k[o] >> np.uint64(32)).astype(np.uint32).view(np.float32)
        S[b, :n[b]], Bx[b, :n[b]], Cl[b, :n[b]] = sc, box[b, :n[b]][o], cls[b, :n[b]][o]
        per.append((k, box[b, :n[b]], cls[b, :n[b]]))
    return n, per, (torch.from_numpy(S).to(DEV), torch.from_numpy(Bx).to(DEV), torch.from_numpy(Cl).to(DEV))


def bench_lists(name, size, B, C, loc_mean, iters, K=100, thr=0.05):
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(2024 + size + C, B, A, C, loc_mean, 2.0)
    t = lambda x: torch.from_numpy(x).to(DEV)
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    ops.dense_decode(t(maps.loc_logits), t(maps.cls_logits), t(maps.box_raw), off, sc, size, size, thr, cand,
                     mode="candidate_first")
    n, per, padded = padded_lists(cand, B)
    n_sub = min(32, max(2, -(-cand.capacity // 2048)))
    split = cand.capacity >= ops.SPLIT_NMS_FROM and B * n_sub <= 296          # what dense_postprocess picks
    res = dict(workload=name, image=size, batch=B, classes=C, K=K, list_lengths=dict(min=int(n.min()), mean=float(n.mean()),
               max=int(n.max())), capacity=int(cand.capacity), ms={})
    res["ms"]["hard_nms_topk"] = cuda_ms(lambda: ops.nms_topk(cand, B, 0.5, K), iters)
    if split:
        res["ms"]["hard_nms_topk_split"] = cuda_ms(lambda: ops.nms_topk(cand, B, 0.5, K, split=True), iters)
    for label, method, nt, sigma in SOFT:
        out = ops.soft_nms_topk(cand, B, method, nt, sigma, thr, K)
        res["ms"][label] = cuda_ms(lambda: ops.soft_nms_topk(cand, B, method, nt, sigma, thr, K, out=out), iters)
        res["ms"][label + "_torch_loop"] = cuda_ms(lambda: torch_loop(*padded, method, nt, sigma, thr, K), max(2, iters // 10), 1)
        t0 = time.perf_counter()
        for key, box, cls in per:
            sno.soft_nms_candidates(key, box, cls, method, nt, sigma, thr, K)
        res["ms"][label + "_host_oracle"] = (time.perf_counter() - t0) * 1e3
        # the kernel's detections equal the oracle's (spot check on the first image)
        num, s_, c_, b_ = (x.cpu().numpy() for x in out)
        w = sno.soft_nms_candidates(*per[0], method, nt, sigma, thr, K)
        res.setdefault("equal_to_oracle_image0", {})[label] = bool(num[0] == w[0] and (s_[0] == w[1]).all() and (b_[0] == w[3]).all())
    return res


def bench_standalone(iters, n=30000, max_out=1000):
    boxes, scores, classes = synth.nms_candidates_np(3, n, 1024, 1)
    tb, ts, tc = (torch.from_numpy(x).to(DEV) for x in (boxes, scores, classes))
    res = dict(workload="standalone_30000_one_class", n=n, max_output=max_out, ms={})
    res["ms"]["hard_batched_nms"] = cuda_ms(lambda: ops.batched_nms(tb, ts, tc, 0.5), iters)
    res["hard_kept"] = int(ops.batched_nms(tb, ts, tc, 0.5).numel())
    seg = torch.tensor([0, n], dtype=torch.int32, device=DEV)
    for label, method, nt, sigma in SOFT:
        res["ms"][label] = cuda_ms(lambda: ops.batched_soft_nms(tb, ts, tc, max_out, method, nt, sigma, 0.001, seg_offsets=seg),
                                   iters)
        keep, ks = ops.batched_soft_nms(tb, ts, tc, max_out, method, nt, sigma, 0.001)
        res["ms"][label + "_torch_loop"] = cuda_ms(lambda: torch_loop(ts[None], tb[None], tc[None], method, nt, sigma, 0.001,
                                                                      max_out), 2, 1)
        t0 = time.perf_counter()
        wk, ws = sno.soft_nms(boxes, scores, classes, method, nt, sigma, 0.001, max_out)
        res["ms"][label + "_host_oracle"] = (time.perf_counter() - t0) * 1e3
        res.setdefault("equal_to_oracle", {})[label] = bool(np.array_equal(keep.cpu().numpy(), wk) and
                                                            np.array_equal(ks.cpu().numpy(), ws))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_soft_nms needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), host_cpu_count=os.cpu_count(),
                  host_oracle_threads=1, iters=args.iters, workloads=[])
    for spec in (("cfg1", 640, 64, 80, -6.0), ("crowd", 1024, 8, 80, -2.0), ("crowd_one_class", 1024, 8, 1, -2.0)):
        result["workloads"].append(bench_lists(*spec, iters=args.iters))
        print(json.dumps(result["workloads"][-1]), flush=True)
    result["workloads"].append(bench_standalone(args.iters))
    print(json.dumps(result["workloads"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(json.dumps(dict(gpu=result["gpu"], host_cpu_count=result["host_cpu_count"])))


if __name__ == "__main__":
    main()
