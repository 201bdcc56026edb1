"""DIoU-NMS timings against the hard NMS (CUDA events, after warm-up) on the same inputs, hard and DIoU alternated
round by round in one process.

    python tools/bench_diou_nms.py [--iters 20] [--rounds 3] [--out result.json]

Workloads: the candidate lists of cfg1 (640^2, B=64, C=80, a few hundred candidates per image), the crowd (1024^2, B=8,
thousands of candidates per image) with 80 classes and with one class — single-CTA top-K entry and the class-split
entry, which dense_postprocess picks there — and stand-alone batched NMS of 10 000 and 30 000 boxes with 1 and 80
classes (the whole-GPU bitmask path).  K = 100, threshold 0.5 for both tests.  The inputs are seeded synthetic head
outputs / boxes; list lengths and kept counts are printed with the times, with the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import diou_nms_oracle as dno  # noqa: E402
from sihl_b200 import ops, synth  # noqa: E402

DEV = "cuda:0"
THR = 0.5


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


def alternate(fns: dict, iters: int, rounds: int) -> dict:
    """Median over `rounds` of the per-call time of each function, the functions taking turns every round."""
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(cuda_ms(fn, iters))
    return {k: statistics.median(v) for k, v in times.items()}


def bench_lists(name, size, B, C, loc_mean, iters, rounds, K=100):
    levels = synth.level_sizes(size, size)
    off, sc, anchors = ops.anchor_tables(levels, size, size, DEV)
    A = anchors.shape[0]
    maps = synth.dense_maps_np(2024 + size + C, B, A, C, loc_mean, 2.0)
    t = lambda x: torch.from_numpy(x).to(DEV)
    cand = ops.CandidateBuffers.allocate(B, A, DEV)
    ops.dense_decode(t(maps.loc_logits), t(maps.cls_logits), t(maps.box_raw), off, sc, size, size, 0.05, cand,
                     mode="candidate_first")
    n = cand.count.cpu().numpy()
    n_sub = min(32, max(2, -(-cand.capacity // 2048)))
    split = cand.capacity >= ops.SPLIT_NMS_FROM and B * n_sub <= 296          # what dense_postprocess picks
    fns = {}
    for overlap in ("iou", "diou"):
        label = "hard" if overlap == "iou" else "diou"
        out = ops.nms_topk(cand, B, THR, K, overlap=overlap)
        fns[f"{label}_nms_topk"] = lambda out=out, overlap=overlap: ops.nms_topk(cand, B, THR, K, out=out, overlap=overlap)
        if split:
            fns[f"{label}_nms_topk_split"] = lambda out=out, overlap=overlap: ops.nms_topk(cand, B, THR, K, out=out, split=True,
                                                                                          overlap=overlap)
    res = dict(workload=name, image=size, batch=B, classes=C, K=K, threshold=THR, capacity=int(cand.capacity),
               list_lengths=dict(min=int(n.min()), mean=float(n.mean()), max=int(n.max())),
               ms=alternate(fns, iters, rounds))
    hard, diou = ops.nms_topk(cand, B, THR, K), ops.nms_topk(cand, B, THR, K, overlap="diou")
    res["mean_detections"] = dict(hard=float(hard[0].float().mean()), diou=float(diou[0].float().mean()))
    # spot check: image 0 against the oracle (visit order = (score desc, location asc), i.e. index order by location)
    key, box, cls = (x[0, :n[0]].cpu().numpy() for x in (cand.key, cand.box, cand.cls))
    key = key.view(np.uint64)
    perm = np.argsort(np.uint64(0xFFFFFFFF) - (key & np.uint64(0xFFFFFFFF)), kind="stable")
    scores = (key >> np.uint64(32)).astype(np.uint32).view(np.float32)
    want = perm[dno.batched_diou_nms(box[perm], scores[perm], cls[perm].astype(np.int64), THR)][:K]
    res["diou_equal_to_oracle_image0"] = bool(int(diou[0][0]) == want.size and
                                              np.array_equal(diou[3][0, :want.size].cpu().numpy(), box[want]))
    return res


def bench_standalone(n, C, iters, rounds):
    boxes, scores, classes = synth.nms_candidates_np(3 + C, n, 1024, C)
    tb, ts, tc = (torch.from_numpy(x).to(DEV) for x in (boxes, scores, classes))
    seg = torch.tensor([0, n], dtype=torch.int32, device=DEV)
    fns = {f"{'hard' if o == 'iou' else 'diou'}_batched_nms":
           (lambda o=o: ops.batched_nms(tb, ts, tc, THR, seg_offsets=seg, overlap=o)) for o in ("iou", "diou")}
    res = dict(workload=f"standalone_{n}_{C}_classes", n=n, classes=C, threshold=THR, ms=alternate(fns, iters, rounds))
    keep = ops.batched_nms(tb, ts, tc, THR, overlap="diou").cpu().numpy()
    res["kept"] = dict(hard=int(ops.batched_nms(tb, ts, tc, THR).numel()), diou=int(keep.size))
    res["diou_equal_to_oracle"] = bool(np.array_equal(keep, dno.batched_diou_nms(boxes, scores, classes, THR)))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_diou_nms needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), iters=args.iters, rounds=args.rounds, workloads=[])
    for spec in (("cfg1", 640, 64, 80, -6.0), ("crowd", 1024, 8, 80, -2.0), ("crowd_one_class", 1024, 8, 1, -2.0)):
        result["workloads"].append(bench_lists(*spec, iters=args.iters, rounds=args.rounds))
        print(json.dumps(result["workloads"][-1]), flush=True)
    for n in (10000, 30000):
        for C in (1, 80):
            result["workloads"].append(bench_standalone(n, C, args.iters, args.rounds))
            print(json.dumps(result["workloads"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(json.dumps(dict(gpu=result["gpu"])))


if __name__ == "__main__":
    main()
