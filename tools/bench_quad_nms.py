"""Quadrilateral NMS timings (CUDA events, after warm-up): ops.batched_quad_nms against ops.batched_nms on the quads'
AABBs for the same inputs (what a user of the quadrilateral head could do before), alternated round by round in one
process, and against the host oracle (tests/host_quad_shim.cpp, greedy with an AABB pre-reject, one CPU thread).

    python tools/bench_quad_nms.py [--iters 20] [--rounds 3] [--out profiles/quad_nms_bench.json]

Workloads (seeded synth.quad_candidates_np, threshold 0.5): 64 images x 100 and x 1 000 quads in one segment-form
call; one image of 10 000 and 30 000 quads with 1 and 80 classes; 90 000 quads with 80 classes.  Kept counts of both
arms, whether the GPU keep list equals the oracle's, and the card's name and power limit are recorded with the times.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import quad_reference as qr  # noqa: E402
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


def bench(name, sizes, C, size, iters, rounds):
    parts = [synth.quad_candidates_np(1000 * len(sizes) + i + C, m, size, C) for i, m in enumerate(sizes)]
    quads, scores, classes = (np.concatenate([p[k] for p in parts]) for k in range(3))
    boxes = np.concatenate([quads.min(1), quads.max(1)], 1).astype(np.float32)
    seg = np.zeros(len(sizes) + 1, np.int32)
    seg[1:] = np.cumsum(sizes)
    tq, tb, ts, tc, tseg = (torch.from_numpy(x).to(DEV) for x in (quads, boxes, scores, classes, seg))
    fns = dict(quad_nms=lambda: ops.batched_quad_nms(tq, ts, tc, THR, seg_offsets=tseg),
               aabb_batched_nms=lambda: ops.batched_nms(tb, ts, tc, THR, seg_offsets=tseg))
    res = dict(workload=name, images=len(sizes), quads=int(seg[-1]), classes=C, image_size=size, threshold=THR,
               ms=alternate(fns, iters, rounds))
    kq, cq = (x.cpu().numpy() for x in ops.batched_quad_nms(tq, ts, tc, THR, seg_offsets=tseg))
    _, cb = ops.batched_nms(tb, ts, tc, THR, seg_offsets=tseg)
    res["kept"] = dict(quad_nms=int(cq.sum()), aabb_batched_nms=int(cb.sum()))
    t0 = time.perf_counter()
    want = [qr.batched_quad_nms(quads[s:e], scores[s:e], classes[s:e], THR) + s for s, e in zip(seg[:-1], seg[1:])]
    res["host_oracle_one_thread_ms"] = (time.perf_counter() - t0) * 1e3
    res["equal_to_oracle"] = bool(all(np.array_equal(kq[s:s + c], w) for s, c, w in zip(seg[:-1], cq, want)))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_quad_nms needs a CUDA device")
    qr.shim()                                                     # compile the host oracle outside the timed calls
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), iters=args.iters, rounds=args.rounds,
                  timing="CUDA events around iters back-to-back calls after 3 warm-up calls; median of rounds, arms "
                         "alternated; inputs stay resident in L2 between calls", workloads=[])
    specs = [("64_images_x_100", [100] * 64, 80, 1024), ("64_images_x_1000", [1000] * 64, 80, 1024),
             ("10000_1_class", [10000], 1, 4096), ("10000_80_classes", [10000], 80, 4096),
             ("30000_1_class", [30000], 1, 4096), ("30000_80_classes", [30000], 80, 4096),
             ("90000_80_classes", [90000], 80, 4096)]
    for spec in specs:
        result["workloads"].append(bench(*spec, iters=args.iters, rounds=args.rounds))
        print(json.dumps(result["workloads"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(json.dumps(dict(gpu=result["gpu"])))


if __name__ == "__main__":
    main()
