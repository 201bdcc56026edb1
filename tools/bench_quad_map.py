"""Polygon-IoU COCO matching timings (CUDA events, after warm-up): ops.quad_map_match against ops.map_match on the
quads' AABBs for the same inputs (what a user of the quadrilateral head could do before), alternated round by round in
one process; DetectionMAP(iou_type="quad").compute() on the host; and the host oracle (tests/quad_map_reference.py: the
COCOeval loop in Python on the host build of the hull IoU, one CPU thread) for reference.

    python tools/bench_quad_map.py [--iters 20] [--rounds 3] [--out profiles/quad_map_bench.json]

Workloads (seeded synth.quad_map_batch_np: rotated-rectangle ground truth, detections = jittered copies of it plus
parallel-line decoys and random rectangles; the 10 COCO thresholds and 4 area ranges): 64 images x 100 detections x 100
ground-truth quads with 80 classes; 16 images x 1 000 x 500 with one class (a crowded text page); 256 images x 100 x 20
with 80 classes.  Whether the GPU tables equal the oracle's on the images it timed, and the card's name and power limit
are recorded with the times.
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

import quad_map_reference as qm  # noqa: E402
from sihl_b200 import metrics, ops, synth  # noqa: E402

DEV = "cuda:0"


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


def bench(name, B, K, G, C, oracle_images, iters, rounds):
    dq, ds, dc, gq, gc, go = synth.quad_map_batch_np(B * 7 + K + G, B, K, G, C)
    db = np.concatenate([dq.min(2), dq.max(2)], -1).astype(np.float32)
    gb = np.concatenate([gq.min(1), gq.max(1)], -1).astype(np.float32)
    tdq, tds, tdc, tgq, tgc, tgo, tdb, tgb = (torch.from_numpy(x).to(DEV) for x in (dq, ds, dc, gq, gc, go, db, gb))
    fns = dict(quad_map_match=lambda: ops.quad_map_match(tdq, tds, tdc, tgq, tgc, tgo),
               aabb_map_match=lambda: ops.map_match(tdb, tds, tdc, tgb, tgc, tgo))
    res = dict(workload=name, images=B, detections_per_image=K, gt_per_image=G, classes=C,
               same_class_pairs=int(sum(int((dc[b][:, None] == gc[go[b]:go[b + 1]][None]).sum()) for b in range(B))),
               ms=alternate(fns, iters, rounds))
    got = {k: v.cpu().numpy() for k, v in ops.quad_map_match(tdq, tds, tdc, tgq, tgc, tgo).items()}
    aabb = ops.map_match(tdb, tds, tdc, tgb, tgc, tgo)
    res["matched_at_iou_0.5_area_all"] = dict(quad=int((got["dt_match"][:, 0, 0] >= 0).sum()),
                                              aabb=int((aabb["dt_match"][:, 0, 0] >= 0).sum()))
    # DetectionMAP.compute() on the host (accumulate + summarize over the tables of this batch)
    m = metrics.DetectionMAP(sync_dist=False, iou_type="quad")
    m.update_batch(tds, tdc, tdq, tgq, tgc, np.diff(go).tolist())
    torch.cuda.synchronize()
    host = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        summary = m.compute()
        host.append((time.perf_counter() - t0) * 1e3)
    res["detection_map_compute_host_ms"] = statistics.median(host)
    res["map"] = float(summary["map"])
    # the host oracle on the first `oracle_images` images
    t0 = time.perf_counter()
    want = [qm.match_image_quads(dq[b], ds[b], dc[b], gq[go[b]:go[b + 1]], gc[go[b]:go[b + 1]], ops.COCO_IOU_THRESHOLDS,
                                 ops.COCO_AREA_RANGES) for b in range(oracle_images)]
    res["host_oracle_one_thread_ms_per_image"] = (time.perf_counter() - t0) * 1e3 / oracle_images
    res["oracle_images"] = oracle_images
    ok = True
    for b, w in enumerate(want):
        g0 = go[b]
        ok &= np.array_equal(got["det_order"][b], w["order"])
        ok &= np.array_equal(np.where(got["dt_match"][b] >= 0, got["dt_match"][b] - g0, -1), w["dt_match"])
        ok &= np.array_equal(got["dt_ignore"][b], w["dt_ignore"])
        ok &= np.array_equal(got["gt_ignore"][:, g0:go[b + 1]], w["gt_ignore"])
    res["equal_to_oracle"] = bool(ok)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_quad_map needs a CUDA device")
    qm.shim()                                                     # compile the host oracle outside the timed calls
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), iters=args.iters, rounds=args.rounds,
                  timing="CUDA events around iters back-to-back calls after 3 warm-up calls; median of rounds, arms "
                         "alternated; inputs stay resident in L2 between calls; each call includes its output and "
                         "workspace allocations from torch's caching allocator", workloads=[])
    specs = [("64_images_x_100_x_100_80_classes", 64, 100, 100, 80, 8),
             ("16_images_x_1000_x_500_1_class", 16, 1000, 500, 1, 1),
             ("256_images_x_100_x_20_80_classes", 256, 100, 20, 80, 16)]
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
