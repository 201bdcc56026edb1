"""COCO crowd-region / annotated-area matching timings (CUDA events, after warm-up): the plain entries
(ops.map_match / ops.quad_map_match) against the _crowd entries (the same call with gt_crowd and gt_area) on the same
inputs, alternated round by round in one process.

    python tools/bench_map_crowd.py [--iters 20] [--rounds 3] [--out profiles/map_crowd_bench.json]

Workloads (seeded synth.map_crowd_batch_np: ground truth and detections of synth.quad_map_batch_np, ~10 % of the gts
turned into large crowd regions with a cluster of small detections inside each, area annotations with zeros and values
near the 32^2 / 96^2 boundaries; the 10 COCO thresholds and 4 area ranges): 64 images x 100 detections x 100 gt boxes
with 80 classes, and 16 images x 1 000 x 500 quads with one class (a text page with "don't care" regions).  Whether the
_crowd tables equal the oracle's on the images it checked, and the card's name and power limit, are recorded with the
times.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

import crowd_map_reference as cr  # noqa: E402
import quad_map_reference as qm  # noqa: E402
from sihl_b200 import ops, synth  # noqa: E402

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


def bench(name, geometry, B, K, G, C, oracle_images, iters, rounds):
    det, ds, dc, gt, gc, go, crowd, area = synth.map_crowd_batch_np(B * 7 + K + G, B, K, G, C, geometry=geometry)
    t = [torch.from_numpy(np.ascontiguousarray(x)).to(DEV) for x in (det, ds, dc, gt, gc, go, crowd, area)]
    match = ops.map_match if geometry == "box" else ops.quad_map_match
    fns = dict(plain=lambda: match(*t[:6]), crowd=lambda: match(*t[:6], gt_crowd=t[6], gt_area=t[7]))
    res = dict(workload=name, geometry=geometry, images=B, detections_per_image=K, gt_per_image=G, classes=C,
               crowd_gts=int(crowd.sum()), total_gts=int(go[-1]), ms=alternate(fns, iters, rounds))
    got = {k: v.cpu().numpy() for k, v in fns["crowd"]().items()}
    plain = {k: v.cpu().numpy() for k, v in fns["plain"]().items()}
    hits = got["dt_match"][:, 0, 0]
    res["matched_at_iou_0.5_area_all"] = dict(plain=int((plain["dt_match"][:, 0, 0] >= 0).sum()),
                                              crowd=int((hits >= 0).sum()),
                                              crowd_on_crowd_regions=int(crowd[hits[hits >= 0]].sum()))
    ok = True
    for b in range(oracle_images):
        g0, g1 = go[b], go[b + 1]
        if geometry == "box":
            w = cr.match_image_boxes(det[b], ds[b], dc[b], gt[g0:g1], gc[g0:g1], ops.COCO_IOU_THRESHOLDS,
                                     ops.COCO_AREA_RANGES, gt_crowd=crowd[g0:g1], gt_area=area[g0:g1])
        else:
            w = cr.match_image_quads(det[b], ds[b], dc[b], gt[g0:g1], gc[g0:g1], ops.COCO_IOU_THRESHOLDS,
                                     ops.COCO_AREA_RANGES, gt_crowd=crowd[g0:g1], gt_area=area[g0:g1])
        ok &= np.array_equal(got["det_order"][b], w["order"])
        ok &= np.array_equal(np.where(got["dt_match"][b] >= 0, got["dt_match"][b] - g0, -1), w["dt_match"])
        ok &= np.array_equal(got["dt_ignore"][b], w["dt_ignore"])
        ok &= np.array_equal(got["gt_ignore"][:, g0:g1], w["gt_ignore"])
    res["oracle_images"] = oracle_images
    res["equal_to_oracle"] = bool(ok)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_map_crowd needs a CUDA device")
    qm.shim(); cr.shim()                                          # compile the host oracle outside the timed calls
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    result = dict(gpu=smi[0] if smi else torch.cuda.get_device_name(0), iters=args.iters, rounds=args.rounds,
                  timing="CUDA events around iters back-to-back calls after 3 warm-up calls; median of rounds, arms "
                         "alternated; inputs stay resident in L2 between calls; each call includes its output and "
                         "workspace allocations from torch's caching allocator and, for the crowd arm, the conversion "
                         "of gt_crowd to uint8", workloads=[])
    specs = [("64_images_x_100_x_100_80_classes_boxes", "box", 64, 100, 100, 80, 4),
             ("16_images_x_1000_x_500_1_class_quads", "quad", 16, 1000, 500, 1, 1)]
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
