"""Box voting timings: the NMS alone against the NMS followed by the voting pass (CUDA events, after warm-up), on the
same inputs, the two alternated round by round in one process, for the hard and the DIoU selection.

    python tools/bench_box_vote.py [--iters 20] [--rounds 3] [--out result.json]

Workloads are those of tools/bench_diou_nms.py: the candidate lists of cfg1 (640^2, B=64, C=80, a few hundred
candidates per image), the crowd (1024^2, B=8, thousands of candidates per image) with 80 classes and with one class —
single-CTA top-K entry and the class-split entry, which dense_postprocess picks there — and stand-alone batched NMS of
10 000 and 30 000 boxes with 1 and 80 classes.  K = 100, threshold 0.5.  Each warp of the voting pass scans its whole
list, so its work is (detections x list length) class tests, of which the same-class ones also take the overlap test:
both counts are printed beside the times.  The voted boxes are checked against oracle/box_vote_oracle.py (1 ulp) in the
same run, and the card's name and power limit are read in the same run.
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

from oracle import box_vote_oracle as bvo  # noqa: E402
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


def within_one_ulp(got, want) -> bool:
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    d = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    return bool(d.size == 0 or d.max() <= 1)


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
    fns, checks, work = {}, {}, {}
    cls_all = cand.cls.cpu().numpy()
    for overlap in ("iou", "diou"):
        label = "hard" if overlap == "iou" else "diou"
        for entry in (False, True) if split else (False,):
            tag = f"{label}_nms_topk" + ("_split" if entry else "")
            out = ops.nms_topk(cand, B, THR, K, split=entry, overlap=overlap)

            def nms(out=out, entry=entry, overlap=overlap):
                ops.nms_topk(cand, B, THR, K, out=out, split=entry, overlap=overlap)

            def nms_vote(out=out, entry=entry, overlap=overlap):
                ops.nms_topk(cand, B, THR, K, out=out, split=entry, overlap=overlap)
                ops.box_vote_topk(cand, B, THR, out, overlap=overlap)

            fns[tag] = nms
            fns[tag + "+vote"] = nms_vote
        out = ops.nms_topk(cand, B, THR, K, overlap=overlap)
        ops.box_vote_topk(cand, B, THR, out, overlap=overlap)
        num, classes = out[0].cpu().numpy(), out[2].cpu().numpy()
        work[label] = dict(detections=int(num.sum()), class_tests=int((num * np.minimum(n, cand.capacity)).sum()),
                           overlap_tests=int(sum((cls_all[b, :n[b]][None, :] == classes[b, :num[b], None]).sum()
                                                 for b in range(B))))
        # image 0 against the oracle
        want = bvo.topk_vote(cand.key[:1].cpu().numpy(), cand.box[:1].cpu().numpy(), cand.cls[:1].cpu().numpy(),
                             n[:1], THR, K, overlap)
        checks[f"{label}_vote_image0_within_1ulp_of_oracle"] = bool(
            int(num[0]) == int(want[0][0]) and within_one_ulp(out[3][0].cpu().numpy(), want[3][0]))
    ms = alternate(fns, iters, rounds)
    added = {k: ms[k + "+vote"] - ms[k] for k in fns if not k.endswith("+vote")}
    return dict(workload=name, image=size, batch=B, classes=C, K=K, threshold=THR, capacity=int(cand.capacity),
                list_lengths=dict(min=int(n.min()), mean=float(n.mean()), max=int(n.max())), ms=ms, added_ms=added,
                vote_work=work, **checks)


def bench_standalone(n, C, iters, rounds):
    boxes, scores, classes = synth.nms_candidates_np(3 + C, n, 1024, C)
    tb, ts, tc = (torch.from_numpy(x).to(DEV) for x in (boxes, scores, classes))
    seg = torch.tensor([0, n], dtype=torch.int32, device=DEV)
    fns, checks, work = {}, {}, {}
    for o in ("iou", "diou"):
        label = "hard" if o == "iou" else "diou"
        fns[f"{label}_batched_nms"] = lambda o=o: ops.batched_nms(tb, ts, tc, THR, seg_offsets=seg, overlap=o)

        def nms_vote(o=o):
            keep, count = ops.batched_nms(tb, ts, tc, THR, seg_offsets=seg, overlap=o)
            ops.batched_box_vote(tb, ts, tc, keep, THR, keep_count=count, seg_offsets=seg, overlap=o)

        fns[f"{label}_batched_nms+vote"] = nms_vote
        keep = ops.batched_nms(tb, ts, tc, THR, overlap=o)
        voted = ops.batched_box_vote(tb, ts, tc, keep, THR, overlap=o).cpu().numpy()
        keep = keep.cpu().numpy()
        want_keep, want = bvo.batched_nms_vote(boxes, scores, classes, THR, o)
        same = np.bincount(classes, minlength=C)
        work[label] = dict(kept=int(keep.size), class_tests=int(keep.size) * n, overlap_tests=int(same[classes[keep]].sum()))
        checks[f"{label}_equal_keep_and_vote_within_1ulp_of_oracle"] = bool(np.array_equal(keep, want_keep) and
                                                                            within_one_ulp(voted, want))
    ms = alternate(fns, iters, rounds)
    added = {k: ms[k + "+vote"] - ms[k] for k in fns if not k.endswith("+vote")}
    return dict(workload=f"standalone_{n}_{C}_classes", n=n, classes=C, threshold=THR, ms=ms, added_ms=added,
                vote_work=work, **checks)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_box_vote needs a CUDA device")
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
