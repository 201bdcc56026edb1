"""Where the pipelined step's time goes, kernel by kernel: a torch.profiler trace (CUDA activities) of the cfg1 step
as bench.py runs it (4 lanes = steps in flight, rotating input sets, one CUDA graph per lane and set), next to the same
kernels run alone (both chains on one stream, one step after another, so no two kernels share the GPU).

Prints one JSON object: the card and its power limit; per kernel its mean duration in the pipeline and alone; how long
k_nms overlaps a dense scan (necessarily another lane's: its own scan precedes it); the scan's duration split by
whether an NMS ran beside it.  The raw traces and the summary go to OUT_DIR (default: a new temporary directory).

    python tools/step_timeline.py [--steps 200] [--out OUT_DIR] [--no-graph]

--no-graph launches the kernels directly instead of replaying graphs, for a profiler that does not resolve graph
nodes into kernels (the output says which was used and how many kernels the trace holds per step)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from bench import IOU_THR, SCORE_THR, TOPK, WORKLOADS  # noqa: E402
from sihl_b200 import ops, synth  # noqa: E402
from sihl_b200.pipeline import DetectionHeadPipeline, StepInputs  # noqa: E402

SHORT = ("k_dense_decode_tma", "k_candidate_decode", "k_nms", "k_assign_select", "k_assign_resolve", "k_pos_loss_tiles")


def short_name(name):
    for s in SHORT:
        if s + "<" in name or s + "(" in name or name.endswith(s):
            return s
    return name.split("(")[0][:60]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as exc:                       # the measurement still stands; say that the card query failed
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({exc})"}


def kernels(trace_path):
    with open(trace_path) as fh:
        ev = json.load(fh)["traceEvents"]
    out = [(short_name(e["name"]), float(e["ts"]), float(e["dur"])) for e in ev
           if e.get("ph") == "X" and e.get("cat") == "kernel"]
    return sorted(out, key=lambda k: k[1])


def overlap(a0, a1, b0, b1):
    return max(0.0, min(a1, b1) - max(a0, b0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--lanes", type=int, default=4)
    ap.add_argument("--out", default=None, help="directory for the traces and summary.json (default: a new temporary directory)")
    ap.add_argument("--no-graph", action="store_true")
    args = ap.parse_args()
    if args.out is None:
        args.out = tempfile.mkdtemp(prefix="step_timeline_")
    os.makedirs(args.out, exist_ok=True)
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    w = WORKLOADS["cfg1"]
    H, W, B, C, G, K = w["height"], w["width"], w["batch"], w["classes"], w["gt"], w["k"]
    levels = synth.level_sizes(H, W)
    A = synth.num_anchors(levels)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    n_sets = max(3, -(-(400 << 20) // (B * A * (C + 5) * 4)))    # >= 3x the L2, as bench.py
    sets = []
    for _ in range(n_sets):
        boxes, classes, offsets = synth.gt_batch_torch(gen, B, H, W, C, G, dev)
        loc, iou, box, cls = synth.dense_maps_torch(gen, B, A, C, dev)
        sets.append(StepInputs(loc, iou, box, cls, ops.GtBatch(boxes, classes, offsets, [G] * B)))
    L = args.lanes
    pipes = [DetectionHeadPipeline(levels, W, H, B, C, B * G, dev, TOPK, K, SCORE_THR, IOU_THR) for _ in range(L)]
    outs = [[pipes[ln].new_outputs() for _ in range(n_sets)] for ln in range(L)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(L)]
    main_stream = torch.cuda.current_stream(dev)
    torch.cuda.synchronize()

    graphs = None
    if not args.no_graph:
        graphs = []
        for ln in range(L):
            with torch.cuda.stream(streams[ln]):
                row = []
                for i in range(n_sets):
                    pipes[ln].step(sets[i], outs[ln][i])
                    torch.cuda.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=streams[ln]):
                        pipes[ln].step(sets[i], outs[ln][i])
                    g.replay()
                    row.append(g)
                graphs.append(row)
        torch.cuda.synchronize()

    def run(s0, n):
        for st in streams:
            st.wait_stream(main_stream)
        for s in range(s0, s0 + n):
            ln, i = s % L, s % n_sets
            if graphs is not None:
                torch.cuda.set_stream(streams[ln])
                graphs[ln][i].replay()
            else:
                with torch.cuda.stream(streams[ln]):
                    pipes[ln].step(sets[i], outs[ln][i])
        torch.cuda.set_stream(main_stream)
        for st in streams:
            main_stream.wait_stream(st)
        torch.cuda.synchronize()

    run(0, args.warmup)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(args.warmup, args.steps)
    e1.record()
    torch.cuda.synchronize()
    step_us_unprofiled = e0.elapsed_time(e1) * 1e3 / args.steps

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(args.warmup, args.steps)
    pipe_trace = os.path.join(args.out, "pipelined.json")
    prof.export_chrome_trace(pipe_trace)

    # alone: both chains on one stream, one kernel at a time
    def serial(n):
        for s in range(n):
            i = s % n_sets
            pipes[0].infer_chain(sets[i], outs[0][i])
            pipes[0].train_chain(sets[i], outs[0][i])
        torch.cuda.synchronize()

    serial(20)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        serial(min(args.steps, 100))
    alone_trace = os.path.join(args.out, "alone.json")
    prof.export_chrome_trace(alone_trace)

    kp, ka = kernels(pipe_trace), kernels(alone_trace)
    per_p, per_a = defaultdict(list), defaultdict(list)
    for n, _, d in kp:
        per_p[n].append(d)
    for n, _, d in ka:
        per_a[n].append(d)
    table = {n: {"count": len(v), "pipelined_us": sum(v) / len(v),
                 "alone_us": (sum(per_a[n]) / len(per_a[n])) if per_a.get(n) else None} for n, v in per_p.items()}

    scans = [(t, t + d) for n, t, d in kp if n == "k_dense_decode_tma"]
    nmss = [(t, t + d) for n, t, d in kp if n == "k_nms"]
    nms_total = sum(b - a for a, b in nmss)
    nms_with_scan = 0.0
    for a0, a1 in nmss:
        # union of the overlaps (at most a few scans are live at once; they do not overlap each other much, so the sum of
        # pairwise overlaps clipped to the NMS duration is a close upper bound of the union)
        nms_with_scan += min(a1 - a0, sum(overlap(a0, a1, b0, b1) for b0, b1 in scans))
    scan_beside_nms = [b1 - b0 for b0, b1 in scans if any(overlap(a0, a1, b0, b1) > 0 for a0, a1 in nmss)]
    scan_no_nms = [b1 - b0 for b0, b1 in scans if not any(overlap(a0, a1, b0, b1) > 0 for a0, a1 in nmss)]
    mean = lambda v: (sum(v) / len(v)) if v else None
    span_us = (kp[-1][1] - kp[0][1]) if kp else 0.0
    res = {
        "card": card(),
        "workload": "cfg1", "lanes": L, "steps": args.steps, "launch": "direct (--no-graph)" if graphs is None else "graph replay",
        "kernels_per_step_in_trace": len(kp) / args.steps,
        "step_us_unprofiled": step_us_unprofiled,
        "step_us_profiled_span": span_us / max(1, args.steps - 1),
        "kernels": table,
        "nms_overlapped_by_scan_fraction": (nms_with_scan / nms_total) if nms_total else None,
        "nms_overlapped_by_scan_us_per_nms": (nms_with_scan / len(nmss)) if nmss else None,
        "scan_us_with_nms_beside": mean(scan_beside_nms), "scans_with_nms_beside": len(scan_beside_nms),
        "scan_us_without_nms_beside": mean(scan_no_nms), "scans_without_nms_beside": len(scan_no_nms),
        "traces": [os.path.abspath(pipe_trace), os.path.abspath(alone_trace)],
    }
    with open(os.path.join(args.out, "summary.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
