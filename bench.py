#!/usr/bin/env python
"""bench.py — det-head images/sec (assign + loss + NMS), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg1] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic head outputs per GPU:
CIoU top-9 assignment + the four loss reductions (train chain) and dense decode + class-aware
NMS (inference chain).  Workload ``cfg1`` = BASELINE.json configs[1]: 640x640, batch 64 per GPU,
P3-P7 (A=8525), 80 classes, 100 gt / image, synthetic maps (SURVEY.md §8d distributions).
Multi-GPU = the same batch per GPU (weak scaling, configs[2]: 512 images on 8 GPUs); the one
exchange, the 8 fp64 loss sums, is done by the loss kernel itself over NVLink peer memory
(``--allreduce nccl``: an NCCL all-reduce node + a finalize launch instead).

Prints ONE JSON line (rank 0):
  ``value``              inputs resident in HBM, CUDA-graph replay, device timed, dense class-map scan
  ``other_decode_mode``  the same step with the candidate-first decode (same outputs), same run
  ``e2e``                the step through the public API from pinned HOST buffers, results read back
                         every step; class / box maps are read in place over PCIe (candidate-first)
  ``e2e_full_upload``    the same with every input tensor uploaded
  ``roofline``           the dominant kernel (k_dense_decode_tma) timed alone against MEASURED_PEAKS.json
  ``roofline_step``      the whole step against SURVEY.md §8d's algorithmic bytes per image
  ``cpu_baseline``       the reference's OWN functions (oracle/ref_path.py over oracle/ref_loader.py: /root/reference or
                         the staged copy oracle/_ref/sihl_src; "port" only if neither exists) on the host cores, all
                         threads, bounded sample; ``gpu_eager_reference``: the same code as torch eager on this GPU

  ``config``             the workload, identical in both arms; ``execution`` (graph, streams, steps in flight, decode
                         mode) and ``workload_stats`` (positives / candidates / detections per image) describe this arm

``--impl reference``: only that CPU arm (rank 0), same metric/unit/config.

``--steps K`` is the number of timed steps of ``value`` (after ``--warmup`` untimed ones).  ``--dump-outputs DIR``: the
StepOutputs of the last of them (rank 0) as ``DIR/<field>.npy``, a few MB at every workload.  The inputs come from fixed
seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "det-head images/sec (assign+loss+NMS)"
UNIT = "images/s"
WORKLOADS = {
    # name: (height, width, batch per GPU, classes, gt per image, max_instances)
    "cfg1": dict(height=640, width=640, batch=64, classes=80, gt=100, k=100, desc="ObjectDetection head 640x640 b64 P3-P7 C80 G100"),
    "cfg0": dict(height=320, width=320, batch=2, classes=10, gt=20, k=100, desc="examples/object_detection.py head 320x320 b2 C10 G20"),
    "crowd": dict(height=1024, width=1024, batch=8, classes=80, gt=500, k=100, desc="dense-crowd 1024x1024 b8 C80 G500"),
    # the same geometry at a batch whose kernels are long enough (4 x 57 MB per scan) that launch + ramp + tail stop dominating:
    # separates "the kernel does not stream at this geometry" from "a 10 us kernel pays 4 us of fixed cost" (DESIGN.md §8)
    "crowd32": dict(height=1024, width=1024, batch=32, classes=80, gt=500, k=100, desc="dense-crowd 1024x1024 b32 C80 G500"),
}
SCORE_THR, IOU_THR, TOPK = 0.05, 0.5, 9
HBM_FALLBACK_GBS = 6650.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg1", choices=sorted(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true", help="launch kernels directly instead of replaying CUDA graphs")
    ap.add_argument("--serial", action="store_true", help="run both chains on one stream")
    ap.add_argument("--lanes", type=int, default=0, help="steps in flight (independent scratch + stream each); 0 = 4 on one GPU, 6 on several")
    ap.add_argument("--decode-mode", default="dense", choices=["dense", "candidate_first"],
                    help="inference chain of the timed step: dense class-map scan (TMA ring, the roofline kernel) or the "
                         "candidate-first gather (same outputs, ~30x fewer bytes at 2 %% candidates)")
    ap.add_argument("--skip-candidate-first", action="store_true", help="do not also time the candidate-first variant")
    ap.add_argument("--allreduce", default="fused", choices=["fused", "nccl"],
                    help="multi-GPU exchange of the 8 loss sums: inside the loss kernel over NVLink peer memory (fused) "
                         "or an NCCL all-reduce node + a finalize launch per step (nccl)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-gpu-eager", action="store_true")
    ap.add_argument("--regions", type=int, default=1,
                    help="split the --steps timed steps into this many regions; the line reports the median region's time "
                         "per step (SURVEY.md §8d), min/max and per-rank times beside it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy "
                         "(float32, or float64 for the fp64 sums)")
    ap.add_argument("--skip-half-maps", action="store_true", help="do not also time the step on bf16 head outputs")
    ap.add_argument("--skip-mlp", action="store_true", help="do not also time the MLP towers in front of the path (row N4)")
    ap.add_argument("--skip-train-tail", action="store_true", help="do not time the drop-in head's training tail with backward")
    ap.add_argument("--e2e-steps", type=int, default=60)
    ap.add_argument("--e2e-lanes", type=int, default=3, help="end-to-end steps in flight (own stream + buffers each)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def config_dict(w, args, world, extra=None):
    from sihl_b200 import synth
    levels = synth.level_sizes(w["height"], w["width"])
    cfg = {
        "workload": f"{args.workload}: {w['desc']}",
        "image": [w["height"], w["width"]], "levels": [list(l) for l in levels], "anchors": synth.num_anchors(levels),
        "batch_per_gpu": w["batch"], "global_batch": w["batch"] * world, "classes": w["classes"], "gt_per_image": w["gt"],
        "max_instances": w["k"], "topk": TOPK, "score_thr": SCORE_THR, "iou_thr": IOU_THR,
        "parallelism": (f"batch-sharded x{world}, 8 fp64 loss sums all-reduced " +
                        ("inside the loss kernel over NVLink peer memory" if args.allreduce == "fused" else "by NCCL"))
        if world > 1 else "single GPU",
        "cache": "rotating input sets, together >= 400 MB (> 3x the 126 MB L2): every step streams from HBM, no flush needed",
    }
    cfg.update(extra or {})
    return cfg


# ----------------------------------------------------------------------------- CPU arm
def reference_kind():
    """Which code the baseline legs run: the reference's own functions ("reference" = /root/reference, "oracle/_ref" =
    the byte-for-byte staged copy that travels to the GPU box) or, if neither exists, the operator-for-operator
    restatement ("port")."""
    from oracle import ref_loader
    return ref_loader.kind() if ref_loader.available() else "port"


def make_reference_pass(w, levels, boxes, classes, loc, iou, box, cls):
    """One pass of the path by the baseline on the given (host or device) tensors -> callable."""
    import torch
    H, W, C, K = w["height"], w["width"], w["classes"], w["k"]
    if reference_kind() != "port":
        from oracle import ref_path
        path = ref_path.ReferencePath(levels, H, W, C, boxes, classes, loc, iou, box, cls, K)
        return lambda: path.one_pass(SCORE_THR, IOU_THR)
    from oracle import torch_restatement as tr

    def one_pass():
        with torch.no_grad():
            tr.train_losses(levels, W, H, boxes, classes, loc, iou, box, cls, TOPK)
            tr.dense_postprocess(levels, W, H, loc, box, cls, SCORE_THR, IOU_THR, K)
    return one_pass


def cpu_reference_images_per_sec(w, sample, steps, warmup, seed=1234, budget_s=150.0):
    """The reference's own implementation of the path on the host cores (torch CPU, all threads): its unmodified
    ``ObjectDetection.training_step`` — anchors, the per-image ``bbox_matching`` loop, compaction, four losses (ref
    object_detection.py:124-217) — on synthetic head outputs, + dense decode + ``torchvision.ops.batched_nms`` (the
    NMS extension; the reference has no NMS).  ``sample`` images per pass, shrunk only if steps x sample would exceed
    ``budget_s`` of host time."""
    import torch
    from sihl_b200 import synth

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    H, W, C, G = w["height"], w["width"], w["classes"], w["gt"]
    levels = synth.level_sizes(H, W)
    A = synth.num_anchors(levels)

    def make(n):
        gt = synth.gt_batch_np(seed, n, H, W, C, G, ragged=False)
        maps = synth.dense_maps_np(seed + 1, n, A, C)
        boxes = [torch.from_numpy(b.copy()) for b, _ in gt.per_image()]
        classes = [torch.from_numpy(c.copy()) for _, c in gt.per_image()]
        t = torch.from_numpy
        return make_reference_pass(w, levels, boxes, classes, t(maps.loc_logits), t(maps.iou_preds), t(maps.box_raw),
                                   t(maps.cls_logits))

    probe = make(1)
    probe()
    t0 = time.perf_counter(); probe(); t_img = time.perf_counter() - t0
    sample = max(1, min(sample, w["batch"], int(budget_s / max((steps + warmup) * t_img, 1e-9))))
    one_pass = make(sample)
    for _ in range(warmup):
        one_pass()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_pass()
    elapsed = time.perf_counter() - t0
    return dict(value=sample * steps / elapsed, seconds=elapsed, sample_images=sample, cores=cores, steps=steps,
                kind=reference_kind())


REFERENCE_WHAT = ("the reference's unmodified ObjectDetection.training_step (assign + losses, ref object_detection.py:124-217) "
                  "on synthetic head outputs + dense decode + torchvision.ops.batched_nms")


def run_reference_arm(args, w, world, rank):
    if rank != 0:
        return
    steps, warmup = max(args.steps, 1), max(args.warmup, 0)
    r = cpu_reference_images_per_sec(w, w["batch"], steps, warmup)
    sample = (f"{r['sample_images']} of {w['batch']} images per step of {args.workload}: {REFERENCE_WHAT}; torch "
              f"{r['cores']} threads, {steps} steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": 1e3 * r["seconds"] / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(w, args, world),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("kind 'reference' / 'oracle/_ref': the reference's own Python functions, imported unmodified (from /root/reference, "
                 "or from the byte-for-byte staged copy oracle/_ref/sihl_src made by oracle/stage_reference.py, which travels to the "
                 "GPU box); kind 'port': oracle/torch_restatement.py, only when neither exists"),
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        self.marks = []

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        self.marks.append(time.perf_counter())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        lo, hi = (self.marks[0], self.marks[-1]) if len(self.marks) >= 2 else (0, float("inf"))
        sm, mx, reasons, allsm = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, cmax = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            allsm.append(clk)
            if lo - 0.06 <= t <= hi + 0.06:
                sm.append(clk); mx.append(cmax)
                for n, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        use = sm or allsm
        return {"sm_mhz": statistics.median(use) if use else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_rank_to_gpu_numa(local_rank, world):
    """Multi-GPU end-to-end runs feed every GPU from pinned host memory: give each rank its own slice of the CPUs that
    are local to its GPU (NVML CPU affinity), BEFORE any pinned buffer is allocated, so that the rank's host thread and
    (first-touch) its pinned pages sit on the GPU's NUMA node and the ranks do not share cores.  Returns what was done."""
    if world <= 1 or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        local = [c for c in range(n_cpu) if (int(words[c // 64]) >> (c % 64)) & 1]
        allowed = sorted(set(local) & set(os.sched_getaffinity(0))) or sorted(os.sched_getaffinity(0))
        # ranks whose GPUs share this CPU set split it evenly (local ranks are 0..world-1 on one node)
        sharing = []
        for r in range(world):
            wr = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(r), (n_cpu + 63) // 64)
            if list(wr) == list(words):
                sharing.append(r)
        per = max(1, len(allowed) // max(1, len(sharing)))
        k = sharing.index(local_rank) if local_rank in sharing else 0
        mine = allowed[k * per:(k + 1) * per] or allowed
        os.sched_setaffinity(0, mine)
        return {"gpu_local_cpus": len(local), "ranks_sharing_them": len(sharing), "bound_to": [mine[0], mine[-1]], "n_bound": len(mine)}
    except Exception as exc:                                  # noqa: BLE001 - affinity is an optimisation, never fatal
        return {"error": str(exc)[:120]}


# ----------------------------------------------------------------------------- our arm
def dump_outputs(directory, out):
    """One ``<field>.npy`` per field of ``out`` (a StepOutputs): float64 for the fp64 loss sums, float32 for the rest; the
    integer fields (gt indices, counts, class ids) are exact in float32."""
    import dataclasses

    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for f in dataclasses.fields(out):
        t = getattr(out, f.name).cpu()
        t = t if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(directory, f.name + ".npy"), t.numpy())


def run_ours(args, w, world, rank, local_rank):
    import torch
    import torch.distributed as dist

    from sihl_b200 import ops, synth
    from sihl_b200.pipeline import LAUNCHES_PER_STEP, DetectionHeadPipeline, StepInputs

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    affinity = bind_rank_to_gpu_numa(local_rank, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    H, W, B, C, G, K = w["height"], w["width"], w["batch"], w["classes"], w["gt"], w["k"]
    levels = synth.level_sizes(H, W)
    # steps in flight: 4 on one GPU; 6 when the loss kernel waits for its peers' sums (measured at 2 GPUs, same box:
    # 4 lanes 39.4 us, 6 lanes 39.0 us, 8 lanes 40.4 us per step; one GPU: 38.60 vs 38.57 us)
    n_lanes = args.lanes if args.lanes > 0 else (4 if world == 1 else 6)
    if args.lanes <= 0 and w["batch"] * synth.num_anchors(levels) < 250_000:
        n_lanes = 8          # small steps (crowd: 8 images) are latency-bound kernel by kernel: 4 lanes 18.7 us, 8 lanes 17.5 us
    A = synth.num_anchors(levels)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + 1000 * rank)
    # rotating input sets: together at least 3x the 126 MB L2, so that every step streams from HBM (3 sets of 188 MB at
    # cfg1; the small workloads need more sets)
    n_sets = min(16, max(3, -(-(400 << 20) // (B * A * (C + 5) * 4))))
    if os.environ.get("SIHL_BENCH_SETS"):                  # developer A/B: more rotating sets than needed
        n_sets = max(n_sets, int(os.environ["SIHL_BENCH_SETS"]))
    sets = []
    for _ in range(n_sets):
        boxes, classes, offsets = synth.gt_batch_torch(gen, B, H, W, C, G, dev)
        loc, iou, box, cls = synth.dense_maps_torch(gen, B, A, C, dev)
        sets.append(StepInputs(loc, iou, box, cls, ops.GtBatch(boxes, classes, offsets, [G] * B)))
    torch.cuda.synchronize()

    multi = world > 1
    use_graph = not args.no_graph
    main = torch.cuda.current_stream(dev)
    _lp = os.environ.get("SIHL_LANE_PRIORITY")            # developer A/B: CUDA priority of the lanes' (train-chain) streams
    lane_streams = [torch.cuda.Stream(device=dev) if _lp is None else torch.cuda.Stream(device=dev, priority=int(_lp))
                    for _ in range(n_lanes)]

    # multi-GPU: one NCCL communicator per lane (collectives of different lanes may be in flight at once)
    groups = [dist.new_group(ranks=list(range(world)), backend="nccl") for _ in range(n_lanes)] if multi else None
    if multi:
        for ln in range(n_lanes):                      # create the communicators eagerly, outside any capture
            dist.all_reduce(torch.zeros(8, dtype=torch.float64, device=dev), group=groups[ln])
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    fused = multi and args.allreduce == "fused"
    exchanges = []

    fallback_note = []

    def attach(pipes):
        """fused exchange: one region per pipeline (= per step in flight); collective across the ranks.  If peer memory
        cannot be set up (no CUDA IPC / P2P between the ranks) every rank learns it and all fall back to NCCL."""
        nonlocal fused
        if fused:
            from sihl_b200.dist import PeerExchange
            try:
                ex = PeerExchange(dev, n_regions=len(pipes) + 1)      # + one region for the device-side start barrier
            except RuntimeError as exc:
                fused = False
                args.allreduce = "nccl"
                fallback_note.append(str(exc))
                return pipes
            exchanges.append(ex)
            for i, pp in enumerate(pipes):
                pp.attach_exchange(ex, i)
                pp.start_barrier = (ex, len(pipes))
        return pipes

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(mode, steps, warmup, n_regions, in_sets=None):
        """Build the lanes for one decode mode, replay `warmup` steps and then `steps` timed steps split into `n_regions`
        regions, return (median region ms per step, pipes, outs, graphs, timing, outputs of the last timed step)."""
        pipes = attach([DetectionHeadPipeline(levels, W, H, B, C, B * G, dev, TOPK, K, SCORE_THR, IOU_THR, decode_mode=mode)
                        for _ in range(n_lanes)])
        # every (lane, input set) pair owns its outputs: steps in flight on different lanes never share a buffer
        outs = [[pipes[ln].new_outputs() for _ in range(n_sets)] for ln in range(n_lanes)]
        torch.cuda.synchronize()
        return _timed_steps(pipes, outs, steps, warmup, n_regions, in_sets if in_sets is not None else sets)

    def _timed_steps(pipes, outs, n_steps, n_warmup, n_regions, sets):
        def full_step(ln, i):
            """One step incl. the cross-GPU exchange: 8 fp64 sums all-reduced between the loss kernels and finalize."""
            out = outs[ln][i]

            def exchange():                               # right after the loss kernels, next to the inference chain
                dist.all_reduce(out.sums, op=dist.ReduceOp.SUM, group=groups[ln])
                pipes[ln].finalize(out)

            separate = multi and not fused                # NCCL all-reduce node + finalize launch after the loss kernel
            if args.serial:
                pipes[ln].infer_chain(sets[i], out); pipes[ln].train_chain(sets[i], out, finalize=not separate)
                if separate:
                    exchange()
            else:
                pipes[ln].step(sets[i], out, finalize=not separate, after_train=exchange if separate else None)

        graphs = None
        if use_graph and not args.serial:
            graphs = []
            for ln in range(n_lanes):
                with torch.cuda.stream(lane_streams[ln]):
                    lane_graphs = []
                    for i in range(n_sets):
                        full_step(ln, i)                       # warm-up outside capture
                        torch.cuda.synchronize()
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g, stream=lane_streams[ln]):
                            full_step(ln, i)                   # NCCL all-reduce is captured as a graph node
                        g.replay()                             # a graph's first launch is slower: keep it out of the timing
                        lane_graphs.append(g)
                    graphs.append(lane_graphs)
            torch.cuda.synchronize()

        def run_step(s):
            """Step s goes to lane s % n_lanes: consecutive steps overlap (the HBM-bound decode of one step runs
            next to the latency-bound assignment / NMS kernels of its neighbours)."""
            ln, i = s % n_lanes, s % n_sets
            if graphs is not None:
                # set_stream, not the `with torch.cuda.stream(...)` context manager: enqueueing a step costs the host
                # ~11 us with the latter, which is all of cfg0's step; issue_done() puts the main stream back
                torch.cuda.set_stream(lane_streams[ln])
                graphs[ln][i].replay()
            else:
                with torch.cuda.stream(lane_streams[ln]):
                    full_step(ln, i)

        def issue_done():
            torch.cuda.set_stream(main)

        def drain():
            for ln in range(n_lanes):
                main.wait_stream(lane_streams[ln])

        def fork():
            for st in lane_streams:
                st.wait_stream(main)

        fork()
        for s in range(n_warmup):
            run_step(s)
        issue_done()
        drain()
        # n_steps timed steps in R regions (sizes differ by at most one).  Every region: host barrier + synchronize on
        # both sides, and — with the fused exchange — a DEVICE-side barrier enqueued in front of the start event, so that
        # all GPUs enter the region within an NVLink round trip of each other and the host barrier's rank skew stays
        # outside it.  Reported per step: the median region of the max-over-ranks times, min / max, and every
        # rank's median.
        start_barrier = getattr(pipes[0], "start_barrier", None) if fused else None
        R = max(1, min(n_regions, n_steps))
        sizes = [n_steps // R + (r < n_steps % R) for r in range(R)]
        per_region, step_no, host_issue = [], n_warmup, []
        for n in sizes:
            barrier()
            if sampler: sampler.mark()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if start_barrier is not None:
                start_barrier[0].device_barrier(start_barrier[1], main)
            e0.record(main)
            for st in lane_streams:                        # the lanes start behind the start event itself (same-box A/B
                st.wait_event(e0)                          # against fork(): no difference, 40.54 vs 40.56 us at 20 steps)
            h0 = time.perf_counter()
            for s in range(step_no, step_no + n):
                run_step(s)
            host_issue.append((time.perf_counter() - h0) * 1e3 / n)
            issue_done()
            step_no += n
            drain()
            e1.record(main)
            barrier()
            if sampler: sampler.mark()
            per_region.append(e0.elapsed_time(e1) / n)
        mine = torch.tensor(per_region, dtype=torch.float64, device=dev)
        if multi:
            allr = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            allr = torch.stack(allr)                        # [rank, region]
        else:
            allr = mine.view(1, -1)
        region_max = allr.max(dim=0).values                 # max over ranks, per region
        ms = float(region_max.median().item())
        timing = {"regions": len(per_region), "steps_per_region": sizes, "ms_per_step_median": ms,
                  "ms_per_step_min": float(region_max.min().item()),
                  "ms_per_step_max": float(region_max.max().item()),
                  "per_rank_ms_per_step_median": allr.median(dim=1).values.tolist(),
                  "start": "device-side barrier over NVLink peer memory" if start_barrier is not None else "host barrier",
                  # host wall time to ENQUEUE one step (rank 0, median region): the step is device-bound while this is
                  # well below ms_per_step
                  "host_issue_ms_per_step": sorted(host_issue)[len(host_issue) // 2]}
        last = step_no - 1
        return ms, pipes, outs, graphs, timing, outs[last % n_lanes][last % n_sets]

    ms, pipes, outs, graphs, timing, last_out = timed_steps(args.decode_mode, args.steps, max(args.warmup, 3), args.regions)
    pipe = pipes[0]
    value = B * world / (ms * 1e-3)
    outs0 = outs[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_out)

    # ---- sanity of what was timed (not timed): losses finite, detections present
    losses = outs0[0].losses.cpu().tolist()
    P_bar = float(outs0[0].sums[6].item()) / (B * (world if multi else 1))
    cand_mean = None      # measured in the stand-alone decode loop below (k_nms* zero the counters they consume)
    det_mean = float(outs0[0].num_instances.float().mean().item())

    # ---- fused exchange vs NCCL: the same step with an NCCL all-reduce + finalize launch must give the same losses
    allreduce_check = None
    if fused:
        chk = DetectionHeadPipeline(levels, W, H, B, C, B * G, dev, TOPK, K, SCORE_THR, IOU_THR, decode_mode=args.decode_mode)
        chk_out = chk.new_outputs()
        chk.step(sets[0], chk_out, finalize=False)
        dist.all_reduce(chk_out.sums, op=dist.ReduceOp.SUM)
        chk.finalize(chk_out)
        torch.cuda.synchronize()
        allreduce_check = {"nccl_losses": chk_out.losses.cpu().tolist(),
                           "fused_equals_nccl": bool(torch.allclose(chk_out.losses, outs0[0].losses, rtol=1e-6, atol=0))}
        del chk, chk_out

    # ---- the other decode variant on the same inputs (same outputs; reported next to `value`, never instead of it)
    other = None
    if not args.skip_candidate_first:
        other_mode = "candidate_first" if args.decode_mode == "dense" else "dense"
        o_steps = max(3, min(args.steps, 1000))
        o_ms, o_pipes, o_outs, _, _, _ = timed_steps(other_mode, o_steps, max(min(args.warmup, 100), 3), min(args.regions, 3))
        same = all(torch.equal(a, b) for a, b in zip(
            (outs0[0].num_instances, outs0[0].scores, outs0[0].classes, outs0[0].boxes, outs0[0].assignment),
            (o_outs[0][0].num_instances, o_outs[0][0].scores, o_outs[0][0].classes, o_outs[0][0].boxes, o_outs[0][0].assignment)))
        other = {"decode_mode": other_mode, "value": B * world / (o_ms * 1e-3), "unit": UNIT, "steps": o_steps,
                 "ms_per_step": o_ms, "outputs_equal_to_timed_mode": bool(same)}
        del o_pipes, o_outs

    def both_e2e(smp, rows):
        """`e2e` = host maps read in place (candidate-first pipelines); `e2e_full_upload` = every map uploaded."""
        from sihl_b200.pipeline import DetectionHeadPipeline as _P
        n_e2e = max(1, args.e2e_lanes)
        mk = lambda mode: attach([_P(levels, W, H, B, C, B * G, dev, TOPK, K, SCORE_THR, IOU_THR, decode_mode=mode)
                                  for _ in range(n_e2e)])
        e2e_sets = sets[:min(len(sets), 3)]                     # rotating pinned host sets (3 x 188 MB at cfg1)
        full, _ = run_e2e(args, mk(args.decode_mode), e2e_sets, world, multi, dev, smp)
        ref = (outs0[0].num_instances, outs0[0].scores, outs0[0].classes, outs0[0].boxes, outs0[0].assignment,
               outs0[0].rel_iou)
        sparse, cf_out = run_e2e(args, mk("candidate_first"), e2e_sets, world, multi, dev, smp, host_maps=True,
                                 gathered_rows=rows)
        got = (cf_out.num_instances, cf_out.scores, cf_out.classes, cf_out.boxes, cf_out.assignment, cf_out.rel_iou)
        sparse["outputs_equal_to_resident_run"] = bool(all(torch.equal(a, b) for a, b in zip(ref, got)))
        sparse["losses"] = cf_out.losses.cpu().tolist()
        return sparse, full

    if rank != 0:
        # the other ranks only take part in the collective part of the end-to-end measurement
        if not args.skip_e2e:
            both_e2e(None, 0.0)
        for ex in exchanges:
            ex.check()                                   # raises if any in-kernel wait for a peer ever timed out
            ex.close()
        return

    # ---- roofline of the dominant kernel (k_dense_decode), timed alone on the launching stream
    peak, peak_src = measured_peaks()
    # >= 400 launches and >= 10 ms inside the timed region, after 100 untimed launches: the first few hundred launches
    # of a process run up to 25 % slower than the steady state (measured at the crowd workload: 17.5 us for the first
    # 400 launches, 14.2 us afterwards, identical code and inputs), which a 60-launch loop would report as the kernel.
    iters, warm = 400, 100
    counts_saved = pipe.cand.count
    scratch = torch.zeros((iters + warm, B), dtype=torch.int32, device=dev)
    settle = []                                       # ms per launch of every 100-launch warm-up batch

    def decode_once(i):
        x = sets[i % n_sets]
        pipe.cand.count = scratch[i]                 # a fresh zeroed counter row per launch: the kernel is timed alone
        ops.dense_decode(x.loc_logits, x.cls_logits, x.box_raw, pipe.offsets, pipe.scales, W, H, SCORE_THR, pipe.cand,
                         zero_counts=False)

    # The launches are back to back on one stream either way.  Default: `warm` of them captured into ONE CUDA graph
    # (first node zeroes their counter rows) and replayed — an eager loop pays ~14 us of Python + ctypes +
    # cudaFuncSetAttribute per call on the host, which is MORE than a 57 MB scan takes on the device (crowd: every ring
    # shape "measured" 13.9 us that way, r02_decode_sweep_crowd.json), so it would time the host.  --no-graph keeps the loop.
    graph = None
    if not args.no_graph:
        scratch.zero_()
        decode_once(0)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            scratch[:warm].zero_()
            for i in range(warm):
                decode_once(i)

    def batch_of_launches(first):
        if graph is not None:
            graph.replay()
        else:
            for i in range(warm):
                decode_once(first + i)

    for _ in range(60):
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        scratch[iters:].zero_()
        w0.record()
        batch_of_launches(iters)
        w1.record()
        torch.cuda.synchronize()
        settle.append(w0.elapsed_time(w1) / warm)
        # at least ~40 ms of back-to-back launches: a 57 MB scan settles only after ~15 ms
        if len(settle) >= 2 and sum(settle) * warm >= 40.0 and abs(settle[-1] - settle[-2]) <= 0.03 * settle[-1]:
            break
    if graph is None:
        scratch.zero_()
    if sampler: sampler.mark()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for j in range(iters // warm):
        batch_of_launches(j * warm)
    k1.record()
    torch.cuda.synchronize()
    if sampler: sampler.mark()
    cand_mean = float(scratch[:warm if graph is not None else iters].float().mean().item())
    k_ms = k0.elapsed_time(k1) / iters
    eager_ms = None
    if graph is not None:                             # the same launches from a Python loop, for comparison with round 1
        scratch.zero_()
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record()
        for i in range(iters):
            decode_once(i)
        x1.record()
        torch.cuda.synchronize()
        eager_ms = x0.elapsed_time(x1) / iters
    pipe.cand.count = counts_saved
    # algorithmic bytes per launch: every class logit and location logit read once (4*A*(C+1) per image), the raw
    # box (16 B) read and key 8 + box 16 + class 4 = 28 B written per candidate.  (SURVEY.md §8d counts 16*A for the
    # raw boxes of every location; the kernel reads them for candidates only, so that figure would overstate it.)
    decode_bytes = B * 4 * A * (C + 1) + B * cand_mean * (16 + 28)
    achieved = decode_bytes / (k_ms * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
            if tj.get("workload") == args.workload:
                traffic = tj.get("k_dense_decode_dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_dense_decode", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": k_ms,
                "algorithmic_bytes_per_launch": decode_bytes, "launches_timed": iters,
                "launch_mode": (f"CUDA graph of {warm} back-to-back launches (+ one memset node), replayed {iters // warm}x"
                                if graph is not None else "eager loop (host time per call included)"),
                "eager_loop_ms_per_launch": eager_ms,
                "warmup_ms_per_launch_by_100": [round(v, 5) for v in settle[:4] + settle[-2:]], "warmup_batches": len(settle)}
    # whole step: train 20A+24G+(16+4C)P + infer 4A(C+1)+16*cand+28K+8 bytes per image — SURVEY.md §8d's figure minus
    # the raw boxes of the locations that are not candidates (never read); the survey's own figure is reported beside it
    step_bytes_survey = 20 * A + 24 * G + (16 + 4 * C) * P_bar + 4 * A * (C + 5) + 28 * K + 8
    step_bytes_per_image = step_bytes_survey - 16 * (A - cand_mean)
    step_gbs = step_bytes_per_image * B / (ms * 1e-3) / 1e9          # per GPU
    roofline_step = {"bytes_per_image": step_bytes_per_image, "achieved": step_gbs, "peak": peak, "unit": "GB/s",
                     "frac": step_gbs / peak, "per_gpu": True, "bytes_per_image_survey_8d": step_bytes_survey,
                     "frac_survey_8d_bytes": step_bytes_survey * B / (ms * 1e-3) / 1e9 / peak}

    # ---- end to end: host (pinned) inputs -> H2D -> step -> D2H of losses + detections, every step
    e2e = e2e_full = None
    if not args.skip_e2e:
        e2e, e2e_full = both_e2e(sampler, B * (P_bar + (cand_mean or 0.0)))

    cpu = None
    if not multi and not args.skip_cpu_baseline:
        r = cpu_reference_images_per_sec(w, B, 20, 1, budget_s=25.0)     # 10-25 s of host work
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
               "sample": f"{r['sample_images']} of {B} images of {args.workload} x {r['steps']} passes: {REFERENCE_WHAT}; "
                         f"{r['cores']} threads"}

    # ---- the same step on bf16 head outputs (what the MLPs emit under precision="16-mixed"): maps read as they are
    half_maps = None
    if not multi and not args.skip_half_maps:
        hsets = [StepInputs(x.loc_logits.bfloat16(), x.iou_preds.bfloat16(), x.box_raw.bfloat16(), x.cls_logits.bfloat16(), x.gt)
                 for x in sets]
        half_maps = {"map_dtype": "bf16", "note": "extra line, never the headline: identical kernels templated on the map type, "
                                                   "half the bytes in the dense scan; losses / detections follow the reference's "
                                                   "half-precision operator semantics (tests/test_gpu_half_maps.py)"}
        for mode in ("dense", "candidate_first"):
            h_steps = max(3, min(args.steps, 1000))
            h_ms, h_pipes, h_outs, _, _, _ = timed_steps(mode, h_steps, max(min(args.warmup, 100), 3), min(args.regions, 3),
                                                         hsets)
            half_maps[mode] = {"value": B / (h_ms * 1e-3), "unit": UNIT, "ms_per_step": h_ms,
                               "losses": h_outs[0][0].losses.cpu().tolist()}
            del h_pipes, h_outs
        del hsets

    # ---- row N4: the per-location MLP towers in FRONT of the path, on the tensor cores (extra line, never the headline)
    mlp_line = None
    if not multi and not args.skip_mlp:
        mlp_line = mlp_towers_line(B * A, C, dev)

    # ---- the drop-in head's training tail WITH gradients (what ObjectDetection.training_step runs around its MLPs)
    train_tail = None
    if not multi and not args.skip_train_tail:
        train_tail = train_tail_with_backward(w, sets[0], levels, dev)

    # ---- the reference's operator sequence as torch eager on THIS GPU (the bar SURVEY.md §2b names)
    eager = None
    if not multi and not args.skip_gpu_eager:
        eager = gpu_eager_reference(w, sets[0], levels, dev)

    for ex in exchanges:
        ex.check()
        ex.close()
    clocks = sampler.stop() if sampler else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        # `config` names the WORKLOAD only and is the same object in both arms (`--impl reference` prints it too); how this
        # arm executes it, and what the synthetic inputs turned out to contain, sit beside it
        "config": config_dict(w, args, world),
        "execution": {"cuda_graph": graphs is not None, "streams_per_step": 1 if args.serial else 2,
                      "steps_in_flight": n_lanes, "decode_mode": args.decode_mode},
        "workload_stats": {"positives_per_image": P_bar, "candidates_per_image": cand_mean,
                           "detections_per_image": det_mean},
        "timing": timing, "train_with_backward": train_tail, "half_maps": half_maps, "mlp_towers": mlp_line,
        "cpu_affinity": affinity,
        "e2e": e2e, "e2e_full_upload": e2e_full, "gpu_launches": (LAUNCHES_PER_STEP + (1 if multi and not fused else 0)) * args.steps,
        "allreduce": (("fused" if fused else "nccl") if multi else None), "allreduce_check": allreduce_check,
        "allreduce_fallback": (fallback_note[0] if fallback_note else None), "roofline": roofline, "roofline_step": roofline_step,
        "other_decode_mode": other, "cpu_baseline": cpu, "gpu_eager_reference": eager, "clocks": clocks,
        "losses_check": losses,
    }
    print(json.dumps(line), flush=True)


def mlp_towers_line(M, C, dev):
    """SURVEY.md §8f N4: the head's four ``ops.MLP(256 -> 256 x 4 -> out, LayerNorm, SiLU)`` towers (ref
    object_detection.py:51-61) over the step's M = B * A locations through ``sihl_od_mlp_hidden`` / ``sihl_od_mlp_out``
    (tcgen05 + TMA + TMEM; bf16 operands, fp32 accumulate / normalise), and one hidden layer as torch eager fp32 (what the
    reference runs) and bf16 autocast.  Inputs rotate over 3 buffers (> L2); CUDA events."""
    import torch
    from torch import nn
    from torchvision import ops as tvops
    from sihl_b200 import ops
    from sihl_b200.mlp_tower import PackedTower, run_tower

    def timeit(fn, iters, warm=3):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    torch.manual_seed(0)
    xs = [torch.randn((M, 256), device=dev).bfloat16() for _ in range(3)]
    ys = [torch.empty((M, 256), dtype=torch.bfloat16, device=dev) for _ in range(2)]
    towers = {n: tvops.MLP(256, [256] * 4 + [o], norm_layer=nn.LayerNorm, activation_layer=nn.SiLU).to(dev).eval()
              for n, o in (("loc", 1), ("iou", 1), ("box", 4), ("cls", C))}
    packed = {n: PackedTower(m).refresh() for n, m in towers.items()}
    w, b, g, be, eps = packed["loc"].hidden[0]
    ms = timeit(lambda i: ops.mlp_hidden(xs[i % 3], w, b, g, be, eps, out=ys[i & 1]), 30, 10)
    peak_hbm, src = measured_peaks()
    byts, flops = M * 1024.0, 2.0 * M * 256 * 256
    line = {"locations": M, "dtype": "bf16 operands, f32 accumulate", "note": "row N4, extra line: inference only; the path's "
            "own kernels have no dense contraction",
            "hidden_layer": {"ms": ms, "algorithmic_bytes": byts, "flops": flops, "gbs": byts / ms / 1e6, "tflops": flops / ms / 1e9,
                             "roofline": {"bound": "hbm", "achieved": byts / ms / 1e6, "peak": peak_hbm, "unit": "GB/s",
                                          "frac": byts / ms / 1e6 / peak_hbm, "peak_source": src}}}
    scratch = (ys[0], ys[1])

    def four(i):
        for n in towers:
            run_tower(packed[n], xs[i % 3], scratch)
    line["four_towers_ms"] = timeit(four, 5, 2)
    line["gpu_launches_per_call"] = 4 * 5
    with torch.no_grad():
        seq = nn.Sequential(towers["loc"][0], towers["loc"][1], towers["loc"][2])
        xf = xs[0].float()
        line["hidden_layer"]["torch_eager_fp32_ms"] = timeit(lambda i: seq(xf), 3, 1)

        def bf(i):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return seq(xs[i % 3])
        line["hidden_layer"]["torch_eager_bf16_autocast_ms"] = timeit(bf, 3, 1)
    # training path of one tower (loc: 4 hidden layers + 1 output column): forward on the tensor cores + recomputing backward
    from sihl_b200.mlp_tower import run_tower_train
    tower = towers["loc"].train()
    xt = xf.requires_grad_(True)
    gy = torch.randn((M, 1), device=dev)

    def train(run):
        def step(i):
            tower.zero_grad(set_to_none=True)
            xt.grad = None
            run(xt).backward(gy)
        return step
    line["tower_forward_backward"] = {"ms": timeit(train(lambda t: run_tower_train(tower, t)), 5, 2),
                                      "torch_eager_fp32_ms": timeit(train(tower), 2, 1),
                                      "precision": "bf16 operands / activations, fp32 accumulation, statistics and parameter gradients"}
    tower.eval()
    del xs, ys, xf, xt, gy
    torch.cuda.empty_cache()
    line["head_training_step"] = head_training_step_line(C, dev, timeit)
    line["note"] = ("row N4, extra line: the step in FRONT of the path (laterals + four MLP towers) on the tensor cores, inference "
                    "and (opt-in, bf16 mixed precision) training; the path's own kernels have no dense contraction")
    return line


def head_training_step_line(C, dev, timeit):
    """The drop-in head's whole ``training_step`` + ``backward`` (ref object_detection.py:124-217 with its laterals and four
    towers, then the hot path) at cfg1's batch on levels 3-5 of a 640x640 input: ``mlp_backend = "tcgen05+train"`` (laterals
    and towers on the tensor cores, bf16 mixed precision) against the identical module with the torch towers in fp32."""
    import torch
    from sihl_b200 import synth
    from sihl_b200.heads import ObjectDetection
    B, size = 64, 640
    torch.manual_seed(0)
    model = ObjectDetection(in_channels=[3, 64, 128, 256, 256, 256], num_classes=C, num_channels=256, num_layers=4).to(dev).train()
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    inputs = [torch.randn((B, c, size // 2 ** l, size // 2 ** l), generator=g, device=dev) if l >= 3 or l == 0
              else torch.empty((B, c, 1, 1), device=dev) for l, c in enumerate(model.in_channels)]
    gt = synth.gt_batch_np(3, B, size, size, C, 100)
    tb = [torch.from_numpy(b_).to(dev) for b_, _ in gt.per_image()]
    tc = [torch.from_numpy(c_).to(dev) for _, c_ in gt.per_image()]
    out = {"batch": B, "image": size, "levels": "3-5", "locations": B * 8400, "gt_per_image": 100,
           "what": "laterals + four towers + assign + losses, forward and backward, wall clock per step (CUDA events)"}

    def step(i):
        model.zero_grad(set_to_none=True)
        loss, _ = model.training_step(inputs, classes=tc, boxes=tb)
        loss.backward()
        return loss
    for backend, iters in (("tcgen05+train", 6), ("torch", 2)):
        model.mlp_backend = backend
        out[backend.replace("+", "_") + "_ms"] = timeit(step, iters, 2)
        out[backend.replace("+", "_") + "_loss"] = float(step(0).detach())
    out["speedup"] = out["torch_ms"] / out["tcgen05_train_ms"]
    del model, inputs
    torch.cuda.empty_cache()
    return out


def train_tail_with_backward(w, x, levels, dev, reps=300):
    """The training tail of the drop-in head with gradients, as ``ObjectDetection.training_step`` + ``backward`` run it
    around the MLPs: ``sihl_od_train_assign`` (select, resolve, compaction) -> ``sihl_od_train_loss`` (one launch) ->
    ``sihl_od_train_loss_bwd`` (one launch): 3 C calls, 5 launches, no host synchronisation.  The MLP outputs are
    synthetic leaf tensors (rows gathered once, outside the timed region).  ``graph``: the step captured once into a CUDA
    graph and replayed, device-timed; ``eager``: host-launched every step, wall clock."""
    import torch
    from sihl_b200 import ops
    from sihl_b200.heads.object_detection import _TrainLoss
    H, W, B, C, G = w["height"], w["width"], w["batch"], w["classes"], w["gt"]
    counts = list(x.gt.counts)
    st0 = ops.train_assign(levels, W, H, x.gt.boxes, x.gt.classes, counts, B, TOPK)
    bx0 = x.box_raw.view(-1, 4).index_select(0, st0.pos_index).contiguous()
    cl0 = x.cls_logits.view(-1, C).index_select(0, st0.pos_index).contiguous()

    def step(gt_offsets=None):
        st = ops.train_assign(levels, W, H, x.gt.boxes, x.gt.classes, None if gt_offsets is not None else counts, B, TOPK,
                              gt_offsets=gt_offsets)
        leaves = [t.detach().requires_grad_(True) for t in (x.loc_logits, x.iou_preds, bx0, cl0)]
        out = _TrainLoss.apply(*leaves, st, None)
        out[4].backward()
        return out, [t.grad for t in leaves]

    out, grads = step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    torch.cuda.synchronize()
    eager_ms = (time.perf_counter() - t0) / reps * 1e3
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(3):
            step(x.gt.offsets)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_grads = step(x.gt.offsets)
    for _ in range(20):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    graph_ms = e0.elapsed_time(e1) / reps
    same = bool(torch.equal(g_out, out) and all(torch.equal(a, b) for a, b in zip(g_grads, grads)))
    return {"what": "assign + positive compaction + 4 losses + backward (drop-in head's own path; MLP outputs are leaf tensors)",
            "ms_per_step": graph_ms, "value": B / (graph_ms * 1e-3), "unit": UNIT, "mode": "CUDA graph replay, device timed",
            "eager_ms_per_step": eager_ms, "eager_value": B / (eager_ms * 1e-3), "graph_equals_eager": same,
            "gpu_launches_per_step": 5, "c_calls_per_step": 3, "host_syncs_per_step": 0,
            "positives": int(st0.pos_total.item()), "row_capacity": st0.capacity, "losses": out.detach().cpu().tolist()}


def gpu_eager_reference(w, x, levels, dev, passes=2):
    """The reference's own code (oracle/ref_path.py: its unmodified ``training_step`` with the per-image Python loop and
    host syncs, + dense decode + torchvision.ops.batched_nms) as torch eager on the same GPU and the same resident
    inputs: the eager-PyTorch bar for this path."""
    import torch
    H, W, B, K, G = w["height"], w["width"], w["batch"], w["k"], w["gt"]
    boxes = [x.gt.boxes[b * G:(b + 1) * G] for b in range(B)]
    classes = [x.gt.classes[b * G:(b + 1) * G] for b in range(B)]
    one_pass = make_reference_pass(w, levels, boxes, classes, x.loc_logits, x.iou_preds, x.box_raw, x.cls_logits)
    best = None
    for _ in range(passes + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        one_pass()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": B / best, "unit": UNIT, "ms_per_step": best * 1e3, "impl_kind": reference_kind(),
            "kind": "torch eager on the same GPU: %s, best of %d" % (REFERENCE_WHAT, passes)}


def run_e2e(args, pipes, xs, world, multi, dev, sampler, host_maps=False, gathered_rows=0.0):
    """End to end through the public API (DetectionHeadPipeline.step) from pinned HOST inputs, every step: inputs
    cross PCIe inside the timed region, losses + detections are read back to the host.  One lane per pipeline in
    `pipes` (own stream, device input slot, outputs, host result buffers): step i runs on lane i % len(pipes), so
    the PCIe traffic of one step overlaps the kernels of its neighbours.  The host inputs ROTATE over the sets `xs`
    (step i reads set i % len(xs)), so no step re-reads what the previous one left in a cache.

    host_maps=False: all seven input tensors are uploaded (copy stream), any decode mode.
    host_maps=True (pipelines in candidate-first mode): only the location / IoU maps and the gt are uploaded; the class
    and box maps stay in pinned host memory and the kernels read the rows they need (positives, candidates) in place
    over PCIe.  `gathered_rows` = positives + candidates per step, to count those bytes.
    Returns (result dict, outputs of lane 0 for set 0)."""
    import torch
    import torch.distributed as dist

    from sihl_b200 import ops
    from sihl_b200.pipeline import StepInputs

    n = max(args.e2e_steps, 2)
    L, S = len(pipes), len(xs)
    fields = lambda x: (x.loc_logits, x.iou_preds, x.box_raw, x.cls_logits, x.gt.boxes, x.gt.classes, x.gt.offsets)
    hosts = [[t.cpu().pin_memory() for t in fields(x)] for x in xs]
    host = hosts[0]
    copied = [i for i in range(len(host)) if not (host_maps and i in (2, 3))]
    h2d = sum(host[i].numel() * host[i].element_size() for i in copied)
    if host_maps:
        h2d += int(gathered_rows * (host[3].shape[-1] * 4 + 16))       # rows read in place: C class logits + raw box
    copy = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    lanes = []
    for pipe in pipes:
        d = [torch.empty_like(t, device=dev) if i in copied else None for i, t in enumerate(host)]
        out = pipe.new_outputs()
        results = (out.losses, out.num_instances, out.scores, out.classes, out.boxes)
        # one StepInputs per host set: the uploaded tensors are shared, host-resident maps point at that set's buffers
        slots = [StepInputs(d[0], d[1], d[2] if d[2] is not None else hosts[k][2], d[3] if d[3] is not None else hosts[k][3],
                            ops.GtBatch(d[4], d[5], d[6], list(xs[k].gt.counts))) for k in range(S)]
        lanes.append(dict(pipe=pipe, out=out, results=results, stream=torch.cuda.Stream(device=dev), slots=slots, dev=d,
                          res_host=[torch.empty_like(t, device="cpu").pin_memory() for t in results],
                          ready=torch.cuda.Event(), done=torch.cuda.Event()))
    d2h = sum(t.numel() * t.element_size() for t in lanes[0]["res_host"])

    def upload(ln, k):
        with torch.cuda.stream(copy):
            copy.wait_event(ln["done"])                 # the step that last read this slot has finished
            for i in copied:
                ln["dev"][i].copy_(hosts[k][i], non_blocking=True)
            ln["ready"].record(copy)

    def one(i, total):
        ln = lanes[i % L]
        st, pipe, out = ln["stream"], ln["pipe"], ln["out"]
        with torch.cuda.stream(st):
            st.wait_event(ln["ready"])
            separate = multi and pipe._exchange is None      # no fused exchange attached: NCCL all-reduce + finalize
            pipe.step(ln["slots"][i % S], out, finalize=not separate)
            if separate:
                dist.all_reduce(out.sums, op=dist.ReduceOp.SUM)
                pipe.finalize(out)
            ln["done"].record(st)
            if i + L < total:
                upload(ln, (i + L) % S)                  # refill this lane's slot for step i+L while its neighbours compute
            for h, d in zip(ln["res_host"], ln["results"]):
                h.copy_(d, non_blocking=True)

    for ln in lanes:
        ln["done"].record(main)
    torch.cuda.synchronize()
    # warm-up (L steps), timed n steps, then ONE untimed step of set 0 on lane 0 (the outputs the caller compares);
    # the uploads of the first L steps of a phase are inside its region
    ms = 0.0
    for phase, count in (("warm", L), ("timed", n), ("check", 1)):
        if multi:
            dist.barrier()
        torch.cuda.synchronize()
        if phase == "timed" and sampler: sampler.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        copy.wait_event(e0)
        for j, ln in enumerate(lanes):
            ln["stream"].wait_event(e0)
            upload(ln, j % S)
        for i in range(count):
            one(i, count)
        for ln in lanes:
            main.wait_stream(ln["stream"])
        e1.record(main)
        torch.cuda.synchronize()
        if phase == "timed":
            if sampler: sampler.mark()
            ms = e0.elapsed_time(e1)
    if multi:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    note = ("pinned host inputs; location / IoU maps + gt uploaded, class and box maps read in place over PCIe: only the "
            "rows of the positives and of the candidates cross the bus (candidate-first decode)"
            if host_maps else "pinned host inputs, all maps uploaded on a copy stream; PCIe-bound")
    res = {"value": pipes[0].B * world * n / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": n, "ms_per_step": ms / n, "decode_mode": pipes[0].decode_mode, "host_maps": bool(host_maps),
           "steps_in_flight": L, "host_input_sets": S, "note": note}
    return res, lanes[0]["out"]


def main():
    args = parse_args()
    w = WORKLOADS[args.workload]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, w, world, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, w, world, rank, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
