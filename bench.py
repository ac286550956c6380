#!/usr/bin/env python
"""bench.py -- post-head path throughput (Detect decode + per-task NMS) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic raw head tensors: BASELINE.json config 3 (3 task heads
20/19/12 classes, 640x640 -> 8400 anchors, B=64 images per GPU, fp16, val settings conf 0.001 / iou 0.6 / multi_label /
max_nms 30000 / max_det 300).  N>1: every rank owns B images (weak scaling; N=8 is config 5, B=512) and the padded
detections of every batch reach rank 0 inside the timed region.

How the timed region runs (cerberusdet_b200/pipeline.py): a two-stage software pipeline replayed from CUDA graphs --
step k decodes batch k while the NMS of batch k-1 runs beside it (one stream: the NMS kernel releases its dependents at
entry and the decode launch carries the programmatic-serialization attribute); a final flush does the last NMS, so K
steps are exactly K decode launches + K NMS launches.  32 of the K steps (16 when K < 128) are "instrumented" replays of the
same two kernels in serial order with timing events recorded by the graph itself around each kernel: that is where
`roofline` (the decode kernel alone on the GPU) comes from; they cost ~13 us more than an overlapped step each.

`--dump-outputs DIR` writes what the last timed step delivered (rank 0) as DIR/detections.npy (float32 [tasks, images,
max_det, 6], rows past each count zeroed) and DIR/counts.npy (float32 [tasks, images]); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput; `e2e` = the host-buffer public API (pinned H2D
of the raw heads + D2H of the detections inside the timed region); `roofline` = decode kernel vs the measured HBM peak;
`cpu_baseline` = the reference's own code (oracle/_ref) on this box's host cores on a bounded sample; extras (N=1):
`surface` (the reference-facing drop-in calls -> list[Tensor]), `serial` (no overlap), `gpu_eager_reference` (the
reference's code on this same GPU), `planted` (realistic regime, IoU pairs/s), `config5_strong` (B=512 split over N).
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from untouched (it may be read-only)

import torch  # noqa: E402

NCS = [20, 19, 12]  # voc / objects365_animals / objects365_tableware (reference data/*.yaml)
IMGSZ = 640
ANCHORS = 8400
B_PER_GPU = 64
NMS_KW = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)  # reference val.py:139,318
METRIC = "post-proc images/s (3 tasks, 640^2, B=64 per GPU): Detect decode + per-task NMS"
CPU_SAMPLE_IMAGES = 3  # cpu_baseline: ~1.2 s per (image, task) segment on 16 cores -> ~10 s of CPU work
TIMED_SLOTS = 32       # instrumented steps inside the timed region; 16 when --steps < 128 (still >= 16 whenever steps >= 17)
REFERENCE_BUDGET_S = 240.0


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _decode_bytes_per_image(ncs, anchors, elt):
    return sum((64 + nc) * elt * anchors + (4 + nc) * elt * anchors for nc in ncs)


class ClockSampler:
    """SM clock + throttle reasons of one GPU while the timed region runs (NVML, ~2 ms period;
    falls back to polling nvidia-smi)."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self.nvml, self.h = None, None
        self.stop = threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _init_nvml(self):
        """Open the NVML handle on the caller's thread, BEFORE the timed region: nvmlInit alone can take longer than
        the ~50 ms the default run is timed for, which would leave the sampler without a single sample."""
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")  # NVML enumerates physical GPUs
        phys = self.index
        if vis:
            try:
                phys = int(vis.split(",")[self.index])
            except (ValueError, IndexError):
                phys = self.index
        self.nvml, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))

    def _sample_nvml(self):
        self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)))
        mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        for name, bit in self.BAD.items():
            if mask & bit:
                self.reasons.add(name)

    def _run_nvml(self):
        while not self.stop.is_set():
            self._sample_nvml()
            self.stop.wait(0.002)
        self._sample_nvml()  # one more under load: the caller stops the sampler before it synchronises

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.sm.append(float(parts[0]))
                    self.max_mhz = float(parts[1])
                    self.reasons.update(n for i, n in enumerate(names) if parts[2 + i].lower().startswith("active"))
            except Exception:
                pass
            self.stop.wait(0.05)

    def _run(self):
        try:
            if self.h is None:
                raise RuntimeError("no NVML")
            self._run_nvml()
        except Exception:
            self._run_smi()

    def __enter__(self):
        try:
            self._init_nvml()
        except Exception:
            self.h = None
        self.th.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"], "samples": 0}
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


# ------------------------------------------------------------------------------------------------ CPU reference legs
class CpuReference:
    """The reference's CPU implementation of the path on ONE (image, task) segment: its own Detect eval branch and its
    own non_max_suppression (one image per call) when the reference tree travelled with the snapshot (oracle/_ref,
    kind "reference"); otherwise the oracle port (same torch ops + torchvision.ops.nms, kind "port")."""

    def __init__(self):
        from cerberusdet_b200.synth import STRIDES

        self.strides = STRIDES
        self.runner = None
        try:
            from oracle.ref_run import ReferenceRunner, reference_available

            if reference_available():
                self.runner = ReferenceRunner(STRIDES)
        except Exception as exc:  # pragma: no cover - depends on the box
            print(f"[bench] reference tree unusable ({type(exc).__name__}: {exc}); timing the oracle port", file=sys.stderr)
        self.kind = "reference" if self.runner is not None else "port"

    def segment(self, heads_cpu, image, task):
        t0 = time.perf_counter()
        lv = [x[image : image + 1] for x in heads_cpu[task]]
        if self.runner is not None:
            self.runner.segment(lv, NCS[task], **NMS_KW)
        else:
            from oracle import ref_port as rp

            rp.nms_port(rp.decode_port(lv, NCS[task], self.strides), greedy="torchvision", **NMS_KW)
        return time.perf_counter() - t0

    def describe(self):
        return ("the reference's own Detect eval branch + non_max_suppression (oracle/_ref, unmodified), one image per call"
                if self.runner is not None else "oracle port: torch CPU ops + torchvision.ops.nms")


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation on the host cores.  Each step is a bounded sample of the
    workload: one (image, task) segment = 1/3 image, the task rotating with the step."""
    if rank != 0:
        return
    from cerberusdet_b200.synth import synth_heads

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cpu = CpuReference()
    heads = synth_heads(range(CPU_SAMPLE_IMAGES), NCS, IMGSZ, torch.float16, "iid", cfg=3)
    t_begin = time.perf_counter()
    for k in range(args.warmup):
        cpu.segment(heads, 0, k % 3)
    times = []
    for k in range(args.steps):
        times.append(cpu.segment(heads, 0, k % 3))
        if time.perf_counter() - t_begin > REFERENCE_BUDGET_S and len(times) >= 3:
            break  # keep the arm inside a few minutes whatever K the caller asked for
    tot, done = sum(times), len(times)
    val = (done / 3.0) / tot
    sample = (f"one (image, task) segment (= 1/3 image) of the B=64 batch per step, task rotating; "
              f"{done} of {args.steps} steps run; {cpu.describe()}")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
        "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * tot / done,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": _config(args.gpus),
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": cpu.kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _config(n):
    return {"workload": "BASELINE config 3 per GPU: 3 task heads (nc 20/19/12), 640x640 (8400 anchors), "
                        f"B={B_PER_GPU} images per GPU, fp16 raw head tensors, conf 0.001 / iou 0.6 / multi_label / "
                        "max_nms 30000 / max_det 300",
            "global_batch": B_PER_GPU * n, "tasks": 3, "anchors": ANCHORS, "regime": "iid (SURVEY 8d R-dense)",
            "l2": "inputs (261 MB raw heads per step) exceed the 126 MB L2; no explicit flush",
            "parallelism": f"image-sharded x{n}, padded detections of every batch delivered to rank 0" if n > 1 else "single GPU"}


# ------------------------------------------------------------------------------------------------ extras (rank 0, N = 1)
def _time_loop(fn, iters, sync):
    sync()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    sync()
    return (time.perf_counter() - t0) / iters


def surface_line(heads_dev, dev):
    """The reference-facing surface, eagerly, as a caller of the drop-in uses it: per task one Detect-decode call
    (what the patched Detect.forward runs after the conv towers) and one non_max_suppression(y, ...) call returning
    list[Tensor[n_i, 6]] -- including the counts device->host sync and the per-image views."""
    from cerberusdet_b200 import ops
    from cerberusdet_b200.nms import non_max_suppression
    from cerberusdet_b200.synth import STRIDES

    def once():
        outs = []
        for lv in heads_dev:
            y = ops.decode_heads([lv], STRIDES)[0]
            outs.append(non_max_suppression(y, **NMS_KW))
        return outs

    for _ in range(3):
        outs = once()
    assert all(len(o) == B_PER_GPU and o[0].shape[1] == 6 for o in outs)
    s = _time_loop(once, 20, lambda: torch.cuda.synchronize(dev))

    def once_batched():  # all task heads in one decode launch + one NMS launch, then the same list[Tensor] views
        ys = ops.decode_heads(heads_dev, STRIDES)
        dets, counts = ops.nms_batched(ys, **NMS_KW)
        n = counts.tolist()
        return [[dets[t, i, : n[t][i]] for i in range(B_PER_GPU)] for t in range(len(NCS))]

    for _ in range(3):
        once_batched()
    s2 = _time_loop(once_batched, 20, lambda: torch.cuda.synchronize(dev))
    return {"value": B_PER_GPU / s, "unit": "images/s", "ms_per_batch": 1e3 * s,
            "what": "eager, per task: decode_heads (patched Detect.forward's decode) + non_max_suppression(y, conf, iou, "
                    "multi_label=True, max_det=300) -> list[Tensor[n,6]] incl. the counts sync; no CUDA graph",
            "batched_all_tasks": {"value": B_PER_GPU / s2, "unit": "images/s", "ms_per_batch": 1e3 * s2,
                                  "what": "eager ops.decode_heads(all tasks) + ops.nms_batched + counts.tolist() + views"}}


def eager_reference_line(heads_dev, dev, budget_s=40.0):
    """Same-GPU baseline (BASELINE.md section 3): the reference's own Python (Detect eval branch + non_max_suppression
    with torchvision's CUDA kernel) on this B200, eagerly, one image per NMS call, on a bounded sample of the batch."""
    from cerberusdet_b200.synth import STRIDES

    try:
        from oracle.ref_run import ReferenceRunner, reference_available

        runner = ReferenceRunner(STRIDES) if reference_available() else None
    except Exception:
        runner = None
    if runner is None:
        from oracle import ref_port as rp
    n_img = 8
    sample = [[x[:n_img].contiguous() for x in lv] for lv in heads_dev]

    def once():
        for t, lv in enumerate(sample):
            if runner is not None:
                runner.segment(lv, NCS[t], **NMS_KW)
            else:
                y = rp.decode_port(lv, NCS[t], STRIDES)
                for i in range(n_img):
                    rp.nms_port(y[i : i + 1], greedy="torchvision", **NMS_KW)

    once()
    torch.cuda.synchronize(dev)
    t0, reps = time.perf_counter(), 0
    while reps < 5 and time.perf_counter() - t0 < budget_s:
        once()
        reps += 1
    torch.cuda.synchronize(dev)
    s = (time.perf_counter() - t0) / reps
    return {"value": n_img / s, "unit": "images/s", "ms_per_image": 1e3 * s / n_img, "kind": "reference" if runner is not None else "port",
            "sample": f"images 0..{n_img - 1} of the batch x 3 task heads, {reps} repetitions, eager PyTorch + torchvision CUDA NMS on the same GPU"}


def planted_line(dev):
    """R-planted regime (SURVEY 8d realism check): trained-detector-like clusters, B=16.  Kernel times from graph replays
    and the NMS kernel's own counters (IoU tests, candidates consumed)."""
    from cerberusdet_b200 import ops
    from cerberusdet_b200.synth import STRIDES, synth_heads

    out = {}
    for regime, bsz in (("planted", 16), ("iid", B_PER_GPU)):
        heads = [[x.to(dev) for x in lv] for lv in synth_heads(range(bsz), NCS, IMGSZ, torch.float16, regime, cfg=3)]
        ys = ops.decode_heads(heads, STRIDES)
        _, counts, stats = ops.nms_statistics(ys, **NMS_KW)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
            ys2 = ops.decode_heads(heads, STRIDES)
            ops.nms_batched(ys2, **NMS_KW)
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        both_us = e0.elapsed_time(e1) * 1e3 / 20
        gd = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s), torch.cuda.graph(gd, stream=s):
            ops.decode_heads(heads, STRIDES)
        torch.cuda.current_stream().wait_stream(s)
        gd.replay()
        e0.record()
        for _ in range(20):
            gd.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        dec_us = e0.elapsed_time(e1) * 1e3 / 20
        nms_us = both_us - dec_us
        pairs, consumed = int(stats[..., 0].sum()), int(stats[..., 1].sum())
        out[regime] = {"batch": bsz, "segments": bsz * len(NCS), "decode_plus_nms_us": round(both_us, 1), "nms_us": round(nms_us, 1),
                       "iou_pairs": pairs, "iou_pairs_per_s": pairs / (nms_us * 1e-6), "candidates_consumed": consumed,
                       "max_consumed_in_a_segment": int(stats[..., 1].max()), "mean_kept": float(counts.float().mean()),
                       "segments_per_s": bsz * len(NCS) / (nms_us * 1e-6)}
    return out


def head_tail_line(dev, reps=10):
    """SURVEY 8f row 3 at the bench shape (B=64, 3 task heads, 640x640) with yolov8x head widths (c2 = 80, c3 = 320): the
    fused tcgen05 kernel (last 1x1 convolutions of both towers + concat + decode, cerb_head_tail) against what the
    reference runs on the same GPU (18 cuDNN 1x1 convolutions + 9 torch.cat + the decode kernel) -- CUDA-graph replays,
    events around the replay.  Roofline: HBM (inputs read once + y and the score summary written)."""
    import torch.nn.functional as F

    from cerberusdet_b200 import ops
    from cerberusdet_b200.synth import STRIDES

    B, c2, c3 = B_PER_GPU, 80, 320
    hw = [(IMGSZ // int(s), IMGSZ // int(s)) for s in STRIDES]
    gen = torch.Generator(device=dev).manual_seed(3)
    mk = lambda *shape, std=1.0: (torch.randn(*shape, generator=gen, device=dev) * std).half()  # noqa: E731
    box = [[mk(B, c2, h, w) for h, w in hw] for _ in NCS]
    cls = [[mk(B, c3, h, w) for h, w in hw] for _ in NCS]
    bw = [[mk(64, c2, 1, 1, std=3.0 / c2**0.5) for _ in hw] for _ in NCS]
    bb = [[mk(64) for _ in hw] for _ in NCS]
    cw = [[mk(n, c3, 1, 1, std=2.0 / c3**0.5) for _ in hw] for n in NCS]
    cb = [[mk(n) - 5.0 for _ in hw] for n in NCS]

    def unfused():
        raw = [[torch.cat((F.conv2d(box[t][l], bw[t][l], bb[t][l]), F.conv2d(cls[t][l], cw[t][l], cb[t][l])), 1) for l in range(3)]
               for t in range(len(NCS))]
        return ops.decode_heads(raw, STRIDES)

    def fused():
        return ops.head_tail(box, cls, bw, bb, cw, cb, STRIDES)

    def timed(fn):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
            fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
            keep = fn()
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(3):
            g.replay()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            torch.cuda.synchronize(dev)
            ts.append(a.elapsed_time(b))
        del keep
        return statistics.median(ts)

    in_bytes = B * ANCHORS * 2 * (c2 + c3) * len(NCS)
    out_bytes = sum(B * ANCHORS * 2 * (4 + n) + B * n * (ANCHORS // 8) * 2 for n in NCS)
    raw_bytes = sum(B * ANCHORS * 2 * (64 + n) for n in NCS)
    fused_ms, unfused_ms = timed(fused), timed(unfused)
    peak, peak_src = _peaks()
    gbps = (in_bytes + out_bytes) / (fused_ms * 1e-3) / 1e9
    return {"kernel": "head_tail_kernel (tcgen05.mma kind::f16, TMA, TMEM; csrc/head_tail.cu)",
            "what": "last 1x1 convs of both towers (c2=80 -> 64, c3=320 -> nc) + concat + decode, B=64, 3 task heads, 640x640, fp16",
            "fused_ms": fused_ms, "reference_sequence_same_gpu_ms": unfused_ms, "speedup": unfused_ms / fused_ms,
            "images_per_s": B / (fused_ms * 1e-3), "algorithmic_bytes": in_bytes + out_bytes,
            "raw_head_bytes_never_written_or_reread": 2 * raw_bytes,
            "roofline": {"bound": "hbm", "achieved": gbps, "peak": peak, "unit": "GB/s", "frac": gbps / peak, "peak_source": peak_src}}


def dump_outputs(out_dir, result):
    """``result`` = (dets [T, B, max_det, 6] float32, counts [T, B] int32) as a caller of the pipeline receives them.
    Rows past each count are padding the kernel leaves unwritten, so they are zeroed to make two runs comparable."""
    import numpy as np

    dets, counts = (x.cpu() for x in result)
    dets = dets.clone()
    dets[torch.arange(dets.shape[2]).view(1, 1, -1) >= counts.unsqueeze(-1)] = 0.0
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "detections.npy"), dets.numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "counts.npy"), counts.numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the surface / eager-reference / planted / serial / config-5 lines")
    ap.add_argument("--serial", action="store_true", help="decode -> NMS of the same batch back to back (no overlap) in the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the detections and counts of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist

    from cerberusdet_b200 import ops
    from cerberusdet_b200.api import postprocess_host
    from cerberusdet_b200.pipeline import PostHeadPipeline
    from cerberusdet_b200.shard import make_delivery
    from cerberusdet_b200.synth import STRIDES, synth_heads

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    images = range(rank * B_PER_GPU, (rank + 1) * B_PER_GPU)
    heads_host = synth_heads(images, NCS, IMGSZ, torch.float16, "iid", cfg=3, pin=True)
    heads_dev = [[x.to(dev, non_blocking=True) for x in lv] for lv in heads_host]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: the NMS kernel writes each batch's padded detections where the delivery to rank 0 picks them up: straight
    # into rank 0's memory over NVLink (peer-mapped symmetric memory) or, failing that, into a packed local buffer that
    # one asynchronous NCCL gather moves.  Two buffers alternate with the pipeline's two output slots.
    delivery = make_delivery(len(NCS), B_PER_GPU, NMS_KW["max_det"], dev, prefer_peer=not args.serial) if world > 1 else None
    if os.environ.get("CERB_DELIVERY") == "none":  # diagnostic only (tools/): N independent replicas, nothing reaches rank 0
        delivery = None
    outs = delivery.outs if delivery is not None else None

    steps = args.steps
    # instrumented steps: parity must match the step index; spread evenly over the timed region, never step 0
    n_timed = 0 if args.serial else min(TIMED_SLOTS if steps >= 128 else 16, max(steps - 1, 0))
    timed_at = sorted({1 + (i * (steps - 1)) // n_timed for i in range(n_timed)}) if n_timed else []
    pipe = PostHeadPipeline(heads_dev, STRIDES, NMS_KW, outs=outs, timed_parities=[k & 1 for k in timed_at], overlap=not args.serial,
                            delivery=delivery, timed_steps=timed_at)
    slot_of = {k: i for i, k in enumerate(timed_at)}

    def run_steps(n, timed=False):
        """n pipeline steps + flush; every finished batch is handed to the delivery (N > 1)."""
        pipe.k, pipe.pending = 0, None
        for k in range(n):
            if delivery is not None:
                delivery.before_write((k - 1) & 1 if pipe.overlap else k & 1)
            done = pipe.step(timed=slot_of.get(k) if timed else None)
            if delivery is not None and done is not None:
                delivery.after_write(done)
        if delivery is not None and pipe.overlap and n:
            delivery.before_write((n - 1) & 1)
        done = pipe.flush()
        if delivery is not None and done is not None:
            delivery.after_write(done)
        if delivery is not None:
            delivery.drain()

    # ---- correctness, outside the timed region: the pipeline's detections == the plain two-call path, bit for bit;
    # N > 1: what rank 0 received from every rank == the single-GPU result on that rank's images
    run_steps(3)
    barrier()
    ys_chk = ops.decode_heads(heads_dev, STRIDES)
    d_chk, c_chk = ops.nms_batched(ys_chk, **NMS_KW)
    last = (3 - 1) & 1
    assert torch.equal(pipe.outs[last][1], c_chk) and torch.equal(pipe.outs[last][0], d_chk), "pipeline != direct calls"
    equality = {"pipeline_equals_direct_calls": True}
    if world > 1 and delivery is not None and os.environ.get("CERB_SIDE", "branch") != "off":
        got = delivery.result(last)  # rank 0: (dets[T, world*B, max_det, 6], counts[T, world*B])
        for r in range(1, world):     # every shard's inputs travel to rank 0 once; rank 0 recomputes it alone
            shard = [[torch.empty_like(x) for x in lv] for lv in heads_dev] if rank == 0 else None
            for t in range(len(NCS)):
                for l in range(3):
                    if rank == r:
                        dist.send(heads_dev[t][l], dst=0)
                    elif rank == 0:
                        dist.recv(shard[t][l], src=r)
            if rank == 0:
                d1, c1 = ops.nms_batched(ops.decode_heads(shard, STRIDES), **NMS_KW)
                sl = slice(r * B_PER_GPU, (r + 1) * B_PER_GPU)
                assert torch.equal(got[1][:, sl], c1) and torch.equal(got[0][:, sl], d1), f"rank {r}'s detections differ from the 1-GPU result"
            del shard
        if rank == 0:
            assert torch.equal(got[1][:, :B_PER_GPU], c_chk) and torch.equal(got[0][:, :B_PER_GPU], d_chk)
            equality["n_gpu_equals_1_gpu"] = True
            equality["delivery"] = delivery.kind
        barrier()
    del ys_chk, d_chk, c_chk

    run_steps(args.warmup)
    barrier()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        t_start.record()
        run_steps(steps, timed=True)
        t_end.record()
        barrier()
    elapsed_ms = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:  # the last batch sits in outs slot (steps - 1) & 1, as in the check above
        # barrier() above ended in torch.cuda.synchronize(), which waits for every stream of the device, so the
        # pipeline's last NMS (and, N > 1, the delivery's collect) has finished writing this slot
        last = (steps - 1) & 1
        dump_outputs(args.dump_outputs, delivery.result(last) if delivery is not None else pipe.outs[last])
    samples = [pipe.timed_ms(i) for i in range(len(timed_at))]
    nms_ms, dec_ms = [s[0] for s in samples], [s[1] for s in samples]
    per_rank = None
    if world > 1:
        mine = torch.tensor([elapsed_ms, sum(dec_ms) / max(len(dec_ms), 1), sum(nms_ms) / max(len(nms_ms), 1)], device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [[round(float(v), 5) for v in t.tolist()] for t in allr]  # [elapsed ms, decode ms, NMS ms] of every rank
        elapsed_ms = max(r[0] for r in per_rank)

    # ---- the same engine without the instrumented steps (outside the timed region, reported beside `value`): what K steps
    # cost when none of them is serialised for the roofline brackets -- the steady state of a long stream of batches
    steady = None
    if not args.serial:
        ss_steps = 200
        run_steps(10)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        run_steps(ss_steps)
        s1.record()
        barrier()
        ss_ms = s0.elapsed_time(s1)
        if world > 1:
            tt = torch.tensor([ss_ms], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ss_ms = float(tt.item())
        steady = {"steps": ss_steps, "ms_per_step": ss_ms / ss_steps, "value": B_PER_GPU * world * ss_steps / (ss_ms * 1e-3), "unit": "images/s",
                  "what": "the timed region's loop without instrumented steps (every step overlapped), max over ranks; not the headline"}

    # ---- end to end through the host-buffer API (pinned host in, pinned host out)
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        postprocess_host(heads_host, STRIDES, device=dev, **NMS_KW)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out_dets, out_counts = postprocess_host(heads_host, STRIDES, device=dev, **NMS_KW)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    h2d = sum(x.numel() * x.element_size() for lv in heads_host for x in lv)
    d2h = out_dets.numel() * 4 + out_counts.numel() * 4

    # ---- config 5 as stated (strong scaling): B = 512 split over the N ranks (the 64 synthetic images tiled)
    cfg5 = None
    if not args.no_extras:
        b5 = 512 // world
        heads5 = [[x.repeat(b5 // B_PER_GPU, 1, 1, 1) if b5 >= B_PER_GPU else x[:b5].contiguous() for x in lv] for lv in heads_dev]
        deliv5 = make_delivery(len(NCS), b5, NMS_KW["max_det"], dev) if world > 1 else None
        pipe5 = PostHeadPipeline(heads5, STRIDES, NMS_KW, outs=deliv5.outs if deliv5 else None, delivery=deliv5)
        s5 = 40

        def run5(n):
            pipe5.k, pipe5.pending = 0, None
            for k in range(n):
                if deliv5 is not None:
                    deliv5.before_write((k - 1) & 1)
                done = pipe5.step()
                if deliv5 is not None and done is not None:
                    deliv5.after_write(done)
            if deliv5 is not None:
                deliv5.before_write((n - 1) & 1)
            done = pipe5.flush()
            if deliv5 is not None:
                deliv5.after_write(done)
                deliv5.drain()

        run5(5)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run5(s5)
        e1.record()
        barrier()
        ms5 = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms5], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms5 = float(tt.item())
        cfg5 = {"global_batch": 512, "batch_per_gpu": b5, "steps": s5, "ms_per_step": ms5 / s5, "value": 512 * s5 / (ms5 * 1e-3),
                "unit": "images/s", "scaling": "strong", "data": "the 64 synthetic images of rank 0..N-1 tiled to B=512"}
        del pipe5, heads5, deliv5
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = _peaks()
        elt = 2
        bytes_per_launch = B_PER_GPU * _decode_bytes_per_image(NCS, ANCHORS, elt)
        line = {
            "metric": METRIC, "value": B_PER_GPU * world * steps / (elapsed_ms * 1e-3), "unit": "images/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": elapsed_ms / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": _config(world),
        }
        if dec_ms:
            dec_avg_ms = sum(dec_ms) / len(dec_ms)
            achieved = bytes_per_launch / (dec_avg_ms * 1e-3) / 1e9
            traffic = None
            tp = os.path.join(ROOT, "profiles", "decode_traffic.json")
            if os.path.exists(tp):
                with open(tp) as f:
                    traffic = json.load(f).get("dram_bytes_per_launch")
            line["roofline"] = {
                "kernel": "decode_pipe_kernel<__half,8,2,1>", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "frac_of_nominal_8000": achieved / 8000.0,
                "algorithmic_bytes_per_launch": bytes_per_launch, "decode_ms_avg": dec_avg_ms,
                "decode_ms_median": statistics.median(dec_ms), "decode_ms_max": max(dec_ms), "nms_ms_avg": sum(nms_ms) / len(nms_ms),
                "nms_ms_median": statistics.median(nms_ms), "timed_launches": len(dec_ms),
                "how": "CUDA events recorded by the step graph itself around each kernel, serial order, on "
                       f"{len(dec_ms)} steps spread over the timed region"}
        line["e2e"] = {"value": B_PER_GPU * world * e2e_steps / e2e_s, "unit": "images/s", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "steps": e2e_steps}
        line["gpu_launches"] = 2 * steps  # one decode_pipe_kernel + one nms_kernel per step, nothing else of ours
        line["launch_mode"] = "cuda_graphs, serial" if args.serial else ("cuda_graphs, one stream per step: NMS(k-1), then decode(k) launched programmatically "
                                                                        "beside it (griddepcontrol / programmatic stream serialization)")
        line["clocks"] = clk.summary()
        line["equality"] = equality
        if steady is not None:
            line["steady_state"] = steady
            line["instrumented_steps"] = len(dec_ms)
        if per_rank is not None:
            line["per_rank_ms"] = {"elapsed": [r[0] for r in per_rank], "decode_instrumented": [r[1] for r in per_rank],
                                   "nms_instrumented": [r[2] for r in per_rank]}
        if cfg5 is not None:
            line["config5_strong"] = cfg5
        if not args.no_extras and world == 1:
            # the same K-step loop without the overlap (decode -> NMS of the same batch, one stream, PDL edge)
            ser = PostHeadPipeline(heads_dev, STRIDES, NMS_KW, overlap=False)
            for _ in range(10):
                ser.step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(100):
                ser.step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 100
            line["serial"] = {"ms_per_step": ms, "value": B_PER_GPU / (ms * 1e-3), "unit": "images/s"}
            del ser
            try:
                line["surface"] = surface_line(heads_dev, dev)
            except Exception as exc:  # pragma: no cover
                line["surface"] = {"error": f"{type(exc).__name__}: {exc}"}
            try:
                line["planted"] = planted_line(dev)
            except Exception as exc:  # pragma: no cover
                line["planted"] = {"error": f"{type(exc).__name__}: {exc}"}
            try:
                line["head_tail"] = head_tail_line(dev)
            except Exception as exc:  # pragma: no cover
                line["head_tail"] = {"error": f"{type(exc).__name__}: {exc}"}
            try:
                line["gpu_eager_reference"] = eager_reference_line(heads_dev, dev)
            except Exception as exc:  # pragma: no cover
                line["gpu_eager_reference"] = {"error": f"{type(exc).__name__}: {exc}"}
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            cpu = CpuReference()
            cpu_heads = [[x[:CPU_SAMPLE_IMAGES].clone() for x in lv] for lv in heads_host]
            cpu.segment(cpu_heads, 0, 0)  # warm-up
            secs = sum(cpu.segment(cpu_heads, i, t) for i in range(CPU_SAMPLE_IMAGES) for t in range(3))
            line["cpu_baseline"] = {"value": CPU_SAMPLE_IMAGES / secs, "unit": "images/s", "cores": cores, "kind": cpu.kind,
                                    "sample": f"images 0..{CPU_SAMPLE_IMAGES - 1} of the same batch, all 3 task heads, once "
                                              f"({secs:.1f} s; {cpu.describe()})"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
