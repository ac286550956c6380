"""bf16 against fp16 on the post-head kernels, on the GPU: decode and NMS kernel times (CUDA events, L2 overwritten
between timed calls, the two dtypes alternated in the same process), the NMS counters (IoU tests and candidates consumed
per segment, ``ops.nms_statistics``) and the path a bf16 user had before the kernels took bf16: the reference's decode
ops + one ``non_max_suppression`` per image (torchvision's CUDA NMS) on the same GPU, on a sample of the batch.

    python tools/microbench_bf16.py [--configs cfg3 cfg4] [--reps 30] [--out FILE]

Config 3: 3 tasks (20/19/12), B = 64, 640 x 640; config 4: the same heads, B = 16, 1280 x 1280; both at the validation
settings (conf 0.001, IoU 0.6, multi-label, max_det 300).  Prints one JSON line per (config, dtype) and one for the
eager path; ``--out`` also writes them there.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from cerberusdet_b200 import ops  # noqa: E402
from cerberusdet_b200.synth import STRIDES, synth_heads  # noqa: E402

NCS = [20, 19, 12]
KW = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
CFG = {"cfg3": (64, 640), "cfg4": (16, 1280)}


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def time_alternating(fns, reps, flush):
    """{name: median microseconds}: every repetition runs each function once, in turn, after overwriting the L2."""
    ts = {k: [] for k in fns}
    for _ in range(3):
        for fn in fns.values():
            fn()
    for _ in range(reps):
        for k, fn in fns.items():
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b) * 1e3)
    return {k: statistics.median(v) for k, v in ts.items()}


def eager_reference(heads_dev, n_img=8, budget_s=30.0):
    """The reference's decode ops + per-image non_max_suppression (torchvision CUDA NMS), eagerly, on images 0..n_img-1."""
    from oracle import ref_port as rp

    sample = [[x[:n_img].contiguous() for x in lv] for lv in heads_dev]

    def once():
        for t, lv in enumerate(sample):
            y = rp.decode_port(lv, NCS[t], STRIDES)
            for i in range(n_img):
                rp.nms_port(y[i:i + 1], greedy="torchvision", **KW)

    once()
    torch.cuda.synchronize()
    t0, reps = time.perf_counter(), 0
    while reps < 5 and time.perf_counter() - t0 < budget_s:
        once()
        reps += 1
    torch.cuda.synchronize()
    s = (time.perf_counter() - t0) / reps
    return {"images_per_s": round(n_img / s, 2), "ms_per_image": round(1e3 * s / n_img, 2), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["cfg3", "cfg4"])
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = [{"card": card(), "torch": torch.__version__}]
    print(json.dumps(lines[0]), flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # twice the 126 MB L2
    for name in a.configs:
        B, imgsz = CFG[name]
        dev, ys = {}, {}
        for dt in (torch.float16, torch.bfloat16):
            heads = synth_heads(range(B), NCS, imgsz, dt, "iid", cfg=3)
            dev[dt] = [[x.cuda() for x in lv] for lv in heads]
            del heads
            ys[dt] = ops.decode_heads(dev[dt], STRIDES)
        fns = {}
        for dt, tag in ((torch.float16, "fp16"), (torch.bfloat16, "bf16")):
            fns["decode_" + tag] = (lambda d=dt: ops.decode_heads(dev[d], STRIDES))
            fns["nms_" + tag] = (lambda d=dt: ops.nms_batched(ys[d], **KW))
        med = time_alternating(fns, a.reps, flush)
        A = sum(x.shape[2] * x.shape[3] for x in dev[torch.float16][0])
        nbytes = B * sum((64 + nc + 4 + nc) * 2 * A for nc in NCS)
        for dt, tag in ((torch.float16, "fp16"), (torch.bfloat16, "bf16")):
            dets, counts, stats = ops.nms_statistics(ys[dt], **KW)
            st = stats.double()
            line = {"cfg": name, "dtype": tag, "B": B, "imgsz": imgsz,
                    "decode_us": round(med["decode_" + tag], 1), "decode_GBps": round(nbytes / med["decode_" + tag] / 1e3, 1),
                    "nms_us": round(med["nms_" + tag], 1),
                    "iou_tests_per_segment": round(float(st[..., 0].mean()), 1),
                    "consumed_per_segment": round(float(st[..., 1].mean()), 1),
                    "consumed_max": int(stats[..., 1].max()), "kept_per_segment": round(float(counts.double().mean()), 1)}
            lines.append(line)
            print(json.dumps(line), flush=True)
        if name == "cfg3":
            line = {"cfg": name, "dtype": "bf16", "path": "eager reference ops, per-image NMS",
                    **eager_reference(dev[torch.bfloat16])}
            lines.append(line)
            print(json.dumps(line), flush=True)
        del dev, ys
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
