"""Validation mAP statistics (``ap_per_class``, reference utils/metrics.py:56-120): the GPU path against the numpy
restatement of the reference on the same machine's host cores, at VOC size (1.49 M detections x 10 IoU columns, 20
classes) and Objects365 size (80 000 images x 300 detections = 24 M rows, 365 Zipf-skewed classes).  Stats come from
``tests/ap_port.make_stats``: TP probability rises with ``conf`` and the 10 columns are nested.

    python tools/microbench_ap.py [--out profiles/ap_per_class.md] [--iters 10]

- kernels: CUDA events around ``cerb_ap_per_class`` alone (inputs resident, workspace allocated), median;
- device op: ``ops.ap_per_class`` on device tensors (NaN check, ``torch.unique``, the copy of nc values to the host,
  workspace allocation, the kernels), host clock to a synchronise, median;
- drop-in: ``val_stats.ap_per_class`` from numpy in to numpy out (H2D copies of the stats, the op, the host tail), median;
- numpy: the reference's text (``tests/ap_port.ap_per_class_verbatim``), host clock, one run (the 24 M case takes
  minutes).
Every shape is run once before it is timed.  The drop-in's outputs are compared with the port's at both sizes."""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402
import torch  # noqa: E402

import ap_port  # noqa: E402
from cerberusdet_b200 import _lib, ops, val_stats  # noqa: E402

SIZES = [("VOC", 1_490_000, 20), ("Objects365", 24_000_000, 365)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def kernel_ms(tp, conf, pred_cls, target_cls, iters):
    lib = _lib.load()
    classes, nt = torch.unique(target_cls, sorted=True, return_counts=True)
    classes_h, nt_h = classes.cpu(), nt.cpu()
    n, K = tp.shape
    nc = classes.numel()
    ap = torch.empty((nc, K), dtype=torch.float64, device="cuda")
    p = torch.empty((nc, 1000), dtype=torch.float64, device="cuda")
    r = torch.empty((nc, 1000), dtype=torch.float64, device="cuda")
    ws_bytes = int(lib.cerb_ap_workspace_bytes(n, K, nc))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def run():
        _lib.check(lib.cerb_ap_per_class(tp.data_ptr(), K, conf.data_ptr(), pred_cls.data_ptr(), n, classes_h.data_ptr(),
                                         nt_h.data_ptr(), nc, 1e-16, ap.data_ptr(), p.data_ptr(), r.data_ptr(), ws.data_ptr(),
                                         ws_bytes, stream))

    run()
    times = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), ws_bytes


def wall_ms(fn, iters):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t) * 1e3)
    return statistics.median(times)


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--out", default=os.path.join(ROOT, "profiles", "ap_per_class.md"))
    ap_.add_argument("--iters", type=int, default=10)
    args = ap_.parse_args()
    name, limits = card()
    rows = []
    for label, n, nc in SIZES:
        stats = ap_port.make_stats(n, nc, seed=0)
        names = {k: str(k) for k in range(nc)}
        dev = [torch.from_numpy(a).cuda() for a in stats]
        k_ms, ws_bytes = kernel_ms(*dev, args.iters)
        op_ms = wall_ms(lambda: ops.ap_per_class(*dev), args.iters)
        got = val_stats.ap_per_class(*stats, names=names)
        dropin_ms = wall_ms(lambda: val_stats.ap_per_class(*stats, names=names), args.iters)
        want = ap_port.ap_per_class_port(*stats, names)
        same = all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(got, want))
        t = time.perf_counter()
        ap_port.ap_per_class_verbatim(*stats, names)
        numpy_ms = (time.perf_counter() - t) * 1e3
        rows.append((label, n, nc, k_ms, op_ms, dropin_ms, numpy_ms, ws_bytes, same))
        print(label, f"kernels {k_ms:.2f} ms, op {op_ms:.2f} ms, drop-in {dropin_ms:.1f} ms, numpy {numpy_ms:.0f} ms, "
              f"bit-equal to the port: {same}", flush=True)
    lines = [
        "# Validation mAP statistics (`ap_per_class`) on the B200",
        "",
        f"Measured with `tools/microbench_ap.py` on **{name}** (power limit, max SM clock: {limits}); the numpy column on the "
        f"same machine's host cores ({os.cpu_count()} logical CPUs).  K = 10 IoU columns; stats from `tests/ap_port.make_stats` "
        "(Zipf-distributed classes, TP probability rising with `conf`, nested columns).",
        "",
        f"- kernels: CUDA events around `cerb_ap_per_class` alone, median of {args.iters};",
        f"- device op: `ops.ap_per_class` on device tensors (NaN check, `torch.unique`, nc values to the host, workspace, kernels), host clock to a synchronise, median of {args.iters};",
        f"- drop-in: `val_stats.ap_per_class` from numpy in to numpy out, H2D copies and the host tail included, median of {args.iters};",
        "- numpy: the reference's text (`tests/ap_port.ap_per_class_verbatim`), one run.",
        "",
        "| stats | rows | classes | kernels (ms) | device op (ms) | drop-in (ms) | numpy (ms) | drop-in speed-up | workspace (MB) | drop-in = port |",
        "|---|---|---|---|---|---|---|---|---|---|",
    ]
    for label, n, nc, k_ms, op_ms, dropin_ms, numpy_ms, ws_bytes, same in rows:
        lines.append(f"| {label} | {n:,} | {nc} | {k_ms:.2f} | {op_ms:.2f} | {dropin_ms:.1f} | {numpy_ms:.0f} | "
                     f"{numpy_ms / dropin_ms:.0f}x | {ws_bytes / 2**20:.0f} | {'bit-equal' if same else 'DIFFERENT'} |")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
