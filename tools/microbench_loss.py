"""Box-regression loss term (BboxLoss.forward, reference utils/loss.py:12-44): the fused kernels (``ops.bbox_loss``,
forward + backward) against the reference's ops run eagerly on the same GPU (tests/bbox_loss_port.py: one torch op per
reference op, five boolean-mask indexings and their host synchronisations included).  Training shape: B=64, 640x640
(8400 anchors on 80/40/20 levels), positives from seeded ground truths through the assigner (``ops.tal_assign``).

    python tools/microbench_loss.py [--out profiles/bbox_loss.md] [--batch 64]

Fused: CUDA events around forward + backward, L2 overwritten between iterations (a 256 MB buffer), median of the
iterations.  Reference: host clock around forward + backward + synchronise, median.  The backward kernel is also timed
alone; its algorithmic bytes are the fg_mask read, the dense gradient writes and the positive anchors' inputs."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
import torch  # noqa: E402

import bbox_loss_port as lp  # noqa: E402
from cerberusdet_b200 import _lib, ops  # noqa: E402

LEVELS, STRIDES = [(80, 80), (40, 40), (20, 20)], [8, 16, 32]
HBM_MEASURED_GBS = 6531.9  # the B200's measured HBM peak (MEASURED_PEAKS.json where present; DESIGN §4.1)
try:
    with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as _f:
        HBM_MEASURED_GBS = float(json.load(_f)["hbm_gbs"])
except (OSError, KeyError, ValueError):
    pass


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def fused_step(c):
    pd = c["pred_dist"].detach().requires_grad_(True)
    pb = c["pred_bboxes"].detach().requires_grad_(True)
    li, ld = ops.bbox_loss(**dict(c, pred_dist=pd, pred_bboxes=pb))
    torch.autograd.backward((li, ld))


def reference_step(c):
    pd = c["pred_dist"].detach().requires_grad_(True)
    pb = c["pred_bboxes"].detach().requires_grad_(True)
    li, ld = lp.bbox_loss_port(**dict(c, pred_dist=pd, pred_bboxes=pb))
    torch.autograd.backward((li, ld))


def time_events(fn, flush, n=50, warm=5):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return statistics.median(ts)


def time_host(fn, flush, n=30, warm=5):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e6)
    return statistics.median(ts)


def bwd_kernel(c, code):
    """One cerb_bbox_loss_bwd launch on the case (the op's backward without autograd around it)."""
    lib = _lib.load()
    B, A, C = (int(v) for v in c["target_scores"].shape)
    gd, gb = torch.empty_like(c["pred_dist"]), torch.empty_like(c["pred_bboxes"])
    g = torch.ones(2, device="cuda")
    tss = c["target_scores_sum"]
    ptr = lambda k: c[k].data_ptr()  # noqa: E731
    stream = torch.cuda.current_stream().cuda_stream

    def run():
        rc = lib.cerb_bbox_loss_bwd(ptr("pred_dist"), ptr("pred_bboxes"), ptr("anchor_points"), ptr("target_bboxes"),
                                    ptr("target_scores"), ptr("fg_mask"), tss.data_ptr(), 1.0, B, A, C, 16, code,
                                    g.data_ptr(), g[1:].data_ptr(), gd.data_ptr(), gb.data_ptr(), stream)
        _lib.check(rc)

    return run


# mode: (prediction dtype, dtype code); "amp" and "bf16" run under autocast of that dtype
MODES = {"fp32": (torch.float32, _lib.CERB_F32), "amp": (torch.float16, _lib.CERB_F16), "bf16": (torch.bfloat16, _lib.CERB_BF16)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bbox_loss.md"))
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--modes", default="fp32,amp", help="comma-separated: fp32, amp (fp16 autocast), bf16 (bf16 autocast)")
    args = ap.parse_args()
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rows = []
    for C in (20, 80):
        for mode in args.modes.split(","):
            dtype, code = MODES[mode]
            c = lp.loss_case(5, args.batch, LEVELS, STRIDES, C, 20, dtype=dtype, ops=ops)
            amp = torch.autocast("cuda", dtype=dtype, enabled=mode != "fp32")
            with amp:
                fused = time_events(lambda: fused_step(c), flush)
                ref = time_host(lambda: reference_step(c), flush)
            bwd = time_events(bwd_kernel(c, code), flush)
            B, A = c["fg_mask"].shape
            npos = int(c["fg_mask"].sum())
            s = c["pred_dist"].element_size()
            # fg_mask, dense grad_pred_dist + grad_pred_bboxes writes, per positive: 64 bins + box + anchor + target box + score row
            nbytes = B * A * (1 + 64 * s + 4 * s) + npos * (64 * s + 4 * s + 2 * s + 16 + 4 * C)
            rows.append(dict(classes=C, mode=mode, positives=npos, fused_fwd_bwd_us=round(fused, 1), reference_fwd_bwd_us=round(ref, 1),
                             speedup=round(ref / fused, 1), bwd_kernel_us=round(bwd, 1), bwd_bytes=nbytes,
                             bwd_GBps=round(nbytes / bwd / 1e3, 1), bwd_frac_of_measured_hbm=round(nbytes / bwd / 1e3 / HBM_MEASURED_GBS, 3)))
            print(json.dumps(rows[-1]), flush=True)
    lines = [
        "# Box-regression loss term (`ops.bbox_loss`) on the B200",
        "",
        f"Measured with `tools/microbench_loss.py` on **{name}** (power limit, max SM clock: {power}).  "
        f"B={args.batch}, 640x640 (8400 anchors), 20 ground truths per image through `ops.tal_assign`; \"fp32\" = every tensor "
        "fp32, \"amp\" = the trainer's fp16 autocast case, \"bf16\" = its bf16 autocast case.",
        "",
        "- fused: `ops.bbox_loss` forward + backward (two kernels + the workspace memset), CUDA events, L2 overwritten between "
        "iterations, median of 50.",
        "- reference: the reference's ops run eagerly on the same GPU (`tests/bbox_loss_port.py`, five boolean-mask indexings, "
        "each a host synchronisation), host clock around forward + backward + synchronise, median of 30.",
        f"- backward kernel alone: algorithmic bytes (fg_mask, the dense gradients, the positives' inputs) over its time, as a "
        f"share of the measured HBM peak, {HBM_MEASURED_GBS / 1000:.2f} TB/s (DESIGN §4.1).",
        "",
        "| classes | mode | positives | fused fwd+bwd (us) | reference fwd+bwd (us) | speed-up | bwd kernel (us) | bwd GB/s | share of measured HBM |",
        "|---|---|---|---|---|---|---|---|---|",
    ]
    for r in rows:
        lines.append(f"| {r['classes']} | {r['mode']} | {r['positives']} | {r['fused_fwd_bwd_us']} | {r['reference_fwd_bwd_us']} | "
                     f"{r['speedup']}x | {r['bwd_kernel_us']} | {r['bwd_GBps']} | {r['bwd_frac_of_measured_hbm']:.0%} |")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
