"""TAL assigner: cerb_tal_assign (three launches) against the reference's own TaskAlignedAssigner.forward on the same GPU
(eager PyTorch, oracle/_ref; where that tree is absent, oracle/ref_port.tal_assign_port, its op-by-op restatement),
training shape 640x640 (8400 anchors).  Engineering numbers for DESIGN.md, not bench values.
    python tools/microbench_tal.py [--batch 64] [--boxes 20] [--classes 20] [--dtype fp32|fp16|bf16]
fp16 and bf16 are the scores of the trainer under autocast of that dtype; both sides run under it."""
import argparse
import json
import os
import sys
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from cerberusdet_b200 import ops  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from oracle.ref_import import load_reference, reference_available  # noqa: E402


def timeit(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--boxes", type=int, default=20)
    ap.add_argument("--classes", type=int, default=20)
    ap.add_argument("--dtype", choices=("fp32", "fp16", "bf16"), default="fp32")
    args = ap.parse_args()
    dt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    c = {k: v.cuda() for k, v in rp.tal_case(5, args.batch, [(80, 80), (40, 40), (20, 20)], [8, 16, 32], args.classes, args.boxes,
                                             score_dtype=dt).items()}
    amp = torch.autocast("cuda", dtype=dt, enabled=args.dtype != "fp32")
    res = {"gpu": torch.cuda.get_device_name(0), "batch": args.batch, "boxes": args.boxes, "classes": args.classes,
           "anchors": 8400, "scores": args.dtype}
    with amp:
        res["kernel_us"] = round(timeit(lambda: ops.tal_assign(**c, topk=10, num_classes=args.classes)), 1)
    if reference_available():
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            load_reference()
        from cerberusdet.utils.tal import TaskAlignedAssigner

        asg = TaskAlignedAssigner(topk=10, num_classes=args.classes, alpha=0.5, beta=6.0).cuda()
        fwd = getattr(TaskAlignedAssigner.forward, "_cerb_reference", TaskAlignedAssigner.forward)
        with amp:
            res["reference_eager_us"] = round(timeit(lambda: fwd(asg, c["pd_scores"], c["pd_bboxes"], c["anc_points"],
                                                                c["gt_labels"], c["gt_bboxes"], c["mask_gt"]), reps=10), 1)
        res["speedup"] = round(res["reference_eager_us"] / res["kernel_us"], 1)
    else:  # without the reference tree: its ops as oracle/ref_port.py restates them, eagerly on the same GPU
        with amp, torch.device("cuda"):
            res["port_eager_us"] = round(timeit(lambda: rp.tal_assign_port(**c, topk=10, num_classes=args.classes), reps=10), 1)
        res["speedup_vs_port"] = round(res["port_eager_us"] / res["kernel_us"], 1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
