"""Validation confusion matrix: the reference's ``ConfusionMatrix.process_batch`` text per image on CUDA tensors, the
drop-in (``val_stats.make_confusion_process_batch``) per image, and ``ops.confusion_matrix_batch`` per batch of 32, on a
VOC-size run (4952 images, nc 20) and an Objects365-size run (nc 365).  Detections are what NMS leaves at the validation
settings (conf 0.001, max_det 300): 300 rows per image, most of them below the matrix's conf 0.25.  Each arm is timed with
the host clock up to a device synchronise; the kernel with CUDA events; synchronisations per image with
``torch.cuda.set_sync_debug_mode``.  Writes a markdown table (``--out``).

    python tools/microbench_confusion.py --out profiles/confusion_matrix.md
"""
import argparse
import os
import subprocess
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import confusion_port as cp  # noqa: E402

from cerberusdet_b200 import ops, val_stats  # noqa: E402


def make_run(n_images, nc, mean_labels, seed, max_det=300):
    """Per image: labels (Poisson count around ``mean_labels``, at least 1) and ``max_det`` detections with NMS-like
    confidences (a few high, most near the 0.001 floor), in batches of 32 as the validation loop holds them."""
    rng = np.random.default_rng(seed)
    batches = []
    for b0 in range(0, n_images, 32):
        B = min(32, n_images - b0)
        dets = torch.zeros((B, max_det, 6))
        labs, offsets = [], [0]
        for b in range(B):
            M = int(min(max(rng.poisson(mean_labels), 1), 200))
            d, lab = cp.image_case(rng, M, max_det, nc)
            d[:, 4] = torch.from_numpy(np.sort(rng.random(max_det) ** 6)[::-1].copy()).clamp(min=0.001)
            dets[b] = d
            labs.append(lab)
            offsets.append(offsets[-1] + M)
        batches.append((dets.cuda(), torch.full((B,), max_det, dtype=torch.int32, device="cuda"), torch.cat(labs).cuda(),
                        torch.tensor(offsets, dtype=torch.int32, device="cuda"), offsets))
    return batches


def per_image(batches):
    for dets, counts, labels, _, offsets in batches:
        for b in range(dets.shape[0]):
            yield dets[b], labels[offsets[b] : offsets[b + 1]]


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def syncs(fn):
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            fn()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    return sum("synchroniz" in str(x.message) for x in w)


def bench(name, n_images, nc, mean_labels, ref_sample, seed):
    batches = make_run(n_images, nc, mean_labels, seed)
    images = list(per_image(batches))
    dropin = val_stats.make_confusion_process_batch(cp.ConfusionMatrixVerbatim.process_batch)
    ref_cm, drop_cm = cp.ConfusionMatrixVerbatim(nc), cp.ConfusionMatrixVerbatim(nc)
    out = torch.zeros((nc + 1, nc + 1), dtype=torch.int64, device="cuda")

    def run_ref(cm, imgs):
        for d, lab in imgs:
            cm.process_batch(d, lab)

    def run_drop(cm, imgs):
        for d, lab in imgs:
            dropin(cm, d, lab)

    def run_batched():
        for dets, counts, labels, offs, _ in batches:
            ops.confusion_matrix_batch(dets, counts, labels, offs, nc, out=out)

    # warm-up every arm on a few images / one batch
    run_ref(cp.ConfusionMatrixVerbatim(nc), images[:4])
    run_drop(cp.ConfusionMatrixVerbatim(nc), images[:4])
    ops.confusion_matrix_batch(*batches[0][:4], nc)
    sample = images[:ref_sample]
    t_ref = timed(lambda: run_ref(ref_cm, sample))
    t_drop = timed(lambda: run_drop(drop_cm, images))
    out.zero_()
    t_batch = timed(run_batched)
    # kernel time: events around the batched launches, many passes
    passes = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(passes):
        run_batched()
    e1.record()
    torch.cuda.synchronize()
    t_kernel = e0.elapsed_time(e1) / 1e3 / passes
    # the three agree (the sample is tie-free in practice; the drop-in and the op use one tie rule)
    check = cp.ConfusionMatrixVerbatim(nc)
    run_drop(check, sample)
    agree_ref = np.array_equal(check.matrix, ref_cm.matrix)
    agree_op = np.array_equal(out.cpu().numpy(), (passes + 1) * drop_cm.matrix)
    s_ref = syncs(lambda: run_ref(cp.ConfusionMatrixVerbatim(nc), images[:50])) / 50
    s_drop = syncs(lambda: run_drop(cp.ConfusionMatrixVerbatim(nc), images[:50])) / 50
    s_batch = syncs(run_batched)
    kept = sum(int((d[:, 4] > 0.25).sum()) for d, _ in images[:500]) / min(500, len(images))
    labels_per = sum(int(lab.shape[0]) for _, lab in images) / len(images)
    n = len(images)
    return dict(name=name, n=n, nc=nc, labels=labels_per, kept=kept, ref_sample=len(sample),
                ref_ms=1e3 * t_ref / len(sample), drop_ms=1e3 * t_drop / n, batch_ms=1e3 * t_batch / n,
                ref_run=t_ref / len(sample) * n, drop_run=t_drop, batch_run=t_batch, kernel_run=t_kernel,
                kernel_batch_us=1e6 * t_kernel / len(batches), s_ref=s_ref, s_drop=s_drop, s_batch=s_batch / n,
                agree_ref=agree_ref, agree_op=agree_op)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--voc-images", type=int, default=4952)
    ap.add_argument("--o365-images", type=int, default=80000)
    ap.add_argument("--ref-sample", type=int, default=1000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("microbench_confusion: needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    rows = [bench("VOC size", a.voc_images, 20, 2.4, a.ref_sample, 0),
            bench("Objects365 size", a.o365_images, 365, 15.0, a.ref_sample, 1)]
    lines = [f"# Validation confusion matrix (`tools/microbench_confusion.py`)", "",
             f"Card: {card} (name, power limit; `nvidia-smi` in the same run).  torch {torch.__version__}.", "",
             "Detections per image: 300 (NMS at conf 0.001, max_det 300), confidences mostly near the floor; "
             "`ConfusionMatrix(nc)` defaults conf 0.25, iou_thres 0.45.  Host clock to a synchronise for each arm; the "
             "reference arm runs on the first `sample` images and is scaled to the run.  Kernel time: CUDA events around "
             "the batched launches (20 passes).  Synchronisations: `torch.cuda.set_sync_debug_mode`.", "",
             "| run | images | nc | labels / image | dets > 0.25 / image | reference text / image | drop-in / image | "
             "batched op (32) / image | reference text / run | drop-in / run | batched op / run | kernel / run | kernel / batch "
             "| syncs / image: ref, drop-in, batched | results agree |",
             "|---|---|---|---|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append(f"| {r['name']} | {r['n']} | {r['nc']} | {r['labels']:.1f} | {r['kept']:.1f} | {r['ref_ms']:.3f} ms "
                     f"(sample {r['ref_sample']}) | {r['drop_ms']:.3f} ms | {r['batch_ms'] * 1e3:.2f} µs | {r['ref_run']:.2f} s | "
                     f"{r['drop_run']:.3f} s | {r['batch_run'] * 1e3:.2f} ms | {r['kernel_run'] * 1e3:.3f} ms | "
                     f"{r['kernel_batch_us']:.1f} µs | {r['s_ref']:.1f}, {r['s_drop']:.1f}, {r['s_batch']:.1f} | "
                     f"{r['agree_ref'] and r['agree_op']} |")
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
