"""Letterbox preprocessing (``cerb_letterbox``; reference cerberusdet_preprocessor.py:42-74) on the GPU: kernel time,
bandwidth, the upload of the raw images and the whole path from numpy in to device tensor out, against the reference
recipe on one host thread.

    python tools/microbench_letterbox.py [--out profiles/letterbox.md] [--iters 20]

- kernel: CUDA events around one ``cerb_letterbox`` call on device-resident images (called through ctypes with the
  arguments prepared), after a 512 MB write that evicts the 126 MB L2, median;
- bandwidth: the source rows the resize reads plus the output written, over the kernel time, next to a device-to-device
  ``copy_`` of 1 GiB timed the same way (read + write bytes);
- upload: CUDA events around the host-to-device copy of the batch's raw bytes from one pinned buffer, median;
- end to end: ``preprocess.letterbox_images`` from a list of numpy images to the device tensor (staging into pinned
  memory, upload, kernel), host clock to a synchronise, median; the reference recipe (cv2 letterbox, cvtColor,
  transpose, np.stack, upload, ``.half()``, ``/ 255``) on one host thread the same way, when cv2 is installed.
The outputs of both paths are compared for every workload."""
import argparse
import ctypes
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

import letterbox_port as lp  # noqa: E402
from cerberusdet_b200 import _lib  # noqa: E402
from cerberusdet_b200.preprocess import letterbox_geometry, letterbox_images  # noqa: E402

MIXED = [(1080, 1920), (720, 1280), (480, 640), (1920, 1080), (375, 500), (1200, 1600), (640, 640), (2160, 3840)]
WORKLOADS = [("64 x 1920x1080 -> 640 (downscale)", [(1080, 1920)] * 64),
             ("64 mixed sizes -> 640 (8 each of " + ", ".join(f"{w}x{h}" for h, w in MIXED) + ")", MIXED * 8),
             ("64 x 500x333 -> 640 (upscale)", [(333, 500)] * 64)]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def event_ms(fn, iters, flush=None):
    fn()
    times = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


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


def rows_read(h, uh):
    """Source rows the resize of h rows to uh reads (all of them for a copy or the 2x area path)."""
    if uh == h or h == 2 * uh:
        return h
    s = np.floor(((np.arange(uh) + 0.5) * (1.0 / (uh / h)) - 0.5).astype(np.float32)).astype(np.int64)
    return len(set(np.clip(s, 0, h - 1).tolist()) | set(np.clip(s + 1, 0, h - 1).tolist()))


def reference_recipe(images, new_shape):
    import cv2

    out = []
    for im in images:
        x = lp.letterbox_verbatim(im, new_shape, auto=False)[0]
        x = cv2.cvtColor(x, cv2.COLOR_BGR2RGB).transpose(2, 0, 1)
        out.append(np.ascontiguousarray(x))
    t = torch.from_numpy(np.stack(out)).to("cuda").half()
    t /= 255.0
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "letterbox.md"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    name, limits = card()
    try:
        import cv2  # noqa: F401

        have_cv2 = True
    except ImportError:
        have_cv2 = False
    lib = _lib.load()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    big = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    big2 = torch.empty_like(big)
    copy_ms = event_ms(lambda: big2.copy_(big), args.iters)
    copy_tbs = 2 * big.numel() / copy_ms / 1e9
    del big, big2
    rng = np.random.default_rng(0)
    rows = []
    for label, sizes in WORKLOADS:
        ims = [lp.random_image(rng, h, w) for h, w in sizes]
        geoms = [letterbox_geometry(h, w, 640) for h, w in sizes]
        B = len(ims)
        pinned = torch.empty(sum(im.nbytes for im in ims), dtype=torch.uint8, pin_memory=True)
        o = 0
        for im in ims:
            pinned[o:o + im.nbytes].numpy()[:] = im.reshape(-1)
            o += im.nbytes
        dev_buf = torch.empty(pinned.numel(), dtype=torch.uint8, device="cuda")
        up_ms = event_ms(lambda: dev_buf.copy_(pinned, non_blocking=True), args.iters)
        dev, o = [], 0
        for im in ims:
            dev.append(dev_buf[o:o + im.nbytes].view(im.shape))
            o += im.nbytes
        out = torch.empty((B, 3, 640, 640), dtype=torch.float16, device="cuda")
        cargs = (_lib.ptr_array([d.data_ptr() for d in dev]), _lib.int_array([h for h, _ in sizes]), _lib.int_array([w for _, w in sizes]),
                 (ctypes.c_long * B)(*[3 * w for _, w in sizes]), _lib.int_array([g.unpad_h for g in geoms]),
                 _lib.int_array([g.unpad_w for g in geoms]), _lib.int_array([g.top for g in geoms]), _lib.int_array([g.left for g in geoms]),
                 B, 640, 640, _lib.CERB_F16, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        k_ms = event_ms(lambda: _lib.check(lib.cerb_letterbox(*cargs)), args.iters, flush)
        read = sum(rows_read(h, g.unpad_h) * 3 * w for (h, w), g in zip(sizes, geoms))
        written = out.numel() * out.element_size()
        e2e_ms = wall_ms(lambda: letterbox_images(ims, 640), max(3, args.iters // 4))
        got = letterbox_images(ims, 640)[0]
        if have_cv2:
            ref_ms = wall_ms(lambda: reference_recipe(ims, 640), 3)
            want = reference_recipe(ims, 640)
        else:
            ref_ms = None
            want = torch.from_numpy(np.stack([lp.letterbox_port(im, (g.unpad_h, g.unpad_w, g.top, g.left, 640, 640))
                                              for im, g in zip(ims, geoms)])).cuda().half() / 255.0
        same = torch.equal(got, want)
        raw = pinned.numel()
        rows.append((label, B, raw, read, written, k_ms, up_ms, e2e_ms, ref_ms, same, have_cv2))
        print(label, f"kernel {k_ms * 1e3:.1f} us ({(read + written) / k_ms / 1e9:.2f} TB/s), upload {up_ms:.2f} ms "
              f"({raw / up_ms / 1e6:.1f} GB/s), end to end {e2e_ms:.1f} ms, reference {ref_ms} ms, equal: {same}", flush=True)
        del dev_buf, dev, out, pinned
    lines = [
        "# Letterbox preprocessing (`cerb_letterbox`) on the B200",
        "",
        f"Measured with `tools/microbench_letterbox.py` on **{name}** (power limit, max SM clock: {limits}); host side on the "
        f"same machine ({os.cpu_count()} logical CPUs).  fp16 output `[64, 3, 640, 640]`, `auto=False`; images from "
        "`tests/letterbox_port.random_image`.",
        "",
        f"- kernel: CUDA events around one `cerb_letterbox` call on device-resident images, a 512 MB write before each "
        f"to evict L2, median of {args.iters};",
        "- bandwidth: source rows the resize reads + output written, over the kernel time; measured copy peak: device-to-"
        f"device `copy_` of 1 GiB, read + write = **{copy_tbs:.2f} TB/s**;",
        f"- upload: host-to-device copy of the raw uint8 images from one pinned buffer, CUDA events, median of {args.iters};",
        "- end to end: `preprocess.letterbox_images` from a list of numpy images to the device tensor (staging into pinned "
        "memory on one host thread, one upload, one launch), host clock to a synchronise;",
        "- reference recipe: per image cv2 `letterbox` + `cvtColor` + `transpose`, then `np.stack`, upload, `.half()`, `/ 255`, "
        "on one host thread, host clock to a synchronise.",
        "",
        "| workload | raw MB | kernel (us) | kernel GB/s (share of copy peak) | upload (ms) | upload GB/s | end to end (ms) | reference recipe (ms) | speed-up | same tensor |",
        "|---|---|---|---|---|---|---|---|---|---|",
    ]
    for label, B, raw, read, written, k_ms, up_ms, e2e_ms, ref_ms, same, cv in rows:
        bw = (read + written) / k_ms / 1e6
        ref = f"{ref_ms:.0f}" if ref_ms is not None else "not measured (no cv2)"
        sp = f"{ref_ms / e2e_ms:.1f}x" if ref_ms is not None else "-"
        lines.append(f"| {label} | {raw / 1e6:.0f} | {k_ms * 1e3:.0f} | {bw:.0f} ({bw / 1e3 / copy_tbs:.2f}) | {up_ms:.2f} | "
                     f"{raw / up_ms / 1e6:.1f} | {e2e_ms:.1f} | {ref} | {sp} | "
                     f"{('bit-equal to the reference recipe' if cv else 'bit-equal to the port') if same else 'DIFFERENT'} |")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
