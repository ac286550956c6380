"""Write tests/golden/letterbox_cv2.npz: seeded source images and the reference ``letterbox``'s output for them, made
with cv2 (the GPU tests compare the kernel against these bytes on machines without cv2).  Run: python tools/gen_golden_letterbox.py"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import letterbox_port as lp  # noqa: E402

# (h, w, new_shape, auto, scaleup): downscale, upscale, exact 2x (INTER_AREA), auto padding, 1-pixel-tall and -wide
# sources, odd pads, and scaleup=False (same size: no resize, pad only)
CASES = [(120, 160, 64, False, True), (33, 50, 96, False, True), (64, 64, 32, False, True), (40, 56, 64, True, True),
         (1, 37, 48, False, True), (45, 1, 48, False, True), (37, 53, [64, 96], False, True), (50, 70, 96, False, False)]


def main():
    import cv2

    rng = np.random.default_rng(2024)
    arrays, meta = {}, []
    for k, (h, w, new_shape, auto, scaleup) in enumerate(CASES):
        im = lp.random_image(rng, h, w)
        out, _, _ = lp.letterbox_verbatim(im, new_shape, auto=auto, scaleup=scaleup)
        arrays[f"src_{k}"], arrays[f"out_{k}"] = im, out
        meta.append({"new_shape": new_shape, "auto": auto, "scaleup": scaleup})
    arrays["meta"] = np.array(json.dumps({"cv2": cv2.__version__, "cases": meta}))
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "letterbox_cv2.npz"), **arrays)


if __name__ == "__main__":
    main()
