"""numpy restatement of the letterbox the kernel of ``csrc/letterbox.cu`` computes, and the reference's own text.

``letterbox_verbatim`` is the reference's ``letterbox`` (cerberusdet/data/augmentations.py:59-90) for the arguments the
inference preprocessor uses (no ``scaleFill``).  ``resize_linear_port`` is cv2's ``INTER_LINEAR`` resize of a uint8
HWC image restated in integer numpy (imgproc/src/resize.cpp): the coefficient tables, the exact horizontal pass, the
fixed-point vertical pass and the switch to ``INTER_AREA`` for an exact 2x downscale.  ``letterbox_port`` puts the two
together as the kernel does: uint8 BGR HWC in, the letterboxed RGB CHW uint8 image out."""
from __future__ import annotations

import numpy as np

PAD = 114


def letterbox_verbatim(im, new_shape=(640, 640), color=(114, 114, 114), auto=True, scaleup=True, stride=32):
    import cv2

    shape = im.shape[:2]  # current shape [height, width]
    if isinstance(new_shape, int):
        new_shape = (new_shape, new_shape)
    r = min(new_shape[0] / shape[0], new_shape[1] / shape[1])
    if not scaleup:
        r = min(r, 1.0)
    ratio = r, r
    new_unpad = int(round(shape[1] * r)), int(round(shape[0] * r))
    dw, dh = new_shape[1] - new_unpad[0], new_shape[0] - new_unpad[1]
    if auto:
        dw, dh = np.mod(dw, stride), np.mod(dh, stride)
    dw /= 2
    dh /= 2
    if shape[::-1] != new_unpad:
        im = cv2.resize(im, new_unpad, interpolation=cv2.INTER_LINEAR)
    top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
    left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
    im = cv2.copyMakeBorder(im, top, bottom, left, right, cv2.BORDER_CONSTANT, value=color)
    return im, ratio, (dw, dh)


def _coeffs(dst: int, src: int):
    """cv2's per-output-index source index and 11-bit weights: fx = (float)((d + 0.5) * scale - 0.5), sx = floor(fx),
    fx -= sx, weights rint((1 - fx) * 2048) and rint(fx * 2048) (``saturate_cast<short>``).  ``clamp`` applies the
    horizontal border rule (fx = 0 at both ends); the vertical pass keeps the weights and clamps the rows instead."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    return s, f


def _weights(f):
    w0 = np.rint((np.float32(1.0) - f).astype(np.float32) * np.float32(2048)).astype(np.int64)
    w1 = np.rint(f * np.float32(2048)).astype(np.int64)
    return w0, w1


def resize_linear_port(im: np.ndarray, out_w: int, out_h: int) -> np.ndarray:
    """``cv2.resize(im, (out_w, out_h), interpolation=cv2.INTER_LINEAR)`` for a uint8 [h, w, 3] image."""
    h, w = im.shape[:2]
    if (out_w, out_h) == (w, h):
        return im.copy()
    src = im.astype(np.int64)
    if w == 2 * out_w and h == 2 * out_h:  # is_area_fast with a 2x2 kernel: cv2 switches to INTER_AREA
        s = src[0::2, 0::2] + src[0::2, 1::2] + src[1::2, 0::2] + src[1::2, 1::2]
        return ((s + 2) >> 2).astype(np.uint8)
    sx, fx = _coeffs(out_w, w)
    left, right = sx < 0, sx >= w - 1
    fx = np.where(left | right, np.float32(0), fx).astype(np.float32)
    sx = np.clip(sx, 0, w - 1)
    a0, a1 = _weights(fx)
    x1 = np.minimum(sx + 1, w - 1)
    hrow = src[:, sx] * a0[None, :, None] + src[:, x1] * a1[None, :, None]  # [h, out_w, 3], exact
    sy, fy = _coeffs(out_h, h)
    b0, b1 = _weights(fy)
    y0, y1 = np.clip(sy, 0, h - 1), np.clip(sy + 1, 0, h - 1)
    r0, r1 = hrow[y0], hrow[y1]
    v = ((((r0 >> 4) * b0[:, None, None]) >> 16) + (((r1 >> 4) * b1[:, None, None]) >> 16) + 2) >> 2
    return np.clip(v, 0, 255).astype(np.uint8)


def letterbox_port(im: np.ndarray, geometry) -> np.ndarray:
    """uint8 BGR [h, w, 3] -> the letterboxed uint8 RGB [3, out_h, out_w] for ``geometry`` =
    ``(unpad_h, unpad_w, top, left, out_h, out_w)``."""
    uh, uw, top, left, out_h, out_w = geometry
    out = np.full((out_h, out_w, 3), PAD, dtype=np.uint8)
    out[top:top + uh, left:left + uw] = resize_linear_port(im, uw, uh)
    return np.ascontiguousarray(out[:, :, ::-1].transpose(2, 0, 1))


def random_image(rng: np.random.Generator, h: int, w: int) -> np.ndarray:
    """A uint8 BGR image with smooth areas, edges and noise (every rounding path of the resize gets exercised)."""
    yy, xx = np.mgrid[0:h, 0:w]
    base = (np.sin(xx[..., None] * rng.uniform(0.01, 0.3, 3) + yy[..., None] * rng.uniform(0.01, 0.3, 3)) * 127.5 + 127.5)
    noise = rng.integers(0, 256, (h, w, 3))
    mix = np.where(rng.random((h, w, 1)) < 0.3, noise, base)
    return np.clip(mix, 0, 255).astype(np.uint8)
