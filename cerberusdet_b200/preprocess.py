"""Letterbox preprocessing on the GPU: the inference front end of the reference's ``CerberusPreprocessor.preprocess``
(cerberusdet/cerberusdet_preprocessor.py:42-74) -- per image ``letterbox`` (data/augmentations.py:59-90: cv2
``INTER_LINEAR`` resize + constant 114 border), BGR -> RGB, HWC -> CHW, stack, upload, ``/255`` -- as one upload and
one kernel launch for the whole batch (``ops.letterbox``, ``csrc/letterbox.cu``).

``letterbox_geometry`` is the reference's shape arithmetic, ``letterbox_images`` the batched pipeline.  The pixels equal
cv2's bit for bit, and the normalised values equal what the reference's ``/255`` on the GPU gives (INTEGRATION §2).
"""
from __future__ import annotations

from typing import List, NamedTuple, Sequence, Tuple, Union

import numpy as np
import torch

from . import ops


class LetterboxGeometry(NamedTuple):
    """What the reference ``letterbox`` decides for one image: ``ratio`` and ``pad`` = ``(dw, dh)`` as it returns them,
    the resized size ``unpad_w`` x ``unpad_h`` and the border widths it passes to ``cv2.copyMakeBorder``."""

    ratio: Tuple[float, float]
    pad: Tuple[float, float]
    unpad_w: int
    unpad_h: int
    top: int
    bottom: int
    left: int
    right: int

    @property
    def out_shape(self) -> Tuple[int, int]:
        """``(height, width)`` of the letterboxed image."""
        return self.unpad_h + self.top + self.bottom, self.unpad_w + self.left + self.right


def letterbox_geometry(h: int, w: int, new_shape: Union[int, Sequence[int]] = 640, stride: int = 32, auto: bool = False,
                       scaleup: bool = True) -> LetterboxGeometry:
    """The shape arithmetic of the reference ``letterbox`` (data/augmentations.py:59-90) for an ``h`` x ``w`` image, in
    the same Python float operations: ``r = min(...)`` (``min(r, 1)`` without ``scaleup``), round-half-even of the
    scaled sizes, ``np.mod(d, stride)`` with ``auto``, the halved padding and ``int(round(d -/+ 0.1))`` borders."""
    shape = (int(h), int(w))
    if isinstance(new_shape, int):
        new_shape = (new_shape, new_shape)
    r = min(new_shape[0] / shape[0], new_shape[1] / shape[1])
    if not scaleup:
        r = min(r, 1.0)
    new_unpad = int(round(shape[1] * r)), int(round(shape[0] * r))
    dw, dh = new_shape[1] - new_unpad[0], new_shape[0] - new_unpad[1]
    if auto:
        dw, dh = np.mod(dw, stride), np.mod(dh, stride)
    dw /= 2
    dh /= 2
    return LetterboxGeometry((r, r), (dw, dh), new_unpad[0], new_unpad[1], int(round(dh - 0.1)), int(round(dh + 0.1)),
                             int(round(dw - 0.1)), int(round(dw + 0.1)))


def letterbox_images(images: Sequence[Union[np.ndarray, torch.Tensor]], new_shape: Union[int, Sequence[int]] = 640,
                     stride: int = 32, auto: bool = False, scaleup: bool = True, half: bool = True,
                     device: Union[str, torch.device] = "cuda") -> Tuple[torch.Tensor, List[Tuple[int, int]]]:
    """Letterbox a batch of uint8 BGR ``[h, w, 3]`` images (numpy arrays as ``cv2.imread`` returns them, or CUDA tensors
    of that layout, used in place) into one ``[B, 3, H, W]`` RGB tensor on ``device``, float16 with ``half`` else
    float32, scaled by 1/255.  Host images go up in one copy from one pinned buffer; the batch is one kernel launch.

    Returns ``(tensor, shapes)`` with ``shapes[i] = (h_i, w_i)``, the ``original_shape`` list
    ``CerberusDetInference.predict`` takes.  ``auto=True`` pads to a multiple of ``stride`` per image; images that then
    get different sizes raise ``ValueError`` (the reference's ``np.stack`` fails on them too)."""
    if len(images) == 0:
        raise ValueError("letterbox_images needs at least one image")
    device = torch.device(device)
    if device.type != "cuda":
        raise TypeError(f"letterbox_images runs on a CUDA device (cerberusdet_b200 has no CPU path), got {device}")
    shapes, geoms = [], []
    for i, im in enumerate(images):
        if im.ndim != 3 or im.shape[2] != 3 or im.dtype not in (np.uint8, torch.uint8):
            raise TypeError(f"image {i}: expected a uint8 [h, w, 3] BGR image, got {im.dtype} {tuple(im.shape)}")
        h, w = int(im.shape[0]), int(im.shape[1])
        g = letterbox_geometry(h, w, new_shape, stride, auto, scaleup)
        if g.unpad_w <= 0 or g.unpad_h <= 0:
            raise ValueError(f"image {i}: {h}x{w} scales to an empty {g.unpad_h}x{g.unpad_w} image")
        shapes.append((h, w))
        geoms.append(g)
    out_hw = geoms[0].out_shape
    if any(g.out_shape != out_hw for g in geoms):
        raise ValueError(f"letterboxed images differ in size ({sorted({g.out_shape for g in geoms})}); with auto=True "
                         "every image of a batch must pad to the same shape")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    host = [i for i, im in enumerate(images) if not torch.is_tensor(im)]
    src = list(images)
    if host:
        sizes = [int(images[i].nbytes) for i in host]
        staged = torch.empty((sum(sizes),), dtype=torch.uint8, pin_memory=True)
        flat = staged.numpy()
        o = 0
        for i, n in zip(host, sizes):
            flat[o:o + n].reshape(images[i].shape)[...] = images[i]
            o += n
        dev_buf = staged.to(device, non_blocking=True)
        o = 0
        for i, n in zip(host, sizes):
            src[i] = dev_buf[o:o + n].view(images[i].shape)
            o += n
    out = ops.letterbox(src, [(g.unpad_h, g.unpad_w, g.top, g.left) for g in geoms], out_hw,
                        torch.float16 if half else torch.float32)
    return out, shapes
