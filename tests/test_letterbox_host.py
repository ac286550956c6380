"""CPU tests of the letterbox preprocessing (``cerb_letterbox``, ``ops.letterbox``, ``preprocess``): the numpy port of
the kernel's arithmetic against cv2 and the reference's ``letterbox`` text, the geometry, the goldens the GPU tests use,
the ABI's argument checks and its ctypes prototype.  No kernel is launched here."""
import ctypes
import json
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import letterbox_port as lp  # noqa: E402

from cerberusdet_b200.preprocess import letterbox_geometry  # noqa: E402


def _shapes(n=60, seed=0):
    """Seeded (h, w, new_shape, auto, scaleup) cases: downscale, upscale, identity, exact 2x, 1-pixel-wide and -tall
    sources, odd pads, auto with stride 32 and scaleup=False."""
    rng = np.random.default_rng(seed)
    fixed = [(1080, 1920, 640, False, True), (720, 1280, 640, False, True), (700, 1000, 640, False, True),
             (1280, 1280, 640, False, True), (500, 333, 640, False, True), (150, 100, 640, False, True),
             (640, 480, 640, False, True), (480, 640, 640, False, True), (1, 100, 64, False, True), (100, 1, 64, False, True),
             (1, 60, 64, False, True), (60, 1, 64, False, True),
             (1, 1, 32, False, True), (64, 128, 64, False, True), (37, 53, (64, 96), False, True), (45, 61, 96, True, True),
             (500, 375, 320, True, True), (100, 150, 640, False, False), (900, 700, 640, False, False)]
    out = list(fixed)
    while len(out) < n:
        k = len(out)
        h, w = int(rng.integers(2, 900)), int(rng.integers(2, 900))
        ns = int(rng.choice([96, 160, 320, 416])) if k % 3 else (int(rng.integers(2, 14)) * 32, int(rng.integers(2, 14)) * 32)
        out.append((h, w, ns, k % 4 == 0, k % 5 != 0))
    return out


@pytest.mark.parametrize("case", _shapes(), ids=lambda c: f"{c[0]}x{c[1]}-{c[2]}-auto{int(c[3])}-up{int(c[4])}")
def test_port_equals_cv2_letterbox(case):
    pytest.importorskip("cv2")
    h, w, ns, auto, scaleup = case
    rng = np.random.default_rng(h * 7919 + w)
    im = lp.random_image(rng, h, w)
    ref, ratio, pad = lp.letterbox_verbatim(im, ns, auto=auto, scaleup=scaleup)
    g = letterbox_geometry(h, w, ns, 32, auto, scaleup)
    assert g.ratio == ratio and g.pad == pad and g.out_shape == ref.shape[:2]
    got = lp.letterbox_port(im, (g.unpad_h, g.unpad_w, g.top, g.left, *g.out_shape))
    assert np.array_equal(got, np.ascontiguousarray(ref[:, :, ::-1].transpose(2, 0, 1)))


def test_port_covers_every_resize_mode():
    kinds = set()
    for h, w, ns, auto, scaleup in _shapes():
        g = letterbox_geometry(h, w, ns, 32, auto, scaleup)
        kinds.add("same" if (g.unpad_h, g.unpad_w) == (h, w) else "area" if (h, w) == (2 * g.unpad_h, 2 * g.unpad_w)
                  else "up" if g.unpad_w > w else "down")
        kinds.add("odd_pad") if (g.top + g.bottom) % 2 or (g.left + g.right) % 2 else None
    assert kinds == {"same", "area", "up", "down", "odd_pad"}


def test_geometry_matches_reference_arithmetic_on_many_sizes():
    rng = np.random.default_rng(3)
    for _ in range(3000):
        h, w = int(rng.integers(1, 4000)), int(rng.integers(1, 4000))
        ns = int(rng.choice([320, 640, 1280])) if rng.random() < 0.7 else (int(rng.integers(1, 40)) * 32, int(rng.integers(1, 40)) * 32)
        auto, scaleup = bool(rng.random() < 0.5), bool(rng.random() < 0.7)
        g = letterbox_geometry(h, w, ns, 32, auto, scaleup)
        s = (ns, ns) if isinstance(ns, int) else ns
        r = min(s[0] / h, s[1] / w)
        r = r if scaleup else min(r, 1.0)
        uw, uh = int(round(w * r)), int(round(h * r))
        dw, dh = s[1] - uw, s[0] - uh
        if auto:
            dw, dh = dw % 32, dh % 32
        assert (g.unpad_w, g.unpad_h, g.ratio) == (uw, uh, (r, r))
        assert g.pad == (dw / 2, dh / 2) and g.top + g.bottom == dh and g.left + g.right == dw


def test_geometry_rounds_half_to_even():
    # w * r = 0.5 * odd: Python's round goes to the even neighbour, as the reference's int(round(...)) does
    g = letterbox_geometry(10, 5, 1, 32, False, True)  # r = 0.1, w * r = 0.5 -> 0
    assert g.unpad_w == 0 and g.unpad_h == 1
    g = letterbox_geometry(8, 12, 10, 32, False, True)  # r = 10 / 12, h * r = 6.666.. ; pad 10 - 7 = 3 -> 1 + 2
    assert (g.top, g.bottom) == (1, 2)


def test_goldens_are_the_port():
    data = np.load(os.path.join(HERE, "golden", "letterbox_cv2.npz"))
    meta = json.loads(str(data["meta"]))
    for k, m in enumerate(meta["cases"]):
        im, want = data[f"src_{k}"], data[f"out_{k}"]
        g = letterbox_geometry(im.shape[0], im.shape[1], m["new_shape"] if isinstance(m["new_shape"], int) else tuple(m["new_shape"]),
                               32, m["auto"], m["scaleup"])
        got = lp.letterbox_port(im, (g.unpad_h, g.unpad_w, g.top, g.left, *g.out_shape))
        assert np.array_equal(got, np.ascontiguousarray(want[:, :, ::-1].transpose(2, 0, 1))), k


def test_reciprocal_constant_of_the_kernel():
    # letterbox.cu multiplies by fp32(1 / 255) given as its bit pattern
    assert np.array(np.float32(1) / np.float32(255)).view(np.uint32) == 0x3B808081
    src = open(os.path.join(os.path.dirname(HERE), "cerberusdet_b200", "csrc", "letterbox.cu")).read()
    assert "0x3b808081" in src


# ------------------------------------------------------------------------------------------ the C ABI, without a GPU
def test_letterbox_prototype_matches_header():
    from cerberusdet_b200 import _lib

    text = open(os.path.join(os.path.dirname(HERE), "include", "cerb_post.h")).read()
    m = re.search(r"(\w+)\s+cerb_letterbox\(([^)]*)\);", text)
    assert m
    fn = getattr(_lib.load(), "cerb_letterbox")
    assert fn.restype is ctypes.c_int and m.group(1) == "int"
    scalar = {"int": ctypes.c_int, "long": ctypes.c_long}
    params = [" ".join(p.split()) for p in m.group(2).split(",")]
    assert len(params) == len(fn.argtypes)
    for p, t in zip(params, fn.argtypes):
        if p.startswith("const void* const*"):
            assert t is ctypes.POINTER(ctypes.c_void_p), p
        elif p.startswith("void*"):
            assert t is ctypes.c_void_p, p
        elif "*" in p:
            assert t is ctypes.POINTER(scalar[p.split()[1].rstrip("*")]), p
        else:
            assert t is scalar[p.split()[0]], p


def test_letterbox_abi_validation_without_gpu():
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    ia = lambda *v: (ctypes.c_int * len(v))(*v)  # noqa: E731

    def call(B=2, h=(100, 80), w=(120, 60), pitch=(360, 180), uh=(50, 64), uw=(60, 48), top=(7, 0), left=(2, 8),
             out_h=64, out_w=64, dtype=_lib.CERB_F16, src=(256, 512), out=256):
        return lib.cerb_letterbox((ctypes.c_void_p * 2)(*src), ia(*h), ia(*w), (ctypes.c_long * 2)(*pitch), ia(*uh), ia(*uw),
                                  ia(*top), ia(*left), B, out_h, out_w, dtype, out, None)

    def refused(fragment, **kw):
        return call(**kw) == _lib.CERB_EINVAL and fragment in lib.cerb_last_error()

    assert refused(b"negative batch", B=-1)
    assert refused(b"output size", out_h=0) and refused(b"output size", out_w=-3)
    assert refused(b"dtype", dtype=7)
    assert refused(b"image 1 has size", h=(100, 0))
    assert refused(b"image 0 has size", w=(0, 60))
    assert refused(b"row pitch", pitch=(359, 180))
    assert refused(b"empty", uw=(0, 48))
    assert refused(b"does not fit", top=(15, 0))  # 15 + 50 > 64
    assert refused(b"does not fit", left=(2, 17))  # 17 + 48 > 64
    assert refused(b"does not fit", top=(-1, 0))
    assert refused(b"image 1 is null", src=(256, 0))
    assert refused(b"null argument", out=None)
    assert call(B=0) == 0  # nothing to do, nothing launched


def test_ops_letterbox_refuses_cpu_and_bad_input():
    import torch

    from cerberusdet_b200 import ops, preprocess

    with pytest.raises(TypeError):
        ops.letterbox([torch.zeros(10, 10, 3, dtype=torch.uint8)], [(10, 10, 0, 0)], (10, 10))
    with pytest.raises(TypeError):
        preprocess.letterbox_images([np.zeros((10, 10, 3), np.uint8)], 32, device="cpu")
    with pytest.raises(TypeError):
        preprocess.letterbox_images([np.zeros((10, 10, 4), np.uint8)], 32)
    with pytest.raises(TypeError):
        preprocess.letterbox_images([np.zeros((10, 10, 3), np.float32)], 32)
    with pytest.raises(ValueError):
        preprocess.letterbox_images([], 32)


def test_letterbox_images_refuses_auto_batches_of_different_shapes():
    from cerberusdet_b200 import preprocess

    ims = [np.zeros((480, 640, 3), np.uint8), np.zeros((640, 480, 3), np.uint8)]
    with pytest.raises(ValueError, match="differ in size"):
        preprocess.letterbox_images(ims, 640, auto=True)
