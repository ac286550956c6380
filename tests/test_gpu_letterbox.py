"""GPU tests of the letterbox preprocessing (``csrc/letterbox.cu``, ``ops.letterbox``, ``preprocess.letterbox_images``):
the kernel against the numpy port of cv2's arithmetic and against the cv2 goldens, bit for bit, with the normalisation
that torch computes for the reference's own ``/ 255`` on the same GPU."""
import json
import os

import numpy as np
import pytest
import torch

import letterbox_port as lp
from test_letterbox_host import _shapes

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _expected(port_chw: np.ndarray, dtype) -> torch.Tensor:
    """The reference's tensor for a letterboxed uint8 image: upload, ``.half()`` / ``.float()``, ``/ 255`` on the GPU."""
    x = torch.from_numpy(np.ascontiguousarray(port_chw)).cuda()
    return (x.half() if dtype == torch.float16 else x.float()) / 255.0


def _port_batch(images, new_shape, auto=False, scaleup=True):
    from cerberusdet_b200.preprocess import letterbox_geometry

    out = []
    for im in images:
        g = letterbox_geometry(im.shape[0], im.shape[1], new_shape, 32, auto, scaleup)
        out.append(lp.letterbox_port(im, (g.unpad_h, g.unpad_w, g.top, g.left, *g.out_shape)))
    return np.stack(out)


@pytest.mark.parametrize("half", [True, False])
def test_normalisation_equals_torch_division_for_all_256_values(half):
    from cerberusdet_b200 import ops

    dt = torch.float16 if half else torch.float32
    v = torch.arange(256, dtype=torch.uint8).reshape(16, 16, 1).expand(16, 16, 3).contiguous().cuda()
    got = ops.letterbox([v], [(16, 16, 0, 0)], (16, 16), dt)[0, 0].reshape(-1)  # same size: no resize, R = the value
    x = torch.arange(256, dtype=torch.uint8).cuda()
    x = x.half() if half else x.float()
    for want in (x / 255.0, x / 255):
        assert torch.equal(got.view(torch.int16 if half else torch.int32), want.view(torch.int16 if half else torch.int32))
    y = x.clone()
    y /= 255.0
    assert torch.equal(got, y)


@pytest.mark.parametrize("half", [True, False])
def test_kernel_equals_port_on_every_case(half):
    from cerberusdet_b200.preprocess import letterbox_images

    dt = torch.float16 if half else torch.float32
    for h, w, ns, auto, scaleup in _shapes():
        im = lp.random_image(np.random.default_rng(h * 7919 + w), h, w)
        got, shapes = letterbox_images([im], ns, auto=auto, scaleup=scaleup, half=half)
        want = _expected(_port_batch([im], ns, auto, scaleup), dt)
        assert shapes == [(h, w)] and got.dtype == dt
        assert torch.equal(got, want), (h, w, ns, auto, scaleup, (got != want).float().mean().item())


@pytest.mark.parametrize("half", [True, False])
def test_kernel_equals_port_mixed_batch_of_64(half):
    from cerberusdet_b200.preprocess import letterbox_images

    rng = np.random.default_rng(7)
    sizes = [(1080, 1920), (720, 1280), (1280, 1280), (500, 333), (640, 640), (1, 90), (90, 1)]
    sizes += [(int(rng.integers(2, 1300)), int(rng.integers(2, 1300))) for _ in range(64 - len(sizes))]
    ims = [lp.random_image(rng, h, w) for h, w in sizes]
    dt = torch.float16 if half else torch.float32
    got, shapes = letterbox_images(ims, 640, half=half)
    assert shapes == sizes and tuple(got.shape) == (64, 3, 640, 640)
    want = _expected(_port_batch(ims, 640), dt)
    assert torch.equal(got, want)
    # device-resident input, used in place: the same bits; and strided rows (a crop of a wider frame)
    dev = [torch.from_numpy(im).cuda() for im in ims]
    assert torch.equal(letterbox_images(dev, 640, half=half)[0], got)
    wide = torch.from_numpy(np.concatenate([ims[0], ims[0][:, :100]], axis=1)).cuda()[:, :1920]
    assert wide.stride(0) == 3 * 2020
    assert torch.equal(letterbox_images([wide], 640, half=half)[0], got[:1])
    # two runs, identical bits
    assert torch.equal(letterbox_images(ims, 640, half=half)[0], got)


def test_kernel_equals_cv2_goldens():
    from cerberusdet_b200.preprocess import letterbox_images

    data = np.load(os.path.join(HERE, "golden", "letterbox_cv2.npz"))
    for k, m in enumerate(json.loads(str(data["meta"]))["cases"]):
        ns = m["new_shape"] if isinstance(m["new_shape"], int) else tuple(m["new_shape"])
        for half in (True, False):
            got, _ = letterbox_images([data[f"src_{k}"]], ns, auto=m["auto"], scaleup=m["scaleup"], half=half)
            want = _expected(data[f"out_{k}"][:, :, ::-1].transpose(2, 0, 1)[None], torch.float16 if half else torch.float32)
            assert torch.equal(got, want), (k, m)


def test_more_images_than_one_launch_takes():
    from cerberusdet_b200.preprocess import letterbox_images

    rng = np.random.default_rng(9)
    ims = [lp.random_image(rng, int(rng.integers(10, 90)), int(rng.integers(10, 90))) for _ in range(300)]
    got, _ = letterbox_images(ims, 64, half=False)
    assert torch.equal(got, _expected(_port_batch(ims, 64), torch.float32))


def test_cuda_graph_replays_on_fresh_inputs():
    from cerberusdet_b200 import ops
    from cerberusdet_b200.preprocess import letterbox_geometry

    rng = np.random.default_rng(11)
    sizes = [(480, 640), (300, 500), (1080, 1920)]
    geoms = [letterbox_geometry(h, w, 320) for h, w in sizes]
    geo = [(g.unpad_h, g.unpad_w, g.top, g.left) for g in geoms]
    static = [torch.from_numpy(lp.random_image(rng, h, w)).cuda() for h, w in sizes]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.letterbox(static, geo, (320, 320))  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = ops.letterbox(static, geo, (320, 320))
    for _ in range(2):
        fresh = [lp.random_image(rng, h, w) for h, w in sizes]
        for dst, im in zip(static, fresh):
            dst.copy_(torch.from_numpy(im))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, _expected(_port_batch(fresh, 320), torch.float16))
        assert torch.equal(out, ops.letterbox(static, geo, (320, 320)))


def test_opcheck():
    from cerberusdet_b200 import ops

    rng = np.random.default_rng(5)
    ims = [torch.from_numpy(lp.random_image(rng, h, w)).cuda() for h, w in ((40, 60), (64, 32))]
    for dt in (torch.float16, torch.float32):
        torch.library.opcheck(ops.letterbox_op, (ims, [32, 48, 8, 0, 64, 32, 0, 8], [64, 48], dt))


def test_ops_letterbox_refuses_bad_arguments():
    from cerberusdet_b200 import ops

    im = torch.zeros(40, 60, 3, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError, match="does not fit"):
        ops.letterbox([im], [(40, 60, 10, 0)], (40, 60))
    with pytest.raises(TypeError):
        ops.letterbox([im.float()], [(40, 60, 0, 0)], (40, 60))
    with pytest.raises(TypeError):
        ops.letterbox([im], [(40, 60, 0, 0)], (40, 60), torch.bfloat16)


@pytest.mark.parametrize("half", [False, True])
def test_letterbox_images_feed_predict_like_the_host_letterbox(half):
    from test_gpu_dropin import TwoTaskModel

    from cerberusdet_b200.inference import CerberusDetInference
    from cerberusdet_b200.preprocess import letterbox_images

    torch.manual_seed(3)
    eng = CerberusDetInference(model=TwoTaskModel().cuda(), device="cuda:0", conf_thres=0.25, iou_thres=0.45, half=half, img_size=64)
    rng = np.random.default_rng(13)
    ims = [lp.random_image(rng, h, w) for h, w in ((480, 640), (360, 200), (128, 128), (1080, 1920))]
    x, shapes = letterbox_images(ims, 128, half=half)
    x_host = _expected(_port_batch(ims, 128), torch.float16 if half else torch.float32)
    got = eng.predict(x, original_shape=shapes, max_det=50)
    want = eng.predict(x_host, original_shape=[im.shape[:2] for im in ims], max_det=50)
    assert got == want and sum(len(r) for r in got) > 0
