"""bf16 on the REAL reference: ``patch.install()`` against the unmodified ``Detect`` and ``non_max_suppression``, with a
bf16 model and with an fp32 model under bf16 autocast -- the bf16 counterpart of tests/test_gpu_reference.py.  Skipped
where the reference tree (``/root/reference`` or its copy ``oracle/_ref``) is absent.

The reference's candidate sort (utils/general.py:459) is an unstable argsort and bf16 scores tie heavily, so the
reference runs with ``stable=True`` forced on ``Tensor.argsort`` (as oracle/gen_golden.py does), one image per call.
The small NMS cases run it on a CPU copy (torchvision's CPU kernel: the IoU convention the kernels follow); the 1280 x 1280
Detect case runs it on the GPU, as tests/test_gpu_reference.py does (torchvision's CUDA kernel differs only for an IoU
exactly equal to the fp32 image of the threshold, INTEGRATION.md section 6), so that its time limit is not hit.
"""
import os
import sys
import warnings

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_import import reference_available  # noqa: E402

from cerberusdet_b200.synth import STRIDES, synth_prediction  # noqa: E402
from test_gpu_bf16 import check_decode_bf16  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not reference_available(), reason="needs the reference tree (/root/reference or oracle/_ref)")]
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def ref():
    from oracle.ref_import import load_reference

    os.environ.setdefault("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD", "1")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return load_reference()


@pytest.fixture()
def patch(ref):
    from cerberusdet_b200 import patch as p

    p.uninstall()
    yield p
    p.uninstall()


def _stable_reference_nms(nms, pred, cpu=True, **kw):
    """The reference function per image (on a CPU copy by default), with its argsort forced stable (canonical tie
    order)."""
    from oracle.gen_golden import _StableArgsort

    out = []
    for i in range(pred.shape[0]):
        with _StableArgsort(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            x = pred[i:i + 1]
            out.append(nms(x.cpu() if cpu else x, **kw)[0].cpu())
    return out


@pytest.mark.parametrize("mode", ["model", "autocast"])
def test_real_detect_and_nms_patched_vs_reference_bf16(ref, patch, mode):
    """The reference's own Detect (real conv towers, cuDNN) in bf16 at a 1280 x 1280 input (P3 anchor centres round):
    after install() the same instance returns the same raw levels bit for bit, takes the decode kernel (its score summary
    is attached to y) and agrees with the reference's y within the bf16 bounds; the patched non_max_suppression on that y
    equals the unmodified reference's (stable sort) bit for bit."""
    from cerberusdet_b200 import ops

    torch.manual_seed(20)
    m = ref.yolo.Detect(nc=20, ch=(64, 128, 256))
    m.stride = torch.tensor(STRIDES)
    m.bias_init()
    for seq in m.cv3:
        torch.nn.init.normal_(seq[-1].weight, std=0.5)
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(5)
    feats = [torch.randn(2, c, 1280 // int(s), 1280 // int(s), generator=g).cuda() for c, s in zip((64, 128, 256), STRIDES)]
    if mode == "model":
        m = m.bfloat16()
        feats = [f.bfloat16() for f in feats]
    ctx = (lambda: torch.autocast("cuda", dtype=BF16)) if mode == "autocast" else (lambda: torch.autocast("cuda", enabled=False))
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    reference_nms = ref.general.non_max_suppression
    with torch.no_grad(), warnings.catch_warnings(), ctx():
        warnings.simplefilter("ignore")
        y_ref, x_ref = m([f.clone() for f in feats])
        info = patch.install()
        assert "cerberusdet.models.yolo.Detect.forward" in info["patched"]
        m.shape = None
        y, x = m([f.clone() for f in feats])
        got = ref.general.non_max_suppression(y, **kw)
    assert y.dtype == y_ref.dtype == BF16 and y.shape == y_ref.shape
    assert ops.find_summary(y) is not None, "the patched forward did not run the decode kernel"
    for a, b in zip(x, x_ref):
        assert torch.equal(a, b)
    ok, msg = check_decode_bf16(y, y_ref, [t.shape[2:] for t in x], STRIDES)
    assert ok, msg
    want = _stable_reference_nms(reference_nms, y, cpu=False, **kw)
    assert sum(r.shape[0] for r in want) > 0
    for a, b in zip(got, want):
        assert a.dtype == b.dtype == torch.float32 and torch.equal(a.cpu(), b)


@pytest.mark.parametrize("kw", [dict(conf_thres=0.25, iou_thres=0.45), dict(conf_thres=0.3, iou_thres=0.45, multi_label=True),
                                dict(conf_thres=0.001, iou_thres=0.6, multi_label=True),
                                dict(conf_thres=0.1, iou_thres=0.5, agnostic=True, max_det=50)])
def test_real_nms_patched_vs_reference_bf16(ref, patch, kw, monkeypatch):
    """A bf16 prediction through the patched name against the unmodified reference function (stable sort): the kernel
    path is taken (the batched NMS is called once) and the rows are equal bit for bit."""
    from cerberusdet_b200 import nms as nms_mod

    pred = synth_prediction(2, 7, 1500, seed=23, dtype=torch.float32, regime="clusters").to(BF16)
    want = _stable_reference_nms(ref.general.non_max_suppression, pred, **kw)
    calls = []
    real = nms_mod.nms_batched
    monkeypatch.setattr(nms_mod, "nms_batched", lambda *a, **k: (calls.append(1), real(*a, **k))[1])
    patch.install()
    got = ref.general.non_max_suppression(pred.cuda(), **kw)
    assert calls == [1], "bf16 fell off the kernel path"
    for a, b in zip(got, want):
        assert a.is_cuda and a.dtype == b.dtype == torch.float32
        assert torch.equal(a.cpu(), b), f"{kw}: {a.shape} vs {b.shape}"
