"""GPU parity of the box-regression loss kernels (``cerb_bbox_loss_fwd/_bwd`` through ``ops.bbox_loss``: BboxLoss.forward,
cerberusdet/utils/loss.py:12-44) against the port (tests/bbox_loss_port.py) run on the same GPU, in fp32 and under fp16
autocast, plus determinism, freedom from host synchronisation, CUDA-graph capture and the ``install(loss=True)`` wiring.

Bounds.  fp32: the per-anchor CIoU term bit for bit (same libdevice as ATen, one rounding per op); the per-anchor DFL
term 1e-5 relative plus a few ulps of 16 times the weight (log_softmax is a difference of terms as large as the logits,
which stay below 16 here); the two scalars 1e-5 relative (ATen's ``.sum()`` adds in another order).  Gradients: each
value is a sum of several paths (intersection, enclosing box, centre distance, aspect ratio; the two cross-entropies), so
its error scales with the paths, not with the sum: the bound is ``rtol * (|want| + S)`` with ``S`` the largest gradient of
the same anchor (boxes) or side (bins), rtol 1e-5.  Autocast: the same per-anchor and scalar bounds (the kernels keep the
reference's half roundings, the log-probabilities of the cross-entropy included); fp16 gradients: the reference rounds
every path's gradient to half and adds them in half, in an order of its own: rtol 1e-3 and one half ulp of ``S``."""
import os
import sys
import warnings

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402
from oracle.ref_import import reference_available  # noqa: E402
from test_loss_host import _host_case, stub_reference  # noqa: E402,F401

pytestmark = pytest.mark.gpu
LEVELS = [(80, 80), (40, 40), (20, 20)]


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    return o


def _grads_close(got, want, rtol, group, half):
    """``|got - want| <= rtol * (|want| + S) (+ one half ulp of S)``, S = max |want| over groups of ``group`` values.
    Returns the worst ``|got - want| / bound``."""
    g, w = got.float().cpu(), want.float().cpu()
    S = w.abs().reshape(-1, group).amax(-1, keepdim=True).expand(-1, group).reshape(w.shape)
    bound = rtol * (w.abs() + S) + 1e-30
    if half:
        bound = bound + torch.exp2(torch.floor(torch.log2(S.clamp(min=2.0**-14))) - 10)  # (2^-24 below half's normal range)
    d = (g - w).abs()
    assert torch.isfinite(g).all()
    ok = d <= bound
    assert ok.all(), f"worst excess {(d - bound).max().item():.3e} of {int((~ok).sum())} values"
    return float((d / bound).max())


def _case(ops, kind, dtype=torch.float32):
    if kind == "train":  # the training shape: 640x640, 8400 anchors
        return lp.loss_case(51, 4, LEVELS, [8, 16, 32], 20, 20, dtype=dtype, ops=ops)
    if kind == "crowded":
        return lp.loss_case(52, 2, LEVELS, [8, 16, 32], 80, 60, dtype=dtype, ops=ops)
    if kind == "one_level":  # 16 anchors, one box
        return lp.loss_case(53, 1, [(4, 4)], [8], 2, 1, dtype=dtype, ops=ops)
    c = lp.loss_case(54, 2, [(20, 20), (10, 10), (5, 5)], [8, 16, 32], 7, 9, dtype=dtype, ops=ops)
    if kind == "none":
        c["fg_mask"] = torch.zeros_like(c["fg_mask"])
        c["target_scores"] = torch.zeros_like(c["target_scores"])
        c["target_scores_sum"] = 1
    elif kind == "all":
        g = torch.Generator().manual_seed(7)
        c["fg_mask"] = torch.ones_like(c["fg_mask"])
        lab = torch.randint(0, 7, c["fg_mask"].shape, generator=g)
        ts = torch.nn.functional.one_hot(lab, 7).float() * torch.rand(*lab.shape, 1, generator=g)
        c["target_scores"] = ts.cuda()
        c["target_scores_sum"] = ts.sum().clamp(min=1).cuda()
    return c


def _run(fn, c, amp=False):
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    args = dict(c, pred_dist=pd, pred_bboxes=pb)
    with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        out = fn(**args)
    li, ld = out[0], out[1]
    gd, gb = torch.autograd.grad((li, ld), (pd, pb), (torch.tensor(0.7, device="cuda"), torch.tensor(1.3, device="cuda")),
                                 allow_unused=True)
    gd = torch.zeros_like(pd) if gd is None else gd
    gb = torch.zeros_like(pb) if gb is None else gb
    return li.detach(), ld.detach(), gd, gb, (out[2] if len(out) > 2 else None)


def _fused_terms(ops):
    def fn(**k):
        per = torch.empty(k["fg_mask"].shape + (2,), device="cuda")
        li, ld = ops.bbox_loss(**k, per_anchor=per)
        return li, ld, per

    return fn


def _scalars_close(a, b, rtol):
    a, b = float(a), float(b)
    assert abs(a - b) <= rtol * abs(b) + 1e-30, (a, b)


@pytest.mark.parametrize("kind", ["train", "crowded", "one_level", "none", "all"])
def test_bbox_loss_fp32_matches_port_on_the_same_gpu(ops, kind):
    c = _case(ops, kind)
    li, ld, gd, gb, per = _run(_fused_terms(ops), c)
    wi, wd, wgd, wgb, wper = _run(lambda **k: lp.bbox_loss_port(**k, terms=True), c)
    assert li.dtype == torch.float32 and li.dim() == 0 and ld.dim() == 0
    assert torch.equal(per[..., 0], wper[..., 0]), "per-anchor CIoU term"
    w = c["target_scores"].sum(-1)
    assert ((per[..., 1] - wper[..., 1]).abs() <= 1e-5 * wper[..., 1].abs() + 4 * 2.0**-19 * w).all(), "per-anchor DFL term"
    _scalars_close(li, wi, 1e-5)
    _scalars_close(ld, wd, 1e-5)
    _grads_close(gb, wgb, 1e-5, 4, False)
    _grads_close(gd, wgd, 1e-5, 16, False)
    if kind == "none":
        assert float(li) == 0.0 and float(ld) == 0.0 and not gd.any() and not gb.any()
    else:
        assert c["fg_mask"].any()
    assert not gd[~c["fg_mask"]].any() and not gb[~c["fg_mask"]].any()


@pytest.mark.parametrize("kind", ["train", "crowded", "one_level", "all"])
def test_bbox_loss_autocast_fp16_matches_port_on_the_same_gpu(ops, kind):
    c = _case(ops, kind, dtype=torch.float16)
    li, ld, gd, gb, per = _run(_fused_terms(ops), c, amp=True)
    wi, wd, wgd, wgb, wper = _run(lambda **k: lp.bbox_loss_port(**k, terms=True), c, amp=True)
    assert torch.equal(per[..., 0], wper[..., 0]), "per-anchor CIoU term"
    w = c["target_scores"].sum(-1)
    assert ((per[..., 1] - wper[..., 1]).abs() <= 1e-5 * wper[..., 1].abs() + 4 * 2.0**-19 * w).all(), "per-anchor DFL term"
    assert gd.dtype == torch.float16 and gb.dtype == torch.float16 and wgd.dtype == torch.float16 and wgb.dtype == torch.float16
    _scalars_close(li, wi, 1e-5)
    _scalars_close(ld, wd, 1e-5)
    _grads_close(gb, wgb, 1e-3, 4, True)
    _grads_close(gd, wgd, 1e-3, 16, True)


@pytest.mark.parametrize("seed", [3, 4])
def test_bbox_loss_crafted_ties_match_autograd(ops, seed):
    """Integer boxes: predicted and target corners coincide (min / max ties), intersections of width exactly 0 (clamp),
    DFL targets on bin edges, at 0 and clamped to 14.99 -- the gradient split must be autograd's."""
    pd, pb, ap, tb, ts, fg = (t.cuda() for t in _host_case(seed, B=4, A=256, ties=True))
    c = dict(pred_dist=pd.float(), pred_bboxes=pb.float(), anchor_points=ap.float(), target_bboxes=tb.float(),
             target_scores=ts.float(), target_scores_sum=ts.float().sum().clamp(min=1), fg_mask=fg)
    assert ((pb == tb) & fg[..., None]).any()
    li, ld, gd, gb, per = _run(_fused_terms(ops), c)
    wi, wd, wgd, wgb, wper = _run(lambda **k: lp.bbox_loss_port(**k, terms=True), c)
    assert torch.equal(per[..., 0], wper[..., 0])
    _scalars_close(li, wi, 1e-5)
    _scalars_close(ld, wd, 1e-5)
    _grads_close(gb, wgb, 1e-5, 4, False)
    _grads_close(gd, wgd, 1e-5, 16, False)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_bbox_loss_is_deterministic_and_sync_free(ops, dtype):
    c = _case(ops, "train", dtype)
    a = _run(ops.bbox_loss, c, amp=dtype == torch.float16)
    b = _run(ops.bbox_loss, c, amp=dtype == torch.float16)
    for x, y in zip(a[:4], b[:4]):
        assert torch.equal(x, y)
    torch.cuda.synchronize()
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    go = torch.ones((), device="cuda")
    prev = torch.cuda.get_sync_debug_mode()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.autocast("cuda", dtype=torch.float16, enabled=dtype == torch.float16):
            li, ld = ops.bbox_loss(**dict(c, pred_dist=pd, pred_bboxes=pb))
        torch.autograd.backward((li, ld), (go, go))
    finally:
        torch.cuda.set_sync_debug_mode(prev)
    torch.cuda.synchronize()
    assert pd.grad is not None and pb.grad is not None


def test_bbox_loss_cuda_graph_replay_equals_eager(ops):
    c = _case(ops, "train")
    static = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in c.items()}
    pd = static["pred_dist"].requires_grad_(True)
    pb = static["pred_bboxes"].requires_grad_(True)
    go = (torch.tensor(0.7, device="cuda"), torch.tensor(1.3, device="cuda"))  # as _run
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up on the capture stream
        for _ in range(2):
            li, ld = ops.bbox_loss(**static)
            torch.autograd.grad((li, ld), (pd, pb), go)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        li, ld = ops.bbox_loss(**static)
        gd, gb = torch.autograd.grad((li, ld), (pd, pb), go)
    fresh = lp.loss_case(61, 4, LEVELS, [8, 16, 32], 20, 12, ops=ops)
    for k, v in fresh.items():
        static[k].detach().copy_(v)
    graph.replay()
    graph.replay()  # the workspace counter must be left ready by every launch
    torch.cuda.synchronize()
    e = _run(ops.bbox_loss, fresh)
    assert torch.equal(li, e[0]) and torch.equal(ld, e[1]) and torch.equal(gd, e[2]) and torch.equal(gb, e[3])


def test_install_loss_takes_the_kernel_path_on_cuda(ops, stub_reference):
    from cerberusdet_b200 import patch

    BboxLoss = stub_reference["cerberusdet.utils.loss"].BboxLoss
    patch.install(loss=True)
    calls = []
    real = ops.bbox_loss
    ops.bbox_loss = lambda *a, **k: (calls.append(1), real(*a, **k))[1]
    try:
        c = _case(ops, "train")
        m = BboxLoss(15, use_dfl=True)
        got = m(*[c[k] for k in ("pred_dist", "pred_bboxes", "anchor_points", "target_bboxes", "target_scores",
                                 "target_scores_sum", "fg_mask")])
        assert len(calls) == 1
        want = lp.bbox_loss_port(**c)
        _scalars_close(got[0], want[0], 1e-5)
        _scalars_close(got[1], want[1], 1e-5)
        m16 = BboxLoss(15, use_dfl=True)
        h = {k: (v.half() if torch.is_tensor(v) and v.dtype == torch.float32 and k in ("pred_dist", "pred_bboxes") else v)
             for k, v in c.items()}
        m16(*[h[k] for k in ("pred_dist", "pred_bboxes", "anchor_points", "target_bboxes", "target_scores",
                             "target_scores_sum", "fg_mask")])  # mixed dtypes outside autocast: the reference's code
        assert len(calls) == 1
        BboxLoss(15, use_dfl=False)(*[c[k] for k in ("pred_dist", "pred_bboxes", "anchor_points", "target_bboxes",
                                                      "target_scores", "target_scores_sum", "fg_mask")])
        assert len(calls) == 1
    finally:
        ops.bbox_loss = real


@pytest.mark.skipif(not reference_available(), reason="needs the reference tree (/root/reference or oracle/_ref)")
@pytest.mark.parametrize("amp", [False, True])
def test_bbox_loss_equals_the_reference_bboxloss_on_this_gpu(ops, amp):
    from oracle.ref_import import load_reference

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        load_reference()
    from cerberusdet.utils.loss import BboxLoss

    from cerberusdet_b200 import patch

    patch.uninstall()
    c = _case(ops, "train", torch.float16 if amp else torch.float32)
    ref = BboxLoss(15, use_dfl=True).cuda()
    wi, wd, wgd, wgb, _ = _run(lambda **k: ref(*k.values()), c, amp=amp)
    try:
        info = patch.install(loss=True)
        assert "cerberusdet.utils.loss.BboxLoss.forward" in info["patched"]
        calls = []
        real = ops.bbox_loss
        ops.bbox_loss = lambda *a, **k: (calls.append(1), real(*a, **k))[1]
        try:
            li, ld, gd, gb, _ = _run(lambda **k: ref(*k.values()), c, amp=amp)
        finally:
            ops.bbox_loss = real
        assert calls, "the kernel path was not taken"
        _scalars_close(li, wi, 1e-5)
        _scalars_close(ld, wd, 1e-5)
        _grads_close(gb, wgb, 1e-3 if amp else 1e-5, 4, amp)
        _grads_close(gd, wgd, 1e-3 if amp else 1e-5, 16, amp)
        cpu = {k: (v.cpu() if torch.is_tensor(v) else v) for k, v in _case(ops, "one_level").items()}
        want = BboxLoss.forward._cerb_reference(ref, *cpu.values())
        assert all(torch.equal(a, b) for a, b in zip(ref(*cpu.values()), want))
    finally:
        patch.uninstall()
    assert not hasattr(BboxLoss.forward, "_cerb_reference")
