"""CPU tests of the box-regression loss term (``ops.bbox_loss``, ``cerb_bbox_loss_fwd/_bwd``, ``install(loss=True)``):
argument validation of the C ABI, the port's autograd gradient against the closed-form gradient the kernels implement, and
the patch's wiring on stand-in reference modules.  No kernel is launched here."""
import ctypes
import math
import os
import sys
import types

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402


def test_bbox_loss_abi_validation_without_gpu():
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    fake, odd = ctypes.c_void_p(256), ctypes.c_void_p(256 + 16)

    def fwd(pd=fake, B=2, A=100, C=5, reg_max=16, dtype=_lib.CERB_F32, ws=fake, ws_bytes=1 << 20):
        return lib.cerb_bbox_loss_fwd(pd, fake, fake, fake, fake, fake, None, 1.0, B, A, C, reg_max, dtype, fake, fake, None, ws,
                                      ws_bytes, None)

    assert fwd(reg_max=8) == _lib.CERB_EINVAL and b"reg_max=8" in lib.cerb_last_error()
    assert fwd(dtype=5) == _lib.CERB_EINVAL and b"dtype" in lib.cerb_last_error()
    assert fwd(pd=odd) == _lib.CERB_EINVAL and b"misaligned" in lib.cerb_last_error()  # 16-byte, not 32-byte aligned rows
    assert fwd(B=1 << 16, A=1 << 16) == _lib.CERB_EINVAL and b"overflow" in lib.cerb_last_error()
    assert fwd(C=0) == _lib.CERB_EINVAL
    assert fwd(ws_bytes=8) == _lib.CERB_ENOSPC and b"workspace" in lib.cerb_last_error()
    # one (loss_iou, loss_dfl) partial pair per CTA of the forward grid (capped at 8 per SM of a B200) after a 16-byte counter
    assert lib.cerb_bbox_loss_workspace_bytes(2, 100) == 16 + 4 * 8
    assert lib.cerb_bbox_loss_workspace_bytes(64, 8400) == 16 + 148 * 8 * 8
    rc = lib.cerb_bbox_loss_bwd(fake, fake, fake, fake, fake, fake, None, 1.0, 2, 100, 5, 16, _lib.CERB_F16, fake, fake, odd,
                                fake, None)
    assert rc == _lib.CERB_EINVAL and b"grad_pred_dist" in lib.cerb_last_error()
    rc = lib.cerb_bbox_loss_bwd(fake, fake, fake, fake, fake, fake, None, 1.0, 2, 100, 5, 16, _lib.CERB_F32, None, fake, fake,
                                fake, None)
    assert rc == _lib.CERB_EINVAL and b"null" in lib.cerb_last_error()
    # an empty batch has nothing to differentiate
    assert lib.cerb_bbox_loss_bwd(None, None, None, None, None, None, None, 1.0, 0, 8400, 5, 16, _lib.CERB_F32, None, None, None,
                                  None, None) == 0


def test_ops_bbox_loss_refuses_cpu_tensors():
    from cerberusdet_b200 import ops

    z = torch.zeros
    with pytest.raises(TypeError):
        ops.bbox_loss(z(1, 4, 64), z(1, 4, 4), z(4, 2), z(1, 4, 4), z(1, 4, 3), 1, z(1, 4, dtype=torch.bool))


# ----------------------------------------------------------------------------- closed-form gradient (what the kernels compute)
def _split_min(a, b, g):  # autograd's share of minimum(a, b) on a: all, half on an exact tie, none
    return torch.where(a < b, g, torch.where(a == b, g / 2, torch.zeros_like(g)))


def _split_max(a, b, g):
    return torch.where(a > b, g, torch.where(a == b, g / 2, torch.zeros_like(g)))


def ciou_grad(p, t, G, eps=1e-7):
    """d(CIoU)/d(box1) * G with alpha a constant, clamp(0) passing the gradient at 0 and min/max ties split in half."""
    px1, py1, px2, py2 = p.unbind(-1)
    tx1, ty1, tx2, ty2 = t.unbind(-1)
    w1, h1 = px2 - px1, py2 - py1 + eps
    w2, h2 = tx2 - tx1, ty2 - ty1 + eps
    ix = torch.minimum(px2, tx2) - torch.maximum(px1, tx1)
    iy = torch.minimum(py2, ty2) - torch.maximum(py1, ty1)
    inter = ix.clamp(0) * iy.clamp(0)
    uni = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / uni
    cw = torch.maximum(px2, tx2) - torch.minimum(px1, tx1)
    ch = torch.maximum(py2, ty2) - torch.minimum(py1, ty1)
    c2 = cw**2 + ch**2 + eps
    dx, dy = tx1 + tx2 - px1 - px2, ty1 + ty2 - py1 - py2
    rho2 = (dx**2 + dy**2) / 4
    at = torch.atan(w2 / h2) - torch.atan(w1 / h1)
    K = 4 / math.pi**2
    v = K * at**2
    alpha = v / (v - iou + (1 + eps))
    g_union = -G * iou / uni
    g_inter = G / uni - g_union
    g_ix = torch.where(ix >= 0, g_inter * iy.clamp(0), torch.zeros_like(G))
    g_iy = torch.where(iy >= 0, g_inter * ix.clamp(0), torch.zeros_like(G))
    gS = -G
    g_c2 = -gS * rho2 / c2**2
    g_dx, g_dy = gS / c2 / 4 * 2 * dx, gS / c2 / 4 * 2 * dy
    g_cw, g_ch = g_c2 * 2 * cw, g_c2 * 2 * ch
    g_r1 = -(gS * alpha * K * 2 * at) / (1 + (w1 / h1) ** 2)
    g_w1 = g_union * h1 + g_r1 / h1
    g_h1 = g_union * w1 - g_r1 * w1 / h1**2
    return torch.stack((
        -g_w1 + _split_max(px1, tx1, -g_ix) + _split_min(px1, tx1, -g_cw) - g_dx,
        -g_h1 + _split_max(py1, ty1, -g_iy) + _split_min(py1, ty1, -g_ch) - g_dy,
        g_w1 + _split_min(px2, tx2, g_ix) + _split_max(px2, tx2, g_cw) - g_dx,
        g_h1 + _split_min(py2, ty2, g_iy) + _split_max(py2, ty2, g_ch) - g_dy), -1)


def bbox_loss_grad(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, tss, fg_mask, g_iou, g_dfl):
    w = target_scores.sum(-1)
    G = -(g_iou / tss) * w
    gb = torch.where(fg_mask[..., None], ciou_grad(pred_bboxes, target_bboxes, G), torch.zeros_like(pred_bboxes))
    target = lp.bbox2dist(anchor_points, target_bboxes, 15)  # [B, A, 4]
    tl = target.long()
    wl = (tl + 1) - target
    wr = 1 - wl
    p = pred_dist.view(*pred_dist.shape[:2], 4, 16).softmax(-1)
    gq = ((g_dfl / tss) * w / 4)[..., None]
    gl, gr = (gq * wl)[..., None], (gq * wr)[..., None]
    oh_l = torch.nn.functional.one_hot(tl, 16).to(p)
    oh_r = torch.nn.functional.one_hot(tl + 1, 16).to(p)
    gd = gl * (p - oh_l) + gr * (p - oh_r)
    gd = torch.where(fg_mask[..., None, None], gd, torch.zeros_like(gd)).view_as(pred_dist)
    return gd, gb


def _host_case(seed, B=3, A=40, C=6, ties=False):
    g = torch.Generator().manual_seed(seed)
    f64 = torch.float64
    ap = torch.rand(A, 2, generator=g, dtype=f64) * 20 + 2
    if ties:  # integer corners: predicted and target corners coincide, targets on bin edges, on 0 and past 14.99
        ap = ap.round() + 0.5
        lt = torch.randint(0, 17, (B, A, 4), generator=g).to(f64)
        tb = torch.cat((ap - lt[..., :2], ap + lt[..., 2:]), -1)
        pb = tb + torch.randint(-1, 2, (B, A, 4), generator=g).to(f64)
        pb = torch.cat((torch.minimum(pb[..., :2], ap), torch.maximum(pb[..., 2:], ap)), -1)
    else:
        lt = torch.rand(B, A, 4, generator=g, dtype=f64) * 14
        tb = torch.cat((ap - lt[..., :2], ap + lt[..., 2:]), -1)
        d = (lt + torch.randn(B, A, 4, generator=g, dtype=f64)).clamp(0, 15)
        pb = torch.cat((ap - d[..., :2], ap + d[..., 2:]), -1)
    fg = torch.rand(B, A, generator=g) < 0.4
    lab = torch.randint(0, C, (B, A), generator=g)
    ts = torch.nn.functional.one_hot(lab, C).to(f64) * torch.rand(B, A, 1, generator=g, dtype=f64) * fg[..., None]
    pd = torch.randn(B, A, 64, generator=g, dtype=f64) * 3
    return pd, pb, ap, tb, ts, fg


@pytest.mark.parametrize("seed,ties", [(1, False), (2, False), (3, True), (4, True)])
def test_port_autograd_gradient_equals_closed_form(seed, ties):
    """The gradient the kernels implement is the reference's autograd gradient (fp64, alpha detached, autograd's tie
    rules); crafted integer boxes put min / max ties, clamp(0) at exactly 0 and DFL targets on bin edges and past 14.99."""
    pd, pb, ap, tb, ts, fg = _host_case(seed, ties=ties)
    tss = ts.sum().clamp(min=1)
    pd.requires_grad_(True)
    pb.requires_grad_(True)
    li, ld = lp.bbox_loss_port(pd, pb, ap, tb, ts, tss, fg)
    g_iou, g_dfl = torch.tensor(0.7, dtype=torch.float64), torch.tensor(1.3, dtype=torch.float64)
    want_d, want_b = torch.autograd.grad((li, ld), (pd, pb), (g_iou, g_dfl))
    got_d, got_b = bbox_loss_grad(pd.detach(), pb.detach(), ap, tb, ts, tss, fg, g_iou, g_dfl)
    assert torch.allclose(got_d, want_d, rtol=1e-10, atol=1e-13)
    assert torch.allclose(got_b, want_b, rtol=1e-10, atol=1e-13)
    if ties:
        eq = (pb.detach() == tb) & fg[..., None]
        assert eq.any(), "the crafted case should contain exact corner ties"


# ----------------------------------------------------------------------------- the patch, on stand-in reference modules
class _RefBboxLoss(torch.nn.Module):
    """Stand-in for the reference's BboxLoss: its forward is the port."""

    def __init__(self, reg_max, use_dfl=False):
        super().__init__()
        self.reg_max, self.use_dfl = reg_max, use_dfl

    def forward(self, pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask):
        if not self.use_dfl:
            return lp.bbox_loss_port(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum,
                                     fg_mask, reg_max=self.reg_max)[0], torch.tensor(0.0)
        return lp.bbox_loss_port(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask,
                                 reg_max=self.reg_max)


@pytest.fixture()
def stub_reference(monkeypatch):
    """The modules ``patch.install(loss=True)`` touches, as stand-ins (the reference tree is not needed)."""
    mods = {}
    for name in ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general",
                 "cerberusdet.utils.loss"):
        mods[name] = types.ModuleType(name)
        monkeypatch.setitem(sys.modules, name, mods[name])
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = lambda *a, **k: None
    mods["cerberusdet.utils.loss"].BboxLoss = type("BboxLoss", (_RefBboxLoss,), {})
    from cerberusdet_b200 import patch

    patch.uninstall()
    yield mods
    patch.uninstall()
    if hasattr(mods["cerberusdet.models.yolo"].Detect, "_cerb_reference_forward"):
        del mods["cerberusdet.models.yolo"].Detect._cerb_reference_forward


def test_install_loss_rebinds_bboxloss_and_keeps_cpu_on_the_reference(stub_reference):
    from cerberusdet_b200 import patch

    BboxLoss = stub_reference["cerberusdet.utils.loss"].BboxLoss
    original = BboxLoss.forward
    pd, pb, ap, tb, ts, fg = (t.float() if t.is_floating_point() else t for t in _host_case(5))
    want = lp.bbox_loss_port(pd, pb, ap, tb, ts, 1, fg)
    info = patch.install(loss=True)
    assert "cerberusdet.utils.loss.BboxLoss.forward" in info["patched"]
    assert BboxLoss.forward is not original and BboxLoss.forward._cerb_reference is original
    assert patch.install(loss=True) == {"already": ["installed"]}  # idempotent
    got = BboxLoss(15, use_dfl=True)(pd, pb, ap, tb, ts, 1, fg)  # CPU tensors: the reference's code, bit for bit
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    got = BboxLoss(15, use_dfl=False)(pd, pb, ap, tb, ts, 1, fg)
    assert torch.equal(got[0], want[0])
    patch.uninstall()
    assert BboxLoss.forward is original
    # composes with the other switches: install(train=...) rebinds other names only, and the loss switch still applies
    info = patch.install()
    assert "cerberusdet.utils.loss.BboxLoss.forward" not in info["patched"]
    info = patch.install(loss=True)
    assert info["patched"] == ["cerberusdet.utils.loss.BboxLoss.forward"]
