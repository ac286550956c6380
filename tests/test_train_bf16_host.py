"""bf16 autocast training through the assigner and the box-regression loss, host side (no GPU).

The rounding rules the bf16 kernels follow, each shown to be observable -- the alternative gives other bits on the
CPU -- so that tests/test_gpu_train_bf16.py, which pins them under ``torch.autocast("cuda", dtype=torch.bfloat16)``
against the ports, is testing a choice:

1. Assigner: CUDA autocast's fp32 op list has ``pow``.  ``bbox_scores.pow(alpha)`` (utils/tal.py:129) on bf16 scores
   runs in fp32 on the widened scores and is not rounded, so bf16 scores give what the same values in fp32 give.  The
   fp16 kernel rounds the power to half -- the reference outside autocast; under fp16 autocast the reference does
   not (DESIGN §7).
2. BboxLoss: w1, h1 (twice), w1 * h1, w1 / h1 and atan(w1 / h1) are bf16; everything that meets a target coordinate is
   fp32; the cross-entropy's log_softmax keeps bf16 (fp32 inside, rounded once) and nll_loss reads it in fp32 -- the
   fp16 rules with bf16 rounding.  An fp32 op rounded once to bf16 is the bf16 op (DESIGN §2, fact 3), which is what
   ``rh<__nv_bfloat16>`` of bbox_loss.cu computes.

Also: the dtype gates of the C ABI for the two calls."""
import ctypes
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402
from test_train_bounds_host import flat_case  # noqa: E402

from cerberusdet_b200 import _lib  # noqa: E402

BF16 = torch.bfloat16


# ------------------------------------------------------------------ rule 1: the assigner's power is not rounded
@pytest.mark.parametrize("alpha", [0.5, 1.0, 0.7])
def test_widened_power_differs_from_the_rounded_power(alpha):
    s = torch.rand(1 << 16, generator=torch.Generator().manual_seed(3)).clamp(min=1e-3).to(BF16)
    wide = s.float().pow(alpha)  # autocast: fp32 pow of the widened score
    rounded = s.pow(alpha).float()  # bf16 tensor op: the power rounded to bf16
    if alpha == 1.0:
        assert torch.equal(wide, rounded)  # x^1 is exact: the rule cannot show here
    else:
        assert int((wide != rounded).sum()) > len(s) // 2
        # and the assigner's metric, score^alpha * overlap^6, keeps the difference
        ov = torch.rand(len(s), generator=torch.Generator().manual_seed(4))
        assert not torch.equal(wide * ov.pow(6.0), rounded * ov.pow(6.0))


def test_bf16_scores_are_exact_in_fp32():
    """The kernels' bf16 path widens the score and then runs the fp32 path: widening is exact, so the fp32 kernel on
    ``scores.float()`` is the same computation."""
    s = torch.rand(1 << 16, generator=torch.Generator().manual_seed(5)).to(BF16)
    assert torch.equal(s.float().to(BF16), s)
    assert torch.equal(s.float().double().float(), s.float())


# ------------------------------------------------------------------ rule 2: the box loss rounds where fp16 does, in bf16
def test_bbox_loss_rounding_points_and_their_effect():
    """On the CPU without autocast the promotion of mixed operands is the same as on the GPU under autocast for every op
    of the CIoU term (none of them is on an autocast list): bf16 where both operands are bf16, fp32 once a target
    coordinate takes part.  Rounding there matters: the fp32 CIoU of the same predictions gives other bits."""
    c = flat_case(7, 2, 512, fg=1.0)
    pb = c["pred_bboxes"].to(BF16)
    t = c["target_bboxes"]
    b1_x1, b1_y1, b1_x2, b1_y2 = pb.chunk(4, -1)
    w1, h1 = b1_x2 - b1_x1, b1_y2 - b1_y1 + 1e-7
    assert w1.dtype == h1.dtype == (w1 * h1).dtype == (w1 / h1).dtype == torch.atan(w1 / h1).dtype == BF16
    assert (w1 * h1 + (t[..., 2:3] - t[..., 0:1])).dtype == torch.float32
    assert (b1_x2.minimum(t[..., 2:3]) - b1_x1.maximum(t[..., 0:1])).dtype == torch.float32
    # an fp32 op on bf16 operands rounded once to bf16 is the bf16 op (what rh<__nv_bfloat16> computes)
    assert torch.equal(w1, (b1_x2.float() - b1_x1.float()).to(BF16))
    assert torch.equal(h1, ((b1_y2.float() - b1_y1.float()).to(BF16).float() + 1e-7).to(BF16))
    assert torch.equal(w1 / h1, (w1.float() / h1.float()).to(BF16))
    assert torch.equal(torch.atan(w1 / h1), torch.atan((w1 / h1).float()).to(BF16))
    iou_bf = lp.bbox_iou_ciou(pb, t)
    iou_32 = lp.bbox_iou_ciou(pb.float(), t)
    assert iou_bf.dtype == torch.float32 and not torch.equal(iou_bf, iou_32)


def test_cross_entropy_log_probabilities_are_rounded_to_bf16():
    """The rule autocast gives ``F.cross_entropy`` on bf16 logits (cross_entropy_loss calls log_softmax with the input's
    dtype; nll_loss is on the fp32 list): the log-probabilities are rounded to bf16 before the fp32 nll.  On the CPU
    log_softmax of bf16 logits is a bf16 tensor too, and its values are not the fp32 log-probabilities.  (The CUDA kernel
    computes in fp32 and rounds once; the CPU one does not, so the bits are pinned on the GPU only.)"""
    x = (torch.randn(4096, 16, generator=torch.Generator().manual_seed(8)) * 3).to(BF16)
    ls = torch.log_softmax(x, 1)
    assert ls.dtype == BF16
    assert int((ls.float() != torch.log_softmax(x.float(), 1)).sum()) > ls.numel() // 2


# ------------------------------------------------------------------ dtype gates
def test_abi_takes_bf16_for_the_assigner_and_the_box_loss():
    lib = _lib.load()
    fake, odd = ctypes.c_void_p(256), ctypes.c_void_p(256 + 2)
    # cerb_tal_assign: bf16 passes the dtype check and stops at the (too small) workspace; an unknown code does not
    for code, want, msg in ((_lib.CERB_BF16, _lib.CERB_ENOSPC, b"workspace"), (5, _lib.CERB_EINVAL, b"dtype")):
        rc = lib.cerb_tal_assign(fake, fake, fake, fake, fake, fake, 2, 100, 5, 3, 10, 0.5, 6.0, 1e-9, code, fake, fake, fake,
                                 fake, fake, fake, 16, None)
        assert rc == want and msg in lib.cerb_last_error(), code

    def fwd(dtype, pb=fake):
        return lib.cerb_bbox_loss_fwd(fake, pb, fake, fake, fake, fake, None, 1.0, 2, 100, 5, 16, dtype, fake, fake, None, fake,
                                      8, None)

    assert fwd(_lib.CERB_BF16) == _lib.CERB_ENOSPC and b"workspace" in lib.cerb_last_error()
    # bf16 box rows are 8 bytes: 2-byte alignment is not enough, as for fp16
    assert fwd(_lib.CERB_BF16, pb=odd) == _lib.CERB_EINVAL and b"misaligned" in lib.cerb_last_error()
    assert fwd(5) == _lib.CERB_EINVAL and b"dtype" in lib.cerb_last_error()
    # the backward: an empty batch is accepted; a grad_pred_bboxes on a 4-byte boundary is not (8-byte rows)
    assert lib.cerb_bbox_loss_bwd(None, None, None, None, None, None, None, 1.0, 0, 8400, 5, 16, _lib.CERB_BF16, None, None,
                                  None, None, None) == 0
    rc = lib.cerb_bbox_loss_bwd(fake, fake, fake, fake, fake, fake, None, 1.0, 2, 100, 5, 16, _lib.CERB_BF16, fake, fake, fake,
                                ctypes.c_void_p(256 + 4), None)
    assert rc == _lib.CERB_EINVAL and b"misaligned" in lib.cerb_last_error()

