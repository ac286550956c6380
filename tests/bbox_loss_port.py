"""Restatement of the reference's box-regression loss term, one torch op per reference op: the checker of
``ops.bbox_loss`` (tests/test_gpu_loss.py, tests/test_loss_host.py, tools/microbench_loss.py).

TEST INFRASTRUCTURE ONLY; nothing under ``cerberusdet_b200/`` imports it.  CerberusDet's ``BboxLoss`` is the
ultralytics-8.0 one (cerberusdet/utils/loss.py:12-44), built by ``Loss.__init__`` as ``BboxLoss(m.reg_max - 1,
use_dfl=True)``, so ``reg_max == 15`` here and the distributions have 16 bins.  ``bbox_iou`` (utils/metrics.py:373-408)
computes CIoU's ``alpha`` under ``torch.no_grad()``; ``ciou_port`` of ``oracle/ref_port.py`` (the assigner's, forward
only) does not, so this module has its own CIoU with the reference's ``no_grad`` -- the forward values are the same.
"""
import math

import torch
import torch.nn.functional as F


def bbox_iou_ciou(box1: torch.Tensor, box2: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """``bbox_iou(box1, box2, xywh=False, CIoU=True)`` (utils/metrics.py:373-408), alpha detached as in the reference."""
    b1_x1, b1_y1, b1_x2, b1_y2 = box1.chunk(4, -1)
    b2_x1, b2_y1, b2_x2, b2_y2 = box2.chunk(4, -1)
    w1, h1 = b1_x2 - b1_x1, b1_y2 - b1_y1 + eps
    w2, h2 = b2_x2 - b2_x1, b2_y2 - b2_y1 + eps
    inter = (b1_x2.minimum(b2_x2) - b1_x1.maximum(b2_x1)).clamp(0) * (b1_y2.minimum(b2_y2) - b1_y1.maximum(b2_y1)).clamp(0)
    union = w1 * h1 + w2 * h2 - inter + eps
    iou = inter / union
    cw = b1_x2.maximum(b2_x2) - b1_x1.minimum(b2_x1)
    ch = b1_y2.maximum(b2_y2) - b1_y1.minimum(b2_y1)
    c2 = cw**2 + ch**2 + eps
    rho2 = ((b2_x1 + b2_x2 - b1_x1 - b1_x2) ** 2 + (b2_y1 + b2_y2 - b1_y1 - b1_y2) ** 2) / 4
    v = (4 / math.pi**2) * torch.pow(torch.atan(w2 / h2) - torch.atan(w1 / h1), 2)
    with torch.no_grad():
        alpha = v / (v - iou + (1 + eps))
    return iou - (rho2 / c2 + v * alpha)


def bbox2dist(anchor_points: torch.Tensor, bbox: torch.Tensor, reg_max: int) -> torch.Tensor:
    """utils/tal.py:208-211."""
    x1y1, x2y2 = bbox.chunk(2, -1)
    return torch.cat((anchor_points - x1y1, x2y2 - anchor_points), -1).clamp(0, reg_max - 0.01)


def df_loss(pred_dist: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """``BboxLoss._df_loss`` (utils/loss.py:37-44)."""
    tl = target.long()
    tr = tl + 1
    wl = tr - target
    wr = 1 - wl
    return (F.cross_entropy(pred_dist, tl.view(-1), reduction="none").view(tl.shape) * wl
            + F.cross_entropy(pred_dist, tr.view(-1), reduction="none").view(tl.shape) * wr).mean(-1, keepdim=True)


def bbox_loss_port(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask,
                   reg_max: int = 15, terms: bool = False):
    """``BboxLoss.forward`` with ``use_dfl=True`` (utils/loss.py:12-35).  Returns ``(loss_iou, loss_dfl)``; with
    ``terms=True`` also the per-anchor ``[B, A, 2]`` float32 tensor of ``(1 - iou) * weight`` and ``DFL * weight``
    (zero at background anchors), the layout of ``ops.bbox_loss(..., per_anchor=)``."""
    weight = torch.masked_select(target_scores.sum(-1), fg_mask).unsqueeze(-1)
    iou = bbox_iou_ciou(pred_bboxes[fg_mask], target_bboxes[fg_mask])
    l_iou = (1.0 - iou) * weight
    loss_iou = l_iou.sum() / target_scores_sum
    target_ltrb = bbox2dist(anchor_points, target_bboxes, reg_max)
    l_dfl = df_loss(pred_dist[fg_mask].view(-1, reg_max + 1), target_ltrb[fg_mask]) * weight
    loss_dfl = l_dfl.sum() / target_scores_sum
    if not terms:
        return loss_iou, loss_dfl
    per = torch.zeros(fg_mask.shape + (2,), dtype=torch.float32, device=fg_mask.device)
    per[fg_mask] = torch.cat((l_iou, l_dfl), -1).detach().float()
    return loss_iou, loss_dfl, per


def loss_case(seed: int, bs: int, level_hw, strides, nc: int, n_gt: int, dtype=torch.float32, device="cuda", ops=None):
    """Seeded inputs of ``BboxLoss.forward`` as ``Loss.__call__`` builds them (utils/loss.py:139-170): ground truths and
    positives from ``oracle.ref_port.tal_case`` through the assigner (``ops.tal_assign`` on the GPU), targets divided by
    the strides (grid units), random DFL logits and predicted boxes whose side distances are the targets' jittered."""
    from oracle import ref_port as rp

    c = {k: v.to(device) for k, v in rp.tal_case(seed, bs, level_hw, strides, nc, n_gt).items()}
    assign = ops.tal_assign if ops is not None else (lambda *a, **k: rp.tal_assign_port(*a, **k)[:5])
    _, tb, ts, fg, _ = assign(**c, topk=10, num_classes=nc)
    st = torch.cat([torch.full((h * w, 1), float(s)) for (h, w), s in zip(level_hw, strides)]).to(device)
    g = torch.Generator().manual_seed(seed + 1000)
    A = st.shape[0]
    ap = (c["anc_points"] / st).to(dtype)
    tb = tb / st
    pred_dist = (torch.randn(bs, A, 64, generator=g) * 3).to(device=device, dtype=dtype)
    apf = ap.float().cpu()
    ltrb = torch.cat((apf - tb.cpu()[..., :2], tb.cpu()[..., 2:] - apf), -1)
    d = (ltrb + torch.randn(bs, A, 4, generator=g) * 0.7).clamp(0, 15)  # what Loss.bbox_decode can return
    pb = torch.cat((apf - d[..., :2], apf + d[..., 2:]), -1).to(device=device, dtype=dtype)
    tss = ts.sum().clamp(min=1)  # max(target_scores.sum(), 1) (loss.py:165) without the host round trip
    return dict(pred_dist=pred_dist, pred_bboxes=pb, anchor_points=ap, target_bboxes=tb, target_scores=ts,
                target_scores_sum=tss, fg_mask=fg)
