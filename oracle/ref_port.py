"""CPU oracle for the CerberusDet post-head path (decode + per-task NMS).

TEST INFRASTRUCTURE ONLY.  Nothing under ``cerberusdet_b200/`` may import this
module; only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs do, and there only as the checker or
the timed CPU baseline -- never as the product path.

It is a restatement of the reference algorithm, stage by stage, on ``torch`` CPU
tensors (the reference itself is pure torch, so the same ATen kernels do the
arithmetic).  Every function cites the reference lines it follows
(paths relative to the reference root).

Parity status: PINNED.  ``oracle/gen_golden.py`` runs the unmodified reference in
the build container and stores its outputs under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this module against them bit for bit.

One deliberate difference from the reference: the candidate sort
(``utils/general.py:459``) is an *unstable* ``argsort`` there, so the order of
equal scores is unspecified.  The oracle fixes the canonical rule
"score descending, then candidate index ascending" (``stable=True``).  On tie-free
inputs both give identical results, which the golden generator asserts.

The greedy suppression itself lives in a third-party dependency that is not in
the reference tree: ``torchvision.ops.nms`` (pinned ``torchvision==0.20.1`` in
``pyproject.toml:52``; call site ``utils/general.py:464``).  ``greedy_nms.c`` restates
its published CPU algorithm in plain C; ``nms_port(..., greedy="c")`` uses that,
``greedy="torchvision"`` calls the installed binary, and the tests require both to
agree.
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

REG_MAX = 16  # models/yolo.py:75  (DFL bins per box side)
MAX_WH = 7680  # utils/general.py:415
MAX_NMS = 30000  # utils/general.py:416

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")
_LIB = os.path.join(_BUILD, "libcerb_oracle.so")
_lib = None


# --------------------------------------------------------------------------- C part
def build_c_oracle(force: bool = False) -> str:
    """Compile ``greedy_nms.c`` (gcc, -O2, no FMA contraction) into ``oracle/_build``."""
    src = os.path.join(_HERE, "greedy_nms.c")
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(src):
        os.makedirs(_BUILD, exist_ok=True)
        cmd = ["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", _LIB, src]
        subprocess.run(cmd, check=True)
    return _LIB


def _c():
    global _lib
    if _lib is None:
        lib = ctypes.CDLL(build_c_oracle())
        lib.oracle_greedy_nms.restype = ctypes.c_long
        lib.oracle_greedy_nms.argtypes = [
            ctypes.c_void_p,  # const float* boxes [n,4]
            ctypes.c_long,  # n
            ctypes.c_double,  # iou threshold
            ctypes.c_void_p,  # long* keep [n]
        ]
        lib.oracle_greedy_nms_topk.restype = ctypes.c_long
        lib.oracle_greedy_nms_topk.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_double, ctypes.c_void_p, ctypes.c_long]
        _lib = lib
    return _lib


def greedy_nms_c(boxes: torch.Tensor, iou_thres: float, max_keep: int = 0) -> torch.Tensor:
    """Greedy suppression over boxes ALREADY in processing order (score-descending).  ``max_keep > 0`` stops after that
    many kept boxes (the same first ``max_keep`` indices as the full run: greedy suppression is causal)."""
    b = np.ascontiguousarray(boxes.detach().cpu().numpy(), dtype=np.float32)
    n = b.shape[0]
    keep = np.empty(max(n, 1), dtype=np.int64)
    k = _c().oracle_greedy_nms_topk(b.ctypes.data, n, float(iou_thres), keep.ctypes.data, int(max_keep))
    return torch.from_numpy(keep[:k].copy())


# --------------------------------------------------------------------------- decode
def anchor_grid(level_hw: Sequence[Sequence[int]], strides: Sequence[float], dtype, device="cpu"):
    """``make_anchors`` (utils/tal.py:181-193) + the transpose at models/yolo.py:94.

    Anchor k of a level with width w sits at (k % w + 0.5, k // w + 0.5) in grid
    units; levels are concatenated in order.  Returns ``anchors[2, A]`` and
    ``strides[1, A]`` in ``dtype``.
    """
    pts, st = [], []
    for (h, w), s in zip(level_hw, strides):
        xs = torch.arange(w, dtype=dtype, device=device) + 0.5
        ys = torch.arange(h, dtype=dtype, device=device) + 0.5
        gy, gx = torch.meshgrid(ys, xs, indexing="ij")
        pts.append(torch.stack((gx, gy), -1).reshape(-1, 2))
        st.append(torch.full((h * w, 1), float(s), dtype=dtype, device=device))
    return torch.cat(pts).transpose(0, 1), torch.cat(st).transpose(0, 1)


def dfl_expectation(box_logits: torch.Tensor) -> torch.Tensor:
    """``DFL.forward`` (models/yolo.py:57-59): softmax over the 16 bins of each side,
    then a frozen 1x1 conv with weights 0..15 (models/yolo.py:52-54).

    ``box_logits`` is ``[B, 64, A]`` with channel = side*16 + bin.  The conv is kept
    as a conv (not a hand-written dot product) so half inputs round exactly where
    the reference's do.
    """
    b, _, a = box_logits.shape
    probs = box_logits.view(b, 4, REG_MAX, a).transpose(2, 1).softmax(1)  # [b,16,4,a]
    w = torch.arange(REG_MAX, dtype=torch.float).view(1, REG_MAX, 1, 1).to(box_logits)
    return F.conv2d(probs, w).view(b, 4, a)


def ltrb_to_xywh(dist: torch.Tensor, anchors: torch.Tensor) -> torch.Tensor:
    """``dist2bbox(xywh=True, dim=1)`` (utils/tal.py:196-205), operation order kept:
    corners first, then centre = (x1y1 + x2y2) / 2 and size = x2y2 - x1y1."""
    lt, rb = dist[:, :2], dist[:, 2:]
    p1 = anchors - lt
    p2 = anchors + rb
    return torch.cat(((p1 + p2) / 2, p2 - p1), 1)


def decode_port(levels: Sequence[torch.Tensor], nc: int, strides: Sequence[float]) -> torch.Tensor:
    """Eval branch of ``Detect.forward`` after the conv towers (models/yolo.py:93-99).

    ``levels[l]`` is the raw head tensor ``[B, 64+nc, H_l, W_l]``.  Returns
    ``y[B, 4+nc, A]`` in the input dtype: (cx, cy, w, h) in pixels, then sigmoid scores.
    """
    bsz = levels[0].shape[0]
    no = 4 * REG_MAX + nc
    dtype = levels[0].dtype
    anchors, stride_row = anchor_grid([t.shape[2:] for t in levels], strides, dtype, levels[0].device)
    flat = torch.cat([t.reshape(bsz, no, -1) for t in levels], 2)  # models/yolo.py:97
    box_logits, cls_logits = flat[:, : 4 * REG_MAX], flat[:, 4 * REG_MAX :]
    dbox = ltrb_to_xywh(dfl_expectation(box_logits), anchors.unsqueeze(0)) * stride_row  # yolo.py:98
    return torch.cat((dbox, cls_logits.sigmoid()), 1)  # yolo.py:99


# --------------------------------------------------------------------------- NMS
def centre_to_corners(b: torch.Tensor) -> torch.Tensor:
    """``xywh2xyxy`` (utils/general.py:272-288); arithmetic stays in the input dtype."""
    half_w = b[..., 2] / 2
    half_h = b[..., 3] / 2
    return torch.stack((b[..., 0] - half_w, b[..., 1] - half_h, b[..., 0] + half_w, b[..., 1] + half_h), -1)


def candidates_port(
    img: torch.Tensor,
    conf_thres: float,
    classes: Optional[Sequence[int]],
    multi_label: bool,
) -> torch.Tensor:
    """Stages N1-N3 for one image ``img[4+nc, A]`` -> fp32 rows (x1,y1,x2,y2,conf,cls).

    utils/general.py:411 (per-anchor prefilter, compare in tensor dtype), :427
    (rows in ascending anchor order), :443 (corners), :444-449 (multi-label
    expansion in anchor-major, class-minor order, or best class with the lowest
    index winning ties), :452-453 (class filter).
    """
    nc = img.shape[0] - 4
    rows = img.transpose(0, 1)  # [A, 4+nc]
    rows = rows[rows[:, 4:].amax(1) > conf_thres]
    if rows.shape[0] == 0:
        return torch.zeros((0, 6))
    box = centre_to_corners(rows[:, :4])
    scores = rows[:, 4:]
    if multi_label and nc > 1:  # utils/general.py:419
        r, c = (scores > conf_thres).nonzero(as_tuple=True)
        det = torch.cat((box[r].float(), scores[r, c].float()[:, None], c.float()[:, None]), 1)
    else:
        conf, c = scores.max(1)
        det = torch.cat((box.float(), conf.float()[:, None], c.float()[:, None]), 1)
        det = det[conf > conf_thres]
    if classes is not None:
        wanted = torch.tensor(list(classes), dtype=torch.float32)
        det = det[(det[:, 5:6] == wanted).any(1)]
    return det


def nms_port(
    prediction: torch.Tensor,
    conf_thres: float = 0.25,
    iou_thres: float = 0.45,
    classes: Optional[Sequence[int]] = None,
    agnostic: bool = False,
    multi_label: bool = False,
    max_det: int = 300,
    max_nms: int = MAX_NMS,
    max_wh: float = MAX_WH,
    greedy: str = "torchvision",
    return_candidates: bool = False,
) -> List[torch.Tensor]:
    """``non_max_suppression`` (utils/general.py:360-481) with ``labels=()``, ``nm=0``.

    No wall-clock time limit (utils/general.py:417,477-479 is a result hazard, not
    part of the algorithm) and a stable candidate sort (see module docstring).
    """
    assert 0 <= conf_thres <= 1, f"Invalid Confidence threshold {conf_thres}"  # :399
    assert 0 <= iou_thres <= 1, f"Invalid IoU {iou_thres}"  # :400
    if isinstance(prediction, (list, tuple)):  # :401-402
        prediction = prediction[0]
    out: List[torch.Tensor] = []
    cands = []
    for img in prediction:
        det = candidates_port(img, conf_thres, classes, multi_label)
        if det.shape[0]:
            order = det[:, 4].argsort(descending=True, stable=True)[:max_nms]  # :459 (canonical ties)
            det = det[order]
            shifted = det[:, :4] + det[:, 5:6] * (0 if agnostic else max_wh)  # :462-463
            if greedy == "torchvision":
                import torchvision

                keep = torchvision.ops.nms(shifted, det[:, 4], iou_thres)  # :464
            else:
                keep = greedy_nms_c(shifted, iou_thres, max_keep=max_det)  # early exit: same first max_det indices
            det_out = det[keep[:max_det]]  # :465,474
        else:
            det_out = det
        out.append(det_out)
        cands.append(det)
    return (out, cands) if return_candidates else out


def postprocess_port(task_levels, ncs, strides, **nms_kw):
    """Whole path for several task heads: decode each head, then NMS each head
    (the per-task loop of cerberusdet_inference.py:125-135)."""
    results = []
    for levels, nc in zip(task_levels, ncs):
        y = decode_port(levels, nc, strides)
        results.append(nms_port(y, **nms_kw))
    return results


# --------------------------------------------------------------------------- training-time sibling decode (SURVEY 8f-4)
def bbox_decode_port(anchor_points: torch.Tensor, pred_dist: torch.Tensor) -> torch.Tensor:
    """``Loss.bbox_decode`` with ``use_dfl`` (utils/loss.py:126-131) followed by ``dist2bbox(xywh=False)``
    (utils/tal.py:196-205): ``pred_dist [B, A, 64]`` (bins of a side contiguous) and ``anchor_points [A, 2]`` ->
    ``[B, A, 4]`` = (x1, y1, x2, y2) in grid units.  Differentiable (the test compares autograd gradients too)."""
    b, a, c = pred_dist.shape
    proj = torch.arange(REG_MAX, dtype=torch.float, device=pred_dist.device)
    dist = pred_dist.view(b, a, 4, c // 4).softmax(3).matmul(proj.type(pred_dist.dtype))
    lt, rb = torch.split(dist, 2, -1)
    return torch.cat((anchor_points - lt, anchor_points + rb), -1)


# --------------------------------------------------------------------------- head tail (SURVEY 8f-3; the checker is ready, the kernel is round 2)
def head_tail_port(box_feats: Sequence[torch.Tensor], cls_feats: Sequence[torch.Tensor], box_w: Sequence[torch.Tensor],
                   box_b: Sequence[torch.Tensor], cls_w: Sequence[torch.Tensor], cls_b: Sequence[torch.Tensor],
                   strides: Sequence[float]) -> Tuple[torch.Tensor, list]:
    """The step right before the path plus the path: the LAST 1x1 convolutions of the two towers of every level
    (``cv2[i][-1]``: c2 -> 64 and ``cv3[i][-1]``: c3 -> nc, models/yolo.py:81-84), the channel concat (yolo.py:89-90) and
    the eval decode (yolo.py:93-99).

    ``box_feats[l]`` ``[B, c2, H_l, W_l]`` / ``cls_feats[l]`` ``[B, c3, H_l, W_l]`` are the inputs of those last
    convolutions; ``box_w[l]`` ``[64, c2, 1, 1]``, ``cls_w[l]`` ``[nc, c3, 1, 1]`` and the biases are their parameters.
    Returns ``(y [B, 4+nc, A], raw levels [B, 64+nc, H_l, W_l])`` like ``Detect.forward`` in eval mode."""
    raw = []
    for l in range(len(box_feats)):
        raw.append(torch.cat((F.conv2d(box_feats[l], box_w[l], box_b[l]), F.conv2d(cls_feats[l], cls_w[l], cls_b[l])), 1))
    nc = int(cls_w[0].shape[0])
    return decode_port(raw, nc, strides), raw


# --------------------------------------------------------------------------- TAL assigner (SURVEY 8f-4: the training-time sibling's caller)
def ciou_port(box1: torch.Tensor, box2: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """``bbox_iou(box1, box2, xywh=False, CIoU=True)`` (utils/metrics.py:373-408), one torch op per reference op."""
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
    v = (4 / math.pi**2) * (torch.atan(w2 / h2) - torch.atan(w1 / h1)).pow(2)
    alpha = v / (v - iou + (1 + eps))
    return iou - (rho2 / c2 + v * alpha)


def tal_assign_port(pd_scores: torch.Tensor, pd_bboxes: torch.Tensor, anc_points: torch.Tensor, gt_labels: torch.Tensor,
                    gt_bboxes: torch.Tensor, mask_gt: torch.Tensor, topk: int = 10, num_classes: int = 80, alpha: float = 0.5,
                    beta: float = 6.0, eps: float = 1e-9, claims: bool = False):
    """``TaskAlignedAssigner.forward`` (utils/tal.py:56-178, with ``select_candidates_in_gts`` :13-28 and
    ``select_highest_overlaps`` :31-53) restated stage by stage.  One thing is made canonical: the reference's
    ``torch.topk`` (:140) leaves the order of EQUAL metrics unspecified; here ties go to the lower anchor index.  That
    only matters when a ground-truth box has fewer than ``topk`` anchors with a positive metric AND anchors inside it
    whose metric is exactly 0 (CIoU <= 0): which of those become positives is arbitrary in the reference.
    ``ambiguous [B, G]`` (last return value) flags those boxes so that tests compare the others.

    Returns ``(target_labels [B, A] int64, target_bboxes [B, A, 4], target_scores [B, A, C], fg_mask [B, A] bool,
    target_gt_idx [B, A] int64, ambiguous [B, G] bool)``; with ``claims=True`` also ``[B, A]`` int64, the number of boxes
    whose top-k claims each anchor before ``select_highest_overlaps`` resolves anchors claimed by several."""
    bs, n_max = pd_scores.size(0), gt_bboxes.size(1)
    A = pd_scores.size(1)
    if n_max == 0:
        return (torch.full_like(pd_scores[..., 0], num_classes), torch.zeros_like(pd_bboxes), torch.zeros_like(pd_scores),
                torch.zeros_like(pd_scores[..., 0]), torch.zeros_like(pd_scores[..., 0]), torch.zeros((bs, 0), dtype=torch.bool))
    # get_box_metrics (:121-130)
    bidx = torch.arange(bs).view(-1, 1).repeat(1, n_max)
    lab = gt_labels.long().squeeze(-1)
    bbox_scores = pd_scores[bidx, :, lab]  # [B, G, A]
    overlaps = ciou_port(gt_bboxes.unsqueeze(2), pd_bboxes.unsqueeze(1)).squeeze(3).clamp(0)
    align_metric = bbox_scores.pow(alpha) * overlaps.pow(beta)
    # select_candidates_in_gts (:13-28)
    lt, rb = gt_bboxes.view(-1, 1, 4).chunk(2, 2)
    deltas = torch.cat((anc_points[None] - lt, rb - anc_points[None]), dim=2).view(bs, n_max, A, -1)
    mask_in_gts = deltas.amin(3).gt_(eps)
    # select_topk_candidates (:132-151), ties to the lower anchor index
    metrics = align_metric * mask_in_gts
    order = torch.sort(metrics, dim=-1, descending=True, stable=True).indices  # stable: equal values keep index order
    topk_idxs = order[..., :topk]
    topk_mask = mask_gt.repeat([1, 1, topk]).bool()
    topk_idxs = torch.where(topk_mask, topk_idxs, 0)
    is_in_topk = F.one_hot(topk_idxs, A).sum(-2)
    is_in_topk = torch.where(is_in_topk > 1, 0, is_in_topk).to(metrics.dtype)
    mask_pos = is_in_topk * mask_in_gts * mask_gt
    n_positive = ((metrics > 0).sum(-1))
    n_zero_inside = ((mask_in_gts > 0) & (metrics == 0)).sum(-1)
    ambiguous = (n_positive < topk) & (n_zero_inside > 0) & (mask_gt.squeeze(-1) > 0)
    # select_highest_overlaps (:31-53)
    fg_mask = mask_pos.sum(-2)
    n_claims = fg_mask.long()
    if fg_mask.max() > 1:
        mask_multi = (fg_mask.unsqueeze(1) > 1).repeat([1, n_max, 1])
        is_max = F.one_hot(overlaps.argmax(1), n_max).permute(0, 2, 1).to(overlaps.dtype)
        mask_pos = torch.where(mask_multi, is_max, mask_pos)
        fg_mask = mask_pos.sum(-2)
    target_gt_idx = mask_pos.argmax(-2)
    # get_targets (:153-178)
    flat_idx = target_gt_idx + torch.arange(bs, dtype=torch.int64)[..., None] * n_max
    target_labels = gt_labels.long().flatten()[flat_idx]
    target_bboxes = gt_bboxes.view(-1, 4)[flat_idx]
    target_scores = F.one_hot(target_labels, num_classes)
    target_scores = torch.where(fg_mask[:, :, None].repeat(1, 1, num_classes) > 0, target_scores, 0)
    # normalise (:103-108)
    align_metric = align_metric * mask_pos
    pos_align = align_metric.amax(-1, keepdim=True)
    pos_ov = (overlaps * mask_pos).amax(-1, keepdim=True)
    norm = (align_metric * pos_ov / (pos_align + eps)).amax(-2).unsqueeze(-1)
    out = (target_labels, target_bboxes, target_scores * norm, fg_mask.bool(), target_gt_idx, ambiguous)
    return out + (n_claims,) if claims else out


def tal_case(seed: int, bs: int, level_hw, strides, nc: int, n_gt: int, noise: float = 4.0, score_dtype=torch.float32):
    """Seeded inputs of ``TaskAlignedAssigner.forward`` as the loss builds them (utils/loss.py:139-162): anchor points in
    pixels, ground-truth boxes (a few of them heavily overlapping, padded per image with ``mask_gt = 0``), predicted
    boxes = for every anchor the first ground truth that contains it, jittered (so overlaps are positive where it
    matters), and sigmoid-like scores."""
    g = torch.Generator().manual_seed(seed)
    pts = []
    for (h, w), s in zip(level_hw, strides):
        sy, sx = torch.meshgrid(torch.arange(h, dtype=torch.float32) + 0.5, torch.arange(w, dtype=torch.float32) + 0.5, indexing="ij")
        pts.append(torch.stack((sx, sy), -1).view(-1, 2) * s)
    anc = torch.cat(pts)
    A = anc.shape[0]
    H, W = level_hw[0][0] * strides[0], level_hw[0][1] * strides[0]
    counts = torch.randint(max(n_gt // 3, 1), n_gt + 1, (bs,), generator=g)
    counts[0] = n_gt
    gt_bboxes = torch.zeros(bs, n_gt, 4)
    gt_labels = torch.zeros(bs, n_gt, 1)
    mask_gt = torch.zeros(bs, n_gt, 1)
    for b in range(bs):
        n = int(counts[b])
        wh = torch.rand(n, 2, generator=g) * torch.tensor([W * 0.35, H * 0.35]) + 12.0
        cxy = torch.rand(n, 2, generator=g) * torch.tensor([W * 0.8, H * 0.8]) + torch.tensor([W * 0.1, H * 0.1])
        if n >= 4:  # two heavily overlapping pairs: anchors claimed by two boxes
            cxy[1] = cxy[0] + 3.0
            wh[1] = wh[0] * 1.1
            cxy[3] = cxy[2] - 2.0
            wh[3] = wh[2] * 0.9
        box = torch.cat((cxy - wh / 2, cxy + wh / 2), 1).clamp(min=0)
        box[:, 2].clamp_(max=W)
        box[:, 3].clamp_(max=H)
        gt_bboxes[b, :n] = box
        gt_labels[b, :n, 0] = torch.randint(0, nc, (n,), generator=g).float()
        mask_gt[b, :n] = 1
    pd_bboxes = torch.zeros(bs, A, 4)
    for b in range(bs):
        n = int(counts[b])
        inside = ((anc[None, :, 0] > gt_bboxes[b, :n, None, 0]) & (anc[None, :, 1] > gt_bboxes[b, :n, None, 1])
                  & (anc[None, :, 0] < gt_bboxes[b, :n, None, 2]) & (anc[None, :, 1] < gt_bboxes[b, :n, None, 3]))  # [n, A]
        first = torch.where(inside.any(0), inside.float().argmax(0), torch.randint(0, n, (A,), generator=g))
        pd_bboxes[b] = gt_bboxes[b, first] + torch.randn(A, 4, generator=g) * noise
    pd_scores = torch.sigmoid(torch.randn(bs, A, nc, generator=g) * 2.0 - 1.0).to(score_dtype)
    return dict(pd_scores=pd_scores, pd_bboxes=pd_bboxes, anc_points=anc, gt_labels=gt_labels, gt_bboxes=gt_bboxes, mask_gt=mask_gt)
