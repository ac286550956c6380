"""Two restatements of the reference's ``ConfusionMatrix`` (cerberusdet/utils/metrics.py:273-370, yolov5's class) and the
case generators of the confusion-matrix tests.

* ``ConfusionMatrixVerbatim``: the reference's text (numpy ``argsort()[::-1]`` / ``unique``, the two Python loops); it
  runs on CPU or CUDA tensors.  Its order on exactly equal IoUs is numpy's unstable sort's, so it is the yardstick on
  tie-free inputs only.
* ``ConfusionMatrixPort``: the same semantics with the canonical tie rule of the kernel -- a detection's best label is the
  highest IoU, then the lowest label index; a label's winner is the highest IoU, then the lowest detection index.

Both compare ``conf`` and ``iou_thres`` in fp32 and take IoU as ``box_iou`` (metrics.py:415-433).
"""
from __future__ import annotations

import numpy as np
import torch


def box_iou(box1: torch.Tensor, box2: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """``[M, 4] x [N, 4]`` xyxy -> ``[M, N]``: inter / (area1 + area2 - inter + eps), one rounding per operation."""
    (a1, a2), (b1, b2) = box1.unsqueeze(1).chunk(2, 2), box2.unsqueeze(0).chunk(2, 2)
    inter = (torch.min(a2, b2) - torch.max(a1, b1)).clamp(0).prod(2)
    return inter / ((a2 - a1).prod(2) + (b2 - b1).prod(2) - inter + eps)


class ConfusionMatrixVerbatim:
    """The reference's class, ``process_batch`` as written there."""

    def __init__(self, nc, conf=0.25, iou_thres=0.45):
        self.matrix = np.zeros((nc + 1, nc + 1))
        self.nc = nc  # number of classes
        self.conf = conf
        self.iou_thres = iou_thres

    def process_batch(self, detections, labels):
        if detections is None:
            gt_classes = labels.int()
            for gc in gt_classes:
                self.matrix[self.nc, gc] += 1  # background FN
            return

        detections = detections[detections[:, 4] > self.conf]
        gt_classes = labels[:, 0].int()
        detection_classes = detections[:, 5].int()
        iou = box_iou(labels[:, 1:], detections[:, :4])

        x = torch.where(iou > self.iou_thres)
        if x[0].shape[0]:
            matches = torch.cat((torch.stack(x, 1), iou[x[0], x[1]][:, None]), 1).cpu().numpy()
            if x[0].shape[0] > 1:
                matches = matches[matches[:, 2].argsort()[::-1]]
                matches = matches[np.unique(matches[:, 1], return_index=True)[1]]
                matches = matches[matches[:, 2].argsort()[::-1]]
                matches = matches[np.unique(matches[:, 0], return_index=True)[1]]
        else:
            matches = np.zeros((0, 3))

        n = matches.shape[0] > 0
        m0, m1, _ = matches.transpose().astype(int)
        for i, gc in enumerate(gt_classes):
            j = m0 == i
            if n and sum(j) == 1:
                self.matrix[detection_classes[m1[j]], gc] += 1  # correct
            else:
                self.matrix[self.nc, gc] += 1  # true background

        if n:
            for i, dc in enumerate(detection_classes):
                if not any(m1 == i):
                    self.matrix[dc, self.nc] += 1  # predicted background


class ConfusionMatrixPort(ConfusionMatrixVerbatim):
    """Same counts with the canonical tie rule (see the module docstring)."""

    def process_batch(self, detections, labels):
        if detections is None:
            for gc in labels.cpu().int().tolist():
                self.matrix[self.nc, gc] += 1
            return
        det, lab = detections.detach().cpu().float(), labels.detach().cpu().float()
        det = det[det[:, 4] > self.conf]
        gc, dc = lab[:, 0].int().tolist(), det[:, 5].int().tolist()
        iou = box_iou(lab[:, 1:], det[:, :4]).numpy()
        above = iou > np.float32(self.iou_thres)
        M, N = iou.shape
        win = {}  # label -> detection
        if M and N:
            best = np.where(above, iou, -np.inf).argmax(0)  # first maximum: the lowest label index
            for d in range(N):  # ascending: a later detection takes a label only with a strictly higher IoU
                if above[best[d], d]:
                    l = int(best[d])
                    if l not in win or iou[l, d] > iou[l, win[l]]:
                        win[l] = d
        for i in range(M):
            self.matrix[dc[win[i]] if i in win else self.nc, gc[i]] += 1
        if win:
            matched = set(win.values())
            for d in range(N):
                if d not in matched:
                    self.matrix[dc[d], self.nc] += 1


def batch_port(dets, counts, labels, offsets, nc, conf=0.25, iou_thres=0.45, cls=ConfusionMatrixPort):
    """The matrix the validation loop builds over a batch (val.py:321-357 layout): per image, no labels -> nothing; labels
    and no detections -> ``process_batch(None, labels[:, 0])``; else ``process_batch(dets, labels)``."""
    cm = cls(nc, conf, iou_thres)
    for b in range(len(counts)):
        lab = labels[offsets[b] : offsets[b + 1]]
        n = int(counts[b])
        if lab.shape[0] == 0:
            continue
        cm.process_batch(None, lab[:, 0]) if n == 0 else cm.process_batch(dets[b, :n], lab)
    return cm.matrix


# ----------------------------------------------------------------------------------------------------- cases
def image_case(rng: np.random.Generator, M: int, N: int, nc: int, size: float = 640.0, crowd: float = 0.0,
               grid: bool = False):
    """One image: ``labels [M, 5]`` and ``detections [N, 6]`` float32 tensors, conf descending as NMS leaves them.  Most
    detections are jittered copies of labels (class kept with probability 0.7); ``crowd`` > 0 packs the labels into a
    small area so that many pairs pass the threshold.  ``grid`` snaps coordinates to integers (exact IoU ties)."""
    span = size * (1.0 - crowd) if crowd else size
    c = rng.uniform(0, span, (M, 2))
    wh = rng.uniform(8, 160, (M, 2))
    lab_boxes = np.concatenate((c - wh / 2, c + wh / 2), 1)
    lab_cls = rng.integers(0, nc, M)
    src = rng.integers(0, max(M, 1), N)
    jitter = rng.normal(0, 6 if not crowd else 10, (N, 4))
    det_boxes = lab_boxes[src] + jitter if M else rng.uniform(0, size, (N, 4))
    rand = rng.random(N) < 0.25
    det_boxes[rand] = np.concatenate((rng.uniform(0, size, (rand.sum(), 2)), rng.uniform(0, size, (rand.sum(), 2))), 1)
    det_boxes = np.concatenate((np.minimum(det_boxes[:, :2], det_boxes[:, 2:]), np.maximum(det_boxes[:, :2], det_boxes[:, 2:])), 1)
    det_cls = np.where(rng.random(N) < 0.7, lab_cls[src] if M else 0, rng.integers(0, nc, N))
    conf = np.sort(rng.uniform(0.001, 1.0, N))[::-1]
    if grid:
        lab_boxes, det_boxes = np.round(lab_boxes / 8) * 8, np.round(det_boxes / 8) * 8
    labels = np.concatenate((lab_cls[:, None], lab_boxes), 1).astype(np.float32)
    dets = np.concatenate((det_boxes, conf[:, None], det_cls[:, None]), 1).astype(np.float32)
    return torch.from_numpy(dets), torch.from_numpy(labels)


def has_ties(dets: torch.Tensor, labels: torch.Tensor, conf=0.25, iou_thres=0.45) -> bool:
    """Whether two above-threshold IoUs of the image are exactly equal (the verbatim text's order is undefined then)."""
    det = dets[dets[:, 4] > conf]
    iou = box_iou(labels[:, 1:], det[:, :4])
    v = iou[iou > iou_thres]
    return v.numel() != v.unique().numel()


def batch_case(seed: int, B: int, nc: int, max_det: int = 300, m_range=(0, 40), n_range=(0, 300), crowd: float = 0.0,
               grid: bool = False, conf_floor: float = 0.001):
    """A padded batch as the validation loop holds it: ``dets [B, max_det, 6]`` (rows past ``counts`` are garbage),
    ``counts [B]`` int32, ``labels [sum M, 5]``, ``offsets`` (B+1 ints)."""
    rng = np.random.default_rng(seed)
    dets = torch.from_numpy(rng.uniform(-50, 700, (B, max_det, 6)).astype(np.float32))  # padding: anything
    counts, labs, offsets = [], [], [0]
    for _ in range(B):
        M = int(rng.integers(m_range[0], m_range[1] + 1))
        N = int(rng.integers(n_range[0], min(n_range[1], max_det) + 1))
        d, lab = image_case(rng, M, N, nc, crowd=crowd, grid=grid)
        d[:, 4] = torch.clamp(d[:, 4], min=conf_floor)
        dets[len(counts), :N] = d
        counts.append(N)
        labs.append(lab)
        offsets.append(offsets[-1] + M)
    return dets, torch.tensor(counts, dtype=torch.int32), torch.cat(labs, 0), offsets
