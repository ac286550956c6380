"""Host restatement of the per-image statistics step that follows NMS in the reference validation loop
(SURVEY section 8f row 2): ``process_batch`` (cerberusdet/val.py:32-54) -- which detections count as correct at each
of the IoU thresholds ``iouv``.

Semantics, per threshold t: the pairs (label l, detection d) with ``iou >= t`` and equal class are sorted by IoU
descending; every detection keeps its first pair (its best label), the survivors -- now ordered by detection index --
are de-duplicated per label keeping the first, i.e. the lowest detection index (val.py:48-51).  The reference sorts with
numpy's unstable default, so exactly equal IoUs have no defined order there; the canonical rule here (and in the CUDA
kernel) is "IoU descending, then label index ascending".

After the loop: ``ap_per_class`` (cerberusdet/utils/metrics.py:56-120), the drop-in whose per-class curves and APs come
from ``ops.ap_per_class`` and whose O(nc * 1000) tail runs here in numpy, and ``make_ap_per_class``, its guarded form for
``patch.install(metrics=True)``.  With ``plots`` on, the loop also feeds ``ConfusionMatrix.process_batch``
(utils/metrics.py:273-370) per image: ``make_confusion_process_batch`` is its drop-in for ``patch.install(confusion=True)``,
and ``validation_batch_statistics(confusion=...)`` its batched form.
"""
from __future__ import annotations

from pathlib import Path
from typing import Optional

import numpy as np
import torch

from .cross_task import pairwise_iou


def match_predictions(detections: torch.Tensor, labels: torch.Tensor, iouv: torch.Tensor) -> torch.Tensor:
    """``detections [N, 6]`` (x1, y1, x2, y2, conf, cls), ``labels [M, 5]`` (cls, x1, y1, x2, y2), ``iouv [K]``
    -> ``correct [N, K]`` bool (val.py:32-54)."""
    n, k = detections.shape[0], iouv.shape[0]
    correct = torch.zeros((n, k), dtype=torch.bool)
    if n == 0 or labels.shape[0] == 0:
        return correct
    det, lab = detections.detach().cpu().float(), labels.detach().cpu().float()
    iou = pairwise_iou(lab[:, 1:], det[:, :4])  # [M, N]
    same = lab[:, 0:1] == det[:, 5]
    masked = torch.where(same, iou, torch.full_like(iou, -1.0))
    best_iou, best_lab = masked.max(0)  # per detection; torch.max returns the first (lowest label) maximum
    iouv = iouv.detach().cpu().float()
    for i in range(k):
        valid = (best_iou >= iouv[i]) & (best_iou >= 0)
        taken = set()
        for d in range(n):  # ascending detection index: the first detection claiming a label keeps it
            if bool(valid[d]):
                l = int(best_lab[d])
                if l not in taken:
                    taken.add(l)
                    correct[d, i] = True
    return correct


def make_process_batch(reference_process_batch):
    """Drop-in for the reference's ``process_batch(detections, labels, iouv)`` (cerberusdet/val.py:32-54), bound onto
    ``cerberusdet.val`` by ``patch.install(val=True)``: the validation loop (val.py:321-357) calls it once per image.
    CUDA tensors go to ``cerb_val_match`` (ONE launch and no host round trip per image, where the reference makes
    ~5 launches and a ``.cpu().numpy()`` sync per IoU threshold -- 10 of them); anything else (CPU tensors, more than
    1024 labels or detections in an image) runs the reference's own function."""
    from . import ops

    cache = {}

    def process_batch(detections, labels, iouv):
        n, m = int(detections.shape[0]), int(labels.shape[0])
        on_path = (detections.is_cuda and labels.is_cuda and detections.dim() == 2 and detections.shape[1] == 6
                   and labels.dim() == 2 and labels.shape[1] == 5 and 0 < n <= 30000 and 0 < m <= 1024)
        if not on_path:
            return reference_process_batch(detections, labels, iouv)
        key = (iouv.data_ptr(), int(iouv.shape[0]), getattr(iouv, "_version", 0))
        host = cache.get(key)
        if host is None:  # the thresholds are one tensor for the whole run (val.py:206): read them once
            cache.clear()
            host = cache[key] = [float(v) for v in iouv.detach().cpu().float().tolist()]
        counts = torch.full((1,), n, dtype=torch.int32, device=detections.device)
        correct = ops.match_batch(detections.float().unsqueeze(0), counts, labels, [0, m], iouv, iouv_host=host)
        return correct[0]

    process_batch._cerb_reference = reference_process_batch
    return process_batch


def batch_statistics(dets: torch.Tensor, counts: torch.Tensor, labels: torch.Tensor, label_offsets, iouv: torch.Tensor):
    """The whole statistics step of one validation batch and one task in a single launch: ``dets [B, max_det, 6]`` /
    ``counts [B]`` straight from ``ops.nms_batched`` (already in native space, see ``ops.cross_task_merge``'s ``scale`` or
    the reference's ``scale_boxes``), ``labels [sum M_b, 5]`` native-space rows with ``label_offsets [B+1]``.
    Returns ``(correct [sum n_b, K] bool, conf [sum n_b], pcls [sum n_b])`` concatenated over the images in order -- the
    first three columns the reference appends to ``stats`` per image (val.py:357) -- as device tensors."""
    from . import ops

    correct = ops.match_batch(dets, counts, labels, label_offsets, iouv)  # [B, max_det, K]
    n = counts.to(torch.int64)
    keep = torch.arange(dets.shape[1], device=dets.device)[None, :] < n[:, None]  # rows below each image's count
    return correct[keep], dets[..., 4][keep], dets[..., 5][keep]


# ------------------------------------------------------------------------------------------------ the whole loop body
def _scale_params(img_hw, ori_shapes, ratio_pads, device):
    """Per-image (1 / gain, pad_x, pad_y, w0, h0) of ``scale_boxes`` (utils/general.py:313-337) as float32 device columns.
    The reference divides a tensor by the Python float ``gain``; on CUDA PyTorch evaluates tensor / scalar as a
    multiplication by the float32 reciprocal (BinaryDivTrueKernel.cu), on the CPU as a true division.  The first column
    therefore holds the reciprocal on CUDA and the gain itself on the CPU, and ``_scale_boxes_batched`` applies it the
    same way -- bit-identical to the reference on both (tests/test_gpu_reference.py, tests/test_host_logic.py)."""
    rows = []
    for shape, rp in zip(ori_shapes, ratio_pads):
        h0, w0 = float(shape[0]), float(shape[1])
        if rp is None:
            gain = min(img_hw[0] / h0, img_hw[1] / w0)
            pad = ((img_hw[1] - w0 * gain) / 2, (img_hw[0] - h0 * gain) / 2)
        else:
            gain, pad = rp[0][0], rp[1]
        rows.append([float(gain), float(pad[0]), float(pad[1]), w0, h0])
    t = torch.tensor(rows, dtype=torch.float64).to(torch.float32).to(device)
    inv_gain = torch.ones((), dtype=torch.float32, device=device) / t[:, 0] if t.is_cuda else t[:, 0]
    return inv_gain, t[:, 1], t[:, 2], t[:, 3], t[:, 4]


def _scale_boxes_batched(boxes, inv_gain, pad_x, pad_y, w0, h0):
    """``scale_boxes`` + ``clip_boxes`` on ``boxes [..., 4]`` whose leading dimension lines up with the parameter columns."""
    shape = (-1,) + (1,) * (boxes.dim() - 2)
    g = inv_gain.view(shape)
    unscale = (lambda v: v * g) if boxes.is_cuda else (lambda v: v / g)
    out = boxes.clone()
    out[..., 0] = unscale(boxes[..., 0] - pad_x.view(shape)).clamp(min=0).minimum(w0.view(shape))
    out[..., 2] = unscale(boxes[..., 2] - pad_x.view(shape)).clamp(min=0).minimum(w0.view(shape))
    out[..., 1] = unscale(boxes[..., 1] - pad_y.view(shape)).clamp(min=0).minimum(h0.view(shape))
    out[..., 3] = unscale(boxes[..., 3] - pad_y.view(shape)).clamp(min=0).minimum(h0.view(shape))
    return out


def validation_batch_statistics(dets: torch.Tensor, counts: torch.Tensor, batch: dict, iouv: torch.Tensor, single_cls: bool = False,
                                confusion: Optional[torch.Tensor] = None):
    """The "Statistics per image" block of the reference validation loop (cerberusdet/val.py:321-357) for a whole batch
    of ONE task: native-space predictions (``scale_boxes``), native-space labels (``xywh2xyxy`` * (w, h, w, h), then
    ``scale_boxes``), ``process_batch`` -- here: a handful of batched elementwise ops and ONE ``cerb_val_match`` launch, no
    host synchronisation, where the reference runs the block per image with ~10 ``.cpu().numpy()`` round trips each.

    ``dets [B, max_det, 6]`` / ``counts [B]``: the padded NMS output of the task (``ops.nms_batched(...)[0][t]``, network
    space); ``batch``: the reference's batch dict (``img``, ``batch_idx``, ``cls``, ``bboxes``, ``ori_shape``, ``ratio_pad``).
    Returns what the loop would have appended to ``stats``: a list of ``(correct [n, K] bool, conf [n], pcls [n], tcls [m])``
    device-tensor tuples in image order -- images with neither predictions nor labels contribute nothing, images without
    predictions an empty first three (val.py:333-338).

    ``confusion``: optional ``int64 [nc+1, nc+1]`` device matrix; the batch's ``ConfusionMatrix(nc).process_batch`` counts
    (the calls the loop makes when ``plots`` is on, default ``conf`` 0.25 / ``iou_thres`` 0.45) are added to it with one
    ``cerb_confusion_matrix`` launch on the same native-space predictions and labels.  A class outside ``[0, nc)`` raises
    ``ValueError`` (the status is read with the counts, so no extra synchronisation)."""
    from . import ops

    dev = dets.device
    B, max_det = int(dets.shape[0]), int(dets.shape[1])
    img_hw = (int(batch["img"].shape[2]), int(batch["img"].shape[3]))
    ratio_pads = batch.get("ratio_pad") or [None] * B
    inv_gain, pad_x, pad_y, w0, h0 = _scale_params(img_hw, batch["ori_shape"], ratio_pads, dev)
    dets = dets.float()
    pred = dets.clone()
    if single_cls:
        pred[..., 5] = 0
    predn = pred.clone()
    predn[..., :4] = _scale_boxes_batched(pred[..., :4], inv_gain, pad_x, pad_y, w0, h0)
    # labels: rows of all images, grouped by image (batch_idx is sorted by construction of the collate function; sort anyway)
    bidx = batch["batch_idx"].to(dev).long().view(-1)
    order = torch.argsort(bidx, stable=True)
    bidx = bidx[order]
    cls = batch["cls"].to(dev).float().view(-1, 1)[order]
    bbox = batch["bboxes"].to(dev).float()[order]
    m_per = torch.bincount(bidx, minlength=B)
    offsets = [0] + torch.cumsum(m_per, 0).tolist()  # (the one host read of this step: B small integers)
    tbox = bbox.clone()  # xywh2xyxy (utils/general.py:272-288)
    tbox[:, 0] = bbox[:, 0] - bbox[:, 2] / 2
    tbox[:, 1] = bbox[:, 1] - bbox[:, 3] / 2
    tbox[:, 2] = bbox[:, 0] + bbox[:, 2] / 2
    tbox[:, 3] = bbox[:, 1] + bbox[:, 3] / 2
    tbox = tbox * torch.tensor((img_hw[1], img_hw[0], img_hw[1], img_hw[0]), device=dev)
    tbox = _scale_boxes_batched(tbox, inv_gain[bidx], pad_x[bidx], pad_y[bidx], w0[bidx], h0[bidx])
    labelsn = torch.cat((cls, tbox), 1)
    correct = ops.match_batch(predn, counts, labelsn, offsets, iouv)  # [B, max_det, K] bool
    if confusion is None:
        n_host = counts.tolist()
    else:
        offsets_d = torch.cat((m_per.new_zeros(1), torch.cumsum(m_per, 0))).to(torch.int32)
        _, status = ops.confusion_matrix_batch(predn, counts, labelsn, offsets_d, int(confusion.shape[0]) - 1, out=confusion)
        host = torch.cat((counts.to(torch.int32).view(-1), status)).tolist()
        n_host, bad = host[:B], [i for i, s in enumerate(host[B:]) if s]
        if bad:
            raise ValueError(f"confusion matrix: images {bad} have a class outside [0, {int(confusion.shape[0]) - 1}) or more than "
                             f"{ops.CM_MAX_LABELS} labels; they were not counted")
    K = int(iouv.shape[0])
    stats = []
    for i in range(B):
        n, tcls = int(n_host[i]), cls[offsets[i] : offsets[i + 1], 0]
        if n == 0:
            if tcls.numel():
                stats.append((torch.zeros((0, K), dtype=torch.bool, device=dev), torch.zeros(0, device=dev), torch.zeros(0, device=dev), tcls))
            continue
        stats.append((correct[i, :n], pred[i, :n, 4], pred[i, :n, 5], tcls))
    return stats


# ------------------------------------------------------------------------------------ mAP statistics (after the loop)
def _smooth(y, f=0.05):
    """Box filter of fraction ``f`` (utils/metrics.py ``smooth``)."""
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def _on_device(x, device):
    return x.to(device) if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x)).to(device)


def ap_per_class(tp, conf, pred_cls, target_cls, plot=False, save_dir=Path(), names=(), eps=1e-16, prefix=""):
    """Drop-in for the reference's ``ap_per_class`` (utils/metrics.py:56-120) with its signature and 7-tuple of numpy
    arrays ``(tp, fp, p, r, f1, ap, unique_classes)``.  Inputs are numpy arrays (copied to the device) or CUDA tensors.
    ``ap`` and the ``p`` / ``r`` curves come from ``ops.ap_per_class``; the O(nc * 1000) tail (f1, ``smooth``, argmax, the
    rounded tp / fp) runs here in numpy, as in the reference.  Equal confidences are ordered by row index, which is
    ``np.argsort(-conf, kind="stable")``; the reference's unstable argsort leaves their order undefined.  Plots are not
    drawn: ``plot=True`` raises (``make_ap_per_class`` sends it to the reference)."""
    from . import ops

    if plot:
        raise ValueError("ap_per_class: plot=True is the reference's (it draws the curves with matplotlib)")
    device = next((x.device for x in (tp, conf, pred_cls, target_cls) if torch.is_tensor(x) and x.is_cuda), torch.device("cuda"))
    tp, conf, pred_cls, target_cls = (_on_device(x, device) for x in (tp, conf, pred_cls, target_cls))
    ap, p, r, unique_classes, nt = (t.cpu().numpy() for t in ops.ap_per_class(tp, conf.reshape(-1), pred_cls.reshape(-1),
                                                                              target_cls.reshape(-1), eps=eps))
    f1 = 2 * p * r / (p + r + eps)
    names = [v for k, v in names.items() if k in unique_classes]  # (used by the reference's plots only)
    names = dict(enumerate(names))
    i = _smooth(f1.mean(0), 0.1).argmax()  # max F1 index
    p, r, f1 = p[:, i], r[:, i], f1[:, i]
    tp = (r * nt).round()  # true positives
    fp = (tp / (p + eps) - tp).round()  # false positives
    return tp, fp, p, r, f1, ap, unique_classes.astype(int)


def _ap_on_path(tp, conf, pred_cls, target_cls, kwargs) -> bool:
    if kwargs.get("plot") or set(kwargs) - {"plot", "save_dir", "names", "eps", "prefix"} or not torch.cuda.is_available():
        return False
    arrays = (tp, conf, pred_cls, target_cls)
    if not all(isinstance(x, np.ndarray) or (torch.is_tensor(x) and x.is_cuda) for x in arrays):
        return False
    if tp.dtype not in (np.bool_, torch.bool) or tp.ndim != 2 or not 1 <= tp.shape[1] <= 32:
        return False
    if any(x.dtype not in (np.float16, np.float32, torch.float16, torch.float32) for x in arrays[1:]):
        return False
    if conf.shape != (tp.shape[0],) or pred_cls.shape != (tp.shape[0],):
        return False
    nan = lambda x: bool(torch.isnan(x).any()) if torch.is_tensor(x) else bool(np.isnan(x).any())  # noqa: E731
    return not (nan(conf) or nan(target_cls))


def make_ap_per_class(reference_ap_per_class):
    """``ap_per_class`` for ``cerberusdet.utils.metrics`` (``patch.install(metrics=True)``): ``DetMetrics.process`` calls
    it once per task at the end of validation (utils/metrics.py:241-246).  Anything off the kernels' path runs the
    reference's own function: ``plot=True`` (the curves are drawn with matplotlib), no CUDA device, ``tp`` not bool or
    with more than 32 IoU columns, float64 scores or classes, NaN in ``conf`` or ``target_cls``, CPU tensors."""

    def ap_per_class_(tp, conf, pred_cls, target_cls, **kwargs):
        if not _ap_on_path(tp, conf, pred_cls, target_cls, kwargs):
            return reference_ap_per_class(tp, conf, pred_cls, target_cls, **kwargs)
        return ap_per_class(tp, conf, pred_cls, target_cls, **kwargs)

    ap_per_class_.__doc__ = ap_per_class.__doc__
    ap_per_class_._cerb_reference = reference_ap_per_class
    return ap_per_class_


# ---------------------------------------------------------------------------------- confusion matrix (with plots on)
def _confusion_on_path(cm, detections, labels) -> bool:
    if not (getattr(detections, "is_cuda", False) and getattr(labels, "is_cuda", False)):  # (None: the reference's first case)
        return False
    if labels.device != detections.device or not detections.dtype == labels.dtype == torch.float32:
        return False
    if detections.dim() != 2 or detections.shape[1] != 6 or labels.dim() != 2 or labels.shape[1] != 5:
        return False
    from .ops import CM_MAX_DETS, CM_MAX_LABELS

    if detections.shape[0] > CM_MAX_DETS or labels.shape[0] > CM_MAX_LABELS:
        return False
    nc, conf, iou = getattr(cm, "nc", None), getattr(cm, "conf", None), getattr(cm, "iou_thres", None)
    if not (isinstance(nc, (int, np.integer)) and 1 <= nc <= 32767 and isinstance(getattr(cm, "matrix", None), np.ndarray)
            and cm.matrix.shape == (nc + 1, nc + 1)):
        return False
    return isinstance(conf, (float, int, np.floating, np.integer)) and isinstance(iou, (float, int, np.floating, np.integer)) \
        and float(iou) >= 0


def make_confusion_process_batch(reference_process_batch):
    """``ConfusionMatrix.process_batch(self, detections, labels)`` (utils/metrics.py:273-370) for
    ``patch.install(confusion=True)``.  float32 CUDA tensors with at most 30000 detections and 1024 labels take ONE
    ``cerb_confusion_matrix`` launch and ONE device-to-host copy of ``1 + M + N`` int32 (the status and the cell of every
    row), applied to ``self.matrix`` with ``np.add.at`` -- the reference synchronises once per label and per detection.
    The instance's ``nc``, ``conf`` and ``iou_thres`` are used.  Equal IoUs resolve to the lowest label index, then the
    lowest detection index (the reference's unstable argsorts leave them undefined).  ``detections=None``, CPU tensors,
    other dtypes, larger images, a negative ``iou_thres`` and a class outside ``[0, nc)`` (seen in the status, before
    ``self.matrix`` is touched) run the reference's own method."""
    from . import ops

    def process_batch(self, detections, labels):
        if not _confusion_on_path(self, detections, labels):
            return reference_process_batch(self, detections, labels)
        host = ops.confusion_cells(detections, labels, int(self.nc), float(self.conf), float(self.iou_thres)).cpu().numpy()
        if host[0]:  # a class numpy would raise or wrap on
            return reference_process_batch(self, detections, labels)
        cells = host[1:][host[1:] >= 0]
        np.add.at(self.matrix, (cells // (self.nc + 1), cells % (self.nc + 1)), 1)

    process_batch._cerb_reference = reference_process_batch
    return process_batch
