"""numpy restatement of the reference's ``ap_per_class`` (cerberusdet/utils/metrics.py:56-120, the YOLOv5 /
ultralytics-8.0 form) and the ``compute_ap`` / ``smooth`` it calls, plus a seeded generator of validation-like
statistics.

``ap_per_class_verbatim`` is the reference text with its default (unstable) ``np.argsort``.  ``ap_per_class_port``
differs in one rule only: equal confidences are ordered by row index (``kind="stable"``), the order the kernels use.
It also takes each class's rows from a class-grouped copy instead of a boolean mask over all rows; the subsequence,
and so every value, is the same (tests/test_ap_host.py checks it against the verbatim text).  ``plot`` is not
restated (the drop-in sends it to the reference)."""
from __future__ import annotations

import numpy as np

_trapz = getattr(np, "trapezoid", None) or np.trapz


def smooth(y, f=0.05):
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def compute_ap(recall, precision):
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    mpre = np.flip(np.maximum.accumulate(np.flip(mpre)))
    x = np.linspace(0, 1, 101)
    ap = _trapz(np.interp(x, mrec, mpre), x)
    return ap, mpre, mrec


def _tail(tp, p, r, ap, unique_classes, nt, names, eps):
    f1 = 2 * p * r / (p + r + eps)
    names = [v for k, v in names.items() if k in unique_classes]
    names = dict(enumerate(names))
    i = smooth(f1.mean(0), 0.1).argmax()
    p, r, f1 = p[:, i], r[:, i], f1[:, i]
    tp = (r * nt).round()
    fp = (tp / (p + eps) - tp).round()
    return tp, fp, p, r, f1, ap, unique_classes.astype(int)


def _class_curves(tp_c, conf_c, n_l, px, eps):
    fpc = (1 - tp_c).cumsum(0)
    tpc = tp_c.cumsum(0)
    recall = tpc / (n_l + eps)
    precision = tpc / (tpc + fpc)
    r = np.interp(-px, -conf_c, recall[:, 0], left=0)
    p = np.interp(-px, -conf_c, precision[:, 0], left=1)
    ap = [compute_ap(recall[:, j], precision[:, j])[0] for j in range(tp_c.shape[1])]
    return ap, p, r


def ap_per_class_verbatim(tp, conf, pred_cls, target_cls, names=None, eps=1e-16):
    """The reference's text (plot=False)."""
    i = np.argsort(-conf)
    tp, conf, pred_cls = tp[i], conf[i], pred_cls[i]
    unique_classes, nt = np.unique(target_cls, return_counts=True)
    nc = unique_classes.shape[0]
    px = np.linspace(0, 1, 1000)
    ap, p, r = np.zeros((nc, tp.shape[1])), np.zeros((nc, 1000)), np.zeros((nc, 1000))
    for ci, c in enumerate(unique_classes):
        i = pred_cls == c
        n_l = nt[ci]
        n_p = i.sum()
        if n_p == 0 or n_l == 0:
            continue
        ap[ci], p[ci], r[ci] = _class_curves(tp[i], conf[i], n_l, px, eps)
    return _tail(tp, p, r, ap, unique_classes, nt, names if names is not None else {}, eps)


def ap_arrays_port(tp, conf, pred_cls, target_cls, eps=1e-16):
    """``(ap, p, r, unique_classes, nt)`` under the tie rule: conf descending, then row index ascending."""
    i = np.argsort(-conf, kind="stable")
    tp, conf, pred_cls = tp[i], conf[i], pred_cls[i]
    g = np.argsort(pred_cls, kind="stable")  # class-grouped; each class keeps its rows' order
    tp, conf, pred_cls = tp[g], conf[g], pred_cls[g]
    unique_classes, nt = np.unique(target_cls, return_counts=True)
    nc = unique_classes.shape[0]
    px = np.linspace(0, 1, 1000)
    ap, p, r = np.zeros((nc, tp.shape[1])), np.zeros((nc, 1000)), np.zeros((nc, 1000))
    lo = np.searchsorted(pred_cls, unique_classes, side="left")
    hi = np.searchsorted(pred_cls, unique_classes, side="right")  # rows with pred_cls == c (-0.0 == 0.0; NaN none)
    for ci in range(nc):
        n_l, n_p = nt[ci], hi[ci] - lo[ci]
        if n_p == 0 or n_l == 0:
            continue
        s = slice(lo[ci], hi[ci])
        ap[ci], p[ci], r[ci] = _class_curves(tp[s], conf[s], n_l, px, eps)
    return ap, p, r, unique_classes, nt


def ap_per_class_port(tp, conf, pred_cls, target_cls, names=None, eps=1e-16):
    ap, p, r, unique_classes, nt = ap_arrays_port(tp, conf, pred_cls, target_cls, eps)
    return _tail(tp, p, r, ap, unique_classes, nt, names if names is not None else {}, eps)


def make_stats(n, nc, K=10, seed=0, zipf=1.1, fp16_conf=False, label_ratio=0.05, unlabelled=0, unpredicted=0):
    """Seeded validation-like statistics ``(tp [n, K] bool, conf [n] f32, pred_cls [n] f32, target_cls [m] f32)``.

    Classes are Zipf-distributed (class 0 the most frequent); a detection is a true-positive candidate with probability
    ``conf``, and its IoU (uniform above 0.5) decides the columns: ``tp[:, j]`` is ``iou >= 0.5 + 0.05 j``, so the
    columns are nested.  Per class, at most ``n_l`` candidates are kept (in row order), as the reference's matching
    guarantees.  ``unlabelled`` extra classes are predicted but never labelled, ``unpredicted`` labelled but never
    predicted.  ``fp16_conf`` rounds the scores to half precision (massive ties)."""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, nc + unlabelled + 1) ** zipf
    pred_cls = rng.choice(nc + unlabelled, size=n, p=w / w.sum()).astype(np.float32)
    conf = rng.random(n, dtype=np.float32)
    if fp16_conf:
        conf = conf.astype(np.float16).astype(np.float32)
    m = max(int(n * label_ratio), nc + unpredicted)
    target_cls = np.concatenate((np.arange(nc + unpredicted), rng.choice(nc, size=m - nc - unpredicted, p=w[:nc] / w[:nc].sum())))
    target_cls = target_cls.astype(np.float32)
    target_cls[nc:nc + unpredicted] += unlabelled  # the labelled-only classes sit above the predicted-only ones
    cand = rng.random(n, dtype=np.float32) < conf
    nt_all = np.bincount(target_cls.astype(np.int64), minlength=nc + unlabelled + unpredicted)
    cls_i = pred_cls.astype(np.int64)
    order = np.argsort(cls_i, kind="stable")
    first = np.searchsorted(cls_i[order], cls_i[order], side="left")
    cum = np.cumsum(cand[order]) - cand[order]  # candidates before each row in class-grouped order
    rank = np.empty(n, dtype=np.int64)
    rank[order] = cum - cum[first]  # ... and before it within its class
    cand &= rank < nt_all[cls_i]
    iou = 0.5 + 0.5 * rng.random(n)
    tp = cand[:, None] & (iou[:, None] >= np.linspace(0.5, 0.95, K)[None, :])
    return tp, conf, pred_cls, target_cls
