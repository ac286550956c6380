"""``install()`` -- make an existing CerberusDet checkout use the B200 path.

What gets rebound (and restored by ``uninstall()``):

* ``cerberusdet.models.yolo.Detect.forward``  -> ``detect.detect_forward`` (the class itself is kept:
  checkpoints pickle it by qualified name);
* the name ``non_max_suppression`` in ``cerberusdet.utils.general`` and in every module that imported it
  by name at import time (``val``, ``detect``, ``cerberusdet_inference`` -- reference val.py:17,
  detect.py:18, cerberusdet_inference.py:10);
* ``cerberusdet.cerberusdet_inference.CerberusDetInference`` -> ``inference.CerberusDetInference``;
* with ``train=True`` also ``cerberusdet.utils.loss.Loss.bbox_decode`` -> ``ops.bbox_decode`` (the training-time
  sibling of the decode, reference utils/loss.py:126-131; forward and backward kernels).  The reference's trainer
  computes the loss under ``amp.autocast`` (trainers/averaging.py:158): there ``softmax`` runs in fp32 on the fp16
  ``pred_dist``, autocast rounds its output to fp16 for the ``matmul`` with ``proj`` (fp32 accumulation, fp16 result) and
  ``dist2bbox`` stays in fp16 -- exactly the half path of the kernels (probabilities rounded to half, one rounding of
  the expectation, one per corner), so fp16 ``pred_dist`` + fp16 anchors under autocast go to the kernels; any other
  dtype mix (fp32 under autocast, anchors of another dtype) keeps the reference's own code;
* with ``loss=True`` ``cerberusdet.utils.loss.BboxLoss.forward`` -> ``ops.bbox_loss`` (the box-regression term the loss
  computes right after the assigner, reference utils/loss.py:12-44: CIoU + DFL in one forward and one backward kernel, no
  host synchronisation).  On the path: ``use_dfl`` with 16 bins, CUDA tensors, and either everything fp32 without
  autocast or the trainer's fp16 autocast case (fp16 ``pred_dist`` / ``pred_bboxes`` / ``anchor_points``, fp32 targets);
  anything else (CPU tensors, ``use_dfl=False``, another ``reg_max``, other dtype mixes, bf16 autocast) keeps the
  reference's own code;
* with ``val=True`` the validation loop's per-image matching (val.py:32-54 ``process_batch``) -> ``ops.match_batch``;
* with ``metrics=True`` ``ap_per_class`` (utils/metrics.py:56-120), which ``DetMetrics.process`` reads as a module global,
  -> ``val_stats.ap_per_class`` (``ops.ap_per_class`` for the per-class curves and APs, the host tail in numpy), in
  ``cerberusdet.utils.metrics`` and in every imported ``cerberusdet.*`` module that imported the name.  ``plot=True``,
  no CUDA device, non-bool ``tp``, more than 32 IoU columns, float64 inputs or NaN scores / classes keep the reference's
  own function.

CUDA fp16/fp32 tensors go to the kernels; anything else (CPU tensors, training mode, masks/labels
arguments) is handed to the reference's own, saved implementation -- the patch never changes what a
non-CUDA run computes.
"""
from __future__ import annotations

import importlib
import sys
from typing import Dict, List, Tuple

_saved: List[Tuple[object, str, object]] = []
_NMS_IMPORTERS = ("cerberusdet.utils.general", "cerberusdet.val", "cerberusdet.detect", "cerberusdet.cerberusdet_inference")


def _set(obj, name, value):
    _saved.append((obj, name, getattr(obj, name)))
    setattr(obj, name, value)


def installed() -> bool:
    return bool(_saved)


def install(import_all: bool = False, train: bool = False, val: bool = False, loss: bool = False,
            metrics: bool = False) -> Dict[str, List[str]]:
    """Patch the reference modules that are importable.  ``import_all`` also imports ``val`` /
    ``detect`` / ``cerberusdet_inference`` (they pull in the whole data pipeline); by default only
    modules already imported, plus ``models.yolo`` and ``utils.general``, are touched.  ``train`` also rebinds
    ``Loss.bbox_decode``, ``TaskAlignedAssigner.forward`` and the loss module's ``make_anchors`` (imports
    ``cerberusdet.utils.loss``), ``loss`` the box-regression term ``BboxLoss.forward`` (imports
    ``cerberusdet.utils.loss``), ``val`` the validation matching (imports ``cerberusdet.val``), ``metrics`` the mAP
    statistics ``ap_per_class`` (imports ``cerberusdet.utils.metrics``).  Calling it again adds
    whatever is not patched yet (e.g. ``install()`` then ``install(train=True)``, then ``install(loss=True)``)."""
    import torch

    from . import detect as _detect
    from . import inference as _inference
    from . import nms as _nms

    done: Dict[str, List[str]] = {"patched": []}
    already = {(id(obj), name) for obj, name, _ in _saved}

    def patch_once(obj, name, value, label):
        if (id(obj), name) in already:
            return
        _set(obj, name, value)
        already.add((id(obj), name))
        done["patched"].append(label)

    yolo = importlib.import_module("cerberusdet.models.yolo")
    general = importlib.import_module("cerberusdet.utils.general")

    det_cls = yolo.Detect
    if not hasattr(det_cls, "_cerb_reference_forward"):
        det_cls._cerb_reference_forward = det_cls.forward
    patch_once(det_cls, "forward", _detect.detect_forward, "cerberusdet.models.yolo.Detect.forward")

    cur = general.non_max_suppression
    if hasattr(cur, "_cerb_reference"):
        non_max_suppression = cur  # already ours: reuse the same wrapper for late-imported modules
    else:
        reference_nms = cur

        def non_max_suppression(prediction, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False,
                                multi_label=False, labels=(), max_det=300, nm=0):
            p = prediction[0] if isinstance(prediction, (list, tuple)) else prediction
            on_path = p.is_cuda and p.dtype in (torch.float16, torch.float32) and not nm and not (labels is not None and len(labels))
            if not on_path:
                return reference_nms(prediction, conf_thres, iou_thres, classes, agnostic, multi_label, labels, max_det, nm)
            return _nms.non_max_suppression(prediction, conf_thres, iou_thres, classes, agnostic, multi_label, labels, max_det, nm)

        non_max_suppression.__doc__ = _nms.non_max_suppression.__doc__
        non_max_suppression._cerb_reference = reference_nms
    for modname in _NMS_IMPORTERS:
        mod = sys.modules.get(modname)
        if mod is None and (import_all or modname == "cerberusdet.utils.general" or (val and modname == "cerberusdet.val")):
            mod = importlib.import_module(modname)
        if mod is not None and hasattr(mod, "non_max_suppression"):
            patch_once(mod, "non_max_suppression", non_max_suppression, f"{modname}.non_max_suppression")

    inf = sys.modules.get("cerberusdet.cerberusdet_inference")
    if inf is None and import_all:
        inf = importlib.import_module("cerberusdet.cerberusdet_inference")
    if inf is not None:
        patch_once(inf, "CerberusDetInference", _inference.CerberusDetInference,
                   "cerberusdet.cerberusdet_inference.CerberusDetInference")
    if train:
        from . import ops as _ops

        loss_mod = importlib.import_module("cerberusdet.utils.loss")
        if not hasattr(loss_mod.Loss.bbox_decode, "_cerb_reference"):
            reference_bbox_decode = loss_mod.Loss.bbox_decode

            def bbox_decode(self, anchor_points, pred_dist):
                on_path = (self.use_dfl and pred_dist.is_cuda and pred_dist.dim() == 3 and pred_dist.shape[-1] == 64
                           and anchor_points.dtype == pred_dist.dtype)
                if on_path and torch.is_autocast_enabled():
                    # autocast: fp32 softmax -> fp16 probabilities -> fp16 matmul (fp32 accumulate): the kernels' half path
                    on_path = pred_dist.dtype == torch.float16 and torch.get_autocast_dtype("cuda") == torch.float16
                elif on_path:
                    on_path = pred_dist.dtype in (torch.float16, torch.float32)
                if not on_path:  # CPU tensors, reg_max != 16, mixed dtypes: the reference's own code
                    return reference_bbox_decode(self, anchor_points, pred_dist)
                return _ops.bbox_decode(anchor_points, pred_dist)

            bbox_decode._cerb_reference = reference_bbox_decode
            patch_once(loss_mod.Loss, "bbox_decode", bbox_decode, "cerberusdet.utils.loss.Loss.bbox_decode")
        # the assigner the loss calls right after (utils/loss.py:160-162): three launches instead of ~60
        tal_mod = importlib.import_module("cerberusdet.utils.tal")
        if not hasattr(tal_mod.TaskAlignedAssigner.forward, "_cerb_reference"):
            reference_assign = tal_mod.TaskAlignedAssigner.forward

            @torch.no_grad()
            def forward(self, pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt):
                on_path = (pd_scores.is_cuda and pd_scores.dtype in (torch.float16, torch.float32) and pd_scores.dim() == 3
                           and pd_bboxes.dtype == torch.float32 and gt_bboxes.dtype == torch.float32 and gt_bboxes.dim() == 3
                           and 0 < gt_bboxes.size(1) <= 1024 and self.topk <= min(16, pd_scores.size(1))
                           and pd_scores.size(2) == self.num_classes)
                if not on_path:  # CPU tensors, no boxes at all (the reference's early return), exotic shapes
                    return reference_assign(self, pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt)
                self.bs, self.n_max_boxes = pd_scores.size(0), gt_bboxes.size(1)  # attributes the reference sets (tal.py:86-87)
                return _ops.tal_assign(pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt, self.topk,
                                       self.num_classes, self.alpha, self.beta, self.eps)

            forward._cerb_reference = reference_assign
            patch_once(tal_mod.TaskAlignedAssigner, "forward", forward, "cerberusdet.utils.tal.TaskAlignedAssigner.forward")
        # make_anchors is rebuilt on every loss call (utils/loss.py:149: ~12 small launches); the result depends on the
        # feature shapes, strides, dtype and device only
        if not hasattr(loss_mod.make_anchors, "_cerb_reference"):
            reference_make_anchors = loss_mod.make_anchors
            cache = {}

            def make_anchors(feats, strides, grid_cell_offset=0.5):
                st = strides.tolist() if torch.is_tensor(strides) and not strides.is_cuda else None
                if st is None or feats is None:  # (a device-resident stride tensor would cost a sync per call to key on)
                    return reference_make_anchors(feats, strides, grid_cell_offset)
                key = (tuple(tuple(f.shape[2:]) for f in feats[: len(st)]), tuple(st), feats[0].dtype, feats[0].device, float(grid_cell_offset))
                hit = cache.get(key)
                if hit is None:
                    if len(cache) > 16:
                        cache.clear()
                    hit = cache[key] = reference_make_anchors(feats, strides, grid_cell_offset)
                return hit

            make_anchors._cerb_reference = reference_make_anchors
            patch_once(loss_mod, "make_anchors", make_anchors, "cerberusdet.utils.loss.make_anchors")
    if loss:
        from . import ops as _ops

        loss_mod = importlib.import_module("cerberusdet.utils.loss")
        if not hasattr(loss_mod.BboxLoss.forward, "_cerb_reference"):
            reference_bbox_loss = loss_mod.BboxLoss.forward

            def bbox_loss_forward(self, pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum,
                                  fg_mask):
                tensors = (pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, fg_mask)
                on_path = (self.use_dfl and self.reg_max == 15 and all(t.is_cuda for t in tensors) and pred_dist.dim() == 3
                           and pred_dist.shape[-1] == 64 and fg_mask.dtype == torch.bool
                           and target_bboxes.dtype == torch.float32 and target_scores.dtype == torch.float32
                           and pred_bboxes.dtype == pred_dist.dtype and anchor_points.dtype == pred_dist.dtype)
                if on_path and torch.is_autocast_enabled("cuda"):
                    # fp16 autocast: half predictions, fp32 targets -- the kernels' half mode
                    on_path = pred_dist.dtype == torch.float16 and torch.get_autocast_dtype("cuda") == torch.float16
                elif on_path:
                    on_path = pred_dist.dtype == torch.float32
                if not on_path:  # CPU tensors, use_dfl=False, reg_max != 15, other dtype mixes: the reference's own code
                    return reference_bbox_loss(self, pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores,
                                               target_scores_sum, fg_mask)
                return _ops.bbox_loss(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum,
                                      fg_mask)

            bbox_loss_forward._cerb_reference = reference_bbox_loss
            patch_once(loss_mod.BboxLoss, "forward", bbox_loss_forward, "cerberusdet.utils.loss.BboxLoss.forward")
    if val:
        from . import val_stats as _val_stats

        val_mod = importlib.import_module("cerberusdet.val")
        if not hasattr(val_mod.process_batch, "_cerb_reference"):
            patch_once(val_mod, "process_batch", _val_stats.make_process_batch(val_mod.process_batch),
                       "cerberusdet.val.process_batch")
    if metrics:
        from . import val_stats as _val_stats

        metrics_mod = importlib.import_module("cerberusdet.utils.metrics")
        cur = metrics_mod.ap_per_class
        ap_per_class = cur if hasattr(cur, "_cerb_reference") else _val_stats.make_ap_per_class(cur)
        for modname, mod in list(sys.modules.items()):
            if (modname == "cerberusdet" or modname.startswith("cerberusdet.")) and hasattr(mod, "ap_per_class") \
                    and mod.ap_per_class is ap_per_class._cerb_reference:
                patch_once(mod, "ap_per_class", ap_per_class, f"{modname}.ap_per_class")
    if not done["patched"]:
        return {"already": ["installed"]}
    return done


def uninstall() -> None:
    while _saved:
        obj, name, value = _saved.pop()
        setattr(obj, name, value)
