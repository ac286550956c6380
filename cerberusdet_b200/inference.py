"""Drop-in for the reference ``CerberusDetInference`` (cerberusdet/cerberusdet_inference.py:18-186).

Same constructor and ``predict`` signatures, same attributes, same return structure
(``List[List[Dict{box, score, label, label_name, task}]]``).  Inside, the per-task Python loop of
the reference (``:125-135``: T calls of ``non_max_suppression``, each looping over the B images with
~25 launches and ~4 host syncs per image) becomes: one decode launch for all task heads, one NMS
launch for all (task, image) segments, one device->host copy.  The tail after NMS (``:140-184``) is
host code (``cross_task.py``), as in the reference.
"""
from __future__ import annotations

import contextlib
import os
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch

from . import cross_task
from ._lib import CERB_ENOSPC, CerbLibraryError
from .detect import _FUSE_FLAG, _RAW_FLAG, FusedHeads, SplitHeads, head_strides
from .ops import cross_task_merge, decode_heads, decode_heads_split, head_tail, nms_batched


def _reference_nms():
    """The reference's own ``non_max_suppression`` (the saved original when ``patch.install()`` rebound the name)."""
    try:
        from cerberusdet.utils import general
    except ImportError as exc:  # stand-alone use without the reference package: there is no CPU path of ours
        raise TypeError("non-CUDA predictions need the reference package (cerberusdet) for its CPU non_max_suppression; "
                        "cerberusdet_b200 has no CPU path") from exc
    fn = general.non_max_suppression
    return getattr(fn, "_cerb_reference", fn)


@contextlib.contextmanager
def raw_heads(model, fuse: bool = False):
    """While active, patched Detect heads return ``(None, SplitHeads)`` -- the conv towers' outputs, not even
    concatenated -- so that all task heads can be decoded together in one launch.  ``fuse=True``: heads that meet the
    fused kernel's preconditions (``detect.can_fuse_tail``) stop before their last 1x1 convolutions and return
    ``(None, FusedHeads)`` instead."""
    heads = [m for m in model.modules() if hasattr(type(m), "_cerb_reference_forward")]
    for m in heads:
        setattr(m, _RAW_FLAG, True)
        setattr(m, _FUSE_FLAG, bool(fuse))
    try:
        yield heads
    finally:
        for m in heads:
            setattr(m, _RAW_FLAG, False)
            setattr(m, _FUSE_FLAG, False)


class CerberusDetInference:
    def __init__(
        self,
        weights: Optional[str] = None,
        device: str = "",
        conf_thres: float = 0.25,
        iou_thres: float = 0.45,
        iou_thres_between_tasks: float = 0.8,
        half: bool = False,
        img_size: int = 640,
        model=None,
    ):
        """``model=`` (extension): use an already built CerberusDet-like module instead of loading
        ``weights`` -- anything whose forward returns ``{task: (pred_or_None, levels)}``."""
        self.conf_thres = conf_thres
        self.iou_thres = iou_thres
        self.iou_thres_between_tasks = iou_thres_between_tasks
        # extension: run the heads' last 1x1 convolutions inside the decode kernel (ops.head_tail) whenever the model
        # is half and its shapes allow it; set to False to keep the convolutions in cuDNN
        self.fuse_head_tail = os.environ.get("CERB_HEAD_TAIL", "1") != "0"
        if model is None:
            from . import patch

            patch.install()
            from cerberusdet.models.experimental import attempt_load  # reference loader (:37)
            from cerberusdet.utils.general import check_img_size
            from cerberusdet.utils.torch_utils import select_device

            self.device = select_device(device)
            model = attempt_load(weights, map_location=self.device)
        else:
            check_img_size = None
            self.device = torch.device(device) if device else next(model.parameters()).device
        self.half = half & (self.device.type != "cpu")
        self.model = model
        if self.half:
            self.model.half()
        self.model.eval()
        self.stride = int(self.model.stride.max())
        self.names: Dict[str, List[str]] = self.model.names if hasattr(self.model, "names") else self.model.module.names
        self.categories_inds_map, self.all_class_names = cross_task.category_maps(self.names)
        # warm-up forward, as in the reference (:51-54)
        size = check_img_size(img_size, s=self.stride) if check_img_size else img_size
        p = next(self.model.parameters())
        self.model(torch.zeros(1, 3, size, size, device=self.device, dtype=p.dtype))

    _get_categories_map = staticmethod(cross_task.category_maps)

    def _head_strides(self, n_levels: int) -> List[float]:
        head = getattr(self, "_cerb_head", None)
        if head is None:
            head = next((m for m in self.model.modules()
                         if hasattr(type(m), "_cerb_reference_forward") or type(m).__name__ == "Detect"), self.model)
            self._cerb_head = head
        return list(head_strides(head))[:n_levels]

    @torch.no_grad()
    def predict(
        self,
        tensor: torch.Tensor,
        original_shape: Union[Tuple[int, int], List[Tuple[int, int]], None] = None,
        max_det: int = 300,
        agnostic_nms: bool = False,
        conf_thres: float = None,
        iou_thres: float = None,
        iou_thres_between_tasks: float = None,
    ) -> List[List[Dict]]:
        conf_thres = self.conf_thres if conf_thres is None else conf_thres
        iou_thres = self.iou_thres if iou_thres is None else iou_thres
        between = self.iou_thres_between_tasks if iou_thres_between_tasks is None else iou_thres_between_tasks

        # 1. forward: every head hands over its raw per-level tensors
        with raw_heads(self.model, fuse=self.fuse_head_tail):
            all_out = self.model(tensor)
        # task order = the order of self.names (categories_inds_map), which is the order the reference's
        # nms_between_tasks regroups the rows in (utils/general.py:497-505) -- the scan below is order-dependent
        tasks = [t for t in self.categories_inds_map if t in all_out] + [t for t in all_out if t not in self.categories_inds_map]
        preds = [all_out[t][0] for t in tasks]
        if any(p is None for p in preds):  # raw mode was honoured: decode all heads in one launch
            levels = [all_out[t][1] for t in tasks]
            if any(isinstance(lv, FusedHeads) for lv in levels) and not all(isinstance(lv, FusedHeads) for lv in levels):
                levels = [lv.to_split() if isinstance(lv, FusedHeads) else lv for lv in levels]
            fused = None
            if all(isinstance(lv, FusedHeads) for lv in levels):  # last 1x1 convs + concat + decode in one kernel
                strides = self._head_strides(len(levels[0].box_feat))
                w = [lv.weights() for lv in levels]
                try:
                    fused = head_tail([lv.box_feat for lv in levels], [lv.cls_feat for lv in levels], [x[0] for x in w],
                                      [x[1] for x in w], [x[2] for x in w], [x[3] for x in w], strides)
                except CerbLibraryError as exc:
                    # the weights and two ring stages of the launch do not fit shared memory (wide c3 at large nc).
                    # That depends on every head of the launch, so the kernel decides; these heads run unfused from now on
                    if exc.code != CERB_ENOSPC:
                        raise
                    self.fuse_head_tail = False
                    levels = [lv.to_split() for lv in levels]
            if fused is not None:
                preds = fused
            elif all(isinstance(lv, SplitHeads) for lv in levels):  # patched heads: no channel concat was made
                strides = self._head_strides(len(levels[0].box))
                preds = decode_heads_split([lv.box for lv in levels], [lv.cls for lv in levels], strides)
            else:
                preds = decode_heads(levels, self._head_strides(len(levels[0])))
        bsz = tensor.shape[0]
        on_path = all(p.is_cuda and p.dtype in (torch.float16, torch.bfloat16, torch.float32) for p in preds)
        if on_path:
            # 2. one NMS launch over all (task, image) segments
            dets, counts = nms_batched(preds, conf_thres, iou_thres, agnostic=agnostic_nms, max_det=max_det)
        else:
            # a CPU (or otherwise off-path) model: the reference's own per-task NMS, as patch.install() promises --
            # the patch never changes what a non-CUDA run computes (cerberusdet_inference.py:125-135)
            ref_nms = _reference_nms()
            rows = [ref_nms(p, conf_thres, iou_thres, agnostic=agnostic_nms, max_det=max_det) for p in preds]
            dets = torch.zeros((len(tasks), bsz, max_det, 6), dtype=torch.float32)
            counts = torch.zeros((len(tasks), bsz), dtype=torch.int32)
            for k, per_image in enumerate(rows):
                for i, r in enumerate(per_image):
                    dets[k, i, : r.shape[0]] = r.detach().float().cpu()
                    counts[k, i] = r.shape[0]
        shapes = None
        if original_shape is not None:
            shapes = original_shape if isinstance(original_shape, list) else [original_shape] * bsz
        results = []
        if on_path and max_det <= 65535:
            # 3. cross-task merge + rescale on the GPU (one launch, one CTA per image), then ONE D2H copy
            offsets = [min(self.categories_inds_map[t].values()) if self.categories_inds_map[t] else 0 for t in tasks]
            scale = None
            if shapes is not None:
                net_h, net_w = int(tensor.shape[2]), int(tensor.shape[3])
                rows = []
                for (oh, ow) in shapes:
                    gain = min(net_h / oh, net_w / ow)  # utils/general.py:330-331
                    rows.append([gain, (net_w - ow * gain) / 2, (net_h - oh * gain) / 2, float(ow), float(oh)])
                scale = torch.tensor(rows, dtype=torch.float64).to(torch.float32)
            merged, mcounts = cross_task_merge(dets, counts, offsets, between, scale)
            merged_h, mcounts_h = merged.cpu(), mcounts.cpu()
            per_image = [merged_h[i, : int(mcounts_h[i])] for i in range(bsz)]
        else:
            # off-path (CPU model): host tail, as in the reference
            dets_h, counts_h = dets.cpu(), counts.cpu()
            per_image = []
            for i in range(bsz):
                per_task = {t: dets_h[k, i, : int(counts_h[k, i])] for k, t in enumerate(tasks)}
                det = cross_task.combine_tasks(per_task, self.categories_inds_map)
                det = cross_task.suppress_between_tasks(det, self.categories_inds_map, between)
                if len(det) > 0 and shapes is not None:
                    det[:, :4] = cross_task.rescale_boxes(tensor.shape[2:], det[:, :4], shapes[i]).round()
                per_image.append(det)
        for det in per_image:
            image_results = []
            for *xyxy, conf, cls in det.tolist():
                c = int(cls)
                task_name = next((t for t, m in self.categories_inds_map.items() if c in m.values()), "unknown")
                image_results.append({"box": [int(v) for v in xyxy], "score": float(conf), "label": c,
                                      "label_name": self.all_class_names[c], "task": task_name})
            results.append(image_results)
        return results
