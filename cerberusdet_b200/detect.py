"""Drop-in for the eval branch of the reference ``Detect.forward``
(cerberusdet/models/yolo.py:87-100).

The reference class must stay the class that checkpoints were pickled with
(utils/models_manager.py:296-308, models/experimental.py:112-122), so nothing here
subclasses it: ``detect_forward`` is bound onto the existing class by
``cerberusdet_b200.patch.install()``.  It takes over exactly one thing -- the decode of
CUDA tensors in eval mode; training mode and non-CUDA tensors run the reference's own
method untouched.
"""
from __future__ import annotations

import torch

from .ops import decode_heads

_RAW_FLAG = "_cerb_raw_heads"  # set by inference.raw_heads(): return the per-level tensors undecoded
_FUSE_FLAG = "_cerb_fuse_tail"  # set by inference.raw_heads(fuse=True): stop BEFORE the last 1x1 convolutions when possible
_STRIDES_ATTR = "_cerb_strides"  # (key, python floats): the head's strides without a device sync per forward


def head_strides(head):
    """``head.stride`` as Python floats.  ``attempt_load(..., map_location=device)`` leaves that tensor on the GPU, where
    every ``float()`` is a blocking device->host copy behind the queued conv towers -- so the floats are read once and
    kept on the module, keyed by the tensor object and its version (a replaced or rewritten stride is re-read)."""
    st = head.stride
    key = (id(st), getattr(st, "_version", 0)) if torch.is_tensor(st) else None
    ent = getattr(head, _STRIDES_ATTR, None)
    if ent is None or ent[0] != key or key is None:
        vals = tuple(float(v) for v in (st.detach().cpu().tolist() if torch.is_tensor(st) else st))
        ent = (key, vals)
        object.__setattr__(head, _STRIDES_ATTR, ent)
    return ent[1]


def _level_cat(self, x):
    # the conv towers belong to the model, not to this path (yolo.py:89-90)
    for i in range(self.nl):
        x[i] = torch.cat((self.cv2[i](x[i]), self.cv3[i](x[i])), 1)
    return x


class SplitHeads:
    """Raw heads of one task with the channel concat of models/yolo.py:89-90 left out: ``box[l]`` = cv2[l]'s output
    ``[B, 64, H_l, W_l]``, ``cls[l]`` = cv3[l]'s ``[B, nc, H_l, W_l]``.  ``ops.decode_heads_split`` reads both."""

    __slots__ = ("box", "cls")

    def __init__(self, box, cls):
        self.box, self.cls = box, cls


class FusedHeads:
    """One task's head stopped one layer earlier still: ``box_feat[l]`` / ``cls_feat[l]`` are the INPUTS of the last 1x1
    convolutions ``cv2[l][-1]`` / ``cv3[l][-1]`` (models/yolo.py:81-84); ``ops.head_tail`` runs those convolutions, the
    concat and the decode in one tcgen05 kernel (SURVEY 8f row 3)."""

    __slots__ = ("box_feat", "cls_feat", "head")

    def __init__(self, box_feat, cls_feat, head):
        self.box_feat, self.cls_feat, self.head = box_feat, cls_feat, head

    def to_split(self):
        """Run the last convolutions the ordinary way (mixed batches of fusable and unfusable heads)."""
        h = self.head
        return SplitHeads([h.cv2[i][-1](f) for i, f in enumerate(self.box_feat)], [h.cv3[i][-1](f) for i, f in enumerate(self.cls_feat)])

    def weights(self):
        h = self.head
        n = len(self.box_feat)
        return ([h.cv2[i][-1].weight for i in range(n)], [h.cv2[i][-1].bias for i in range(n)],
                [h.cv3[i][-1].weight for i in range(n)], [h.cv3[i][-1].bias for i in range(n)])


def can_fuse_tail(head, x) -> bool:
    """The fused kernel's preconditions (include/cerb_post.h: cerb_head_tail): half tensors, every level's H*W a multiple
    of 8, both towers ending in a plain biased 1x1 ``nn.Conv2d`` whose input width is a multiple of 16, nc <= 192."""
    if x[0].dtype != torch.float16 or head.nc > 192 or getattr(head, "reg_max", 16) != 16:
        return False
    for i in range(head.nl):
        if (x[i].shape[2] * x[i].shape[3]) % 8:
            return False
        for seq, n_out in ((head.cv2[i], 64), (head.cv3[i], head.nc)):
            last = seq[-1] if isinstance(seq, torch.nn.Sequential) and len(seq) > 1 else None
            if not (isinstance(last, torch.nn.Conv2d) and last.kernel_size == (1, 1) and last.stride == (1, 1)
                    and last.padding == (0, 0) and last.groups == 1 and last.bias is not None
                    and last.out_channels == n_out and last.in_channels % 16 == 0 and last.weight.dtype == torch.float16):
                return False
    return True


def detect_forward(self, x):
    """``forward(self, x: list[Tensor]) -> (y, x)`` | ``y`` (export) | ``x`` (training).

    ``y`` is ``[B, 4+nc, A]`` in the input dtype, rows cx, cy, w, h (pixels) then sigmoid
    scores -- the reference layout.  ``x`` is mutated in place with the per-level
    concatenations exactly like the reference does (yolo.py:89-90).
    """
    reference_forward = type(self)._cerb_reference_forward
    if self.training or not x[0].is_cuda or x[0].dtype not in (torch.float16, torch.bfloat16, torch.float32):
        return reference_forward(self, x)
    shape = x[0].shape  # BCHW before the convs: the reference's anchor-cache key (yolo.py:88,93)
    if getattr(self, _RAW_FLAG, False):
        # inference engine: nobody reads the concatenated raw tensors, so the towers' outputs are handed over as they
        # are and the decode kernel reads box and class channels from their own tensors (no torch.cat copy) -- or, fused
        # mode, the towers stop before their last 1x1 convolution and one kernel does the rest
        if getattr(self, _FUSE_FLAG, False) and can_fuse_tail(self, x):
            return None, FusedHeads([self.cv2[i][:-1](x[i]) for i in range(self.nl)],
                                    [self.cv3[i][:-1](x[i]) for i in range(self.nl)], self)
        return None, SplitHeads([self.cv2[i](x[i]) for i in range(self.nl)], [self.cv3[i](x[i]) for i in range(self.nl)])
    x = _level_cat(self, x)
    if self.dynamic or self.shape != shape:
        # keep the instance attributes other code reads (and pickles) populated (yolo.py:93-95)
        from .anchors import make_anchor_tensors

        self.anchors, self.strides = make_anchor_tensors([t.shape[2:] for t in x], self.stride, x[0].dtype, x[0].device)
        self.shape = shape
    strides = head_strides(self)
    y = decode_heads([[t if t.is_contiguous() else t.contiguous() for t in x]], strides)[0]
    return y if self.export else (y, x)
