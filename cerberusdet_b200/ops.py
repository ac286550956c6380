"""torch custom ops over the C ABI of ``libcerb_post.so``: ``cerb::decode``, ``cerb::decode_split``, ``cerb::nms``,
``cerb::nms_out`` (writes into caller buffers) and ``cerb::decode_nms``.  The Python wrappers below (``decode_heads``,
``nms_batched``, ...) dispatch through these registered ops, so eager calls, CUDA-graph capture and ``torch.compile``
all reach the same kernels.

PyTorch is plumbing here (device memory, streams); the arithmetic is in ``csrc/decode_pipe.cu`` / ``csrc/decode.cu``
and ``csrc/nms.cu``.  Inputs must be CUDA tensors: a CPU tensor raises ``TypeError`` -- there is no fallback.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib

MAX_WH = 7680.0  # reference utils/general.py:415
MAX_NMS = 30000  # reference utils/general.py:416

_DTYPES = {torch.float16: _lib.CERB_F16, torch.float32: _lib.CERB_F32}


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"cerberusdet_b200 supports float16 and float32 tensors, got {t.dtype}") from None


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise TypeError(f"{what} must be a CUDA tensor (cerberusdet_b200 has no CPU path), got device {t.device}")


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _dense16(x: torch.Tensor) -> torch.Tensor:
    """Contiguous and 16-byte aligned (a contiguous view at an odd storage offset is copied)."""
    x = x.contiguous()
    return x if x.data_ptr() % 16 == 0 else x.clone(memory_format=torch.contiguous_format)


def _summary_len(level_sizes: Sequence[int], elt: int) -> int:
    """Row length of the score summary (``cerb_summary_row_len``), or 0 when a level rules the 128-bit path out."""
    V = 16 // elt
    if any(n % V for n in level_sizes):
        return 0
    n = sum(level_sizes) // V
    return (n + V - 1) // V * V


def _decode_impl(levels: Sequence[torch.Tensor], nc: Sequence[int], strides: Sequence[float],
                 cls_levels: Optional[Sequence[torch.Tensor]] = None,
                 out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
    """Returns ``[y_0 .. y_{T-1}, smax_0 .. smax_{T-1}]``; the score summaries ``smax_t`` are empty
    tensors when the shapes do not allow them (see include/cerb_post.h).  With ``cls_levels`` the heads are split:
    ``levels`` hold the 64 box channels, ``cls_levels`` the class channels (``cerb_decode_split``)."""
    lib = _lib.load()
    T = len(nc)
    if T == 0 or len(levels) % T:
        raise ValueError("levels must hold T*L tensors, task-major")
    L = len(levels) // T
    if cls_levels is not None and len(cls_levels) != len(levels):
        raise ValueError("cls_levels must hold one tensor per box tensor")
    if len(strides) != L:
        raise ValueError(f"expected {L} strides, got {len(strides)}")
    first = levels[0]
    _require_cuda(first, "head tensors")
    code = _dtype_code(first)
    B = first.shape[0]
    H = [int(levels[l].shape[2]) for l in range(L)]
    W = [int(levels[l].shape[3]) for l in range(L)]
    A = sum(h * w for h, w in zip(H, W))
    lv = []
    for t in range(T):
        for l in range(L):
            x = levels[t * L + l]
            if x.device != first.device or x.dtype != first.dtype:
                raise TypeError("all head tensors must share device and dtype")
            cbox = 64 if cls_levels is not None else 64 + nc[t]
            if tuple(x.shape) != (B, cbox, H[l], W[l]):
                raise ValueError(f"task {t} level {l}: expected {(B, cbox, H[l], W[l])}, got {tuple(x.shape)}")
            lv.append(_dense16(x))
    cl = []
    if cls_levels is not None:
        for t in range(T):
            for l in range(L):
                c = cls_levels[t * L + l]
                if c.device != first.device or c.dtype != first.dtype:
                    raise TypeError("all head tensors must share device and dtype")
                if tuple(c.shape) != (B, nc[t], H[l], W[l]):
                    raise ValueError(f"task {t} level {l}: expected class tensor {(B, nc[t], H[l], W[l])}, got {tuple(c.shape)}")
                cl.append(_dense16(c))
    # the score summary exists exactly when every level allows 16-byte vectors (inputs and outputs here are 16-byte
    # aligned by construction), so its shape is a function of the shapes alone -- the fake kernel below relies on that
    R = _summary_len([h * w for h, w in zip(H, W)], first.element_size())
    assert R == 0 or R == int(lib.cerb_summary_row_len(A, code))
    if out is None:
        ys = [torch.empty((B, 4 + nc[t], A), dtype=first.dtype, device=first.device) for t in range(T)]
        sm = [torch.empty((B, nc[t], R), dtype=first.dtype, device=first.device) for t in range(T)]
    else:  # caller-provided static buffers [y_0 .. y_{T-1}, smax_0 .. smax_{T-1}] (CUDA graphs, pipelines)
        if len(out) != 2 * T:
            raise ValueError("out= must hold T prediction buffers followed by T score-summary buffers")
        ys, sm = list(out[:T]), list(out[T:])
        for t in range(T):
            ok = (tuple(ys[t].shape) == (B, 4 + nc[t], A) and tuple(sm[t].shape) == (B, nc[t], R)
                  and all(z.dtype == first.dtype and z.device == first.device and z.is_contiguous() and z.data_ptr() % 16 == 0
                          for z in (ys[t], sm[t])))
            if not ok:
                raise ValueError(f"out= buffers of task {t} must be contiguous, 16-byte aligned [B,4+nc,A] / [B,nc,{R}] {first.dtype} tensors")
    written = ctypes.c_int(0)
    tail = (_lib.int_array(list(nc)), T, L, B, _lib.int_array(H), _lib.int_array(W),
            _lib.float_array([float(s) for s in strides]), code, _lib.ptr_array([y.data_ptr() for y in ys]),
            _lib.ptr_array([x.data_ptr() for x in sm]), ctypes.byref(written), _stream_ptr(first.device))
    with torch.cuda.device(first.device):
        if cls_levels is None:
            rc = lib.cerb_decode(_lib.ptr_array([x.data_ptr() for x in lv]), *tail)
        else:
            rc = lib.cerb_decode_split(_lib.ptr_array([x.data_ptr() for x in lv]), _lib.ptr_array([x.data_ptr() for x in cl]), *tail)
    _lib.check(rc)
    if bool(written.value) != (R > 0 and B > 0):
        raise _lib.CerbLibraryError("cerb_decode: score summary state differs from what the shapes imply")
    return ys + sm


@torch.library.custom_op("cerb::decode", mutates_args=())
def decode_op(levels: Sequence[torch.Tensor], nc: Sequence[int], strides: Sequence[float]) -> List[torch.Tensor]:
    """``[y_0 .. y_{T-1}, smax_0 .. smax_{T-1}]`` from ``T*L`` raw head tensors (task-major); ``smax_t`` has a last
    dimension of 0 when the shapes rule the score summary out."""
    return _decode_impl(levels, nc, strides)


@torch.library.custom_op("cerb::decode_out", mutates_args=("out",))
def decode_out_op(levels: Sequence[torch.Tensor], nc: Sequence[int], strides: Sequence[float], out: Sequence[torch.Tensor]) -> None:
    """``cerb::decode`` writing into caller-provided buffers ``[y_0 .. y_{T-1}, smax_0 .. smax_{T-1}]``."""
    _decode_impl(levels, nc, strides, out=out)


@decode_out_op.register_fake
def _(levels, nc, strides, out):
    return None


@torch.library.custom_op("cerb::decode_split", mutates_args=())
def decode_split_op(box_levels: Sequence[torch.Tensor], cls_levels: Sequence[torch.Tensor], nc: Sequence[int],
                    strides: Sequence[float]) -> List[torch.Tensor]:
    """``cerb::decode`` on split heads (box channels and class channels in their own tensors)."""
    return _decode_impl(box_levels, nc, strides, cls_levels=cls_levels)


def _decode_fake(levels, nc, strides):
    T = len(nc)
    L = len(levels) // T
    B = levels[0].shape[0]
    sizes = [levels[l].shape[2] * levels[l].shape[3] for l in range(L)]
    A = sum(sizes)
    R = _summary_len(sizes, levels[0].element_size())
    return [levels[0].new_empty((B, 4 + nc[t], A)) for t in range(T)] + [
        levels[0].new_empty((B, nc[t], R)) for t in range(T)]


@decode_op.register_fake
def _(levels, nc, strides):
    return _decode_fake(levels, nc, strides)


@decode_split_op.register_fake
def _(box_levels, cls_levels, nc, strides):
    return _decode_fake(box_levels, nc, strides)


def _nms_impl(
    preds: Sequence[torch.Tensor],
    conf_thres: float,
    iou_thres: float,
    classes: Optional[Sequence[int]],
    agnostic: bool,
    multi_label: bool,
    max_det: int,
    max_nms: int,
    max_wh: float,
    smax: Sequence[torch.Tensor],
    out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
    stats: Optional[torch.Tensor] = None,
    deliver=None,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """``deliver`` = a ``_lib.Delivery`` (``cerb_delivery``, include/cerb_post.h) built by ``shard.PeerDelivery``: this
    launch's part in the multi-GPU delivery (``cerb_nms_deliver``)."""
    lib = _lib.load()
    T = len(preds)
    first = preds[0]
    _require_cuda(first, "prediction")
    code = _dtype_code(first)
    B, A = int(first.shape[0]), int(first.shape[2])
    ncs, ps = [], []
    for p in preds:
        if p.device != first.device or p.dtype != first.dtype or p.dim() != 3 or p.shape[0] != B or p.shape[2] != A:
            raise ValueError("all predictions must be [B, 4+nc, A] on one device with one dtype")
        ncs.append(int(p.shape[1]) - 4)
        ps.append(p.contiguous())
    dev = first.device
    if out is not None:
        dets, counts = out
        if (tuple(dets.shape) != (T, B, max_det, 6) or dets.dtype != torch.float32 or not dets.is_contiguous()
                or tuple(counts.shape) != (T, B) or counts.dtype != torch.int32 or not counts.is_contiguous()
                or dets.device != dev or counts.device != dev):
            raise ValueError("out= must be contiguous (dets[T,B,max_det,6] float32, counts[T,B] int32) on the input device")
    else:
        dets = torch.empty((T, B, max_det, 6), dtype=torch.float32, device=dev)  # the kernel writes every row
        counts = torch.empty((T, B), dtype=torch.int32, device=dev)
    ws_bytes = lib.cerb_nms_workspace_bytes(T, B, max_det)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
    cls_arr = _lib.int_array(list(classes)) if classes is not None else None
    sm_arr = None
    if len(smax) == T:
        R = int(lib.cerb_summary_row_len(A, code))
        ok = R > 0 and all(s.is_contiguous() and s.dtype == first.dtype and s.device == dev
                           and tuple(s.shape) == (B, n, R) for s, n in zip(smax, ncs))
        ok = ok and all(p.data_ptr() == q.data_ptr() for p, q in zip(preds, ps))  # no hidden copies
        if ok:
            sm_arr = _lib.ptr_array([s.data_ptr() for s in smax])
    if stats is not None and (stats.dtype != torch.int64 or tuple(stats.shape) != (T, B, 2) or stats.device != dev or not stats.is_contiguous()):
        raise ValueError("stats must be a contiguous int64 [T, B, 2] tensor on the input device")
    head = (_lib.ptr_array([p.data_ptr() for p in ps]), _lib.int_array(ncs), T, B, A, code,
            float(conf_thres), float(iou_thres), cls_arr, len(classes) if classes is not None else 0,
            int(bool(agnostic)), int(bool(multi_label)), int(max_det), int(max_nms), float(max_wh),
            sm_arr,
            dets.data_ptr(), counts.data_ptr(), ws.data_ptr() if ws is not None else None, ws_bytes)
    with torch.cuda.device(dev):
        if deliver is not None:
            if stats is not None or out is None:
                raise ValueError("deliver= needs out= (the peer-mapped slot) and excludes stats=")
            rc = lib.cerb_nms_deliver(*head, ctypes.byref(deliver), _stream_ptr(dev))
        else:
            rc = lib.cerb_nms_stats(*head, stats.data_ptr() if stats is not None else None, _stream_ptr(dev))
    _lib.check(rc)
    return dets, counts


@torch.library.custom_op("cerb::nms", mutates_args=())
def nms_op(
    preds: Sequence[torch.Tensor],
    conf_thres: float,
    iou_thres: float,
    classes: Optional[Sequence[int]],
    agnostic: bool,
    multi_label: bool,
    max_det: int,
    max_nms: int,
    max_wh: float,
    smax: Sequence[torch.Tensor],
) -> Tuple[torch.Tensor, torch.Tensor]:
    """torch custom op over ``_nms_impl``."""
    return _nms_impl(preds, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh, smax)


@nms_op.register_fake
def _(preds, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh, smax):
    T, B = len(preds), preds[0].shape[0]
    return (preds[0].new_empty((T, B, max_det, 6), dtype=torch.float32),
            preds[0].new_empty((T, B), dtype=torch.int32))


@torch.library.custom_op("cerb::nms_out", mutates_args=("dets", "counts"))
def nms_out_op(
    preds: Sequence[torch.Tensor],
    conf_thres: float,
    iou_thres: float,
    classes: Optional[Sequence[int]],
    agnostic: bool,
    multi_label: bool,
    max_det: int,
    max_nms: int,
    max_wh: float,
    smax: Sequence[torch.Tensor],
    dets: torch.Tensor,
    counts: torch.Tensor,
) -> None:
    """``cerb::nms`` writing into caller-provided ``dets[T,B,max_det,6]`` / ``counts[T,B]`` (a gather buffer, a peer
    GPU's mapped memory, a static CUDA-graph buffer)."""
    _nms_impl(preds, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh, smax, (dets, counts))


@nms_out_op.register_fake
def _(preds, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh, smax, dets, counts):
    return None


@torch.library.custom_op("cerb::decode_nms", mutates_args=())
def decode_nms_op(
    levels: Sequence[torch.Tensor],
    nc: Sequence[int],
    strides: Sequence[float],
    conf_thres: float,
    iou_thres: float,
    classes: Optional[Sequence[int]],
    agnostic: bool,
    multi_label: bool,
    max_det: int,
    max_nms: int,
    max_wh: float,
) -> List[torch.Tensor]:
    """Raw head tensors -> ``[dets[T,B,max_det,6], counts[T,B], y_0 .. y_{T-1}]`` in ONE library call
    (``cerb_decode_nms``: both kernels back to back on the current stream, no host work in between)."""
    return _decode_nms_impl(levels, nc, strides, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh)


@decode_nms_op.register_fake
def _(levels, nc, strides, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh):
    T = len(nc)
    B = levels[0].shape[0]
    ys = _decode_fake(levels, nc, strides)[:T]
    return [levels[0].new_empty((T, B, max_det, 6), dtype=torch.float32), levels[0].new_empty((T, B), dtype=torch.int32)] + ys


# ----------------------------------------------------------------------------- score-summary hand-over
_SUMMARY_ATTR = "_cerb_score_summary"


def _remember_summary(y: torch.Tensor, smax: torch.Tensor) -> None:
    """Attach ``smax`` (the decode kernel's score summary of ``y`` as it is right now) to the tensor OBJECT ``y``.
    ``find_summary`` hands it back only for this very object while its version counter is unchanged, so a view, a copy
    or a tensor written in place since never gets a stale summary; the summary dies with ``y``.

    Not tracked (PyTorch keeps no version there): tensors created under ``torch.inference_mode()`` -- they simply get no
    summary and NMS scans the scores itself -- and writes that bypass autograd's bookkeeping (``y.data[...] = ...``, a
    foreign kernel writing through ``data_ptr()``): pass ``use_summary=False`` to ``nms_batched`` after such a write."""
    if y.is_inference():
        return
    setattr(y, _SUMMARY_ATTR, (smax, y._version, y.data_ptr()))


def find_summary(y: torch.Tensor):
    ent = getattr(y, _SUMMARY_ATTR, None)
    if ent is None or y.is_inference():
        return None
    smax, version, ptr = ent
    if y._version != version or y.data_ptr() != ptr or not y.is_contiguous():
        return None
    return smax


# ----------------------------------------------------------------------------- friendly wrappers
def decode_buffers(task_levels: Sequence[Sequence[torch.Tensor]]) -> List[torch.Tensor]:
    """Static output buffers for ``decode_heads(..., out=...)``: ``[y_0 .. y_{T-1}, smax_0 .. smax_{T-1}]``."""
    first = task_levels[0][0]
    B = int(first.shape[0])
    sizes = [int(x.shape[2]) * int(x.shape[3]) for x in task_levels[0]]
    A, R = sum(sizes), _summary_len(sizes, first.element_size())
    ncs = [int(lv[0].shape[1]) - 64 for lv in task_levels]
    return ([torch.empty((B, 4 + n, A), dtype=first.dtype, device=first.device) for n in ncs]
            + [torch.empty((B, n, R), dtype=first.dtype, device=first.device) for n in ncs])


def decode_heads(task_levels: Sequence[Sequence[torch.Tensor]], strides: Sequence[float],
                 out: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
    """``task_levels[t][l]`` = raw head tensor ``[B, 64+nc_t, H_l, W_l]`` -> ``y_t [B, 4+nc_t, A]``
    for every task in one launch (reference Detect.forward eval branch, models/yolo.py:93-99).
    The kernel also leaves a score summary per task, remembered for ``nms_batched``.
    ``out=decode_buffers(task_levels)`` writes into caller-owned static buffers."""
    flat = [x for lv in task_levels for x in lv]
    nc = [int(lv[0].shape[1]) - 64 for lv in task_levels]
    if out is not None:
        decode_out_op(flat, nc, [float(s) for s in strides], list(out))
    else:
        out = decode_op(flat, nc, [float(s) for s in strides])
    T = len(nc)
    ys, sms = out[:T], out[T:]
    for y, sm in zip(ys, sms):
        if sm.shape[-1]:
            _remember_summary(y, sm)
    return ys


def decode_heads_split(task_box_levels: Sequence[Sequence[torch.Tensor]], task_cls_levels: Sequence[Sequence[torch.Tensor]],
                       strides: Sequence[float]) -> List[torch.Tensor]:
    """``decode_heads`` on SPLIT heads: ``task_box_levels[t][l]`` = ``[B, 64, H_l, W_l]`` (the cv2 tower's output),
    ``task_cls_levels[t][l]`` = ``[B, nc_t, H_l, W_l]`` (cv3's) -- the reference's channel concat (models/yolo.py:89-90)
    is never materialised.  Same result, bit for bit, as ``decode_heads`` on the concatenated tensors."""
    nc = [int(lv[0].shape[1]) for lv in task_cls_levels]
    out = decode_split_op([x for lv in task_box_levels for x in lv], [x for lv in task_cls_levels for x in lv], nc,
                          [float(s) for s in strides])
    T = len(nc)
    ys, sms = out[:T], out[T:]
    for y, sm in zip(ys, sms):
        if sm.shape[-1]:
            _remember_summary(y, sm)
    return ys


def _head_tail_impl(box_feats: Sequence[torch.Tensor], cls_feats: Sequence[torch.Tensor], box_w: Sequence[torch.Tensor],
                    box_b: Sequence[torch.Tensor], cls_w: Sequence[torch.Tensor], cls_b: Sequence[torch.Tensor],
                    strides: Sequence[float], T: int) -> List[torch.Tensor]:
    """``cerb_head_tail`` on flat task-major lists of T*L tensors.  Returns ``[y_0 .. y_{T-1}, smax_0 .. smax_{T-1}]``."""
    lib = _lib.load()
    n = len(box_feats)
    if T <= 0 or n % T or any(len(z) != n for z in (cls_feats, box_w, box_b, cls_w, cls_b)):
        raise ValueError("head_tail: every list must hold T*L tensors, task-major")
    L = n // T
    if len(strides) != L:
        raise ValueError(f"expected {L} strides, got {len(strides)}")
    first = box_feats[0]
    _require_cuda(first, "head-tail inputs")
    if first.dtype != torch.float16:
        raise TypeError("head_tail runs on float16 tensors only (tcgen05 kind::f16); use the convolutions + decode_heads_split for float32")
    B = int(first.shape[0])
    H = [int(box_feats[l].shape[2]) for l in range(L)]
    W = [int(box_feats[l].shape[3]) for l in range(L)]
    A = sum(h * w for h, w in zip(H, W))
    c2 = [int(box_feats[t * L].shape[1]) for t in range(T)]
    c3 = [int(cls_feats[t * L].shape[1]) for t in range(T)]
    nc = [int(cls_w[t * L].shape[0]) for t in range(T)]
    keep = []  # dense copies (non-contiguous / misaligned inputs only) must outlive the launch

    def dense(x, shape, what, t, l):
        if x.device != first.device or x.dtype != first.dtype:
            raise TypeError("all head-tail tensors must share device and dtype")
        if tuple(x.shape) != shape and not (x.dim() == 4 and tuple(x.shape) == shape + (1, 1)):
            raise ValueError(f"task {t} level {l}: {what} expected {shape}, got {tuple(x.shape)}")
        d = _dense16(x.reshape(shape))
        if d.data_ptr() != x.data_ptr():
            keep.append(d)
        return d.data_ptr()

    ptrs = [[] for _ in range(6)]
    for t in range(T):
        for l in range(L):
            i = t * L + l
            ptrs[0].append(dense(box_feats[i], (B, c2[t], H[l], W[l]), "box features", t, l))
            ptrs[1].append(dense(cls_feats[i], (B, c3[t], H[l], W[l]), "class features", t, l))
            ptrs[2].append(dense(box_w[i], (64, c2[t]), "box weight", t, l))
            ptrs[3].append(dense(box_b[i], (64,), "box bias", t, l))
            ptrs[4].append(dense(cls_w[i], (nc[t], c3[t]), "class weight", t, l))
            ptrs[5].append(dense(cls_b[i], (nc[t],), "class bias", t, l))
    R = _summary_len([h * w for h, w in zip(H, W)], 2)
    ys = [torch.empty((B, 4 + nc[t], A), dtype=first.dtype, device=first.device) for t in range(T)]
    sm = [torch.empty((B, nc[t], R), dtype=first.dtype, device=first.device) for t in range(T)]
    written = ctypes.c_int(0)
    with torch.cuda.device(first.device):
        rc = lib.cerb_head_tail(*[_lib.ptr_array(p) for p in ptrs], _lib.int_array(c2), _lib.int_array(c3), _lib.int_array(nc),
                                T, L, B, _lib.int_array(H), _lib.int_array(W), _lib.float_array([float(s) for s in strides]),
                                _lib.CERB_F16, _lib.ptr_array([y.data_ptr() for y in ys]),
                                _lib.ptr_array([x.data_ptr() for x in sm]) if R else None, ctypes.byref(written),
                                _stream_ptr(first.device))
    _lib.check(rc)
    for x in keep:  # the kernel is only enqueued: keep temporaries alive on this stream
        x.record_stream(torch.cuda.current_stream(first.device))
    return ys + sm


@torch.library.custom_op("cerb::head_tail", mutates_args=())
def head_tail_op(box_feats: Sequence[torch.Tensor], cls_feats: Sequence[torch.Tensor], box_w: Sequence[torch.Tensor],
                 box_b: Sequence[torch.Tensor], cls_w: Sequence[torch.Tensor], cls_b: Sequence[torch.Tensor],
                 strides: Sequence[float], T: int) -> List[torch.Tensor]:
    return _head_tail_impl(box_feats, cls_feats, box_w, box_b, cls_w, cls_b, strides, T)


@head_tail_op.register_fake
def _(box_feats, cls_feats, box_w, box_b, cls_w, cls_b, strides, T):
    L = len(box_feats) // T
    first = box_feats[0]
    sizes = [int(box_feats[l].shape[2]) * int(box_feats[l].shape[3]) for l in range(L)]
    A, R = sum(sizes), _summary_len(sizes, 2)
    ncs = [int(cls_w[t * L].shape[0]) for t in range(T)]
    return ([first.new_empty((first.shape[0], 4 + n, A)) for n in ncs] + [first.new_empty((first.shape[0], n, R)) for n in ncs])


def head_tail(task_box_feats: Sequence[Sequence[torch.Tensor]], task_cls_feats: Sequence[Sequence[torch.Tensor]],
              task_box_w: Sequence[Sequence[torch.Tensor]], task_box_b: Sequence[Sequence[torch.Tensor]],
              task_cls_w: Sequence[Sequence[torch.Tensor]], task_cls_b: Sequence[Sequence[torch.Tensor]],
              strides: Sequence[float]) -> List[torch.Tensor]:
    """Head-tail fusion (SURVEY 8f row 3): the last 1x1 convolutions of both towers of every (task, level)
    (``cv2[l][-1]``: c2 -> 64, ``cv3[l][-1]``: c3 -> nc; reference models/yolo.py:81-84,89-90) + concat + eval decode
    (yolo.py:93-99) in one tcgen05 kernel.  ``task_box_feats[t][l]`` ``[B, c2, H_l, W_l]`` / ``task_cls_feats[t][l]``
    ``[B, c3, H_l, W_l]`` are the inputs of those convolutions, the weights ``[64, c2(,1,1)]`` / ``[nc, c3(,1,1)]`` and
    biases their parameters.  float16 only.  Returns ``y_t [B, 4+nc_t, A]`` per task (score summaries remembered for
    ``nms_batched`` like ``decode_heads`` does)."""
    flat = lambda z: [x for lv in z for x in lv]  # noqa: E731
    T = len(task_box_feats)
    out = head_tail_op(flat(task_box_feats), flat(task_cls_feats), flat(task_box_w), flat(task_box_b), flat(task_cls_w),
                       flat(task_cls_b), [float(s) for s in strides], T)
    ys, sms = out[:T], out[T:]
    for y, sm in zip(ys, sms):
        if sm.shape[-1]:
            _remember_summary(y, sm)
    return ys


def nms_batched(
    preds: Sequence[torch.Tensor],
    conf_thres: float = 0.25,
    iou_thres: float = 0.45,
    classes: Optional[Sequence[int]] = None,
    agnostic: bool = False,
    multi_label: bool = False,
    max_det: int = 300,
    max_nms: int = MAX_NMS,
    max_wh: float = MAX_WH,
    use_summary: bool = True,
    out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
    deliver=None,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """All task heads, all images, one launch.  Returns padded ``dets[T,B,max_det,6]`` and
    ``counts[T,B]`` (device tensors; no host sync).  Predictions that came out of ``decode_heads``
    unmodified bring their score summary along, which spares the kernel the full score scans.
    ``out=(dets, counts)`` writes into caller-provided buffers (e.g. ``shard.DetectionGatherer``'s)."""
    # reference asserts (utils/general.py:399-400) -- same exception type and wording
    assert 0 <= conf_thres <= 1, f"Invalid Confidence threshold {conf_thres}, valid values are between 0.0 and 1.0"
    assert 0 <= iou_thres <= 1, f"Invalid IoU {iou_thres}, valid values are between 0.0 and 1.0"
    preds = list(preds)
    smax = []
    if use_summary:
        found = [find_summary(p) for p in preds]
        if all(f is not None for f in found):
            smax = found
    args = (preds, float(conf_thres), float(iou_thres), None if classes is None else [int(c) for c in classes],
            bool(agnostic), bool(multi_label), int(max_det), int(max_nms), float(max_wh), smax)
    if deliver is not None:  # multi-GPU: the launch also runs this rank's part of the delivery to rank dst
        return _nms_impl(*args, out=out, deliver=deliver)
    if out is not None:
        nms_out_op(*args, out[0], out[1])
        return out
    return nms_op(*args)


def nms_statistics(preds: Sequence[torch.Tensor], **kw) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """``nms_batched`` plus per-segment counters: returns ``(dets, counts, stats[T, B, 2])`` with the IoU tests made and
    the candidates consumed per (task, image) segment (``cerb_nms_stats``; bench.py's IoU pairs/s)."""
    preds = list(preds)
    T, B = len(preds), int(preds[0].shape[0])
    stats = torch.zeros((T, B, 2), dtype=torch.int64, device=preds[0].device)
    use_summary = kw.pop("use_summary", True)
    found = [find_summary(p) for p in preds] if use_summary else []
    smax = found if found and all(f is not None for f in found) else []
    dets, counts = _nms_impl(preds, float(kw.get("conf_thres", 0.25)), float(kw.get("iou_thres", 0.45)),
                             None if kw.get("classes") is None else [int(c) for c in kw["classes"]], bool(kw.get("agnostic", False)),
                             bool(kw.get("multi_label", False)), int(kw.get("max_det", 300)), int(kw.get("max_nms", MAX_NMS)),
                             float(kw.get("max_wh", MAX_WH)), smax, None, stats)
    return dets, counts, stats


def cross_task_merge(dets: torch.Tensor, counts: torch.Tensor, class_offsets: Sequence[int], iou_thres: float,
                     scale: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Batched GPU form of the reference's per-image tail after NMS (cerberusdet_inference.py:140-155):
    combine the tasks' rows with global class ids, ``nms_between_tasks``, optional ``scale_boxes().round()``.
    ``scale`` is a device ``[B, 5]`` float tensor (gain, pad_x, pad_y, orig_w, orig_h) or None.
    Returns ``merged[B, T*max_det, 6]`` and ``counts[B]`` (device)."""
    lib = _lib.load()
    _require_cuda(dets, "dets")
    T, B, max_det, _ = dets.shape
    dets, counts = dets.contiguous(), counts.contiguous()
    ws_bytes = int(lib.cerb_cross_task_workspace_bytes(T, B, max_det))  # 0 while T*max_det <= 1024
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dets.device) if ws_bytes else None
    out = torch.empty((B, T * max_det, 6), dtype=torch.float32, device=dets.device)
    out_counts = torch.empty((B,), dtype=torch.int32, device=dets.device)
    if scale is not None:
        scale = scale.to(device=dets.device, dtype=torch.float32).contiguous()
        if tuple(scale.shape) != (B, 5):
            raise ValueError("scale must be [B, 5]")
    with torch.cuda.device(dets.device):
        rc = lib.cerb_cross_task_ws(dets.data_ptr(), counts.data_ptr(), T, B, max_det, _lib.int_array([int(o) for o in class_offsets]),
                                    float(iou_thres), scale.data_ptr() if scale is not None else None, out.data_ptr(),
                                    out_counts.data_ptr(), ws.data_ptr() if ws is not None else None, ws_bytes,
                                    _stream_ptr(dets.device))
    _lib.check(rc)
    return out, out_counts


def _decode_nms_impl(levels, nc, strides, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh):
    lib = _lib.load()
    T = len(nc)
    if T == 0 or len(levels) % T:
        raise ValueError("levels must hold T*L tensors, task-major")
    L = len(levels) // T
    if len(strides) != L:
        raise ValueError(f"expected {L} strides, got {len(strides)}")
    first = levels[0]
    _require_cuda(first, "head tensors")
    code = _dtype_code(first)
    B = int(first.shape[0])
    H = [int(levels[l].shape[2]) for l in range(L)]
    W = [int(levels[l].shape[3]) for l in range(L)]
    A = sum(h * w for h, w in zip(H, W))
    lv = []
    for t in range(T):
        for l in range(L):
            x = levels[t * L + l]
            if x.device != first.device or x.dtype != first.dtype or tuple(x.shape) != (B, 64 + nc[t], H[l], W[l]):
                raise ValueError(f"task {t} level {l}: expected {(B, 64 + nc[t], H[l], W[l])} {first.dtype} on {first.device}")
            lv.append(_dense16(x))
    dev = first.device
    ys = [torch.empty((B, 4 + n, A), dtype=first.dtype, device=dev) for n in nc]
    R = _summary_len([h * w for h, w in zip(H, W)], first.element_size())
    sm = [torch.empty((B, n, max(R, 1)), dtype=first.dtype, device=dev) for n in nc]
    dets = torch.empty((T, B, max_det, 6), dtype=torch.float32, device=dev)
    counts = torch.empty((T, B), dtype=torch.int32, device=dev)
    ws_bytes = lib.cerb_nms_workspace_bytes(T, B, max_det)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
    with torch.cuda.device(dev):
        rc = lib.cerb_decode_nms(
            _lib.ptr_array([x.data_ptr() for x in lv]), _lib.int_array(list(nc)), T, L, B, _lib.int_array(H), _lib.int_array(W),
            _lib.float_array([float(s) for s in strides]), code, _lib.ptr_array([y.data_ptr() for y in ys]),
            _lib.ptr_array([x.data_ptr() for x in sm]) if R else None, float(conf_thres), float(iou_thres),
            _lib.int_array(list(classes)) if classes is not None else None, len(classes) if classes is not None else 0,
            int(bool(agnostic)), int(bool(multi_label)), int(max_det), int(max_nms), float(max_wh), dets.data_ptr(),
            counts.data_ptr(), ws.data_ptr() if ws is not None else None, ws_bytes, _stream_ptr(dev))
    _lib.check(rc)
    return [dets, counts] + ys


def decode_nms(task_levels: Sequence[Sequence[torch.Tensor]], strides: Sequence[float], conf_thres: float = 0.25,
               iou_thres: float = 0.45, classes: Optional[Sequence[int]] = None, agnostic: bool = False,
               multi_label: bool = False, max_det: int = 300, max_nms: int = MAX_NMS, max_wh: float = MAX_WH):
    """Raw head tensors -> padded detections in ONE library call (``cerb::decode_nms`` / ``cerb_decode_nms``: both kernels
    back to back on the current stream).  Returns ``(dets[T,B,max_det,6], counts[T,B], ys)``."""
    assert 0 <= conf_thres <= 1, f"Invalid Confidence threshold {conf_thres}, valid values are between 0.0 and 1.0"
    assert 0 <= iou_thres <= 1, f"Invalid IoU {iou_thres}, valid values are between 0.0 and 1.0"
    nc = [int(lv[0].shape[1]) - 64 for lv in task_levels]
    out = decode_nms_op([x for row in task_levels for x in row], nc, [float(s) for s in strides], float(conf_thres),
                        float(iou_thres), None if classes is None else [int(c) for c in classes], bool(agnostic),
                        bool(multi_label), int(max_det), int(max_nms), float(max_wh))
    return out[0], out[1], out[2:]


def match_batch(dets: torch.Tensor, counts: torch.Tensor, labels: torch.Tensor, label_offsets: Sequence[int],
                iouv: torch.Tensor, iouv_host: Optional[Sequence[float]] = None) -> torch.Tensor:
    """Batched GPU form of the reference's ``process_batch`` (val.py:32-54): ``dets [B, max_det, 6]`` /
    ``counts [B]`` of one task in native image space, ``labels [sum M_b, 5]`` (cls, x1, y1, x2, y2) with
    ``label_offsets`` (``B+1`` python ints) -> ``correct [B, max_det, K]`` bool (device)."""
    lib = _lib.load()
    _require_cuda(dets, "dets")
    B, max_det, _ = dets.shape
    offs = [int(o) for o in label_offsets]
    if len(offs) != B + 1:
        raise ValueError("label_offsets must have B+1 entries")
    mmax = max((offs[i + 1] - offs[i] for i in range(B)), default=0)
    if mmax > 1024:
        raise ValueError("match_batch supports at most 1024 labels per image")
    dev = dets.device
    dets, counts = dets.contiguous().float(), counts.contiguous().to(torch.int32)
    labels = labels.to(device=dev, dtype=torch.float32).contiguous()
    offs_d = torch.tensor(offs, dtype=torch.int32, device=dev)
    iou_host = list(iouv_host) if iouv_host is not None else [float(v) for v in iouv.detach().cpu().float().tolist()]
    K = len(iou_host)
    correct = torch.empty((B, max_det, K), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.cerb_val_match(dets.data_ptr(), counts.data_ptr(), B, max_det, labels.data_ptr() if labels.numel() else None,
                                offs_d.data_ptr(), mmax, _lib.float_array(iou_host), K, correct.data_ptr(), _stream_ptr(dev))
    _lib.check(rc)
    return correct.bool()


# ----------------------------------------------------------------------------- training-time sibling decode (SURVEY 8f-4)
class _BboxDecode(torch.autograd.Function):
    """``Loss.bbox_decode`` (reference utils/loss.py:126-131) as one CUDA kernel per direction."""

    @staticmethod
    def forward(ctx, anchor_points: torch.Tensor, pred_dist: torch.Tensor) -> torch.Tensor:
        lib = _lib.load()
        _require_cuda(pred_dist, "pred_dist")
        if pred_dist.dim() != 3 or pred_dist.shape[2] != 64:
            raise ValueError(f"pred_dist must be [B, A, 64] (reg_max 16), got {tuple(pred_dist.shape)}")
        B, A, _ = pred_dist.shape
        if tuple(anchor_points.shape) != (A, 2):
            raise ValueError(f"anchor_points must be [{A}, 2], got {tuple(anchor_points.shape)}")
        if anchor_points.device != pred_dist.device:
            raise TypeError("anchor_points and pred_dist must be on the same device")
        code = _dtype_code(pred_dist)
        x = pred_dist.contiguous()
        ap = anchor_points.to(pred_dist.dtype).contiguous()
        out = torch.empty((B, A, 4), dtype=pred_dist.dtype, device=pred_dist.device)
        with torch.cuda.device(x.device):
            rc = lib.cerb_bbox_decode_fwd(x.data_ptr(), ap.data_ptr(), B * A, A, 16, code, out.data_ptr(), _stream_ptr(x.device))
        _lib.check(rc)
        ctx.save_for_backward(x)
        ctx.code = code
        return out

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        (x,) = ctx.saved_tensors
        lib = _lib.load()
        g = grad_out.to(x.dtype).contiguous()
        grad_in = torch.empty_like(x)
        with torch.cuda.device(x.device):
            rc = lib.cerb_bbox_decode_bwd(x.data_ptr(), g.data_ptr(), x.shape[0] * x.shape[1], 16, ctx.code,
                                          grad_in.data_ptr(), _stream_ptr(x.device))
        _lib.check(rc)
        return None, grad_in


def bbox_decode(anchor_points: torch.Tensor, pred_dist: torch.Tensor) -> torch.Tensor:
    """Drop-in for the reference's ``Loss.bbox_decode(anchor_points, pred_dist)`` with ``use_dfl`` (utils/loss.py:126-131):
    ``pred_dist [B, A, 64]`` -> ``[B, A, 4]`` (x1, y1, x2, y2) in grid units, differentiable w.r.t. ``pred_dist``."""
    return _BboxDecode.apply(anchor_points, pred_dist)


# ----------------------------------------------------------------------------- TAL assigner (SURVEY 8f-4)
def tal_assign(pd_scores: torch.Tensor, pd_bboxes: torch.Tensor, anc_points: torch.Tensor, gt_labels: torch.Tensor,
               gt_bboxes: torch.Tensor, mask_gt: torch.Tensor, topk: int = 10, num_classes: Optional[int] = None,
               alpha: float = 0.5, beta: float = 6.0, eps: float = 1e-9):
    """``TaskAlignedAssigner.forward`` (reference utils/tal.py:56-178) in three launches (``cerb_tal_assign``).
    ``pd_scores [B, A, C]`` fp16 | fp32, ``pd_bboxes [B, A, 4]`` fp32 xyxy pixels, ``anc_points [A, 2]``, ``gt_labels [B, G, 1]``,
    ``gt_bboxes [B, G, 4]``, ``mask_gt [B, G, 1]``.  Returns ``(target_labels [B, A] int64, target_bboxes [B, A, 4],
    target_scores [B, A, C] fp32, fg_mask [B, A] bool, target_gt_idx [B, A] int64)``.  ``G == 0`` is the caller's early
    return in the reference (tal.py:89-93) and raises ``ValueError`` here."""
    lib = _lib.load()
    _require_cuda(pd_scores, "pd_scores")
    B, A, C = (int(v) for v in pd_scores.shape)
    G = int(gt_bboxes.shape[1])
    if num_classes is not None and int(num_classes) != C:
        raise ValueError(f"pd_scores has {C} classes, the assigner {num_classes}")
    if G == 0:
        raise ValueError("tal_assign needs at least one (padded) ground-truth box per image; the reference returns early for none")
    dev = pd_scores.device
    code = _dtype_code(pd_scores)
    f32 = lambda t, shape: t.to(device=dev, dtype=torch.float32).reshape(shape).contiguous()  # noqa: E731
    sc = pd_scores.contiguous()
    pb, an = f32(pd_bboxes, (B, A, 4)), f32(anc_points, (A, 2))
    gl, gb, mg = f32(gt_labels, (B, G)), f32(gt_bboxes, (B, G, 4)), f32(mask_gt, (B, G))
    labels = torch.empty((B, A), dtype=torch.int64, device=dev)
    bboxes = torch.empty((B, A, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((B, A, C), dtype=torch.float32, device=dev)
    fg = torch.empty((B, A), dtype=torch.bool, device=dev)
    gidx = torch.empty((B, A), dtype=torch.int64, device=dev)
    ws_bytes = int(lib.cerb_tal_workspace_bytes(B, A, G, int(topk)))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.cerb_tal_assign(sc.data_ptr(), pb.data_ptr(), an.data_ptr(), gl.data_ptr(), gb.data_ptr(), mg.data_ptr(), B, A, C, G,
                                 int(topk), float(alpha), float(beta), float(eps), code, labels.data_ptr(), bboxes.data_ptr(),
                                 scores.data_ptr(), fg.data_ptr(), gidx.data_ptr(), ws.data_ptr(), ws_bytes, _stream_ptr(dev))
    _lib.check(rc)
    for t in (sc, pb, an, gl, gb, mg, ws):
        t.record_stream(torch.cuda.current_stream(dev))
    return labels, bboxes, scores, fg, gidx


# ----------------------------------------------------------------------------- box-regression loss term (SURVEY 8f-4)
def _dense32(x: torch.Tensor) -> torch.Tensor:
    """Contiguous and 32-byte aligned (the 256-bit row accesses of the training kernels)."""
    x = x.contiguous()
    return x if x.data_ptr() % 32 == 0 else x.clone(memory_format=torch.contiguous_format)


class _BboxLoss(torch.autograd.Function):
    """``BboxLoss.forward`` (reference utils/loss.py:12-44) as one CUDA kernel per direction; differentiable in
    ``pred_dist`` and ``pred_bboxes``."""

    @staticmethod
    def forward(ctx, pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask, per_anchor):
        lib = _lib.load()
        _require_cuda(pred_dist, "pred_dist")
        dev = pred_dist.device
        if pred_dist.dim() != 3 or pred_dist.shape[2] != 64:
            raise ValueError(f"pred_dist must be [B, A, 64] (16 bins per side), got {tuple(pred_dist.shape)}")
        B, A, _ = (int(v) for v in pred_dist.shape)
        C = int(target_scores.shape[-1]) if target_scores.dim() == 3 else -1
        for name, t, shape in (("pred_bboxes", pred_bboxes, (B, A, 4)), ("anchor_points", anchor_points, (A, 2)),
                               ("target_bboxes", target_bboxes, (B, A, 4)), ("target_scores", target_scores, (B, A, C)),
                               ("fg_mask", fg_mask, (B, A))):
            if tuple(t.shape) != shape:
                raise ValueError(f"{name} must be {list(shape)}, got {tuple(t.shape)}")
            if t.device != dev:
                raise TypeError(f"{name} must be on {dev}, got {t.device}")
        code = _dtype_code(pred_dist)
        if pred_bboxes.dtype != pred_dist.dtype or anchor_points.dtype != pred_dist.dtype:
            raise TypeError("pred_dist, pred_bboxes and anchor_points must share one dtype")
        if target_bboxes.dtype != torch.float32 or target_scores.dtype != torch.float32 or fg_mask.dtype != torch.bool:
            raise TypeError("target_bboxes and target_scores must be float32 and fg_mask bool")
        tss_dev, tss_host = None, 1.0
        if torch.is_tensor(target_scores_sum):
            if target_scores_sum.numel() != 1:
                raise ValueError("target_scores_sum must hold one value")
            if target_scores_sum.is_cuda:
                if target_scores_sum.device != dev:
                    raise TypeError(f"target_scores_sum must be on {dev}, got {target_scores_sum.device}")
                tss_dev = target_scores_sum.detach().reshape(()).float()
            else:
                tss_host = float(target_scores_sum)  # a CPU value: no device round trip
        else:
            tss_host = float(target_scores_sum)
        x, pb, ap = _dense32(pred_dist.detach()), pred_bboxes.detach().contiguous(), anchor_points.detach().contiguous()
        tb, ts, fg = target_bboxes.contiguous(), target_scores.contiguous(), fg_mask.contiguous()
        loss_iou = torch.empty((), dtype=torch.float32, device=dev)
        loss_dfl = torch.empty((), dtype=torch.float32, device=dev)
        ws_bytes = int(lib.cerb_bbox_loss_workspace_bytes(B, A))
        ws = torch.zeros((ws_bytes,), dtype=torch.uint8, device=dev)
        if per_anchor is not None and (tuple(per_anchor.shape) != (B, A, 2) or per_anchor.dtype != torch.float32
                                       or not per_anchor.is_contiguous() or per_anchor.device != dev):
            raise ValueError(f"per_anchor must be a contiguous float32 [{B}, {A}, 2] tensor on {dev}")
        tss_ptr = tss_dev.data_ptr() if tss_dev is not None else None
        with torch.cuda.device(dev):
            rc = lib.cerb_bbox_loss_fwd(x.data_ptr(), pb.data_ptr(), ap.data_ptr(), tb.data_ptr(), ts.data_ptr(), fg.data_ptr(),
                                        tss_ptr, tss_host, B, A, C, 16, code, loss_iou.data_ptr(), loss_dfl.data_ptr(),
                                        per_anchor.data_ptr() if per_anchor is not None else None, ws.data_ptr(), ws_bytes,
                                        _stream_ptr(dev))
        _lib.check(rc)
        ctx.save_for_backward(x, pb, ap, tb, ts, fg, tss_dev)
        ctx.meta = (B, A, C, code, tss_dev is not None, tss_host)
        return loss_iou, loss_dfl

    @staticmethod
    def backward(ctx, g_iou, g_dfl):
        x, pb, ap, tb, ts, fg, tss = ctx.saved_tensors
        B, A, C, code, has_tss, tss_host = ctx.meta
        lib = _lib.load()
        dev = x.device
        g_iou = torch.zeros((), dtype=torch.float32, device=dev) if g_iou is None else g_iou.detach().reshape(()).float()
        g_dfl = torch.zeros((), dtype=torch.float32, device=dev) if g_dfl is None else g_dfl.detach().reshape(()).float()
        grad_dist = torch.empty_like(x)
        grad_boxes = torch.empty_like(pb)
        with torch.cuda.device(dev):
            rc = lib.cerb_bbox_loss_bwd(x.data_ptr(), pb.data_ptr(), ap.data_ptr(), tb.data_ptr(), ts.data_ptr(), fg.data_ptr(),
                                        tss.data_ptr() if has_tss else None, tss_host, B, A, C, 16, code, g_iou.data_ptr(),
                                        g_dfl.data_ptr(), grad_dist.data_ptr(), grad_boxes.data_ptr(), _stream_ptr(dev))
        _lib.check(rc)
        return grad_dist, grad_boxes, None, None, None, None, None, None


def bbox_loss(pred_dist: torch.Tensor, pred_bboxes: torch.Tensor, anchor_points: torch.Tensor, target_bboxes: torch.Tensor,
              target_scores: torch.Tensor, target_scores_sum, fg_mask: torch.Tensor,
              per_anchor: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Drop-in for the reference's ``BboxLoss(reg_max=15, use_dfl=True).forward`` (utils/loss.py:12-44):
    ``(loss_iou, loss_dfl)`` as 0-d float32 tensors, differentiable in ``pred_dist [B, A, 64]`` and
    ``pred_bboxes [B, A, 4]``.  No host synchronisation: the foreground mask is read by the kernels, and
    ``target_scores_sum`` (a 0-d CUDA tensor, or a number such as the call site's ``1``) is read on the device.

    Two dtype combinations: everything float32; or the trainer's fp16-autocast case -- ``pred_dist``, ``pred_bboxes`` and
    ``anchor_points`` float16, ``target_bboxes`` / ``target_scores`` float32 -- with the reference's half roundings.
    ``per_anchor`` (float32 ``[B, A, 2]``, optional) receives the per-anchor terms ``(1 - CIoU) * weight`` and
    ``DFL * weight`` (zero at background anchors)."""
    return _BboxLoss.apply(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask, per_anchor)


# ----------------------------------------------------------------------------- validation mAP statistics
def ap_per_class(tp: torch.Tensor, conf: torch.Tensor, pred_cls: torch.Tensor, target_cls: torch.Tensor, eps: float = 1e-16):
    """The GPU part of the reference's ``ap_per_class`` (utils/metrics.py:56-120, with ``compute_ap``) in one
    ``cerb_ap_per_class`` call: ``tp [N, K]`` bool (K <= 32 IoU thresholds), ``conf`` / ``pred_cls [N]`` and
    ``target_cls [M]`` float16 | float32, all CUDA tensors.  Returns device tensors ``(ap [nc, K], p [nc, 1000],
    r [nc, 1000])`` float64 and ``(unique_classes [nc] float32, nt [nc] int64)`` as ``np.unique(target_cls,
    return_counts=True)`` gives them.  Equal confidences are ordered by row index (``np.argsort(-conf, kind="stable")``).

    For callers that hold the statistics on the device (``val_stats.validation_batch_statistics``): concatenate them there
    and call this, with no host round trip for the ``[N, K]`` rows; only ``nc`` class values come to the host.  NaN in
    ``conf`` or ``target_cls`` raises ``ValueError``."""
    lib = _lib.load()
    for t, what in ((tp, "tp"), (conf, "conf"), (pred_cls, "pred_cls"), (target_cls, "target_cls")):
        _require_cuda(t, what)
        if t is not tp and t.dtype not in (torch.float16, torch.float32):
            raise TypeError(f"{what} must be float16 or float32, got {t.dtype}")
    if tp.dtype != torch.bool or tp.dim() != 2:
        raise TypeError(f"tp must be a [N, K] bool tensor, got {tp.dtype} {tuple(tp.shape)}")
    n, K = (int(v) for v in tp.shape)
    if not 1 <= K <= 32:
        raise ValueError(f"tp has {K} IoU thresholds, 1..32 supported")
    if tuple(conf.shape) != (n,) or tuple(pred_cls.shape) != (n,):
        raise ValueError(f"conf and pred_cls must be [{n}], got {tuple(conf.shape)} and {tuple(pred_cls.shape)}")
    dev = tp.device
    conf32, cls32 = conf.to(dev, torch.float32).contiguous(), pred_cls.to(dev, torch.float32).contiguous()
    target = target_cls.to(dev, torch.float32).reshape(-1)
    nan_target, nan_conf = torch.stack((target.isnan().any(), conf32.isnan().any())).tolist()
    if nan_target or nan_conf:
        raise ValueError("target_cls contains NaN" if nan_target else "conf contains NaN")
    classes, nt = torch.unique(target, sorted=True, return_counts=True)
    classes_h, nt_h = classes.cpu(), nt.cpu()
    nc = int(classes.numel())
    tpc = tp.contiguous()
    ap = torch.empty((nc, K), dtype=torch.float64, device=dev)
    p = torch.empty((nc, 1000), dtype=torch.float64, device=dev)
    r = torch.empty((nc, 1000), dtype=torch.float64, device=dev)
    ws_bytes = int(lib.cerb_ap_workspace_bytes(n, K, nc))
    ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.cerb_ap_per_class(tpc.data_ptr(), K, conf32.data_ptr(), cls32.data_ptr(), n, classes_h.data_ptr(),
                                   nt_h.data_ptr(), nc, float(eps), ap.data_ptr(), p.data_ptr(), r.data_ptr(), ws.data_ptr(),
                                   ws_bytes, _stream_ptr(dev))
    _lib.check(rc)
    for t in (tpc, conf32, cls32, ws):
        t.record_stream(torch.cuda.current_stream(dev))
    return ap, p, r, classes, nt
