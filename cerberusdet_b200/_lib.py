"""ctypes binding of ``libcerb_post.so`` (C ABI in ``include/cerb_post.h``).

The library is the product: if it is missing or fails to load, importing the ops
raises -- there is no CPU or eager-PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CERB_LIB") or os.path.join(_HERE, "libcerb_post.so")  # CERB_LIB: tools/ only

CERB_F16, CERB_F32 = 0, 1
CERB_EINVAL, CERB_ECUDA, CERB_ENOSPC = -1, -2, -3

EXPORTS = (
    "cerb_version",
    "cerb_last_error",
    "cerb_decode",
    "cerb_decode_split",
    "cerb_head_tail",
    "cerb_summary_row_len",
    "cerb_nms_workspace_bytes",
    "cerb_nms",
    "cerb_nms_stats",
    "cerb_nms_deliver",
    "cerb_deliver_collect",
    "cerb_deliver_push",
    "cerb_decode_nms",
    "cerb_cross_task",
    "cerb_cross_task_workspace_bytes",
    "cerb_cross_task_ws",
    "cerb_val_match",
    "cerb_bbox_decode_fwd",
    "cerb_bbox_decode_bwd",
    "cerb_tal_workspace_bytes",
    "cerb_tal_assign",
    "cerb_bbox_loss_workspace_bytes",
    "cerb_bbox_loss_fwd",
    "cerb_bbox_loss_bwd",
    "cerb_ap_workspace_bytes",
    "cerb_ap_per_class",
    "cerb_debug_set",
    "cerb_debug_reset",
    "cerb_debug_set_chunking",
    "cerb_debug_set_hist_sample",
)

_lib = None


class Delivery(ctypes.Structure):
    """``cerb_delivery`` of include/cerb_post.h."""

    _fields_ = [("push_src", ctypes.c_void_p), ("push_dst", ctypes.c_void_p), ("push_words", ctypes.c_size_t),
                ("flag_remote", ctypes.c_void_p), ("ack_local", ctypes.c_void_p), ("seq_local", ctypes.c_void_p),
                ("done_local", ctypes.c_void_p), ("collect_flags", ctypes.c_void_p), ("collect_ack", ctypes.c_void_p * 16),
                ("collect_count", ctypes.c_void_p), ("world", ctypes.c_int), ("dst", ctypes.c_int)]


class CerbLibraryError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CerbLibraryError(
            f"{LIB_PATH} not found: build it with `sh cerberusdet_b200/csrc/build.sh` "
            "(or __graft_entry__.build()).  cerberusdet_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    vp, ip, i, d, sz = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_double, ctypes.c_size_t
    vpp = ctypes.POINTER(ctypes.c_void_p)
    fp = ctypes.POINTER(ctypes.c_float)
    lib.cerb_version.restype = i
    lib.cerb_version.argtypes = []
    lib.cerb_last_error.restype = ctypes.c_char_p
    lib.cerb_last_error.argtypes = []
    lib.cerb_decode.restype = i
    lib.cerb_decode.argtypes = [vpp, ip, i, i, i, ip, ip, fp, i, vpp, vpp, ip, vp]
    lib.cerb_decode_split.restype = i
    lib.cerb_decode_split.argtypes = [vpp, vpp, ip, i, i, i, ip, ip, fp, i, vpp, vpp, ip, vp]
    if hasattr(lib, "cerb_head_tail") or "CERB_LIB" not in os.environ:
        lib.cerb_head_tail.restype = i
        lib.cerb_head_tail.argtypes = [vpp] * 6 + [ip, ip, ip, i, i, i, ip, ip, fp, i, vpp, vpp, ip, vp]
    lib.cerb_summary_row_len.restype = sz
    lib.cerb_summary_row_len.argtypes = [i, i]
    lib.cerb_nms_workspace_bytes.restype = sz
    lib.cerb_nms_workspace_bytes.argtypes = [i, i, i]
    lib.cerb_nms.restype = i
    lib.cerb_nms.argtypes = [vpp, ip, i, i, i, i, d, d, ip, i, i, i, i, i, d, vpp, vp, vp, vp, sz, vp]
    if hasattr(lib, "cerb_nms_stats") or "CERB_LIB" not in os.environ:
        lib.cerb_nms_stats.restype = i
        lib.cerb_nms_stats.argtypes = [vpp, ip, i, i, i, i, d, d, ip, i, i, i, i, i, d, vpp, vp, vp, vp, sz, vp, vp]
    if hasattr(lib, "cerb_nms_deliver") or "CERB_LIB" not in os.environ:
        lib.cerb_nms_deliver.restype = i
        lib.cerb_nms_deliver.argtypes = [vpp, ip, i, i, i, i, d, d, ip, i, i, i, i, i, d, vpp, vp, vp, vp, sz, ctypes.POINTER(Delivery), vp]
        lib.cerb_deliver_collect.restype = i
        lib.cerb_deliver_collect.argtypes = [vp, vpp, vp, i, i, vp]
        lib.cerb_deliver_push.restype = i
        lib.cerb_deliver_push.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp]
    lib.cerb_decode_nms.restype = i
    lib.cerb_decode_nms.argtypes = [vpp, ip, i, i, i, ip, ip, fp, i, vpp, vpp, d, d, ip, i, i, i, i, i, d, vp, vp, vp, sz, vp]
    lib.cerb_cross_task.restype = i
    lib.cerb_cross_task.argtypes = [vp, vp, i, i, i, ip, d, vp, vp, vp, vp]
    if hasattr(lib, "cerb_cross_task_ws") or "CERB_LIB" not in os.environ:
        lib.cerb_cross_task_workspace_bytes.restype = sz
        lib.cerb_cross_task_workspace_bytes.argtypes = [i, i, i]
        lib.cerb_cross_task_ws.restype = i
        lib.cerb_cross_task_ws.argtypes = [vp, vp, i, i, i, ip, d, vp, vp, vp, vp, sz, vp]
    lib.cerb_val_match.restype = i
    lib.cerb_val_match.argtypes = [vp, vp, i, i, vp, vp, i, fp, i, vp, vp]
    lg = ctypes.c_long
    lib.cerb_bbox_decode_fwd.restype = i
    lib.cerb_bbox_decode_fwd.argtypes = [vp, vp, lg, i, i, i, vp, vp]
    lib.cerb_bbox_decode_bwd.restype = i
    lib.cerb_bbox_decode_bwd.argtypes = [vp, vp, lg, i, i, vp, vp]
    if hasattr(lib, "cerb_tal_assign") or "CERB_LIB" not in os.environ:
        lib.cerb_tal_workspace_bytes.restype = sz
        lib.cerb_tal_workspace_bytes.argtypes = [i, i, i, i]
        lib.cerb_tal_assign.restype = i
        lib.cerb_tal_assign.argtypes = [vp] * 6 + [i] * 5 + [d, d, d, i] + [vp] * 6 + [sz, vp]
    if hasattr(lib, "cerb_bbox_loss_fwd") or "CERB_LIB" not in os.environ:
        lib.cerb_bbox_loss_workspace_bytes.restype = sz
        lib.cerb_bbox_loss_workspace_bytes.argtypes = [i, i]
        lib.cerb_bbox_loss_fwd.restype = i
        lib.cerb_bbox_loss_fwd.argtypes = [vp] * 7 + [d] + [i] * 5 + [vp] * 4 + [sz, vp]
        lib.cerb_bbox_loss_bwd.restype = i
        lib.cerb_bbox_loss_bwd.argtypes = [vp] * 7 + [d] + [i] * 5 + [vp] * 5
    if hasattr(lib, "cerb_ap_per_class") or "CERB_LIB" not in os.environ:
        lib.cerb_ap_workspace_bytes.restype = sz
        lib.cerb_ap_workspace_bytes.argtypes = [lg, i, i]
        lib.cerb_ap_per_class.restype = i
        lib.cerb_ap_per_class.argtypes = [vp, i, vp, vp, lg, vp, vp, i, d, vp, vp, vp, vp, sz, vp]
    if hasattr(lib, "cerb_debug_set") or "CERB_LIB" not in os.environ:  # (tools/ A/B runs may load an older build)
        lib.cerb_debug_set.restype = i
        lib.cerb_debug_set.argtypes = [ctypes.c_char_p, i]
        lib.cerb_debug_reset.restype = i
        lib.cerb_debug_reset.argtypes = []
    lib.cerb_debug_set_chunking.restype = i
    lib.cerb_debug_set_chunking.argtypes = [i, i]
    lib.cerb_debug_set_hist_sample.restype = i
    lib.cerb_debug_set_hist_sample.argtypes = [i]
    _lib = lib
    return lib


def debug_set(name: str, value: int) -> None:
    """Thread-local test / tools knob (include/cerb_post.h: cerb_debug_set)."""
    check(load().cerb_debug_set(name.encode(), int(value)))


def debug_reset() -> None:
    load().cerb_debug_reset()


def last_error() -> str:
    return load().cerb_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Map a C return code to the exception type the reference would raise."""
    if rc == 0:
        return
    msg = last_error()
    if rc == CERB_EINVAL and msg.startswith("Invalid"):
        raise AssertionError(msg)  # reference: `assert 0 <= conf_thres <= 1` (utils/general.py:399-400)
    if rc == CERB_EINVAL:
        raise ValueError(msg)
    raise CerbLibraryError(f"libcerb_post error {rc}: {msg}")


def int_array(values):
    return (ctypes.c_int * max(len(values), 1))(*values)


def float_array(values):
    return (ctypes.c_float * max(len(values), 1))(*values)


def ptr_array(values):
    return (ctypes.c_void_p * max(len(values), 1))(*values)
