"""ctypes binding of ``libcerb_post.so`` (C ABI in ``include/cerb_post.h``).

The library is the product: if it is missing or fails to load, importing the ops
raises -- there is no CPU or eager-PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CERB_LIB") or os.path.join(_HERE, "libcerb_post.so")  # CERB_LIB: tools/ only

CERB_F16, CERB_F32, CERB_BF16 = 0, 1, 2
CERB_EINVAL, CERB_ECUDA, CERB_ENOSPC = -1, -2, -3

_lib = None


class Delivery(ctypes.Structure):
    """``cerb_delivery`` of include/cerb_post.h."""

    _fields_ = [("push_src", ctypes.c_void_p), ("push_dst", ctypes.c_void_p), ("push_words", ctypes.c_size_t),
                ("flag_remote", ctypes.c_void_p), ("ack_local", ctypes.c_void_p), ("seq_local", ctypes.c_void_p),
                ("done_local", ctypes.c_void_p), ("collect_flags", ctypes.c_void_p), ("collect_ack", ctypes.c_void_p * 16),
                ("collect_count", ctypes.c_void_p), ("world", ctypes.c_int), ("dst", ctypes.c_int)]


_vp, _ip, _i, _d, _sz, _lg = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_double, ctypes.c_size_t, ctypes.c_long
_vpp, _fp = ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_float)
_NMS = [_vpp, _ip, _i, _i, _i, _i, _d, _d, _ip, _i, _i, _i, _i, _i, _d, _vpp, _vp, _vp, _vp, _sz]  # shared head of the cerb_nms* calls

# {name: (restype, argtypes)} of every entry point of include/cerb_post.h
PROTOTYPES = {
    "cerb_version": (_i, []),
    "cerb_last_error": (ctypes.c_char_p, []),
    "cerb_decode": (_i, [_vpp, _ip, _i, _i, _i, _ip, _ip, _fp, _i, _vpp, _vpp, _ip, _vp]),
    "cerb_decode_split": (_i, [_vpp, _vpp, _ip, _i, _i, _i, _ip, _ip, _fp, _i, _vpp, _vpp, _ip, _vp]),
    "cerb_head_tail": (_i, [_vpp] * 6 + [_ip, _ip, _ip, _i, _i, _i, _ip, _ip, _fp, _i, _vpp, _vpp, _ip, _vp]),
    "cerb_summary_row_len": (_sz, [_i, _i]),
    "cerb_nms_workspace_bytes": (_sz, [_i, _i, _i]),
    "cerb_nms": (_i, _NMS + [_vp]),
    "cerb_nms_stats": (_i, _NMS + [_vp, _vp]),
    "cerb_nms_deliver": (_i, _NMS + [ctypes.POINTER(Delivery), _vp]),
    "cerb_deliver_collect": (_i, [_vp, _vpp, _vp, _i, _i, _vp]),
    "cerb_deliver_push": (_i, [_vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "cerb_decode_nms": (_i, [_vpp, _ip, _i, _i, _i, _ip, _ip, _fp, _i, _vpp, _vpp, _d, _d, _ip, _i, _i, _i, _i, _i, _d, _vp, _vp, _vp, _sz, _vp]),
    "cerb_cross_task": (_i, [_vp, _vp, _i, _i, _i, _ip, _d, _vp, _vp, _vp, _vp]),
    "cerb_cross_task_workspace_bytes": (_sz, [_i, _i, _i]),
    "cerb_cross_task_ws": (_i, [_vp, _vp, _i, _i, _i, _ip, _d, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cerb_val_match": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _fp, _i, _vp, _vp]),
    "cerb_confusion_matrix": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _d, _d, _vp, _vp, _vp, _vp]),
    "cerb_bbox_decode_fwd": (_i, [_vp, _vp, _lg, _i, _i, _i, _vp, _vp]),
    "cerb_bbox_decode_bwd": (_i, [_vp, _vp, _lg, _i, _i, _vp, _vp]),
    "cerb_tal_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "cerb_tal_assign": (_i, [_vp] * 6 + [_i] * 5 + [_d, _d, _d, _i] + [_vp] * 6 + [_sz, _vp]),
    "cerb_bbox_loss_workspace_bytes": (_sz, [_i, _i]),
    "cerb_bbox_loss_fwd": (_i, [_vp] * 7 + [_d] + [_i] * 5 + [_vp] * 4 + [_sz, _vp]),
    "cerb_bbox_loss_bwd": (_i, [_vp] * 7 + [_d] + [_i] * 5 + [_vp] * 5),
    "cerb_ap_workspace_bytes": (_sz, [_lg, _i, _i]),
    "cerb_ap_per_class": (_i, [_vp, _i, _vp, _vp, _lg, _vp, _vp, _i, _d, _vp, _vp, _vp, _vp, _sz, _vp]),
    "cerb_letterbox": (_i, [_vpp, _ip, _ip, ctypes.POINTER(_lg), _ip, _ip, _ip, _ip, _i, _i, _i, _i, _vp, _vp]),
    "cerb_debug_set": (_i, [ctypes.c_char_p, _i]),
    "cerb_debug_reset": (_i, []),
    "cerb_debug_set_chunking": (_i, [_i, _i]),
    "cerb_debug_set_hist_sample": (_i, [_i]),
}
EXPORTS = tuple(PROTOTYPES)


class CerbLibraryError(RuntimeError):
    """A library call failed; ``code`` is its C return code (``CERB_ECUDA``, ``CERB_ENOSPC``, ...) or None when the
    error was raised on the Python side."""

    def __init__(self, msg: str, code=None):
        super().__init__(msg)
        self.code = code


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
    for name, (restype, argtypes) in PROTOTYPES.items():
        if "CERB_LIB" in os.environ and not hasattr(lib, name):
            continue  # an older build (tools/ A/B runs): a call to the missing entry point fails where it is made
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
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
    raise CerbLibraryError(f"libcerb_post error {rc}: {msg}", code=rc)


def int_array(values):
    return (ctypes.c_int * max(len(values), 1))(*values)


def float_array(values):
    return (ctypes.c_float * max(len(values), 1))(*values)


def ptr_array(values):
    return (ctypes.c_void_p * max(len(values), 1))(*values)
