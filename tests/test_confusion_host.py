"""Host tests of the validation confusion matrix (no GPU): the canonical port (tests/confusion_port.py) against the
reference's text on tie-free cases, the C ABI's argument checks and ctypes prototype, and ``patch.install(confusion=True)``
with every fallback of the drop-in, on stand-in reference modules."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import confusion_port as cp  # noqa: E402


def _both(dets, labels, nc=20, conf=0.25, iou_thres=0.45):
    a, b = cp.ConfusionMatrixVerbatim(nc, conf, iou_thres), cp.ConfusionMatrixPort(nc, conf, iou_thres)
    a.process_batch(dets, labels)
    b.process_batch(dets, labels)
    return a.matrix, b.matrix


@pytest.mark.parametrize("crowd", [0.0, 0.9, 0.97])
def test_port_equals_reference_text_without_ties(crowd):
    rng = np.random.default_rng(int(crowd * 100))
    checked = fp_counted = 0
    for _ in range(150):
        dets, labels = cp.image_case(rng, int(rng.integers(1, 40)), int(rng.integers(1, 120)), 20, crowd=crowd)
        if cp.has_ties(dets, labels):
            continue
        want, got = _both(dets, labels)
        assert np.array_equal(want, got)
        checked += 1
        fp_counted += want[:20, 20].sum() > 0
    assert checked >= 140 and fp_counted > 0


def test_a_label_keeps_its_highest_iou_detection():
    """The reference's second sort is NOT commented out (unlike val.py's process_batch): label 0 goes to detection 1,
    which overlaps it more, although detection 0 comes first."""
    labels = torch.tensor([[3.0, 0, 0, 100, 100]])
    dets = torch.tensor([[0, 0, 100, 80, 0.9, 5], [0, 0, 100, 95, 0.8, 7]])
    for m in _both(dets, labels):
        assert m[7, 3] == 1 and m[5, 20] == 1 and m.sum() == 2


def test_no_surviving_pair_counts_no_false_positive():
    """The ``if n:`` quirk: detections without any pair above the threshold are not counted as background FPs."""
    labels = torch.tensor([[1.0, 0, 0, 10, 10], [2.0, 50, 50, 60, 60]])
    dets = torch.tensor([[200, 200, 300, 300, 0.9, 4], [5, 5, 30, 30, 0.8, 1]])  # IoU 0 and ~0.16
    for m in _both(dets, labels):
        assert m[20, 1] == 1 and m[20, 2] == 1 and m.sum() == 2


def test_detections_none_all_filtered_and_no_labels():
    labels = torch.tensor([[1.0, 0, 0, 10, 10], [1.0, 5, 5, 20, 20], [4.0, 50, 50, 60, 60]])
    for cls in (cp.ConfusionMatrixVerbatim, cp.ConfusionMatrixPort):
        cm = cls(20)
        cm.process_batch(None, labels[:, 0])
        assert cm.matrix[20, 1] == 2 and cm.matrix[20, 4] == 1 and cm.matrix.sum() == 3
    low = torch.tensor([[0, 0, 10, 10, 0.25, 1], [5, 5, 20, 20, 0.1, 1]])  # conf == 0.25 is filtered: strict >
    for m in _both(low, labels):
        assert m[20, 1] == 2 and m[20, 4] == 1 and m.sum() == 3
    dets = torch.tensor([[0, 0, 10, 10, 0.9, 1]])
    for m in _both(dets, labels[:0]):  # M = 0: nothing at all
        assert m.sum() == 0


def test_batch_rule_is_the_sum_of_the_loops_calls():
    dets, counts, labels, offsets = cp.batch_case(3, 12, 20, max_det=60, m_range=(0, 3), n_range=(0, 60))
    counts[1] = 0  # an image whose predictions NMS dropped
    assert (counts == 0).any() and any(offsets[i] == offsets[i + 1] for i in range(12))
    want = np.zeros((21, 21))
    for b in range(12):
        lab, n = labels[offsets[b] : offsets[b + 1]], int(counts[b])
        if lab.shape[0]:
            cm = cp.ConfusionMatrixPort(20)
            cm.process_batch(dets[b, :n] if n else None, lab if n else lab[:, 0])
            want += cm.matrix
    assert np.array_equal(cp.batch_port(dets, counts, labels, offsets, 20), want)


# ------------------------------------------------------------------------------------------------------ the C ABI
def test_confusion_prototype_matches_header():
    from cerberusdet_b200 import _lib

    text = open(os.path.join(os.path.dirname(HERE), "include", "cerb_post.h")).read()
    m = re.search(r"(\w+)\s+cerb_confusion_matrix\(([^)]*)\);", text)
    assert m and m.group(1) == "int"
    fn = _lib.load().cerb_confusion_matrix
    assert fn.restype is ctypes.c_int
    params = [" ".join(p.split()) for p in m.group(2).split(",")]
    assert len(params) == len(fn.argtypes)
    for p, t in zip(params, fn.argtypes):
        if "*" in p:
            assert t is ctypes.c_void_p, p
        else:
            assert t is {"int": ctypes.c_int, "double": ctypes.c_double}[p.split()[0]], p


def test_confusion_abi_validation_without_gpu():
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)

    def call(B=2, max_det=300, n_labels=10, nc=20, iou=0.45, offsets=fake, status=fake, dets=fake, labels=fake):
        return lib.cerb_confusion_matrix(dets, fake, B, max_det, labels, offsets, n_labels, nc, 0.25, iou, fake, None, status, None)

    def refused(fragment, **kw):
        return call(**kw) == _lib.CERB_EINVAL and fragment in lib.cerb_last_error()

    assert refused(b"negative size", B=-1)
    assert refused(b"negative size", n_labels=-1)
    assert refused(b"max_det=30001", max_det=30001)
    assert refused(b"max_det=-1", max_det=-1)
    assert refused(b"nc=0", nc=0)
    assert refused(b"nc=32768", nc=32768)
    assert refused(b"iou_thres", iou=-0.1)
    assert refused(b"iou_thres", iou=float("nan"))
    assert refused(b"without label_offsets", offsets=None)  # B = 2
    assert refused(b"without label_offsets", offsets=None, B=1, n_labels=1025)
    assert refused(b"null argument", status=None)
    assert refused(b"null argument", dets=None)
    assert refused(b"null argument", labels=None)
    assert call(B=0) == 0  # nothing to do, nothing launched


# ---------------------------------------------------------------------------- the patch, on stand-in reference modules
@pytest.fixture()
def stub_reference(monkeypatch):
    """The modules ``patch.install(confusion=True)`` touches, as stand-ins; ``ConfusionMatrix`` is the reference's text."""
    mods = {}
    for name in ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general",
                 "cerberusdet.utils.metrics"):
        mods[name] = types.ModuleType(name)
        monkeypatch.setitem(sys.modules, name, mods[name])
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = lambda *a, **k: None
    mods["cerberusdet.utils.metrics"].ConfusionMatrix = type("ConfusionMatrix", (cp.ConfusionMatrixVerbatim,),
                                                             {"process_batch": cp.ConfusionMatrixVerbatim.process_batch})
    from cerberusdet_b200 import patch

    patch.uninstall()
    yield mods
    patch.uninstall()
    if hasattr(mods["cerberusdet.models.yolo"].Detect, "_cerb_reference_forward"):
        del mods["cerberusdet.models.yolo"].Detect._cerb_reference_forward


def test_install_confusion_rebinds_process_batch_on_the_class(stub_reference):
    from cerberusdet_b200 import patch

    cls = stub_reference["cerberusdet.utils.metrics"].ConfusionMatrix
    original = cls.process_batch
    info = patch.install(confusion=True)
    assert "cerberusdet.utils.metrics.ConfusionMatrix.process_batch" in info["patched"]
    assert stub_reference["cerberusdet.utils.metrics"].ConfusionMatrix is cls  # the class itself is kept
    assert cls.process_batch is not original and cls.process_batch._cerb_reference is original
    assert patch.install(confusion=True) == {"already": ["installed"]}
    # CPU tensors (everything without a GPU) run the reference's own method: same matrix as the text
    rng = np.random.default_rng(4)
    dets, labels = cp.image_case(rng, 12, 50, 20)
    cm, want = cls(20), cp.ConfusionMatrixVerbatim(20)
    cm.process_batch(dets, labels)
    cm.process_batch(None, labels[:, 0])
    want.process_batch(dets, labels)
    want.process_batch(None, labels[:, 0])
    assert np.array_equal(cm.matrix, want.matrix)
    patch.uninstall()
    assert cls.process_batch is original
    assert not any("ConfusionMatrix" in p for p in patch.install()["patched"])  # a switch of its own
    assert patch.install(confusion=True)["patched"] == ["cerberusdet.utils.metrics.ConfusionMatrix.process_batch"]


class _FakeCuda:
    """Stands in for a CUDA tensor in the guard: only what ``_confusion_on_path`` reads."""

    def __init__(self, t, device="cuda:0"):
        self.t, self.is_cuda, self.device, self.dtype, self.shape = t, True, device, t.dtype, t.shape

    def dim(self):
        return self.t.dim()


@pytest.mark.parametrize("what", ["none", "cpu", "fp16", "fp64_labels", "other_device", "n30001", "m1025", "shape",
                                  "neg_iou", "nc0", "matrix_shape", "status"])
def test_dropin_sends_off_path_calls_to_the_reference(what, monkeypatch):
    from cerberusdet_b200 import ops, val_stats

    calls = []

    def reference(self, detections, labels):
        calls.append(what)
        return "reference"

    dets, labels = cp.image_case(np.random.default_rng(1), 5, 20, 20)
    cm = cp.ConfusionMatrixVerbatim(20)
    d, l = _FakeCuda(dets), _FakeCuda(labels)
    if what == "none":
        d, l = None, _FakeCuda(labels[:, 0])
    elif what == "cpu":
        d, l = dets, labels
    elif what == "fp16":
        d = _FakeCuda(dets.half())
    elif what == "fp64_labels":
        l = _FakeCuda(labels.double())
    elif what == "other_device":
        l = _FakeCuda(labels, "cuda:1")
    elif what == "n30001":
        d = _FakeCuda(torch.zeros(30001, 6))
    elif what == "m1025":
        l = _FakeCuda(torch.zeros(1025, 5))
    elif what == "shape":
        d = _FakeCuda(dets[:, :5])
    elif what == "neg_iou":
        cm.iou_thres = -0.1
    elif what == "nc0":
        cm = cp.ConfusionMatrixVerbatim(0)
    elif what == "matrix_shape":
        cm.matrix = np.zeros((5, 5))
    launched = []

    def cells(detections, labels, nc, conf, iou_thres):  # the kernel's answer: status 1 (a class outside [0, nc))
        launched.append(1)
        return torch.tensor([1] + [-1] * 25, dtype=torch.int32)

    monkeypatch.setattr(ops, "confusion_cells", cells)
    before = cm.matrix.copy()
    fn = val_stats.make_confusion_process_batch(reference)
    assert fn._cerb_reference is reference
    assert fn(cm, d, l) == "reference" and calls == [what]
    assert launched == ([1] if what == "status" else [])
    assert np.array_equal(cm.matrix, before)  # the fallback found the matrix untouched


def test_dropin_applies_cells_with_add_at(monkeypatch):
    from cerberusdet_b200 import ops, val_stats

    dets, labels = cp.image_case(np.random.default_rng(2), 3, 4, 20)
    W = 21
    host = [0, 5 * W + 1, 20 * W + 2, 5 * W + 1, -1, 7 * W + 20, 7 * W + 20, -1]  # status, 3 labels, 4 detections
    monkeypatch.setattr(ops, "confusion_cells", lambda *a: torch.tensor(host, dtype=torch.int32))
    cm = cp.ConfusionMatrixVerbatim(20)
    cm.matrix[0, 0] = 4
    val_stats.make_confusion_process_batch(None)(cm, _FakeCuda(dets), _FakeCuda(labels))
    want = np.zeros((21, 21))
    want[0, 0], want[5, 1], want[20, 2], want[7, 20] = 4, 2, 1, 2
    assert np.array_equal(cm.matrix, want)
