"""GPU tests of the mAP statistics (``cerb_ap_per_class`` / ``ops.ap_per_class`` / the ``val_stats.ap_per_class``
drop-in): every output bit-equal to the numpy port (tests/ap_port.py) under the tie rule "conf descending, then row
index", at VOC and Objects365 sizes, with fp16-derived (massively tied) scores and at the edges."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import ap_port  # noqa: E402

pytestmark = pytest.mark.gpu


def _ops():
    from cerberusdet_b200 import ops

    return ops


def _dropin():
    from cerberusdet_b200 import val_stats

    return val_stats.ap_per_class


def _cuda(*arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def _check_arrays(stats, eps=1e-16):
    tp, conf, pred_cls, target_cls = stats
    got = [t.cpu().numpy() for t in _ops().ap_per_class(*_cuda(tp, conf, pred_cls, target_cls), eps=eps)]
    want = ap_port.ap_arrays_port(tp, conf, pred_cls, target_cls, eps)
    for name, a, b in zip(("ap", "p", "r", "unique_classes", "nt"), got, want):
        assert a.shape == b.shape, name
        assert np.array_equal(a, b), f"{name}: {np.count_nonzero(a != b)} of {a.size} differ, max |d| {np.abs(a - b).max()}"
    return got


def _check_dropin(stats, names=None):
    tp, conf, pred_cls, target_cls = stats
    names = names if names is not None else {k: str(k) for k in range(400)}
    got = _dropin()(tp, conf, pred_cls, target_cls, names=names)
    want = ap_port.ap_per_class_port(tp, conf, pred_cls, target_cls, names)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), f"output {k}"
    return got


def test_voc_size_bit_equal():
    stats = ap_port.make_stats(1_490_000, 20, seed=1, unlabelled=1, unpredicted=1)
    _check_arrays(stats)
    _check_dropin(stats)


def test_objects365_size_bit_equal():
    """80 000 images x 300 detections, 365 Zipf-skewed classes: the drop-in's seven outputs against the port."""
    stats = ap_port.make_stats(24_000_000, 365, seed=2, label_ratio=0.05)
    got = _check_dropin(stats)
    assert got[5].shape == (365, 10) and (got[5][:, 0] > 0).all()


def test_fp16_scores_tie_massively_and_stay_bit_equal():
    stats = ap_port.make_stats(2_000_000, 80, seed=3, fp16_conf=True)
    assert np.unique(stats[1]).size < 20000  # > 99 % of the rows share their score with another row
    _check_arrays(stats)
    _check_dropin(stats)


@pytest.mark.parametrize("K", [1, 32])
def test_k_extremes(K):
    _check_arrays(ap_port.make_stats(50_000, 7, K=K, seed=K))


def test_empty_and_tiny_inputs():
    ops = _ops()
    tp, conf, pred_cls, target_cls = ap_port.make_stats(1000, 5, seed=4)
    # N = 0: every class keeps zero rows
    ap, p, r, uc, nt = ops.ap_per_class(*_cuda(tp[:0], conf[:0], pred_cls[:0], target_cls))
    assert ap.shape == (5, 10) and not ap.any() and not p.any() and not r.any() and nt.sum() == target_cls.size
    _check_dropin((tp[:0], conf[:0], pred_cls[:0], target_cls))
    # nc = 0: no label at all
    ap, p, r, uc, nt = ops.ap_per_class(*_cuda(tp, conf, pred_cls, target_cls[:0]))
    assert ap.shape == (0, 10) and p.shape == (0, 1000) and uc.numel() == 0
    _check_dropin((tp, conf, pred_cls, target_cls[:0]))  # (numpy warns of the mean of an empty slice, as in the reference)
    # a single detection, TP and FP
    for v in (True, False):
        _check_arrays((np.full((1, 10), v), np.array([0.7], np.float32), np.array([2.0], np.float32), np.array([2.0, 2.0, 3.0], np.float32)))


def test_all_tp_and_all_fp_columns():
    tp, conf, pred_cls, _ = ap_port.make_stats(40_000, 6, seed=6)
    tp = tp.copy()
    tp[:, 0] = False  # all FP
    target_cls = np.repeat(np.arange(6, dtype=np.float32), 40_000)  # enough labels that every detection may be a TP
    tp[:, 1] = True  # all TP
    _check_arrays((tp, conf, pred_cls, target_cls))
    _check_dropin((tp, conf, pred_cls, target_cls))


def test_unlabelled_unpredicted_and_non_integer_classes():
    tp, conf, pred_cls, target_cls = ap_port.make_stats(60_000, 9, seed=7, unlabelled=3, unpredicted=3)
    _check_arrays((tp, conf, pred_cls, target_cls))
    shift = lambda c: (c * 0.37 - 1.5).astype(np.float32)  # noqa: E731  non-integer, negative class values
    pc = shift(pred_cls)
    pc[::97] = np.nan  # a NaN class matches nothing
    _check_arrays((tp, conf, pc, shift(target_cls)))


def test_signed_zero_confidences_are_one_value():
    tp, conf, pred_cls, target_cls = ap_port.make_stats(20_000, 4, seed=8)
    conf = conf.copy()
    conf[::3] = 0.0
    conf[1::3] = -0.0
    _check_arrays((tp, conf, pred_cls, target_cls))
    # swapping the zero signs changes nothing: they compare equal, ties go by row index
    conf2 = conf.copy()
    conf2[::3], conf2[1::3] = -0.0, 0.0
    a = [t.cpu() for t in _ops().ap_per_class(*_cuda(tp, conf, pred_cls, target_cls))]
    b = [t.cpu() for t in _ops().ap_per_class(*_cuda(tp, conf2, pred_cls, target_cls))]
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_one_class_holds_most_rows():
    """A class with 70 % of 3 M rows: its segment spans thousands of tiles."""
    tp, conf, pred_cls, target_cls = ap_port.make_stats(3_000_000, 30, seed=9, zipf=3.0)
    assert np.mean(pred_cls == 0) > 0.5
    _check_arrays((tp, conf, pred_cls, target_cls))


def test_same_bits_twice_and_for_numpy_or_cuda_inputs():
    stats = ap_port.make_stats(500_000, 40, seed=10, fp16_conf=True)
    a = [t.cpu() for t in _ops().ap_per_class(*_cuda(*stats))]
    b = [t.cpu() for t in _ops().ap_per_class(*_cuda(*stats))]
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    names = {k: str(k) for k in range(40)}
    from_numpy = _dropin()(*stats, names=names)
    from_cuda = _dropin()(*_cuda(*stats), names=names)
    assert all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(from_numpy, from_cuda))


def test_nan_raises_in_the_op():
    tp, conf, pred_cls, target_cls = ap_port.make_stats(1000, 3, seed=11)
    bad = target_cls.copy()
    bad[0] = np.nan
    with pytest.raises(ValueError, match="target_cls"):
        _ops().ap_per_class(*_cuda(tp, conf, pred_cls, bad))
    bad = conf.copy()
    bad[5] = np.nan
    with pytest.raises(ValueError, match="conf"):
        _ops().ap_per_class(*_cuda(tp, bad, pred_cls, target_cls))


def test_abi_rejects_through_the_library():
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    tp, conf, pred_cls, target_cls = (t for t in _cuda(*ap_port.make_stats(1000, 3, seed=12)))
    n = 1000
    ap = torch.empty((3, 10), dtype=torch.float64, device="cuda")
    pr = torch.empty((2, 3, 1000), dtype=torch.float64, device="cuda")
    need = int(lib.cerb_ap_workspace_bytes(n, 10, 3))
    assert need > 0
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    nl = (ctypes.c_longlong * 3)(5, 5, 5)

    def call(classes, ws_bytes=need, n_=n, K=10):
        return lib.cerb_ap_per_class(tp.data_ptr(), K, conf.data_ptr(), pred_cls.data_ptr(), n_, classes, nl, 3, 1e-16,
                                     ap.data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(), ws.data_ptr(), ws_bytes,
                                     torch.cuda.current_stream().cuda_stream)

    ok = (ctypes.c_float * 3)(0.0, 1.0, 2.0)
    assert call((ctypes.c_float * 3)(1.0, 0.0, 2.0)) == _lib.CERB_EINVAL
    assert call((ctypes.c_float * 3)(0.0, 0.0, 2.0)) == _lib.CERB_EINVAL
    assert call(ok, n_=-5) == _lib.CERB_EINVAL
    assert call(ok, K=33) == _lib.CERB_EINVAL
    assert call(ok, ws_bytes=need - 1) == _lib.CERB_ENOSPC and b"workspace" in lib.cerb_last_error()
    assert call(ok) == 0
    torch.cuda.synchronize()


@pytest.mark.reference
@pytest.mark.skipif(not __import__("oracle.ref_import", fromlist=["x"]).reference_available(), reason="needs the reference tree")
def test_reference_ap_per_class_equals_dropin_without_ties():
    """The unmodified reference ``ap_per_class`` (utils/metrics.py:56-120) on tie-free scores, output by output."""
    from oracle.ref_import import load_reference

    load_reference()
    import cerberusdet.utils.metrics as metrics

    tp, _, pred_cls, target_cls = ap_port.make_stats(300_000, 20, seed=13, unlabelled=1, unpredicted=1)
    conf = np.random.default_rng(13).permutation(np.linspace(1e-4, 1, tp.shape[0], dtype=np.float32))
    assert np.unique(conf).size == conf.size
    names = {k: str(k) for k in range(22)}
    want = metrics.ap_per_class(tp, conf, pred_cls, target_cls, plot=False, names=names)
    got = _dropin()(tp, conf, pred_cls, target_cls, names=names)
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(np.asarray(a), np.asarray(b)), f"output {k}"
