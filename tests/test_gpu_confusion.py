"""GPU tests of the validation confusion matrix (``cerb_confusion_matrix``, ``ops.confusion_matrix_batch``, the
``ConfusionMatrix.process_batch`` drop-in and ``validation_batch_statistics(confusion=...)``): every matrix bit-equal to
the canonical port (tests/confusion_port.py), and to the reference's text where no IoU ties."""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import confusion_port as cp  # noqa: E402

pytestmark = pytest.mark.gpu


def _ops():
    from cerberusdet_b200 import ops

    return ops


def _kernel_batch(dets, counts, labels, offsets, nc, conf=0.25, iou_thres=0.45):
    offs = torch.tensor(offsets, dtype=torch.int32, device="cuda")
    m, status = _ops().confusion_matrix_batch(dets.cuda(), counts.cuda(), labels.cuda(), offs, nc, conf, iou_thres)
    assert m.dtype == torch.int64 and tuple(m.shape) == (nc + 1, nc + 1)
    return m.cpu().numpy(), status.cpu()


def _check_batch(case, nc, conf=0.25, iou_thres=0.45):
    dets, counts, labels, offsets = case
    got, status = _kernel_batch(dets, counts, labels, offsets, nc, conf, iou_thres)
    assert not status.any()
    want = cp.batch_port(dets, counts, labels, offsets, nc, conf, iou_thres)
    assert np.array_equal(got, want), f"{np.count_nonzero(got != want)} cells differ"
    return got


def _dropin():
    from cerberusdet_b200 import val_stats

    return val_stats.make_confusion_process_batch(cp.ConfusionMatrixVerbatim.process_batch)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_voc_like_batches(seed):
    m = _check_batch(cp.batch_case(seed, 32, 20, m_range=(0, 40)), 20)
    assert m[:20, :20].trace() > 0 and m[20, :20].sum() > 0 and m[:20, 20].sum() > 0


def test_objects365_like_batch():
    _check_batch(cp.batch_case(7, 32, 365, m_range=(0, 120)), 365)


def test_crowded_images():
    case = cp.batch_case(8, 16, 20, m_range=(60, 200), n_range=(200, 300), crowd=0.97)
    dets, counts, labels, offsets = case
    iou = cp.box_iou(labels[offsets[0] : offsets[1], 1:], dets[0, : counts[0], :4])
    assert (iou > 0.45).sum() > 300  # many pairs above the threshold per image
    _check_batch(case, 20)
    _check_batch(case, 20, conf=0.001, iou_thres=0.1)


def test_exact_iou_ties_follow_the_canonical_rule():
    case = cp.batch_case(9, 16, 5, m_range=(5, 40), n_range=(50, 300), crowd=0.9, grid=True)
    dets, counts, labels, offsets = case
    assert cp.has_ties(dets[0, : counts[0]], labels[offsets[0] : offsets[1]])
    _check_batch(case, 5)


def test_tie_free_batches_equal_the_reference_text():
    case = cp.batch_case(10, 32, 20, m_range=(1, 30))
    dets, counts, labels, offsets = case
    assert not any(cp.has_ties(dets[b, : counts[b]], labels[offsets[b] : offsets[b + 1]]) for b in range(32))
    got, _ = _kernel_batch(*case, 20)
    assert np.array_equal(got, cp.batch_port(*case, 20, cls=cp.ConfusionMatrixVerbatim))


def test_threshold_equality_follows_torch_on_this_gpu():
    """IoU == fp32(0.45) and conf == fp32(0.25) exactly: not above the thresholds, as torch's own ``>`` decides on CUDA."""
    labels = torch.tensor([[1.0, 0, 0, 20, 20], [2.0, 100, 100, 120, 120]])
    eps = np.nextafter(np.float32(0.25), np.float32(1))
    dets = torch.tensor([[0, 0, 10, 18, 0.9, 3],  # IoU 180 / 400 == fp32(0.45)
                         [100, 100, 110, 118.5, 0.25, 4],  # IoU above 0.45, conf == 0.25: filtered
                         [100, 100, 110, 118.5, float(eps), 5],  # the next float above 0.25: kept
                         [300, 300, 310, 310, 0.5, 6]])
    iou = cp.box_iou(labels[:, 1:].cuda(), dets[:, :4].cuda())
    assert iou[0, 0].item() == np.float32(0.45) and not bool(iou[0, 0] > 0.45)
    assert not bool(dets[1, 4].cuda() > 0.25) and bool(dets[2, 4].cuda() > 0.25)
    want = cp.ConfusionMatrixVerbatim(10)
    want.process_batch(dets.cuda(), labels.cuda())  # the reference's text, with torch's comparisons on this GPU
    got, _ = _kernel_batch(dets[None], torch.tensor([4], dtype=torch.int32), labels, [0, 2], 10)
    assert np.array_equal(got, want.matrix)
    assert got[10, 1] == 1 and got[5, 2] == 1 and got[3, 10] == 1 and got[6, 10] == 1


def test_nan_conf_and_nan_boxes():
    dets, counts, labels, offsets = cp.batch_case(11, 16, 20, m_range=(1, 30))
    dets[:, ::7, 4] = float("nan")
    dets[:, 3::11, 1] = float("nan")
    labels[::9, 3] = float("nan")
    _check_batch((dets, counts, labels, offsets), 20)


def test_largest_image():
    """M = 1024 labels and N = 30000 detections in one image."""
    rng = np.random.default_rng(12)
    d, lab = cp.image_case(rng, 1024, 30000, 80, size=4000.0)
    _check_batch((d[None], torch.tensor([30000], dtype=torch.int32), lab, [0, 1024]), 80, conf=0.001)
    cm = cp.ConfusionMatrixPort(80, 0.001)
    cm.process_batch(d, lab)
    mine = cp.ConfusionMatrixVerbatim(80, 0.001)
    _dropin()(mine, d.cuda(), lab.cuda())
    assert np.array_equal(mine.matrix, cm.matrix)


def test_more_than_1024_labels_sets_the_status():
    dets, counts, labels, offsets = cp.batch_case(13, 3, 20, m_range=(5, 10))
    extra = labels[:1].repeat(1025, 1)
    labels2 = torch.cat((labels[: offsets[2]], extra, labels[offsets[2] :]))  # image 1: its labels and 1025 more
    offsets2 = [0, offsets[1], offsets[2] + 1025, offsets[3] + 1025]
    got, status = _kernel_batch(dets, counts, labels2, offsets2, 20)
    assert status.tolist() == [0, 2, 0]
    rest = torch.cat((labels[: offsets[1]], labels[offsets[2] :]))
    want = cp.batch_port(dets[[0, 2]], counts[[0, 2]], rest, [0, offsets[1], offsets[1] + offsets[3] - offsets[2]], 20)
    assert np.array_equal(got, want)


def test_dropin_equals_the_port_and_the_batched_op_its_sum():
    dets, counts, labels, offsets = cp.batch_case(14, 48, 20, m_range=(0, 30))
    dropin = _dropin()
    mine, port = cp.ConfusionMatrixVerbatim(20), cp.ConfusionMatrixPort(20)
    for b in range(48):
        lab, n = labels[offsets[b] : offsets[b + 1]], int(counts[b])
        if lab.shape[0] == 0:
            continue
        args = (dets[b, :n].cuda(), lab.cuda()) if n else (None, lab[:, 0].cuda())
        dropin(mine, *args)
        port.process_batch(*args)
    assert np.array_equal(mine.matrix, port.matrix)
    got, _ = _kernel_batch(dets, counts, labels, offsets, 20)
    assert np.array_equal(got, mine.matrix)


def test_same_bits_twice_and_out_accumulates():
    case = cp.batch_case(15, 32, 20, crowd=0.9)
    a, sa = _kernel_batch(*case, 20)
    b, sb = _kernel_batch(*case, 20)
    assert np.array_equal(a, b) and torch.equal(sa, sb)
    dets, counts, labels, offsets = case
    out = torch.full((21, 21), 3, dtype=torch.int64, device="cuda")
    offs = torch.tensor(offsets, dtype=torch.int32, device="cuda")
    for _ in range(2):
        m, _ = _ops().confusion_matrix_batch(dets.cuda(), counts.cuda(), labels.cuda(), offs, 20, out=out)
        assert m is out
    assert np.array_equal(out.cpu().numpy(), 2 * a + 3)


def test_cuda_graph_replay_on_fresh_inputs():
    ops = _ops()
    B, max_det, L = 16, 300, 16 * 40
    first = cp.batch_case(16, B, 20, m_range=(40, 40))
    dets, counts = first[0].cuda(), first[1].cuda()
    labels = first[2].cuda()
    offs = torch.tensor(first[3], dtype=torch.int32, device="cuda")
    assert labels.shape[0] == L
    matrix = torch.zeros((21, 21), dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.confusion_matrix_batch(dets, counts, labels, offs, 20, out=matrix)  # warm-up
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        matrix.zero_()
        _, status = ops.confusion_matrix_batch(dets, counts, labels, offs, 20, out=matrix)
    for seed in (17, 18, 19):
        d, c, lab, o = cp.batch_case(seed, B, 20, m_range=(40, 40))
        dets.copy_(d)
        counts.copy_(c)
        labels.copy_(lab)
        offs.copy_(torch.tensor(o, dtype=torch.int32))
        g.replay()
        torch.cuda.synchronize()
        assert not status.any()
        assert np.array_equal(matrix.cpu().numpy(), cp.batch_port(d, c, lab, o, 20)), seed


def test_opcheck():
    dets, counts, labels, offsets = cp.batch_case(20, 4, 20, max_det=50, m_range=(0, 10), n_range=(0, 50))
    args = (dets.cuda(), counts.cuda(), labels.cuda(), torch.tensor(offsets, dtype=torch.int32, device="cuda"), 20, 0.25, 0.45,
            torch.zeros((21, 21), dtype=torch.int64, device="cuda"))
    torch.library.opcheck(torch.ops.cerb.confusion_matrix.default, args)


def test_out_of_range_classes_keep_the_reference_behaviour():
    dets, labels = cp.image_case(np.random.default_rng(21), 10, 40, 20)
    dropin = _dropin()
    for what, value in (("label", 20.0), ("label", -1.0), ("det", 20.0), ("det", -3.0), ("label", 25.0), ("det", 25.0)):
        d, lab = dets.clone(), labels.clone()
        if what == "label":
            lab[2, 0] = value
        else:
            d[0, 5] = value  # the highest-conf detection: always above conf
        _, status = _kernel_batch(d[None], torch.tensor([40], dtype=torch.int32), lab, [0, 10], 20)
        assert status.tolist() == [1]
        want, mine = cp.ConfusionMatrixVerbatim(20), cp.ConfusionMatrixVerbatim(20)
        try:
            want.process_batch(d.cuda(), lab.cuda())
        except IndexError:
            with pytest.raises(IndexError):
                dropin(mine, d.cuda(), lab.cuda())
            continue
        dropin(mine, d.cuda(), lab.cuda())
        assert np.array_equal(mine.matrix, want.matrix), (what, value)


def _syncs(fn):
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            fn()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    return sum("synchroniz" in str(x.message) for x in w)


def test_one_synchronisation_per_dropin_call_none_in_the_batched_op():
    ops = _ops()
    dets, labels = cp.image_case(np.random.default_rng(22), 10, 100, 20)
    d, lab = dets.cuda(), labels.cuda()
    cm = cp.ConfusionMatrixVerbatim(20)
    dropin = _dropin()
    dropin(cm, d, lab)  # warm-up (module load)
    assert _syncs(lambda: dropin(cm, d, lab)) == 1
    assert _syncs(lambda: cp.ConfusionMatrixVerbatim(20).process_batch(d, lab)) > 10  # the reference's text
    bd, bc, bl, bo = (x.cuda() if torch.is_tensor(x) else torch.tensor(x, dtype=torch.int32, device="cuda")
                      for x in cp.batch_case(23, 32, 20))
    out = torch.zeros((21, 21), dtype=torch.int64, device="cuda")
    ops.confusion_matrix_batch(bd, bc, bl, bo, 20, out=out)
    assert _syncs(lambda: ops.confusion_matrix_batch(bd, bc, bl, bo, 20, out=out)) == 0


def test_validation_batch_statistics_feeds_the_matrix():
    from cerberusdet_b200 import ops, val_stats

    dets, counts, labels, offsets = cp.batch_case(24, 8, 20, m_range=(0, 25))
    B = 8
    bidx = torch.cat([torch.full((offsets[b + 1] - offsets[b],), b) for b in range(B)]).float()
    xyxy = labels[:, 1:].clamp(1, 630) / 640
    xywh = torch.cat(((xyxy[:, :2] + xyxy[:, 2:]) / 2, xyxy[:, 2:] - xyxy[:, :2]), 1)
    batch = {"img": torch.zeros(B, 3, 640, 640), "batch_idx": bidx, "cls": labels[:, :1], "bboxes": xywh,
             "ori_shape": [(480, 640)] * B, "ratio_pad": None}
    iouv = torch.linspace(0.5, 0.95, 10, device="cuda")
    seen, real = [], ops.confusion_matrix_batch

    def spy(*a, **k):
        seen.append([x.clone() if torch.is_tensor(x) else x for x in a])
        return real(*a, **k)

    plain = val_stats.validation_batch_statistics(dets.cuda(), counts.cuda(), batch, iouv)
    matrix = torch.zeros((21, 21), dtype=torch.int64, device="cuda")
    ops.confusion_matrix_batch = spy
    try:
        with_cm = val_stats.validation_batch_statistics(dets.cuda(), counts.cuda(), batch, iouv, confusion=matrix)
    finally:
        ops.confusion_matrix_batch = real
    assert len(plain) == len(with_cm) and all(torch.equal(x, y) for s, t in zip(plain, with_cm) for x, y in zip(s, t))
    predn, c, labelsn, offs, nc = seen[0][:5]
    assert nc == 20 and offs.tolist() == offsets
    want = cp.batch_port(predn.cpu(), c.cpu(), labelsn.cpu(), offsets, 20)
    assert want.sum() > 0 and np.array_equal(matrix.cpu().numpy(), want)
    bad = dict(batch, cls=batch["cls"].clone())
    bad["cls"][0] = 20.0
    with pytest.raises(ValueError, match="outside"):
        val_stats.validation_batch_statistics(dets.cuda(), counts.cuda(), bad, iouv, confusion=matrix)


@pytest.mark.reference
@pytest.mark.skipif(not __import__("oracle.ref_import", fromlist=["x"]).reference_available(), reason="needs the reference tree")
def test_reference_confusion_matrix_equals_dropin_without_ties():
    """The unmodified reference ``ConfusionMatrix`` (utils/metrics.py:273-370) against the patched class."""
    from oracle.ref_import import load_reference

    load_reference()
    import cerberusdet.utils.metrics as metrics

    from cerberusdet_b200 import patch

    dets, counts, labels, offsets = cp.batch_case(25, 32, 20, m_range=(1, 30))
    want = metrics.ConfusionMatrix(20)
    for b in range(32):
        want.process_batch(dets[b, : counts[b]].cuda(), labels[offsets[b] : offsets[b + 1]].cuda())
    patch.uninstall()
    patch.install(confusion=True)
    try:
        got = metrics.ConfusionMatrix(20)
        for b in range(32):
            got.process_batch(dets[b, : counts[b]].cuda(), labels[offsets[b] : offsets[b + 1]].cuda())
    finally:
        patch.uninstall()
    assert np.array_equal(got.matrix, want.matrix)
