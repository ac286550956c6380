"""The oracle (oracle/ref_port.py + oracle/greedy_nms.c) against the golden vectors that
oracle/gen_golden.py produced by executing the unmodified reference."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import golden_manifest, golden_names, load_golden, split_rows
from cerberusdet_b200.synth import STRIDES
from oracle import ref_port as rp


ROUNDINGS = 4


def assert_matches_golden(got, want, terms, sum_dtype=None):
    """``got`` equals the golden ``want`` bit for bit, or every element lies within ROUNDINGS roundings of its own value
    in the output dtype plus ROUNDINGS roundings in ``sum_dtype`` (default: the output dtype) of ``terms``, the magnitude
    of what that element is summed from.  CPU convolution, matrix-product and reduction kernels (ATen, MKL, oneDNN)
    choose their summation order by instruction set, CPU vendor and thread count, so on a host other than the one that
    produced the vectors the last bits may differ; the bound is per element, so an error of the port itself (a shifted
    box, a changed logit, a missing bias) does not fit in it (test_golden_bounds_reject_port_errors)."""
    got = got.detach()
    assert got.dtype == want.dtype and got.shape == want.shape
    if torch.equal(got, want):
        return
    eps, sum_eps = torch.finfo(want.dtype).eps, torch.finfo(sum_dtype or want.dtype).eps
    bound = ROUNDINGS * (eps * want.double().abs() + sum_eps * terms.double())
    bad = (got.double() - want.double()).abs() > bound
    assert not bad.any(), (f"{int(bad.sum())} of {bad.numel()} elements differ by more than {ROUNDINGS} roundings of their "
                           f"value and terms, the first at {tuple(bad.nonzero()[0].tolist())}")


def decode_terms(y):
    """Per-element magnitude of the terms of a decoded ``y [B, 4+nc, A]``: the corners (c -+ size/2) that centre and size
    are computed from, |c| + |size|/2, and the sigmoid scores themselves."""
    y = y.double().abs()
    t = y.clone()
    t[:, 0] = t[:, 2] = y[:, 0] + y[:, 2] / 2
    t[:, 1] = t[:, 3] = y[:, 1] + y[:, 3] / 2
    return t


def head_tail_case(g):
    """The inputs of the two convolutions of every level, and per level the magnitude of the terms of each raw output:
    the same convolutions on absolute values.  (CPU convolutions of half tensors sum in float32.)"""
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    args = [[t(f"{k}{i}") for i in range(3)] for k in ("box_feat", "cls_feat", "box_w", "box_b", "cls_w", "cls_b")]
    a = lambda x: x.double().abs()  # noqa: E731
    terms = [torch.cat((F.conv2d(a(bf), a(bw), a(bb)), F.conv2d(a(cf), a(cw), a(cb))), 1) for bf, cf, bw, bb, cw, cb in zip(*args)]
    return args, terms


@pytest.mark.parametrize("name", golden_names("decode"))
def test_decode_port_matches_golden(name):
    g = load_golden(name)
    nc = golden_manifest()[name]["nc"]
    levels = [torch.from_numpy(g[f"level{i}"]) for i in range(3)]
    y = rp.decode_port(levels, nc, STRIDES)
    want = torch.from_numpy(g["y"])
    assert_matches_golden(y, want, decode_terms(want))


@pytest.mark.parametrize("greedy", ["torchvision", "c"])
@pytest.mark.parametrize("name", golden_names("nms"))
def test_nms_port_bit_exact(name, greedy):
    g = load_golden(name)
    kw = dict(golden_manifest()[name]["kwargs"])
    pred = torch.from_numpy(g["pred"])
    want = split_rows(g["rows"], g["counts"])
    got = rp.nms_port(pred, greedy=greedy, **kw)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a.dtype == torch.float32 and a.shape == b.shape
        assert torch.equal(a, b)


def test_greedy_c_matches_torchvision_random():
    import torchvision

    gen = torch.Generator().manual_seed(5)
    for n in (0, 1, 2, 65, 700, 3000):
        c = torch.rand(n, 2, generator=gen) * 200
        wh = torch.rand(n, 2, generator=gen) * 60
        boxes = torch.cat((c - wh / 2, c + wh / 2), 1)
        boxes[n // 2 :] = boxes[n // 2 :].round()  # integer boxes: many exact-equality IoUs
        scores = torch.rand(n, generator=gen).sort(descending=True).values
        for thr in (0.0, 0.1, 0.45, 0.5, 0.6, 0.7, 1.0):
            assert torch.equal(torchvision.ops.nms(boxes, scores, thr), rp.greedy_nms_c(boxes, thr))


def test_threshold_rounding_rules():
    # conf threshold is compared in the tensor dtype (utils/general.py:411)
    h = torch.tensor([0.30005], dtype=torch.float16)
    pred = torch.zeros(1, 5, 1, dtype=torch.float16)
    pred[0, :4, 0] = torch.tensor([10, 10, 4, 4], dtype=torch.float16)
    pred[0, 4, 0] = h
    assert rp.nms_port(pred, conf_thres=0.3)[0].shape[0] == 0  # half(0.3) == 0.30005, not >
    f = torch.tensor(np.float32(0.3))
    pred32 = pred.float()
    pred32[0, 4, 0] = f
    assert rp.nms_port(pred32, conf_thres=0.3)[0].shape[0] == 0
    pred32[0, 4, 0] = torch.tensor(np.nextafter(np.float32(0.3), np.float32(1)))
    assert rp.nms_port(pred32, conf_thres=0.3)[0].shape[0] == 1


def test_asserts_like_reference():
    pred = torch.zeros(1, 6, 4)
    with pytest.raises(AssertionError):
        rp.nms_port(pred, conf_thres=1.5)
    with pytest.raises(AssertionError):
        rp.nms_port(pred, iou_thres=-0.1)


@pytest.mark.parametrize("name", golden_names("model"))
def test_real_model_config1_vectors(name):
    """BASELINE config 1: vectors produced by the real 2-task CerberusDet model graph (random init) on the CPU."""
    g = load_golden(name)
    meta = golden_manifest()[name]
    levels = [torch.from_numpy(g[f"level{i}"]) for i in range(3)]
    y = torch.from_numpy(g["y"])
    assert_matches_golden(rp.decode_port(levels, meta["nc"], STRIDES), y, decode_terms(y))
    for greedy in ("torchvision", "c"):  # selection on the reference's own decoded tensor: bit for bit
        got = rp.nms_port(y, greedy=greedy, **meta["kwargs"])
        want = split_rows(g["rows"], g["counts"])
        assert len(got) == 1 and torch.equal(got[0], want[0])


# ------------------------------------------------------------------ training-time sibling decode (SURVEY 8f-4)
@pytest.mark.parametrize("name", golden_names("train_bbox"))
def test_bbox_decode_port_matches_golden(name):
    """The oracle restatement of Loss.bbox_decode (utils/loss.py:126-131) against vectors the unmodified reference
    produced (oracle/gen_golden_train.py): forward and the autograd gradient (assert_matches_golden)."""
    from oracle import ref_port as rp

    g = load_golden(name)
    pred = torch.from_numpy(g["pred"]).requires_grad_(True)
    anchors = torch.from_numpy(g["anchor_points"])
    out = rp.bbox_decode_port(anchors, pred)
    want, grad_out = torch.from_numpy(g["out"]), torch.from_numpy(g["grad_out"])
    corner_anchor = anchors.double().repeat(1, 2)  # (x, y, x, y) of every anchor
    assert_matches_golden(out, want, corner_anchor.abs() + (want.double() - corner_anchor).abs())  # anchor -+ distance
    (grad_in,) = torch.autograd.grad(out, pred, grad_out)
    # d/dlogit_j of sum_k p_k k: p_j (j - E) per side, E <= REG_MAX - 1
    assert_matches_golden(grad_in, torch.from_numpy(g["grad_in"]), (rp.REG_MAX - 1) * grad_out.abs().repeat_interleave(rp.REG_MAX, -1))


# ------------------------------------------------------------------ head tail (SURVEY 8f-3): the checker, ahead of the kernel
@pytest.mark.parametrize("name", golden_names("headtail"))
def test_head_tail_port_matches_golden(name):
    """Last 1x1 convs of both towers + concat + decode, restated in the oracle, against what the unmodified reference
    Detect module (real conv towers, eval mode) returned for the captured inputs of those convs
    (oracle/gen_golden_headtail.py)."""
    from oracle import ref_port as rp

    g = load_golden(name)
    args, terms = head_tail_case(g)
    y, raw = rp.head_tail_port(*args, (8.0, 16.0, 32.0))
    golden_raw = [torch.from_numpy(g[f"raw{i}"]) for i in range(3)]
    for i in range(3):
        assert_matches_golden(raw[i], golden_raw[i], terms[i], torch.float32)
    if not all(torch.equal(a, b) for a, b in zip(raw, golden_raw)):  # the DFL softmax amplifies a rounding of the raw
        y = rp.decode_port(golden_raw, int(args[4][0].shape[0]), (8.0, 16.0, 32.0))  # levels: decode the reference's own
    want = torch.from_numpy(g["y"])
    assert_matches_golden(y, want, decode_terms(want))


def _tal_case_of(name):
    meta = dict(golden_manifest()[name])
    meta.pop("kind")
    if "score_dtype" in meta:
        meta["score_dtype"] = getattr(torch, meta["score_dtype"])
    return rp.tal_case(**meta), meta


@pytest.mark.parametrize("name", golden_names("tal"))
def test_tal_assign_port_matches_golden(name):
    """oracle/ref_port.tal_assign_port against what the unmodified TaskAlignedAssigner.forward returned on the same seeded
    inputs (oracle/gen_golden_tal.py): all five tensors, bit for bit except the normalised scores (assert_matches_golden:
    products and quotients of overlaps, each score is its own scale)."""
    g = load_golden(name)
    c, meta = _tal_case_of(name)
    labels, bboxes, scores, fg, gidx, ambiguous = rp.tal_assign_port(**c, num_classes=meta["nc"])
    assert torch.equal(labels, torch.from_numpy(g["target_labels"]))
    assert torch.equal(bboxes, torch.from_numpy(g["target_bboxes"]))
    want = torch.from_numpy(g["target_scores"])
    assert_matches_golden(scores, want, want.abs())
    assert torch.equal(fg, torch.from_numpy(g["fg_mask"]))
    assert torch.equal(gidx, torch.from_numpy(g["target_gt_idx"]))
    assert fg.any() and (fg.sum(1) > 0).all()


def test_golden_bounds_reject_port_errors():
    """The per-element bounds of assert_matches_golden do not admit small errors of a port: classes off by one, score
    logits +0.05, centres +4 px on the stride-8 level, sizes +1 px, a missing class-convolution bias."""
    for name in golden_names("decode") + golden_names("model"):
        want = torch.from_numpy(load_golden(name)["y"])
        a0 = (int(golden_manifest()[name]["imgsz"][0]) // 8) * (int(golden_manifest()[name]["imgsz"][1]) // 8)
        rolled = torch.cat((want[:, :4], want[:, 4:].roll(1, 1)), 1)
        wrong = [] if torch.equal(rolled, want) else [rolled]  # (nc = 1, or every class scored alike as in model_cfg1)
        logit = torch.cat((want[:, :4], torch.sigmoid(torch.logit(want[:, 4:].double()) + 0.05).to(want.dtype)), 1)
        centre, size = want.clone(), want.clone()
        centre[:, 0, :a0] += 4
        size[:, 2:4] += 1
        for got in wrong + [logit, centre, size]:
            with pytest.raises(AssertionError):
                assert_matches_golden(got, want, decode_terms(want))
    for name in golden_names("headtail"):
        g = load_golden(name)
        args, terms = head_tail_case(g)
        for i in range(3):
            raw = torch.from_numpy(g[f"raw{i}"])
            no_bias = raw.clone()
            no_bias[:, 64:] -= args[5][i].view(1, -1, 1, 1)
            with pytest.raises(AssertionError):
                assert_matches_golden(no_bias, raw, terms[i], torch.float32)
