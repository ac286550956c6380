"""GPU parity tests: the CUDA path (through the C ABI / custom ops) against the golden
vectors from the reference and against the oracle on seeded inputs."""
import numpy as np
import pytest
import torch

from conftest import golden_manifest, golden_names, load_golden, split_rows
from cerberusdet_b200.synth import STRIDES, level_shapes, synth_heads, synth_prediction
from tol import check_bbox_decode, check_decode

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    yield o
    _lib.load().cerb_debug_set_chunking(0, 0)


def _dev(t):
    return t.cuda(non_blocking=False)


# ------------------------------------------------------------------ decode
@pytest.mark.parametrize("name", golden_names("decode"))
def test_decode_golden(ops, name):
    g = load_golden(name)
    meta = golden_manifest()[name]
    levels = [torch.from_numpy(g[f"level{i}"]) for i in range(3)]
    ref = torch.from_numpy(g["y"])
    y = ops.decode_heads([[_dev(x) for x in levels]], STRIDES)[0]
    assert y.dtype == ref.dtype and tuple(y.shape) == tuple(ref.shape)
    ok, msg = check_decode(y, ref, [x.shape[2:] for x in levels], STRIDES, meta["nc"])
    assert ok, msg


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("imgsz,bsz", [((640, 640), 2), ((96, 72), 3), ((40, 24), 1), ((1280, 1280), 1)])
def test_decode_vs_oracle_multitask(ops, dtype, imgsz, bsz):
    from oracle import ref_port as rp

    ncs = [20, 19, 12]
    if imgsz == (40, 24):
        strides = (8.0,)  # single level, hw = 15: no vector width divides it -> scalar path
    else:
        strides = STRIDES
    heads = synth_heads(range(bsz), ncs, imgsz, dtype, "iid", cfg=21, strides=strides)
    ys = ops.decode_heads([[_dev(x) for x in lv] for lv in heads], strides)
    for t, nc in enumerate(ncs):
        ref = rp.decode_port(heads[t], nc, strides)
        ok, msg = check_decode(ys[t], ref, level_shapes(imgsz, strides), strides, nc)
        assert ok, f"task {t}: {msg}"


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_decode_pipelined_kernel_bit_identical_to_register_kernel(ops, dtype, knobs):
    """decode_pipe.cu (cp.async prefetch, several items per thread) and decode.cu do the same arithmetic: y and the score
    summary must be bit-identical, on ragged item counts (B * hw / VEC not a multiple of the items per CTA), several class
    group remainders (nc % 4 = 0, 3, 1, 2) and more than one class group ring turn (nc = 80)."""
    from cerberusdet_b200 import ops as o

    for ncs, imgsz, bsz in [([20, 19, 12], (640, 640), 3), ([80, 5, 1, 2], (96, 72), 5), ([19], (1280, 736), 1)]:
        heads = synth_heads(range(bsz), ncs, imgsz, dtype, "iid", cfg=77)
        dev = [[_dev(x) for x in lv] for lv in heads]
        knobs("decode_pipe", 0)
        y0 = ops.decode_heads(dev, STRIDES)
        s0 = [o.find_summary(y) for y in y0]
        knobs("decode_pipe", 1)
        y1 = ops.decode_heads(dev, STRIDES)
        s1 = [o.find_summary(y) for y in y1]
        for t in range(len(ncs)):
            assert torch.equal(y0[t], y1[t]), f"y differs: task {t} ncs={ncs} imgsz={imgsz}"
            assert (s0[t] is None) == (s1[t] is None)
            if s0[t] is not None:
                n = y0[t].shape[2] // (8 if dtype == torch.float16 else 4)  # the padding past A / V is never written
                assert torch.equal(s0[t][..., :n], s1[t][..., :n]), f"summary differs: task {t} ncs={ncs}"
    # and against the oracle directly
    from oracle import ref_port as rp

    heads = synth_heads(range(2), [20, 19, 12], (640, 640), dtype, "iid", cfg=21)
    ys = ops.decode_heads([[_dev(x) for x in lv] for lv in heads], STRIDES)
    for t, nc in enumerate([20, 19, 12]):
        ok, msg = check_decode(ys[t], rp.decode_port(heads[t], nc, STRIDES), level_shapes((640, 640), STRIDES), STRIDES, nc)
        assert ok, f"task {t}: {msg}"


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("pipe", ["0", "default"])
def test_decode_split_heads_bit_identical_to_concatenated(ops, dtype, pipe, knobs):
    """cerb_decode_split reads the box channels (cv2 output) and the class channels (cv3 output) from their own tensors
    -- the concat of reference models/yolo.py:89-90 is never made -- and must give the same bits as cerb_decode on the
    concatenated tensors, through both kernels and on the scalar (unaligned) path."""
    from cerberusdet_b200 import ops as o

    if pipe != "default":
        knobs("decode_pipe", int(pipe))
    for ncs, imgsz, bsz, strides in [([20, 19, 12], (640, 640), 2, STRIDES), ([80, 3], (96, 72), 3, STRIDES), ([5], (40, 24), 2, (8.0,))]:
        heads = synth_heads(range(bsz), ncs, imgsz, dtype, "iid", cfg=55, strides=strides)
        dev = [[_dev(x) for x in lv] for lv in heads]
        y0 = ops.decode_heads(dev, strides)
        s0 = [o.find_summary(y) for y in y0]
        box = [[x[:, :64].contiguous() for x in lv] for lv in dev]
        cls = [[x[:, 64:].contiguous() for x in lv] for lv in dev]
        y1 = o.decode_heads_split(box, cls, strides)
        s1 = [o.find_summary(y) for y in y1]
        for t in range(len(ncs)):
            assert torch.equal(y0[t], y1[t]), f"task {t} ncs={ncs} imgsz={imgsz}"
            assert (s0[t] is None) == (s1[t] is None)
            if s0[t] is not None:
                n = y0[t].shape[2] // (8 if dtype == torch.float16 else 4)
                assert torch.equal(s0[t][..., :n], s1[t][..., :n])
    with pytest.raises(ValueError):  # class tensor of another spatial shape
        o.decode_heads_split(box, [[c[:, :, :-1].contiguous() for c in lv] for lv in cls], strides)


def test_decode_rejects_cpu_and_bad_shapes(ops):
    heads = synth_heads(range(1), [20], 64, torch.float32)
    with pytest.raises(TypeError):
        ops.decode_heads(heads, STRIDES)
    bad = [[_dev(x) for x in heads[0]]]
    bad[0][1] = bad[0][1][:, :80].contiguous()  # wrong channel count for nc=20
    with pytest.raises(ValueError):
        ops.decode_heads(bad, STRIDES)


def test_decode_nms_rejects_heads_as_decode_does(ops):
    """decode_nms checks its raw heads as decode does: a dtype mismatch raises TypeError, a wrong shape ValueError."""
    heads = synth_heads(range(1), [20], 64, torch.float32)
    mixed = [[_dev(x) for x in heads[0]]]
    mixed[0][1] = mixed[0][1].half()
    bad = [[_dev(x) for x in heads[0]]]
    bad[0][1] = bad[0][1][:, :80].contiguous()
    for fn in (ops.decode_heads, ops.decode_nms):
        with pytest.raises(TypeError):
            fn(mixed, STRIDES)
        with pytest.raises(ValueError):
            fn(bad, STRIDES)


# ------------------------------------------------------------------ NMS
def _assert_rows_equal(got, want, ctx=""):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        a = a.cpu()
        assert a.dtype == torch.float32
        assert tuple(a.shape) == tuple(b.shape), f"{ctx} image {i}: {tuple(a.shape)} vs {tuple(b.shape)}"
        assert torch.equal(a, b), f"{ctx} image {i}: rows differ"


@pytest.mark.parametrize("minb", [1, 2])
@pytest.mark.parametrize("chunking", [(0, 0), (16, 1), (64, 7), (300, 300)])
@pytest.mark.parametrize("name", golden_names("nms"))
def test_nms_golden_bit_exact(ops, name, chunking, minb, knobs):
    """Every golden vector through both register builds of the NMS kernel (minb 1: 128 registers, used when each segment
    gets its own SM; minb 2: 64 registers, two CTAs per SM) and four chunking settings."""
    from cerberusdet_b200 import _lib
    from cerberusdet_b200.nms import non_max_suppression

    knobs("nms_minb", minb)
    g = load_golden(name)
    if chunking != (0, 0) and g["pred"].shape[2] > 4000 and chunking[0] < 300:
        pytest.skip("tiny chunks on the large vectors only repeat the same paths slowly")
    kw = dict(golden_manifest()[name]["kwargs"])
    assert _lib.load().cerb_debug_set_chunking(*chunking) == 0
    try:
        got = non_max_suppression(_dev(torch.from_numpy(g["pred"])), **kw)
    finally:
        _lib.load().cerb_debug_set_chunking(0, 0)
    _assert_rows_equal(got, split_rows(g["rows"], g["counts"]), name)


CASES = [
    # bsz, nc, anchors, dtype, regime, kwargs
    (3, 20, 2100, torch.float32, "clusters", dict(conf_thres=0.25, iou_thres=0.45)),
    (3, 20, 2100, torch.float16, "clusters", dict(conf_thres=0.25, iou_thres=0.45)),
    (2, 12, 2100, torch.float16, "clusters", dict(conf_thres=0.001, iou_thres=0.6, multi_label=True)),
    (2, 19, 3000, torch.float32, "uniform", dict(conf_thres=0.001, iou_thres=0.7, multi_label=True, max_det=1500)),
    (2, 1, 1500, torch.float32, "clusters", dict(conf_thres=0.05, iou_thres=0.5, multi_label=True)),
    (2, 7, 1000, torch.float16, "clusters", dict(conf_thres=0.0, iou_thres=0.0, max_det=20)),
    (2, 7, 1000, torch.float32, "clusters", dict(conf_thres=0.2, iou_thres=1.0, multi_label=True, max_det=3000)),
    (1, 20, 33600, torch.float16, "clusters", dict(conf_thres=0.001, iou_thres=0.6, multi_label=True)),
    (2, 5, 800, torch.float32, "clusters", dict(conf_thres=0.3, iou_thres=0.45, classes=[4], agnostic=True)),
    (2, 5, 800, torch.float32, "clusters", dict(conf_thres=0.3, iou_thres=0.45, classes=[], multi_label=True)),
]


@pytest.mark.parametrize("minb", [1, 2])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_nms_vs_oracle(ops, case, minb, knobs):
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    knobs("nms_minb", minb)
    bsz, nc, anchors, dtype, regime, kw = CASES[case]
    pred = synth_prediction(bsz, nc, anchors, seed=100 + case, dtype=dtype, regime=regime)
    want = rp.nms_port(pred, greedy="c", **kw)
    got = non_max_suppression(_dev(pred), **kw)
    _assert_rows_equal(got, want, f"case {case}")


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_nms_constant_scores_massive_ties(ops, dtype):
    """Every score identical: > 4096 keys in one radix bin -> deeper refinement; canonical
    order is (anchor, class) ascending."""
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    pred = synth_prediction(1, 3, 6000, seed=77, dtype=torch.float32, regime="uniform")
    pred[:, 4:] = 0.5
    pred[:, 4, ::7] = 0.75
    pred = pred.to(dtype)
    for kw in (dict(conf_thres=0.25, iou_thres=0.45, multi_label=True, max_det=1000),
               dict(conf_thres=0.25, iou_thres=0.45, max_det=300)):
        want = rp.nms_port(pred, greedy="c", **kw)
        got = non_max_suppression(_dev(pred), **kw)
        _assert_rows_equal(got, want, str(kw))


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("multi", [False, True])
def test_nms_wild_boxes_outside_class_window(ops, dtype, multi):
    """Boxes far outside [0, max_wh): class-offset boxes of different classes DO overlap there
    (reference general.py:462-463 quirk), so the per-class shortcut must switch itself off."""
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    pred = synth_prediction(2, 6, 1500, seed=31, dtype=torch.float32, regime="clusters", imgsz=9000.0)
    pred[:, 0:2] -= 1500.0  # centres in [-1500, 7500]: some boxes below -960, some above 6720
    pred[1, 0:2, ::3] += 7680.0  # image 1: a third of the boxes shifted by exactly one class gap
    pred = pred.to(dtype)
    kw = dict(conf_thres=0.05, iou_thres=0.5, multi_label=multi, max_det=300)
    want = rp.nms_port(pred, greedy="c", **kw)
    got = non_max_suppression(_dev(pred), **kw)
    _assert_rows_equal(got, want, "wild")


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("regime", ["iid", "planted"])
@pytest.mark.parametrize("kw", [
    dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300),
    dict(conf_thres=0.25, iou_thres=0.45, max_det=300),
    dict(conf_thres=0.01, iou_thres=0.5, classes=[0, 5, 11], multi_label=True, max_det=40),
    dict(conf_thres=0.05, iou_thres=0.5, classes=[2, 3], agnostic=True, max_det=1200),
])
def test_decode_then_nms_with_score_summary(ops, dtype, regime, kw):
    """decode_heads -> nms_batched (summary-guided) == oracle NMS of the same decoded tensor, and
    == the summary-free kernel path; also after an in-place edit (summary must be dropped)."""
    from oracle import ref_port as rp

    ncs = [20, 12]
    heads = synth_heads(range(3), ncs, (320, 256), dtype, regime, cfg=11)
    ys = ops.decode_heads([[_dev(x) for x in lv] for lv in heads], STRIDES)
    assert all(ops.find_summary(y) is not None for y in ys)
    dets, counts = ops.nms_batched(ys, **kw)
    d0, c0 = ops.nms_batched(ys, use_summary=False, **kw)
    assert torch.equal(c0, counts) and torch.equal(d0, dets)
    ch = counts.cpu()
    for t in range(2):
        want = rp.nms_port(ys[t].cpu(), greedy="c", **kw)
        for b in range(3):
            assert torch.equal(dets[t, b, : ch[t, b]].cpu(), want[b]), (t, b)
    ys[0][:, 4:] *= 0.5  # in-place edit: the remembered summary no longer describes the tensor
    assert ops.find_summary(ys[0]) is None
    dets, counts = ops.nms_batched(ys, **kw)
    ch = counts.cpu()
    want = rp.nms_port(ys[0].cpu(), greedy="c", **kw)
    for b in range(3):
        assert torch.equal(dets[0, b, : ch[0, b]].cpu(), want[b])


def _truncation_prediction(dtype, seed=3):
    """> 30000 multi-label candidates, nearly all inside one heavy cluster (suppressed by its top box)
    plus isolated boxes whose scores straddle the rank-30000 cut: the kept set is sensitive to the exact
    max_nms truncation (utils/general.py:459) and the whole candidate list has to be consumed."""
    g = torch.Generator().manual_seed(seed)
    A, nc = 12000, 4
    y = torch.empty(1, 4 + nc, A)
    y[0, 0] = 320 + torch.randn(A, generator=g)
    y[0, 1] = 320 + torch.randn(A, generator=g)
    y[0, 2] = 200 + torch.randn(A, generator=g)
    y[0, 3] = 200 + torch.randn(A, generator=g)
    y[0, 4:] = torch.rand(nc, A, generator=g) * 0.9 + 0.01
    iso = torch.randperm(A, generator=g)[:60]
    gx = (torch.arange(60) % 10) * 60.0 + 15
    gy = (torch.arange(60) // 10) * 60.0 + 615  # far below the cluster
    y[0, 0, iso], y[0, 1, iso] = gx, gy
    y[0, 2, iso] = 8.0
    y[0, 3, iso] = 8.0
    return y.to(dtype)


@pytest.mark.parametrize("sample", [0, 1, 3, 16])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_nms_max_nms_truncation_full_consumption(ops, dtype, sample):
    from cerberusdet_b200 import _lib
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    pred = _truncation_prediction(dtype)
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    want = rp.nms_port(pred, greedy="c", **kw)
    assert 20 < want[0].shape[0] < 300  # neither trivially empty nor capped by max_det
    assert _lib.load().cerb_debug_set_hist_sample(sample) == 0
    try:
        got = non_max_suppression(_dev(pred), **kw)
    finally:
        _lib.load().cerb_debug_set_hist_sample(0)
    _assert_rows_equal(got, want, f"sample={sample}")


def test_nms_empty_and_edge_batches(ops):
    from cerberusdet_b200.nms import non_max_suppression

    pred = torch.zeros(3, 9, 500, device="cuda")
    out = non_max_suppression(pred, 0.25, 0.45)
    assert len(out) == 3 and all(tuple(o.shape) == (0, 6) and o.dtype == torch.float32 for o in out)
    out = non_max_suppression((pred, None), 0.25, 0.45, max_det=0)
    assert all(tuple(o.shape) == (0, 6) for o in out)
    with pytest.raises(AssertionError):
        non_max_suppression(pred, conf_thres=1.2)
    with pytest.raises(AssertionError):
        non_max_suppression(pred, iou_thres=-0.5)
    with pytest.raises(TypeError):
        non_max_suppression(pred.cpu())
    with pytest.raises(NotImplementedError):
        non_max_suppression(pred, nm=32)


def test_multitask_batched_equals_per_task(ops):
    """One launch over T tasks == T single-task calls (the reference's per-task loop,
    cerberusdet_inference.py:125-135)."""
    from cerberusdet_b200.nms import non_max_suppression

    preds = [_dev(synth_prediction(4, nc, 2100, seed=5 + nc, dtype=torch.float16)) for nc in (20, 19, 12)]
    dets, counts = ops.nms_batched(preds, 0.25, 0.45, max_det=300)
    counts = counts.cpu()
    for t, p in enumerate(preds):
        single = non_max_suppression(p, 0.25, 0.45)
        for b in range(4):
            assert torch.equal(dets[t, b, : counts[t, b]], single[b])


def test_full_size_properties_cfg3(ops):
    """BASELINE config 3 at full size (B=64, 3 tasks, 8400 anchors, val settings): checked
    through size-independent properties, plus a bit-exact spot check of a few segments."""
    from oracle import ref_port as rp

    ncs = [20, 19, 12]
    bsz = 64
    heads = synth_heads(range(bsz), ncs, 640, torch.float16, "iid", cfg=3)
    dev_heads = [[_dev(x) for x in lv] for lv in heads]
    ys = ops.decode_heads(dev_heads, STRIDES)
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    dets, counts = ops.nms_batched(ys, **kw)
    # the score summary left by the decode kernel only steers which groups are read: same bits without it
    d0, c0 = ops.nms_batched(ys, use_summary=False, **kw)
    assert torch.equal(c0, counts) and torch.equal(d0, dets)
    counts_h = counts.cpu()
    assert (counts_h <= 300).all() and (counts_h > 0).all()
    for t in range(3):
        for b in range(bsz):
            d = dets[t, b, : counts_h[t, b]]
            s = d[:, 4]
            assert (s[:-1] >= s[1:]).all()  # score-descending
            assert (s > 0.001).all()
            assert ((d[:, 5] >= 0) & (d[:, 5] < ncs[t])).all()
    # the estimating histogram never changes results: exact histogram gives the same bits
    from cerberusdet_b200 import _lib

    for stride in (1, 16):
        _lib.load().cerb_debug_set_hist_sample(stride)
        try:
            d1, c1 = ops.nms_batched(ys, **kw)
        finally:
            _lib.load().cerb_debug_set_hist_sample(0)
        assert torch.equal(c1, counts) and torch.equal(d1, dets)
    # shard invariance: running images 16..31 alone gives the same rows
    ys_shard = [y[16:32].contiguous() for y in ys]
    d2, c2 = ops.nms_batched(ys_shard, **kw)
    assert torch.equal(c2, counts[:, 16:32]) and torch.equal(d2, dets[:, 16:32])
    # EVERY one of the 192 segments against the oracle fed the SAME decoded tensor (selection must be bit exact)
    dets_h = dets.cpu()
    for t in range(3):
        want = rp.nms_port(ys[t].cpu(), greedy="c", **kw)
        for b in range(bsz):
            assert torch.equal(dets_h[t, b, : counts_h[t, b]], want[b]), f"segment task {t} image {b}"
    # and the decode itself, every image, within the north_star tolerance of the oracle port
    for t, nc in enumerate(ncs):
        ok, msg = check_decode(ys[t], rp.decode_port(heads[t], nc, STRIDES), level_shapes(640, STRIDES), STRIDES, nc)
        assert ok, f"task {t}: {msg}"


# ------------------------------------------------------------------ shapes beyond the BASELINE configs
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("nc,imgsz,strides,bsz", [
    (80, (256, 256), (8.0, 16.0, 32.0), 2),            # COCO-sized head: 3 class chunks in the decode grid
    (365, (128, 192), (8.0, 16.0, 32.0), 1),           # Objects365-full head (reference data/voc_obj365_full.yaml)
    (5, (512, 384), (8.0, 16.0, 32.0, 64.0), 2),       # four levels (P3-P6)
    (1, (1280, 736), (8.0, 16.0, 32.0), 1),            # single class, non-square 1280 input
])
def test_decode_and_nms_other_head_shapes(ops, dtype, nc, imgsz, strides, bsz):
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    heads = synth_heads(range(bsz), [nc], imgsz, dtype, "iid", cfg=31, strides=strides)
    y = ops.decode_heads([[_dev(x) for x in heads[0]]], strides)[0]
    ref = rp.decode_port(heads[0], nc, strides)
    ok, msg = check_decode(y, ref, level_shapes(imgsz, strides), strides, nc)
    assert ok, msg
    for kw in (dict(conf_thres=0.01, iou_thres=0.6, multi_label=True, max_det=300),
               dict(conf_thres=0.1, iou_thres=0.45, max_det=100),
               dict(conf_thres=0.01, iou_thres=0.5, multi_label=True, classes=[0, nc - 1, nc // 2], max_det=50)):
        want = rp.nms_port(y.cpu(), greedy="c", **kw)   # selection is bit exact on the SAME decoded tensor
        got = non_max_suppression(y, **kw)
        _assert_rows_equal(got, want, f"nc={nc} {kw}")


def test_full_size_cfg2_and_cfg4(ops):
    """BASELINE configs 2 (B=32, 2 tasks, best class, conf 0.3) and 4 (B=16, 1280^2, 33600 anchors, multi-label) at
    full size: properties on every segment and EVERY segment bit-exact against the oracle fed the same decoded tensor."""
    from oracle import ref_port as rp

    for ncs, bsz, imgsz, kw in (([20, 19], 32, 640, dict(conf_thres=0.3, iou_thres=0.45, max_det=300)),
                                ([20, 19, 12], 16, 1280, dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300))):
        heads = synth_heads(range(bsz), ncs, imgsz, torch.float16, "iid", cfg=3)
        ys = ops.decode_heads([[_dev(x) for x in lv] for lv in heads], STRIDES)
        dets, counts = ops.nms_batched(ys, **kw)
        ch = counts.cpu()
        assert (ch <= 300).all() and (ch > 0).all()
        s = dets[..., 4]
        for t in range(len(ncs)):
            for b in range(bsz):
                n = int(ch[t, b])
                assert (s[t, b, : n - 1] >= s[t, b, 1:n]).all()
                assert (dets[t, b, n:] == 0).all()          # padding rows are zeroed by the kernel
        dets_h = dets.cpu()
        for t in range(len(ncs)):
            want = rp.nms_port(ys[t].cpu(), greedy="c", **kw)
            for b in range(bsz):
                assert torch.equal(dets_h[t, b, : int(ch[t, b])], want[b]), f"imgsz {imgsz} segment task {t} image {b}"


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_decode_nms_single_call_equals_two_calls(ops, dtype):
    heads = synth_heads(range(4), [20, 19, 12], (320, 320), dtype, "iid", cfg=41)
    dev = [[_dev(x) for x in lv] for lv in heads]
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    d1, c1, ys1 = ops.decode_nms(dev, STRIDES, **kw)
    ys2 = ops.decode_heads(dev, STRIDES)
    d2, c2 = ops.nms_batched(ys2, **kw)
    assert all(torch.equal(a, b) for a, b in zip(ys1, ys2))
    assert torch.equal(c1, c2) and torch.equal(d1, d2)


@pytest.mark.parametrize("name", golden_names("model"))
def test_real_model_config1_vectors_gpu(ops, name):
    """BASELINE config 1 on the GPU path: raw head tensors of the real 2-task CerberusDet model -> decode within
    tolerance of the model's own y; NMS of the model's y bit-exact (> 30000 near-tied fp32 candidates)."""
    from cerberusdet_b200.nms import non_max_suppression

    g = load_golden(name)
    meta = golden_manifest()[name]
    levels = [torch.from_numpy(g[f"level{i}"]) for i in range(3)]
    ref_y = torch.from_numpy(g["y"])
    y = ops.decode_heads([[_dev(x) for x in levels]], STRIDES)[0]
    ok, msg = check_decode(y, ref_y, [x.shape[2:] for x in levels], STRIDES, meta["nc"])
    assert ok, msg
    got = non_max_suppression(_dev(ref_y), **meta["kwargs"])
    _assert_rows_equal(got, split_rows(g["rows"], g["counts"]), name)


# ------------------------------------------------------------------ training-time sibling decode (SURVEY 8f-4)
@pytest.mark.parametrize("name", golden_names("train_bbox"))
def test_bbox_decode_golden_forward_and_backward(ops, name):
    """Loss.bbox_decode (reference utils/loss.py:126-131) through the C ABI against vectors from the unmodified reference."""
    g = load_golden(name)
    ap = _dev(torch.from_numpy(g["anchor_points"]))
    pred = _dev(torch.from_numpy(g["pred"])).requires_grad_(True)
    out = ops.bbox_decode(ap, pred)
    ref = torch.from_numpy(g["out"])
    assert out.dtype == ref.dtype and tuple(out.shape) == tuple(ref.shape)
    ok, msg = check_bbox_decode(out.detach(), ref, gmax=float(g["anchor_points"].max()) + 16.0)
    assert ok, "forward: " + msg
    go = torch.from_numpy(g["grad_out"])
    (gi,) = torch.autograd.grad(out, pred, _dev(go))
    ok, msg = check_bbox_decode(gi, torch.from_numpy(g["grad_in"]), grad=True, grad_out=go)
    assert ok, "backward: " + msg


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("bsz,imgsz,scale", [(16, 640, 3.0), (2, 1280, 8.0), (1, 64, 20.0)])
def test_bbox_decode_vs_oracle(ops, dtype, bsz, imgsz, scale):
    """Seeded logits at BASELINE sizes (8400 / 33600 anchors) against the oracle port and its autograd gradient;
    also the unaligned (storage offset) path and linearity of the backward in grad_out."""
    from oracle import ref_port as rp

    shapes = level_shapes((imgsz, imgsz), STRIDES)
    anchors, _ = rp.anchor_grid(shapes, STRIDES, dtype)
    ap = anchors.transpose(0, 1).contiguous()  # [A, 2]
    A = ap.shape[0]
    gen = torch.Generator().manual_seed(1000 + imgsz + bsz)
    pred = (torch.randn(bsz, A, 64, generator=gen) * scale).to(dtype)
    go = torch.randn(bsz, A, 4, generator=gen).to(dtype)
    p_ref = pred.clone().requires_grad_(True)
    want = rp.bbox_decode_port(ap, p_ref)
    (want_g,) = torch.autograd.grad(want, p_ref, go)

    p_dev = _dev(pred).requires_grad_(True)
    out = ops.bbox_decode(_dev(ap), p_dev)
    ok, msg = check_bbox_decode(out.detach(), want.detach(), gmax=float(ap.max()) + 16.0)
    assert ok, "forward: " + msg
    (gi,) = torch.autograd.grad(out, p_dev, _dev(go))
    ok, msg = check_bbox_decode(gi, want_g, grad=True, grad_out=go)
    assert ok, "backward: " + msg

    # a contiguous view at an odd element offset takes the scalar-load path: same bits
    buf = torch.empty(pred.numel() + 1, dtype=dtype, device="cuda")
    view = buf[1:].view(bsz, A, 64)
    view.copy_(pred)
    assert view.data_ptr() % 16 != 0 and view.is_contiguous()
    v = view.detach().requires_grad_(True)
    out2 = ops.bbox_decode(_dev(ap), v)
    assert torch.equal(out2, out)
    (gi2,) = torch.autograd.grad(out2, v, _dev(go))
    assert torch.equal(gi2, gi)

    if dtype == torch.float32:  # backward is linear in grad_out: doubling it doubles every (normal) gradient exactly
        p3 = _dev(pred).requires_grad_(True)
        (gi3,) = torch.autograd.grad(ops.bbox_decode(_dev(ap), p3), p3, _dev(go) * 2)
        assert ((gi3 - gi * 2).abs() <= 1e-38).all()  # exact, except that subnormal results lose bits


def test_bbox_decode_rejects_bad_arguments(ops):
    ap = torch.zeros(10, 2)
    with pytest.raises(TypeError):
        ops.bbox_decode(ap, torch.zeros(1, 10, 64))  # CPU tensor: no fallback
    with pytest.raises(ValueError):
        ops.bbox_decode(ap.cuda(), torch.zeros(1, 10, 32, device="cuda"))  # reg_max != 16
    with pytest.raises(ValueError):
        ops.bbox_decode(ap.cuda(), torch.zeros(1, 11, 64, device="cuda"))  # anchor count mismatch
    out = ops.bbox_decode(torch.zeros(0, 2, device="cuda"), torch.zeros(2, 0, 64, device="cuda"))
    assert tuple(out.shape) == (2, 0, 4)


# ------------------------------------------------------------------ the bench's launch mode: one CUDA graph (decode -> NMS, PDL edge)
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_cuda_graph_replay_equals_eager(ops, dtype):
    """bench.py replays decode -> NMS as ONE captured CUDA graph; the NMS kernel is launched with programmatic stream
    serialization, so inside the graph it hangs off the decode kernel by a programmatic dependency.  Replays on fresh
    inputs (copied into the captured buffers) must give exactly the eager results, replay after replay."""
    ncs, imgsz, bsz = [20, 19, 12], (640, 640), 4
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    batches = [synth_heads(range(k * bsz, (k + 1) * bsz), ncs, imgsz, dtype, "iid", cfg=3) for k in range(3)]
    static = [[_dev(x).clone() for x in lv] for lv in batches[0]]
    eager = []
    for heads in batches:
        ys = ops.decode_heads([[_dev(x) for x in lv] for lv in heads], STRIDES)
        d, c = ops.nms_batched(ys, **kw)
        eager.append((d.clone(), c.clone()))
    for _ in range(2):  # warm-up on the side stream, as torch asks for before a capture
        ops.nms_batched(ops.decode_heads(static, STRIDES), **kw)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            ys = ops.decode_heads(static, STRIDES)
            d_static, c_static = ops.nms_batched(ys, **kw)
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(2):
        for k, heads in enumerate(batches):
            for lv_s, lv in zip(static, heads):
                for xs, x in zip(lv_s, lv):
                    xs.copy_(_dev(x))
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(c_static, eager[k][1]), f"counts differ: replay {rep} batch {k}"
            assert torch.equal(d_static, eager[k][0]), f"rows differ: replay {rep} batch {k}"
