"""bfloat16 heads through the post-head path on the GPU: decode, NMS, the drop-in surfaces and the training-time box
decode, each against the reference's own op sequence (oracle/ref_port.py) run in bf16 -- the decode and the box decode
on the same GPU, the NMS selection on the same decoded tensor."""
import math

import pytest
import torch

from cerberusdet_b200.synth import STRIDES, level_shapes, synth_heads, synth_prediction

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    yield o
    _lib.load().cerb_debug_set_chunking(0, 0)
    _lib.load().cerb_debug_set_hist_sample(0)


def _ulp(x, mant_bits=7):
    """bf16 ulp of |x| (elementwise tensor or float); the smallest normal's ulp below it."""
    if isinstance(x, torch.Tensor):
        e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
        return torch.exp2(e - mant_bits)
    return 2.0 ** (math.floor(math.log2(x)) - mant_bits)


def check_decode_bf16(y, ref, level_hw, strides):
    """The fp16 rule of tests/tol.py with bf16's ulp: boxes within 2^-7 relative plus 2 ulps of the level's largest corner
    coordinate (times the stride), scores within one bf16 ulp, at least 98 % of all outputs bit-identical."""
    yf, rf = y.float().cpu(), ref.float().cpu()
    if not torch.isfinite(yf).all():
        return False, "non-finite output"
    off = 0
    for (h, w), s in zip(level_hw, strides):
        n = h * w
        atol = s * 2.0 * _ulp(max(h, w) + 16.0)
        d = (yf[:, :4, off:off + n] - rf[:, :4, off:off + n]).abs()
        bound = 2.0 ** -7 * rf[:, :4, off:off + n].abs() + atol
        if (d > bound).any():
            return False, f"box mismatch level@{off}: worst excess {(d - bound).max().item():.3e}"
        off += n
    d = (yf[:, 4:] - rf[:, 4:]).abs()
    if (d > _ulp(rf[:, 4:])).any():
        return False, f"score mismatch: worst {d.max().item():.3e}"
    same = (y.cpu() == ref.cpu()).float().mean().item()
    if same < 0.98:
        return False, f"only {same:.4f} of the outputs bit-identical"
    return True, f"{same:.5f} bit-identical"


# ------------------------------------------------------------------ the bf16 facts, against torch on this GPU
def test_bf16_facts_on_gpu():
    ac = torch.arange(160, dtype=BF16, device="cuda") + 0.5
    assert ac[128].item() == 128.0 and ac[129].item() == 130.0 and int((ac.double().cpu() != torch.arange(160).double() + 0.5).sum()) == 32
    for conf, r in ((0.001, 0.00099945068359375), (0.3, 0.30078125), (0.45, 0.44921875), (0.6, 0.6015625)):
        s = torch.tensor([r], dtype=BF16, device="cuda")
        assert not bool((s > conf).item())
        assert bool((s.nextafter(torch.ones_like(s)) > conf).item())


# ------------------------------------------------------------------ decode
NCS = [1, 12, 19, 20, 80]


@pytest.mark.parametrize("imgsz", [640, 1280])
def test_decode_bf16_vs_port(ops, imgsz, knobs):
    """Both kernels, concatenated and split heads, against decode_port in bf16 on the GPU (at 1280 the P3 anchor centres
    round); the two kernels and the two head layouts bit-identical to each other, score summaries included."""
    from oracle import ref_port as rp

    heads = synth_heads(range(2), NCS, imgsz, BF16, "iid", cfg=9)
    dev = [[x.cuda() for x in lv] for lv in heads]
    box = [[x[:, :64].contiguous() for x in lv] for lv in dev]
    cls = [[x[:, 64:].contiguous() for x in lv] for lv in dev]
    runs = {}
    for pipe in (0, 1):
        knobs("decode_pipe", pipe)
        for layout in ("cat", "split"):
            ys = ops.decode_heads(dev, STRIDES) if layout == "cat" else ops.decode_heads_split(box, cls, STRIDES)
            runs[(pipe, layout)] = (ys, [ops.find_summary(y) for y in ys])
    ys0, s0 = runs[(1, "cat")]
    assert all(y.dtype == BF16 for y in ys0) and all(s is not None for s in s0)
    for key, (ys, ss) in runs.items():
        for t in range(len(NCS)):
            assert torch.equal(ys[t], ys0[t]), f"{key} task {t}: y differs"
            n = ys[t].shape[2] // 8  # the padding past A / V is never written
            assert torch.equal(ss[t][..., :n], s0[t][..., :n]), f"{key} task {t}: summary differs"
    for t, nc in enumerate(NCS):
        ref = rp.decode_port(dev[t], nc, STRIDES)
        assert ref.dtype == BF16
        ok, msg = check_decode_bf16(ys0[t], ref, level_shapes(imgsz, STRIDES), STRIDES)
        assert ok, f"imgsz {imgsz} nc {nc}: {msg}"
        # the summary is the maximum of each 8-anchor score vector
        sm = ys0[t][:, 4:].float().reshape(2, nc, -1, 8).amax(-1)
        assert torch.equal(s0[t][..., : sm.shape[-1]].float(), sm)


# ------------------------------------------------------------------ NMS fed the same y
def _rows_equal(dets, counts, want, ctx):
    ch = counts.cpu()
    for b, w in enumerate(want):
        got = dets[b, : ch[b]].cpu()
        assert tuple(got.shape) == tuple(w.shape), f"{ctx} image {b}: {tuple(got.shape)} vs {tuple(w.shape)}"
        assert torch.equal(got, w), f"{ctx} image {b}: rows differ"


FLAGS = [
    dict(conf_thres=0.25, iou_thres=0.45),
    dict(conf_thres=0.3, iou_thres=0.45, multi_label=True),
    dict(conf_thres=0.001, iou_thres=0.6, multi_label=True),
    dict(conf_thres=0.001, iou_thres=0.7, multi_label=True, max_det=3000),
    dict(conf_thres=0.05, iou_thres=0.5, agnostic=True, max_det=1000),
    dict(conf_thres=0.01, iou_thres=0.5, classes=[0, 3, 7], multi_label=True, max_det=40),
    dict(conf_thres=0.3, iou_thres=0.45, classes=[4], agnostic=True),
    dict(conf_thres=0.2, iou_thres=0.45, classes=[]),
    dict(conf_thres=0.0, iou_thres=0.0, max_det=20),
    dict(conf_thres=0.2, iou_thres=1.0, multi_label=True, max_det=3000),
]


@pytest.mark.parametrize("minb", [1, 2])
@pytest.mark.parametrize("regime", ["clusters", "uniform"])
@pytest.mark.parametrize("case", range(len(FLAGS)))
def test_nms_bf16_bit_exact(ops, case, regime, minb, knobs):
    """Every flag set, both register builds, on a bf16 prediction whose scores tie heavily (128 values per binade); the
    scores equal to bf16(conf) must not pass."""
    from oracle import ref_port as rp

    knobs("nms_minb", minb)
    kw = FLAGS[case]
    pred = synth_prediction(3, 8, 2400, seed=40 + case, dtype=torch.float32, regime=regime)
    pred[:, 4, ::5] = float(torch.tensor(kw["conf_thres"]).to(BF16))  # exactly bf16(conf): never a candidate
    pred = pred.to(BF16)
    want = rp.nms_port(pred, greedy="c", **kw)
    dets, counts = ops.nms_batched([pred.cuda()], **kw)
    _rows_equal(dets[0], counts[0], want, f"{kw} {regime}")


def test_nms_bf16_constant_scores_take_radix_refinement(ops):
    """Every score equal: one level-0 radix bin holds more keys than a chunk can sort, so the kernel must refine by
    deeper digits; cerb_nms_stats shows more candidates consumed than one chunk holds, all from that one bin."""
    from oracle import ref_port as rp

    pred = synth_prediction(2, 3, 6000, seed=77, dtype=torch.float32, regime="uniform")
    pred[:, 4:] = 0.5
    pred[:, 4, ::7] = 0.75
    pred = pred.to(BF16)
    for kw in (dict(conf_thres=0.25, iou_thres=0.45, multi_label=True, max_det=3000),
               dict(conf_thres=0.25, iou_thres=0.45, max_det=300)):
        want = rp.nms_port(pred, greedy="c", **kw)
        dets, counts = ops.nms_batched([pred.cuda()], **kw)
        _rows_equal(dets[0], counts[0], want, str(kw))
    kw = dict(conf_thres=0.6, iou_thres=1.0, multi_label=True, max_det=10000, max_nms=30000)
    pred[:, 4:] = 0.5
    pred[:, 4:, ::2] = 0.75  # 9000 keys of score 0.75 per image: one level-0 digit, > 4096 keys
    # the precondition the counter argument rests on: per image, more candidates than one chunk (4096) can sort, and
    # every candidate's key shares its top 12 bits (the level-0 digit = the fp32 score bits >> 20) -- so consuming more
    # than 4096 of them is only possible through the deeper radix levels
    for b in range(pred.shape[0]):
        sc = pred[b, 4:].float()
        cand = sc[sc > float(torch.tensor(kw["conf_thres"]).to(BF16))]
        assert cand.numel() > 4096
        assert torch.unique(cand.view(torch.int32) >> 20).numel() == 1
    dets, counts, stats = ops.nms_statistics([pred.cuda()], **kw)
    want = rp.nms_port(pred, greedy="c", **kw)
    _rows_equal(dets[0], counts[0], want, "refine")
    assert int(stats[0, :, 1].min()) > 4096


def _truncation_prediction_bf16(seed=3):
    g = torch.Generator().manual_seed(seed)
    A, nc = 12000, 4
    y = torch.empty(1, 4 + nc, A)
    y[0, 0] = 320 + torch.randn(A, generator=g)
    y[0, 1] = 320 + torch.randn(A, generator=g)
    y[0, 2] = 200 + torch.randn(A, generator=g)
    y[0, 3] = 200 + torch.randn(A, generator=g)
    y[0, 4:] = torch.rand(nc, A, generator=g) * 0.9 + 0.01
    iso = torch.randperm(A, generator=g)[:60]
    y[0, 0, iso], y[0, 1, iso] = (torch.arange(60) % 10) * 60.0 + 15, (torch.arange(60) // 10) * 60.0 + 615
    y[0, 2, iso] = 8.0
    y[0, 3, iso] = 8.0
    return y.to(BF16)


@pytest.mark.parametrize("sample", [0, 1, 3, 16])
def test_nms_bf16_exact_max_nms_truncation(ops, sample):
    """> 30000 candidates whose tied bf16 scores straddle the max_nms cut: the canonical order decides which are in."""
    from cerberusdet_b200 import _lib
    from oracle import ref_port as rp

    pred = _truncation_prediction_bf16()
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    want = rp.nms_port(pred, greedy="c", **kw)
    assert 20 < want[0].shape[0] < 300
    assert _lib.load().cerb_debug_set_hist_sample(sample) == 0
    try:
        dets, counts = ops.nms_batched([pred.cuda()], **kw)
    finally:
        _lib.load().cerb_debug_set_hist_sample(0)
    _rows_equal(dets[0], counts[0], want, f"sample={sample}")


@pytest.mark.parametrize("cfg", ["cfg3", "cfg4"])
def test_decode_nms_bf16_config_shapes_every_segment(ops, cfg):
    """Config 3 (B=64, 640) and config 4 (B=16, 1280) at the validation settings: every (task, image) segment equals the
    port on the same y; with and without the score summary, sampled and exact histograms, and the single-call
    decode_nms, all equal."""
    from cerberusdet_b200 import _lib
    from oracle import ref_port as rp

    B, imgsz = (64, 640) if cfg == "cfg3" else (16, 1280)
    ncs = [20, 19, 12]
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    heads = synth_heads(range(B), ncs, imgsz, BF16, "iid", cfg=3)
    dev = [[x.cuda() for x in lv] for lv in heads]
    del heads
    ys = ops.decode_heads(dev, STRIDES)
    dets, counts, stats = ops.nms_statistics(ys, **kw)
    d1, c1 = ops.nms_batched(ys, use_summary=False, **kw)
    assert torch.equal(d1, dets) and torch.equal(c1, counts)
    for sample in (1, 8):
        assert _lib.load().cerb_debug_set_hist_sample(sample) == 0
        try:
            d2, c2 = ops.nms_batched(ys, use_summary=False, **kw)
        finally:
            _lib.load().cerb_debug_set_hist_sample(0)
        assert torch.equal(d2, dets) and torch.equal(c2, counts), f"hist_sample {sample}"
    d3, c3, ys3 = ops.decode_nms(dev, STRIDES, **kw)
    assert torch.equal(d3, dets) and torch.equal(c3, counts)
    assert all(torch.equal(a, b) for a, b in zip(ys3, ys))
    assert int(stats[..., 1].min()) > 0
    for t in range(len(ncs)):
        want = rp.nms_port(ys[t].cpu(), greedy="c", **kw)
        _rows_equal(dets[t], counts[t], want, f"{cfg} task {t}")


# ------------------------------------------------------------------ surfaces
def test_opcheck_and_compile_bf16(ops):
    from torch.library import opcheck

    heads = synth_heads(range(2), [5, 3], (128, 192), BF16, "iid", cfg=4)  # every level a multiple of 8: with summaries
    flat = [x.cuda() for lv in heads for x in lv]
    box = [x[:, :64].contiguous() for x in flat]
    cls = [x[:, 64:].contiguous() for x in flat]
    nms_args = (0.01, 0.5, None, False, True, 100, 30000, 7680.0)
    # as tests/test_gpu_ops.py: schema, fake kernels and dispatch registrations (the summaries' padding is never written,
    # so an output-equality replay of an allocation-returning op compares uninitialised bytes)
    tests = ("test_schema", "test_faketensor", "test_autograd_registration")
    opcheck(torch.ops.cerb.decode.default, (flat, [5, 3], list(STRIDES)), test_utils=tests)
    opcheck(torch.ops.cerb.decode_split.default, (box, cls, [5, 3], list(STRIDES)), test_utils=tests)
    out = ops.decode_op(flat, [5, 3], list(STRIDES))
    opcheck(torch.ops.cerb.decode_out.default, (flat, [5, 3], list(STRIDES), [torch.empty_like(z) for z in out]), test_utils=tests)
    ys, sm = out[:2], out[2:]
    opcheck(torch.ops.cerb.nms.default, (ys, *nms_args, sm), test_utils=tests)
    opcheck(torch.ops.cerb.nms.default, (ys, *nms_args, []), test_utils=tests)
    dets = torch.empty((2, 2, 100, 6), device="cuda")
    counts = torch.empty((2, 2), dtype=torch.int32, device="cuda")
    opcheck(torch.ops.cerb.nms_out.default, (ys, *nms_args, sm, dets, counts), test_utils=tests)
    opcheck(torch.ops.cerb.decode_nms.default, (flat, [5, 3], list(STRIDES), *nms_args), test_utils=tests)

    def step(levels):
        y = ops.decode_op(levels, [5, 3], list(STRIDES))
        return ops.nms_op(y[:2], *nms_args, y[2:])

    got = torch.compile(step, backend="aot_eager", fullgraph=True)(flat)
    want = step(flat)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_cuda_graph_decode_nms_bf16(ops):
    heads = synth_heads(range(4), [20, 12], 320, BF16, "iid", cfg=5)
    dev = [[x.cuda() for x in lv] for lv in heads]
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    bufs = ops.decode_buffers(dev)
    out = (torch.empty((2, 4, 300, 6), device="cuda"), torch.empty((2, 4), dtype=torch.int32, device="cuda"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            ys = ops.decode_heads(dev, STRIDES, out=bufs)
            ops.nms_batched(ys, out=out, **kw)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ys = ops.decode_heads(dev, STRIDES, out=bufs)
        ops.nms_batched(ys, out=out, **kw)
    fresh = synth_heads(range(4, 8), [20, 12], 320, BF16, "iid", cfg=5)
    for lv, nv in zip(dev, fresh):
        for x, n in zip(lv, nv):
            x.copy_(n)
    g.replay()
    torch.cuda.synchronize()
    ye = ops.decode_heads(dev, STRIDES)
    de, ce = ops.nms_batched(ye, **kw)
    assert all(torch.equal(a, b) for a, b in zip(ys, ye))
    assert torch.equal(out[1], ce)
    for t in range(2):
        for b in range(4):
            n = int(ce[t, b])
            assert torch.equal(out[0][t, b, :n], de[t, b, :n])


@pytest.fixture()
def patched():
    from cerberusdet_b200.detect import detect_forward
    from test_gpu_dropin import Detect

    Detect._cerb_reference_forward = Detect.forward
    orig = Detect.forward
    Detect.forward = detect_forward
    yield Detect
    Detect.forward = orig
    del Detect._cerb_reference_forward


@pytest.mark.parametrize("mode", ["model", "autocast"])
def test_detect_and_nms_patched_vs_unpatched_bf16(patched, mode):
    """The drop-in Detect.forward + non_max_suppression against the class's own forward (the port) + the port's NMS, with
    a bf16 model and with an fp32 model under bf16 autocast: the decode kernel ran (the score summary it leaves is
    attached to y), the decode within the bf16 bounds, selection bit for bit on the patched y."""
    from cerberusdet_b200 import ops
    from cerberusdet_b200.nms import non_max_suppression
    from oracle import ref_port as rp

    torch.manual_seed(0)
    head = patched(12, (8, 8, 8)).cuda().eval()
    for m in head.cv3:
        torch.nn.init.normal_(m.weight, std=1.5)
        torch.nn.init.constant_(m.bias, -3.0)
    feats = [torch.randn(2, 8, 160 // k, 160 // k, device="cuda") for k in (1, 2, 4)]
    ctx = torch.autocast("cuda", dtype=BF16) if mode == "autocast" else torch.autocast("cuda", enabled=False)
    if mode == "model":
        head = head.bfloat16()
        feats = [f.bfloat16() for f in feats]
    with torch.no_grad(), ctx:
        y, x = head([f.clone() for f in feats])
        y_ref, _ = patched._cerb_reference_forward(head, [f.clone() for f in feats])
        rows = non_max_suppression(y, 0.001, 0.6, multi_label=True)
    assert y.dtype == BF16 and y_ref.dtype == BF16
    assert ops.find_summary(y) is not None, "the patched forward did not run the decode kernel"
    assert ops.find_summary(y_ref) is None
    ok, msg = check_decode_bf16(y, y_ref, [t.shape[2:] for t in x], STRIDES)
    assert ok, msg
    want = rp.nms_port(y.cpu(), 0.001, 0.6, multi_label=True, greedy="c")
    assert len(rows) == 2 and sum(r.shape[0] for r in rows) > 0
    for r, w in zip(rows, want):
        assert r.dtype == torch.float32 and torch.equal(r.cpu(), w)


def test_installed_nms_wrapper_takes_bf16(monkeypatch):
    """patch.install() on stand-in reference modules: the rebound ``non_max_suppression`` sends a bf16 CUDA prediction
    to the kernel (the saved reference function is not called) and returns the port's rows bit for bit; a bf16 CPU
    prediction still goes to the reference's own function."""
    import sys
    import types

    from cerberusdet_b200 import patch
    from oracle import ref_port as rp

    ref_calls = []

    def reference_nms(prediction, *a, **k):
        ref_calls.append(prediction.dtype)
        return []

    names = ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general")
    mods = {n: types.ModuleType(n) for n in names}
    for n, m in mods.items():
        monkeypatch.setitem(sys.modules, n, m)
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = reference_nms
    patch.uninstall()
    patch.install()
    try:
        nms = mods["cerberusdet.utils.general"].non_max_suppression
        assert nms is not reference_nms and nms._cerb_reference is reference_nms
        pred = synth_prediction(3, 6, 2000, seed=12, dtype=torch.float32, regime="clusters").to(BF16)
        for kw in (dict(conf_thres=0.25, iou_thres=0.45), dict(conf_thres=0.001, iou_thres=0.6, multi_label=True)):
            got = nms(pred.cuda(), **kw)
            want = rp.nms_port(pred, greedy="c", **kw)
            assert len(got) == 3 and sum(r.shape[0] for r in got) > 0
            for r, w in zip(got, want):
                assert r.is_cuda and r.dtype == torch.float32 and torch.equal(r.cpu(), w)
        assert ref_calls == []
        nms(pred, 0.25, 0.45)  # CPU tensors: the reference's own code
        assert ref_calls == [BF16]
    finally:
        patch.uninstall()


def test_inference_bf16_model_equals_reference_nms_path(patched, monkeypatch):
    """CerberusDetInference with a bf16 model takes the split-head decode and the batched NMS kernel (counted; the
    reference NMS must not run) and returns what the port's NMS + the host tail give on the same decoded tensors."""
    from cerberusdet_b200 import cross_task as ct
    from cerberusdet_b200 import inference as inf
    from cerberusdet_b200.inference import CerberusDetInference
    from oracle import ref_port as rp
    from test_gpu_dropin import TwoTaskModel

    calls = []
    for name in ("decode_heads_split", "nms_batched", "cross_task_merge"):
        real = getattr(inf, name)
        monkeypatch.setattr(inf, name, lambda *a, _r=real, _n=name, **k: (calls.append(_n), _r(*a, **k))[1])

    def no_reference():
        raise AssertionError("the reference NMS ran: bf16 fell off the kernel path")

    monkeypatch.setattr(inf, "_reference_nms", no_reference)
    torch.manual_seed(1)
    model = TwoTaskModel().cuda().bfloat16()
    eng = CerberusDetInference(model=model, device="cuda:0", conf_thres=0.25, iou_thres=0.45, half=False, img_size=64)
    x = torch.rand(3, 3, 96, 128, device="cuda").bfloat16()
    shapes = [(480, 640), (96, 128), (300, 500)]
    calls.clear()  # (the engine's warm-up forward)
    got = eng.predict(x, original_shape=shapes, max_det=50)
    assert calls == ["decode_heads_split", "nms_batched", "cross_task_merge"], calls
    with torch.no_grad():
        out = eng.model(x)
    per_task = {t: rp.nms_port(y.cpu(), 0.25, 0.45, max_det=50, greedy="c") for t, (y, _) in out.items()}
    assert all(y.dtype == BF16 for y, _ in out.values())
    for i in range(3):
        det = ct.combine_tasks({t: per_task[t][i] for t in per_task}, eng.categories_inds_map)
        det = ct.suppress_between_tasks(det, eng.categories_inds_map, 0.8)
        if len(det):
            det[:, :4] = ct.rescale_boxes((96, 128), det[:, :4], shapes[i]).round()
        want = [{"box": [int(v) for v in r[:4]], "score": float(r[4]), "label": int(r[5])} for r in det.tolist()]
        assert len(got[i]) == len(want)
        for g, w in zip(got[i], want):
            assert g["box"] == w["box"] and g["label"] == w["label"] and g["score"] == w["score"]
    assert sum(len(r) for r in got) > 0


# ------------------------------------------------------------------ training-time box decode
def _check_bbox_decode_bf16(out, ref, grad=False, grad_out=None, gmax=None):
    """tests/tol.py check_bbox_decode with bf16's ulp: rtol 2^-7, forward + 1 ulp(gmax), at most 2 % + 8 flips."""
    of, rf = out.float().cpu(), ref.float().cpu()
    if not torch.isfinite(of).all():
        return False, "non-finite output"
    rtol = 2.0 ** -7
    if not grad:
        bound = rtol * rf.abs() + _ulp(gmax)
    else:
        g = grad_out.float().cpu().abs()
        bound = rtol * rf.abs() + rtol * 16.0 * g.repeat_interleave(16, dim=-1) + 1e-7
    d = (of - rf).abs()
    if (d > bound).any():
        return False, f"mismatch: worst excess {(d - bound).max().item():.3e}"
    if not grad:
        n = (out.cpu() != ref.cpu()).sum().item()
        if n > 0.02 * ref.numel() + 8:
            return False, f"too many 1-ulp flips: {n}/{ref.numel()}"
    return True, "ok"


@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("imgsz", [640, 1280])
def test_bbox_decode_bf16_forward_and_grad(ops, autocast, imgsz):
    from oracle import ref_port as rp

    hw = level_shapes((imgsz, imgsz), STRIDES)
    anchors, _ = rp.anchor_grid(hw, STRIDES, BF16, "cuda")
    anchors = anchors.transpose(0, 1).contiguous()  # [A, 2]
    A = anchors.shape[0]
    g = torch.Generator(device="cuda").manual_seed(imgsz + int(autocast))
    pd = (torch.randn(2, A, 64, device="cuda", generator=g) * 3).to(BF16)
    grad_out = torch.randn(2, A, 4, device="cuda", generator=g).to(BF16)
    ctx = torch.autocast("cuda", dtype=BF16) if autocast else torch.autocast("cuda", enabled=False)
    x0, x1 = pd.clone().requires_grad_(), pd.clone().requires_grad_()
    with ctx:
        out = ops.bbox_decode(anchors, x0)
        ref = rp.bbox_decode_port(anchors, x1)
    assert out.dtype == BF16 and ref.dtype == BF16
    ok, msg = _check_bbox_decode_bf16(out, ref, gmax=max(max(h, w) for h, w in hw) + 16.0)
    assert ok, f"forward: {msg}"
    out.backward(grad_out)
    ref.backward(grad_out)
    assert x0.grad.dtype == BF16
    ok, msg = _check_bbox_decode_bf16(x0.grad, x1.grad, grad=True, grad_out=grad_out)
    assert ok, f"backward: {msg}"


def test_patched_loss_bbox_decode_takes_bf16(ops, monkeypatch):
    """install(train=True) on stand-in reference modules: ``Loss.bbox_decode`` sends bf16 pred_dist + bf16 anchors to the
    kernel with and without bf16 autocast; a pred_dist dtype other than the autocast dtype keeps the reference's code."""
    import sys
    import types

    from cerberusdet_b200 import patch
    from oracle import ref_port as rp

    ref_calls = []

    class Loss:
        use_dfl = True

        def bbox_decode(self, anchor_points, pred_dist):
            ref_calls.append(pred_dist.dtype)
            return rp.bbox_decode_port(anchor_points, pred_dist)

    names = ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general",
             "cerberusdet.utils.loss", "cerberusdet.utils.tal")
    mods = {n: types.ModuleType(n) for n in names}
    for n, m in mods.items():
        monkeypatch.setitem(sys.modules, n, m)
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = lambda *a, **k: None
    mods["cerberusdet.utils.loss"].Loss = Loss
    mods["cerberusdet.utils.loss"].make_anchors = lambda feats, strides, grid_cell_offset=0.5: None
    mods["cerberusdet.utils.tal"].TaskAlignedAssigner = type("TaskAlignedAssigner", (), {"forward": lambda self, *a: None})
    kernel_calls = []
    real = ops.bbox_decode
    monkeypatch.setattr(ops, "bbox_decode", lambda a, p: (kernel_calls.append(p.dtype), real(a, p))[1])
    patch.uninstall()
    patch.install(train=True)
    try:
        anchors = (torch.rand(300, 2, device="cuda") * 40).to(BF16)
        pd = torch.randn(2, 300, 64, device="cuda").to(BF16)
        me = Loss()
        out = Loss.bbox_decode(me, anchors, pd)
        with torch.autocast("cuda", dtype=BF16):
            out_ac = Loss.bbox_decode(me, anchors, pd)
        assert kernel_calls == [BF16, BF16] and ref_calls == []
        assert torch.equal(out, out_ac) and out.dtype == BF16
        with torch.autocast("cuda", dtype=torch.float16):
            Loss.bbox_decode(me, anchors, pd)  # bf16 pred_dist under fp16 autocast: the reference's code
        with torch.autocast("cuda", dtype=BF16):
            Loss.bbox_decode(me, anchors.half(), pd.half())  # fp16 pred_dist under bf16 autocast: likewise
        assert kernel_calls == [BF16, BF16] and ref_calls == [BF16, torch.float16]
    finally:
        patch.uninstall()
