"""bf16 autocast training through the assigner and the box-regression loss: ``ops.tal_assign`` with bf16 scores,
``ops.bbox_loss`` with bf16 predictions, the chain logits -> ``bbox_decode`` -> assigner -> loss -> backward, and the
``install(train=True, loss=True)`` gates -- all under ``torch.autocast("cuda", dtype=torch.bfloat16)``, the trainer's
case.  The references are the ports (oracle/ref_port.py, tests/bbox_loss_port.py) run on CUDA tensors under the same
autocast, so autocast's own op lists decide every rounding point; tests/test_train_bf16_host.py states the rules.

Bounds.  Assigner: every output bit for bit against the port on the images the port marks unambiguous, and bf16
scores give exactly what the same values in fp32 give on every image.  Box loss: the per-anchor CIoU term bit for bit,
the per-anchor DFL term and the scalars as in test_gpu_train_scale.py; gradients within ``bf16_grads_ratio`` (one bf16
ulp, see there).  Chain: the logit gradient within 20 bf16 ulps, fp16's 2e-2 of test_gpu_train_scale.py scaled by
bf16's 8 fewer bits (the decode's backward rounds differently from the port's by design)."""
import math
import os
import sys
import warnings

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from oracle.ref_import import reference_available  # noqa: E402
from test_gpu_train_scale import _dfl_ratio, _edge_case, _finite_rows  # noqa: E402
from test_loss_host import _RefBboxLoss  # noqa: E402
from test_train_bounds_host import MAX_CHANGED_F16, flat_case, scalar_ratio  # noqa: E402

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16
LEVELS = [(80, 80), (40, 40), (20, 20)]
STRIDES = [8, 16, 32]
GO = (0.7, 1.3)  # incoming gradients of loss_iou and loss_dfl
NAMES = ("target_labels", "target_bboxes", "target_scores", "fg_mask", "target_gt_idx")


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    return o


# the share of box-gradient values allowed to differ from the port's at all (measured on a B200: up to 24 % with every
# anchor in the foreground).  A predicted coordinate's gradient has up to four contributions (w1 or h1, the intersection,
# the enclosing box, the centre distance); the kernel adds them in fp32 and rounds once, autograd rounds its running sum
# to bf16 after each addition.  In fp16 most of these gradients are subnormal, where the additions are exact, and fewer
# than MAX_CHANGED_F16 of them differ; in bf16 they are normal numbers.  The per-element bound holds either way.
MAX_CHANGED_BF16_BOX = 0.35


def bf16_grads_ratio(got, want, group, max_changed=MAX_CHANGED_F16):
    """bf16 gradients against the port: ``|got - want| <= 2^-7 (|want| + S) + ulp(S)`` per element, ``S`` the largest
    ``|want|`` of its group (a box's 4 sides, a side's 16 bins) and ``ulp(S) = 2^(floor(log2 S) - 7)`` bf16's ulp there;
    and at most ``max_changed`` of the values differ at all.  This is test_gpu_loss.py's fp16 bound (1e-3 ~ one fp16
    ulp, plus half an ulp of S) with bf16's ulp; the count catches a rounding made in the wrong place on every value,
    which one ulp per element would let through (``MAX_CHANGED_BF16_BOX`` for the box gradients).  Returns
    ``(worst ratio, changed fraction)``."""
    g, w = got.float().cpu(), want.float().cpu()
    assert torch.isfinite(g).all()
    S = w.abs().reshape(-1, group).amax(-1, keepdim=True).expand(-1, group).reshape(w.shape)
    ulp = torch.exp2(torch.floor(torch.log2(S.clamp(min=2.0**-126))) - 7)
    bound = 2.0**-7 * (w.abs() + S) + ulp
    d = (g - w).abs()
    ok = d <= bound
    assert ok.all(), f"worst excess {(d - bound).max().item():.3e} of {int((~ok).sum())} values"
    frac = float((got.cpu() != want.cpu()).float().mean())
    assert frac <= max_changed, f"{frac:.2%} of the bf16 gradient values differ from the port's (limit {max_changed:.0%})"
    return float((d / bound).max()), frac


# ----------------------------------------------------------------------------- 1. the rounding points, pinned
def test_autocast_rounding_points_on_the_gpu():
    """What the reference's ops do under CUDA autocast, bf16 and fp16 (autocast's op lists do not depend on the dtype).
    tests/test_train_bf16_host.py shows that each rule is observable: the alternatives give other bits."""
    g = torch.Generator(device="cuda").manual_seed(1)
    s = torch.rand(1 << 16, device="cuda", generator=g).clamp(min=1e-3)
    for dt in (BF16, torch.float16):
        x = s.to(dt)
        with torch.autocast("cuda", dtype=dt):
            p = x.pow(0.5)  # the assigner's bbox_scores.pow(alpha) (utils/tal.py:129)
        assert p.dtype == torch.float32 and torch.equal(p, x.float().pow(0.5)), dt
        assert not torch.equal(p, x.pow(0.5).float()), dt  # outside autocast the power is rounded to the score dtype
    # BboxLoss: predictions bf16, targets fp32
    a = (torch.rand(4096, device="cuda", generator=g) * 40).to(BF16)
    b = a + (torch.rand(4096, device="cuda", generator=g) * 9 + 0.5).to(BF16)
    t = torch.rand(4096, device="cuda", generator=g) * 40
    with torch.autocast("cuda", dtype=BF16):
        w1 = b - a
        h1 = b - a + 1e-7
        assert w1.dtype == h1.dtype == (w1 * h1).dtype == (w1 / h1).dtype == torch.atan(w1 / h1).dtype == BF16
        assert (b - t).dtype == (w1 * h1 + t).dtype == (torch.atan(t / t) - torch.atan(w1 / h1)).dtype == torch.float32
        logits = (torch.randn(2048, 16, device="cuda", generator=g) * 3).to(BF16)
        tgt = torch.randint(0, 16, (2048,), device="cuda", generator=g)
        ce = torch.nn.functional.cross_entropy(logits, tgt, reduction="none")
    assert ce.dtype == torch.float32
    # log_softmax keeps bf16 (rounded once), nll_loss reads it in fp32
    ls = torch.log_softmax(logits, 1)
    assert ls.dtype == BF16 and torch.equal(ce, -ls.float().gather(1, tgt[:, None])[:, 0])
    assert not torch.equal(ce, -torch.log_softmax(logits.float(), 1).gather(1, tgt[:, None])[:, 0])


# ----------------------------------------------------------------------------- 2. the assigner
def _port_on_gpu(c, nc, topk, slice_=8):
    """``tal_assign_port`` on CUDA tensors under bf16 autocast, image slice by image slice (it materialises
    [B, G, topk, A]): the five outputs and the per-image ambiguity flag."""
    per_image = ("pd_scores", "pd_bboxes", "gt_labels", "gt_bboxes", "mask_gt")
    parts = []
    for s in range(0, c["pd_scores"].shape[0], slice_):
        sub = {k: (v[s:s + slice_] if k in per_image else v) for k, v in c.items()}
        with torch.device("cuda"), torch.autocast("cuda", dtype=BF16):
            out = rp.tal_assign_port(**sub, topk=topk, num_classes=nc)
        parts.append(out[:5] + (out[5].any(-1),))
    return tuple(torch.cat(t) for t in zip(*parts))


def _kernel_assign(ops, c, nc, topk):
    with torch.autocast("cuda", dtype=BF16):
        return ops.tal_assign(**c, topk=topk, num_classes=nc)


@pytest.mark.parametrize("name,bs,level_hw,nc,G,topk", [
    ("B4x8400", 4, LEVELS, 20, 20, 10),                                 # the training shape of test_gpu_tal.py
    ("B64x8400", 64, LEVELS, 20, 30, 10),                               # the trainer's batch
    ("B64_topk16", 64, LEVELS, 20, 30, 16),                             # the largest topk
    ("G1024", 2, LEVELS, 12, 1024, 16),                                 # the most boxes, 640 x 640
    ("small", 3, [(12, 20), (6, 10), (3, 5)], 3, 4, 10),                # fewer than topk anchors inside most boxes
])
def test_tal_assign_bf16_equals_the_port_under_bf16_autocast(ops, name, bs, level_hw, nc, G, topk, record_property):
    """Unambiguous images bit for bit.  With 1024 boxes on one image every image has a box with fewer than topk
    positive-metric anchors and zero-metric ones inside (ambiguous in the reference); there the port's tie rule, which
    the kernels share, is compared on every image."""
    c = {k: v.cuda() for k, v in rp.tal_case(700 + G + topk, bs, level_hw, STRIDES, nc, G, score_dtype=BF16).items()}
    assert c["pd_scores"].dtype == BF16
    got = _kernel_assign(ops, c, nc, topk)
    *want, ambiguous = _port_on_gpu(c, nc, topk)
    clean = (~ambiguous).nonzero().flatten().cpu()
    record_property(f"{name}:clean_images", len(clean))
    if name == "G1024":
        clean = torch.arange(bs)
    elif name != "small":  # (boxes with fewer than topk anchors inside are the ambiguous kind)
        assert len(clean) >= bs // 2, "the seeded case should be unambiguous for most images"
    for n, a, b in zip(NAMES, got, want):
        assert a.dtype == b.dtype and a.shape == b.shape, n
        a, b = a.cpu()[clean], b.cpu()[clean]
        assert torch.equal(a, b), f"{n}: {int((a != b).sum())} values differ"
    assert got[3].any()
    # the widen-then-fp32 rule: bf16 scores are the fp32 path on the same values, on every image
    wide = _kernel_assign(ops, dict(c, pd_scores=c["pd_scores"].float()), nc, topk)
    for n, a, b in zip(NAMES, got, wide):
        assert a.dtype == b.dtype and torch.equal(a, b), n


def test_tal_assign_bf16_is_deterministic_sync_free_and_graph_replayable(ops):
    nc, topk = 20, 10
    c = {k: v.cuda() for k, v in rp.tal_case(720, 8, LEVELS, STRIDES, nc, 24, score_dtype=BF16).items()}
    a, b = _kernel_assign(ops, c, nc, topk), _kernel_assign(ops, c, nc, topk)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    torch.cuda.synchronize()
    prev = torch.cuda.get_sync_debug_mode()
    torch.cuda.set_sync_debug_mode("error")
    try:
        _kernel_assign(ops, c, nc, topk)
    finally:
        torch.cuda.set_sync_debug_mode(prev)
    static = {k: v.clone() for k, v in c.items()}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _kernel_assign(ops, static, nc, topk)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = _kernel_assign(ops, static, nc, topk)
    for seed in (721, 722):
        fresh = {k: v.cuda() for k, v in rp.tal_case(seed, 8, LEVELS, STRIDES, nc, 24, score_dtype=BF16).items()}
        for k, v in fresh.items():
            static[k].copy_(v)
        graph.replay()
        torch.cuda.synchronize()
        e = _kernel_assign(ops, fresh, nc, topk)
        assert all(torch.equal(x, y) for x, y in zip(out, e)), seed


# ----------------------------------------------------------------------------- 3. the box-regression loss
def _cuda(c):
    half = ("pred_dist", "pred_bboxes", "anchor_points")
    return {k: (v.to("cuda", BF16) if k in half else v.cuda()) for k, v in c.items()}


def _run(fn, c, per=True, tss=None):
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    args = dict(c, pred_dist=pd, pred_bboxes=pb)
    if tss is not None:
        args["target_scores_sum"] = tss
    with torch.autocast("cuda", dtype=BF16):
        out = fn(**args)
    gd, gb = torch.autograd.grad(out[:2], (pd, pb), tuple(torch.tensor(g, device="cuda") for g in GO), allow_unused=True)
    gd = torch.zeros_like(pd) if gd is None else gd
    gb = torch.zeros_like(pb) if gb is None else gb
    return out[0].detach(), out[1].detach(), gd, gb, (out[2] if per else None)


def _kernel_fn(ops):
    def fn(**k):
        per = torch.empty(k["fg_mask"].shape + (2,), device="cuda")
        li, ld = ops.bbox_loss(**k, per_anchor=per)
        return li, ld, per

    return fn


def _port_fn(**k):
    return lp.bbox_loss_port(**k, terms=True)


def compare_with_port(ops, c, rec, tag):
    li, ld, gd, gb, per = _run(_kernel_fn(ops), c)
    wi, wd, wgd, wgb, wper = _run(_port_fn, c)
    assert gd.dtype == gb.dtype == wgd.dtype == wgb.dtype == BF16 and li.dtype == torch.float32
    n_rows = c["fg_mask"].numel()
    tss = c["target_scores_sum"]
    m = {"ciou_mismatch": int((per[..., 0] != wper[..., 0]).sum()), "dfl": _dfl_ratio(per, wper, c),
         "scalar_iou": scalar_ratio(li, per[..., 0], tss, n_rows), "scalar_dfl": scalar_ratio(ld, per[..., 1], tss, n_rows),
         "port_iou": abs(float(li) - float(wi)) / (1e-5 * abs(float(wi)) + 1e-30),
         "port_dfl": abs(float(ld) - float(wd)) / (1e-5 * abs(float(wd)) + 1e-30)}
    ok = _finite_rows(gb, wgb)
    m["grad_box"], m["changed_box"] = bf16_grads_ratio(gb[ok], wgb[ok], 4, MAX_CHANGED_BF16_BOX)
    m["grad_dist"], m["changed_dist"] = bf16_grads_ratio(gd, wgd, 16)
    for k, v in m.items():
        rec(f"{tag}:{k}", v)
    assert m["ciou_mismatch"] == 0, f"{m['ciou_mismatch']} per-anchor CIoU terms differ from the port's"
    assert m["dfl"] <= 1.0, "per-anchor DFL term"
    assert m["scalar_iou"] <= 1.0 and m["scalar_dfl"] <= 1.0, "scalars off the kernel's own per-anchor terms"
    assert m["port_iou"] <= 1.0 and m["port_dfl"] <= 1.0, "scalars off the port's"
    assert not gd[~c["fg_mask"]].any() and not gb[~c["fg_mask"]].any()
    return li, ld, gd, gb, per


@pytest.mark.parametrize("kind", ["train", "crowded", "one_level", "all"])
def test_bbox_loss_bf16_matches_the_port_under_bf16_autocast(ops, kind, record_property):
    from test_gpu_loss import _case

    c = _case(ops, kind, dtype=BF16)
    assert c["pred_dist"].dtype == BF16 and c["target_bboxes"].dtype == torch.float32
    compare_with_port(ops, c, record_property, kind)


@pytest.mark.parametrize("fg", [0.04, 1.0])
def test_bbox_loss_bf16_at_the_trainer_shape(ops, fg, record_property):
    compare_with_port(ops, _cuda(flat_case(164, 64, 8400, fg=fg)), record_property, "B64x8400")


@pytest.mark.parametrize("kind", ["C1", "C3", "C365", "logits", "near160", "dfl_edges", "degenerate"])
def test_bbox_loss_bf16_edge_inputs_match_the_port(ops, kind, record_property):
    """test_gpu_train_scale.py's fp16 edges (logits x12): fewer than four classes and many, logits far below the
    maximum, coordinates near 160 grid units (bf16's ulp is 1 there), DFL targets on bin edges, degenerate boxes."""
    c = _edge_case(kind, True)
    if kind == "degenerate":  # targets on bf16 values, so that a bf16 prediction can equal its target
        tb = c["target_bboxes"].to(BF16).float()
        k = torch.arange(tb.shape[1]) % 4
        c["target_bboxes"] = tb
        c["pred_bboxes"][:, k == 2] = tb[:, k == 2]
    c = _cuda(c)
    if kind == "degenerate":
        assert (c["pred_bboxes"] == c["target_bboxes"].to(BF16)).all(-1)[c["fg_mask"]].any()
    compare_with_port(ops, c, record_property, kind)


def test_bbox_loss_bf16_tss_forms_and_misaligned_pred_dist_give_the_same_bits(ops, record_property):
    c = _cuda(flat_case(400, 8, 4096, fg=0.2))
    ref = _run(_kernel_fn(ops), c)
    tss = c["target_scores_sum"]
    for form in (float(tss), tss.cpu()):
        got = _run(_kernel_fn(ops), c, tss=form)
        assert all(torch.equal(x, y) for x, y in zip(got, ref)), type(form)
    n = c["pred_dist"].numel()
    buf = torch.zeros(n + 8, dtype=BF16, device="cuda")
    view = buf[4:4 + n].view_as(c["pred_dist"])
    view.copy_(c["pred_dist"])
    assert view.data_ptr() % 32 != 0 and view.is_contiguous()
    got = _run(_kernel_fn(ops), dict(c, pred_dist=view))
    assert all(torch.equal(x, y) for x, y in zip(got, ref))


def test_bbox_loss_bf16_is_deterministic_sync_free_and_graph_replayable(ops):
    B, A = 64, 8400
    c = _cuda(flat_case(201, B, A))
    a, b = _run(_kernel_fn(ops), c), _run(_kernel_fn(ops), c)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    torch.cuda.synchronize()
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    go = torch.ones((), device="cuda")
    prev = torch.cuda.get_sync_debug_mode()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.autocast("cuda", dtype=BF16):
            li, ld = ops.bbox_loss(**dict(c, pred_dist=pd, pred_bboxes=pb))
        torch.autograd.backward((li, ld), (go, go))
    finally:
        torch.cuda.set_sync_debug_mode(prev)
    torch.cuda.synchronize()
    assert pd.grad.dtype == BF16 and pb.grad.dtype == BF16
    static = {k: v.clone() for k, v in c.items()}
    spd = static["pred_dist"].requires_grad_(True)
    spb = static["pred_bboxes"].requires_grad_(True)
    gos = tuple(torch.tensor(g, device="cuda") for g in GO)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            with torch.autocast("cuda", dtype=BF16):
                li, ld = ops.bbox_loss(**static)
            torch.autograd.grad((li, ld), (spd, spb), gos)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        with torch.autocast("cuda", dtype=BF16):
            li, ld = ops.bbox_loss(**static)
        gd, gb = torch.autograd.grad((li, ld), (spd, spb), gos)
    for seed in (202, 203):
        fresh = _cuda(flat_case(seed, B, A))
        for k, v in fresh.items():
            static[k].detach().copy_(v)
        graph.replay()
        graph.replay()  # the workspace ticket must be left ready by every launch
        torch.cuda.synchronize()
        e = _run(_kernel_fn(ops), fresh)
        assert torch.equal(li, e[0]) and torch.equal(ld, e[1]) and torch.equal(gd, e[2]) and torch.equal(gb, e[3])


# ----------------------------------------------------------------------------- 4. the training chain
def test_training_chain_bf16_matches_the_ports(ops, record_property):
    """test_gpu_train_scale.py's chain at B=16, 640 under bf16 autocast: head logits -> bbox_decode -> assigner -> box
    loss -> backward to the logits, kernels against the ports (the assigner's port on the GPU under the same autocast).
    The port chain carries the kernel decode's box values forward (the decodes' last bits differ by design) and sends
    the gradient back through its own decode."""
    B, nc = 16, 20
    c = rp.tal_case(600, B, LEVELS, STRIDES, nc, 20)
    g = torch.Generator().manual_seed(601)
    A = c["anc_points"].shape[0]
    dist = (torch.randn(B, A, 64, generator=g) * 3).to("cuda", BF16)
    cls = (torch.randn(B, A, nc, generator=g) * 2 - 1).to("cuda", BF16)
    anc, st = rp.anchor_grid(LEVELS, STRIDES, BF16, "cuda")
    ap, st = anc.t().contiguous(), st.t().contiguous()
    gt = {k: c[k].cuda() for k in ("gt_labels", "gt_bboxes", "mask_gt")}

    def chain(decode, assign, loss, boxes=None):
        pd = dist.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=BF16):
            pb = decode(ap, pd)
            if boxes is not None:
                pb = boxes + (pb - pb.detach())
            args = dict(pd_scores=cls.detach().sigmoid(), pd_bboxes=(pb.detach() * st).type(gt["gt_bboxes"].dtype),
                        anc_points=ap * st, **gt)
            assert args["pd_scores"].dtype == BF16
            out = assign(args)
            tb = out[1] / st
            tss = out[2].sum().clamp(min=1)
            li, ld = loss(pd, pb, ap, tb, out[2], tss, out[3])
        (gd,) = torch.autograd.grad((li, ld), (pd,), tuple(torch.tensor(v, device="cuda") for v in GO))
        return out, li.detach(), ld.detach(), gd, pb.detach()

    kout, ki, kd, kg, kpb = chain(ops.bbox_decode, lambda a: ops.tal_assign(**a, topk=10, num_classes=nc), ops.bbox_loss)
    ambiguous = []

    def port_assign(a):
        out = _port_on_gpu(a, nc, 10)
        ambiguous.append(out[5])
        return out[:5]

    pout, pi, pdl, pg, ppb = chain(rp.bbox_decode_port, port_assign, lp.bbox_loss_port, boxes=kpb)
    assert torch.equal(ppb, kpb) and ppb.dtype == BF16
    clean = (~ambiguous[0]).nonzero().flatten()
    record_property("chain:clean_images", len(clean))
    assert len(clean) >= B // 2
    for n, a, b in zip(NAMES, kout, pout):
        assert torch.equal(a[clean], b[clean]), n
    same = all(torch.equal(a, b) for a, b in zip(kout, pout))
    record_property("chain:same_assignment", same)
    if same:  # the loss saw the same assignment in both chains (ambiguous images included: same tie rule)
        for a, b, tag in ((ki, pi, "iou"), (kd, pdl, "dfl")):
            r = abs(float(a) - float(b)) / (1e-5 * abs(float(b)))
            record_property(f"chain:scalar_{tag}", r)
            assert r <= 1.0, tag
        rtol = 20 * 2.0**-7
        w, gk = pg.float().cpu(), kg.float().cpu()
        S = w.abs().reshape(-1, 16).amax(-1, keepdim=True).expand(-1, 16).reshape(w.shape)
        bound = rtol * (w.abs() + S) + torch.exp2(torch.floor(torch.log2(S.clamp(min=2.0**-126))) - 7)
        r = float(((gk - w).abs() / bound).max())
        record_property("chain:grad_logits", r)
        assert torch.isfinite(gk).all() and r <= 1.0


# ----------------------------------------------------------------------------- 5. install() gates, on stand-in modules
@pytest.fixture()
def stub_modules(monkeypatch):
    import types

    from cerberusdet_b200 import patch

    ref_calls = []

    class TaskAlignedAssigner:
        def __init__(self, topk=10, num_classes=80, alpha=0.5, beta=6.0, eps=1e-9):
            self.topk, self.num_classes, self.alpha, self.beta, self.eps = topk, num_classes, alpha, beta, eps

        def __call__(self, *a):
            return type(self).forward(self, *a)

        def forward(self, pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt):
            ref_calls.append(("assign", pd_scores.dtype))
            with torch.device(pd_scores.device):
                return rp.tal_assign_port(pd_scores, pd_bboxes, anc_points, gt_labels, gt_bboxes, mask_gt, self.topk,
                                          self.num_classes, self.alpha, self.beta, self.eps)[:5]

    class BboxLoss(_RefBboxLoss):
        def forward(self, pred_dist, *a):
            ref_calls.append(("loss", pred_dist.dtype))
            return super().forward(pred_dist, *a)

    class Loss:
        use_dfl = True

        def bbox_decode(self, anchor_points, pred_dist):
            return rp.bbox_decode_port(anchor_points, pred_dist)

    names = ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general",
             "cerberusdet.utils.loss", "cerberusdet.utils.tal")
    mods = {n: types.ModuleType(n) for n in names}
    for n, m in mods.items():
        monkeypatch.setitem(sys.modules, n, m)
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = lambda *a, **k: None
    mods["cerberusdet.utils.loss"].Loss = Loss
    mods["cerberusdet.utils.loss"].BboxLoss = BboxLoss
    mods["cerberusdet.utils.loss"].make_anchors = lambda feats, strides, grid_cell_offset=0.5: None
    mods["cerberusdet.utils.tal"].TaskAlignedAssigner = TaskAlignedAssigner
    patch.uninstall()
    yield mods, ref_calls
    patch.uninstall()


def _ctx(dtype):
    return torch.autocast("cuda", dtype=dtype) if dtype is not None else torch.autocast("cuda", enabled=False)


def test_install_sends_bf16_autocast_to_both_kernels_and_every_other_mix_to_the_reference(ops, stub_modules, monkeypatch):
    from cerberusdet_b200 import patch

    from test_gpu_loss import _case

    mods, ref_calls = stub_modules
    nc = 7
    a = {k: v.cuda() for k, v in rp.tal_case(41, 2, [(20, 20), (10, 10), (5, 5)], STRIDES, nc, 9).items()}
    asg = mods["cerberusdet.utils.tal"].TaskAlignedAssigner(topk=10, num_classes=nc)
    order = ("pd_scores", "pd_bboxes", "anc_points", "gt_labels", "gt_bboxes", "mask_gt")
    lc = _case(ops, "one_level")
    kernel_calls = []
    real_assign, real_loss = ops.tal_assign, ops.bbox_loss
    monkeypatch.setattr(ops, "tal_assign", lambda *a, **k: (kernel_calls.append(("assign", a[0].dtype)), real_assign(*a, **k))[1])
    monkeypatch.setattr(ops, "bbox_loss", lambda *a, **k: (kernel_calls.append(("loss", a[0].dtype)), real_loss(*a, **k))[1])
    info = patch.install(train=True, loss=True)
    assert "cerberusdet.utils.tal.TaskAlignedAssigner.forward" in info["patched"]
    assert "cerberusdet.utils.loss.BboxLoss.forward" in info["patched"]
    bl = mods["cerberusdet.utils.loss"].BboxLoss(15, use_dfl=True)
    lorder = ("pred_dist", "pred_bboxes", "anchor_points", "target_bboxes", "target_scores", "target_scores_sum", "fg_mask")

    def assign(dtype, ac):
        with _ctx(ac):
            return asg(*[a[k].to(dtype) if k == "pd_scores" else a[k] for k in order])

    def loss(dtype, ac):
        with _ctx(ac):
            return bl(*[lc[k].to(dtype) if k in ("pred_dist", "pred_bboxes", "anchor_points") else lc[k] for k in lorder])

    # bf16 autocast, the trainer's case: both kernels
    got_a = assign(BF16, BF16)
    got_l = loss(BF16, BF16)
    assert kernel_calls == [("assign", BF16), ("loss", BF16)] and ref_calls == []
    with torch.device("cuda"), torch.autocast("cuda", dtype=BF16):
        want_a = rp.tal_assign_port(*[a[k].to(BF16) if k == "pd_scores" else a[k] for k in order], 10, nc)[:5]
    assert all(torch.equal(x, y) for x, y in zip(got_a, want_a))
    with torch.autocast("cuda", dtype=BF16):
        want_l = lp.bbox_loss_port(*[lc[k].to(BF16) if k in ("pred_dist", "pred_bboxes", "anchor_points") else lc[k]
                                     for k in lorder])
    for x, y in zip(got_l, want_l):
        assert abs(float(x) - float(y)) <= 1e-5 * abs(float(y)) + 1e-30
    # the excluded mixes: bf16 outside autocast, bf16 under fp16 autocast, fp16 under bf16 autocast (the loss)
    kernel_calls.clear()
    assign(BF16, None)
    assign(BF16, torch.float16)
    loss(BF16, None)
    loss(BF16, torch.float16)
    loss(torch.float16, BF16)
    assert kernel_calls == []
    assert ref_calls == [("assign", BF16), ("assign", BF16), ("loss", BF16), ("loss", BF16), ("loss", torch.float16)]
    # the cases that took the kernels before still do
    ref_calls.clear()
    assign(torch.float32, None)
    assign(torch.float16, torch.float16)
    loss(torch.float32, None)
    loss(torch.float16, torch.float16)
    assert kernel_calls == [("assign", torch.float32), ("assign", torch.float16), ("loss", torch.float32),
                            ("loss", torch.float16)] and ref_calls == []


# ----------------------------------------------------------------------------- 6. against the reference itself
@pytest.mark.skipif(not reference_available(), reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_reference_assigner_and_bboxloss_under_bf16_autocast_patched_vs_unpatched(ops):
    from oracle.ref_import import load_reference

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        load_reference()
    from cerberusdet.utils.loss import BboxLoss
    from cerberusdet.utils.tal import TaskAlignedAssigner

    from cerberusdet_b200 import patch
    from test_gpu_loss import _case

    patch.uninstall()
    nc, bs = 20, 8
    c = rp.tal_case(31, bs, LEVELS, STRIDES, nc, 24, score_dtype=BF16)
    ambiguous = rp.tal_assign_port(**{k: (v.float() if k == "pd_scores" else v) for k, v in c.items()}, num_classes=nc)[5]
    clean = [i for i in range(bs) if not bool(ambiguous[i].any())]
    assert len(clean) >= bs // 2
    d = {k: v.cuda() for k, v in c.items()}
    asg = TaskAlignedAssigner(topk=10, num_classes=nc, alpha=0.5, beta=6.0).cuda()
    args = [d[k] for k in ("pd_scores", "pd_bboxes", "anc_points", "gt_labels", "gt_bboxes", "mask_gt")]
    lc = _case(ops, "train", dtype=BF16)
    ref = BboxLoss(15, use_dfl=True).cuda()
    with torch.autocast("cuda", dtype=BF16):
        want_a = asg(*args)
    wi, wd, wgd, wgb, _ = _run(lambda **k: ref(*k.values()), lc, per=False)
    try:
        patch.install(train=True, loss=True)
        calls = []
        real_a, real_l = ops.tal_assign, ops.bbox_loss
        ops.tal_assign = lambda *a, **k: (calls.append("assign"), real_a(*a, **k))[1]
        ops.bbox_loss = lambda *a, **k: (calls.append("loss"), real_l(*a, **k))[1]
        try:
            with torch.autocast("cuda", dtype=BF16):
                got_a = asg(*args)
            li, ld, gd, gb, _ = _run(lambda **k: ref(*k.values()), lc, per=False)
        finally:
            ops.tal_assign, ops.bbox_loss = real_a, real_l
        assert calls == ["assign", "loss"]
        for n, a, b in zip(NAMES, got_a, want_a):
            assert torch.equal(a[clean], b[clean]), n
        for a, b in ((li, wi), (ld, wd)):
            assert abs(float(a) - float(b)) <= 1e-5 * abs(float(b)) + 1e-30
        bf16_grads_ratio(gb, wgb, 4, MAX_CHANGED_BF16_BOX)
        bf16_grads_ratio(gd, wgd, 16)
    finally:
        patch.uninstall()
    assert math.isfinite(float(li))
