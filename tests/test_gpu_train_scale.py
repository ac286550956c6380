"""The training-loss kernels at the trainer's sizes and at their numeric edges: the box-regression loss
(``ops.bbox_loss``), the TAL assigner (``ops.tal_assign``) and the chain head logits -> ``ops.bbox_decode`` ->
assigner -> loss -> backward that ``Loss.__call__`` (reference utils/loss.py:139-170) composes.  References: the loss
port (tests/bbox_loss_port.py) and the closed-form fp64 gradient (tests/test_loss_host.py) run on the same GPU, the
assigner port (oracle/ref_port.py) on the CPU.  The comparators and their derivations are in
tests/test_train_bounds_host.py, which also shows that each of them rejects small errors.

Bounds.  Per anchor: the CIoU term bit for bit; the DFL term ``1e-5 |want| + 4 ulp(R) * weight`` with ``R`` the
largest spread ``max - min`` of the anchor's logits over its sides, at least 16 (log_softmax is a difference of terms
that large; the bound of test_gpu_loss.py, which assumes logits below 16).  Scalars: ``loss * tss`` against the fp64
sum of the kernel's own per-anchor column within the summation-tree bound (``scalar_ratio``), and the port's scalar
within 1e-5.  fp32 gradients: every value within ``2 u e`` of the float64 closed form and ``4 u e`` of the port, ``e``
the first-order error bound of its float32 evaluation (``grad_error_bound``): it grows with the terms a value is made
of, so a value whose paths cancel (a predicted box equal to its target; a softmax near 1 at the target bin) is bounded
by the size of those paths, not by the residue.  fp16 gradients: ``_grads_close`` against the port, 1e-3 and one half
ulp, and at most ``MAX_CHANGED_F16`` of the values may differ.  The chain's logit gradient adds the decode's backward,
which rounds differently from the port's by design (tol.check_bbox_decode): ``_grads_close`` at rtol 1e-4 in fp32 and
2e-2 in fp16 (under autocast the reference's softmax backward runs on unrounded fp32 probabilities).
Every measured ratio is recorded as a test property (``--junitxml``)."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from test_gpu_loss import _grads_close  # noqa: E402
from test_loss_host import _host_case  # noqa: E402
from test_train_bounds_host import (MAX_CHANGED_F16, assign_ratio, flat_case, grad_bound_ratio,  # noqa: E402
                                    grad_error_bound, half_grads_ratio, scalar_ratio)

pytestmark = pytest.mark.gpu
LEVELS = [(80, 80), (40, 40), (20, 20)]
STRIDES = [8, 16, 32]
GO = (0.7, 1.3)  # incoming gradients of loss_iou and loss_dfl


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    return o


def _cuda(c, dtype=torch.float32):
    """Move a loss case to the GPU; ``pred_dist``, ``pred_bboxes`` and ``anchor_points`` in ``dtype`` (fp16 = the
    trainer's autocast case), the targets float32."""
    half = ("pred_dist", "pred_bboxes", "anchor_points")
    return {k: (v.to("cuda", dtype) if k in half else v.cuda()) for k, v in c.items()}


def _kernel(ops, c, amp, pd=None, tss=None):
    pd = c["pred_dist"].clone().requires_grad_(True) if pd is None else pd
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    per = torch.empty(c["fg_mask"].shape + (2,), device="cuda")
    args = dict(c, pred_dist=pd, pred_bboxes=pb)
    if tss is not None:
        args["target_scores_sum"] = tss
    with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        li, ld = ops.bbox_loss(**args, per_anchor=per)
    gd, gb = torch.autograd.grad((li, ld), (pd, pb), tuple(torch.tensor(g, device="cuda") for g in GO))
    return li.detach(), ld.detach(), gd, gb, per


def _port(c, amp):
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        li, ld, per = lp.bbox_loss_port(**dict(c, pred_dist=pd, pred_bboxes=pb), terms=True)
    gd, gb = torch.autograd.grad((li, ld), (pd, pb), tuple(torch.tensor(g, device="cuda") for g in GO), allow_unused=True)
    gd = torch.zeros_like(pd) if gd is None else gd
    gb = torch.zeros_like(pb) if gb is None else gb
    return li.detach(), ld.detach(), gd, gb, per


def _dfl_ratio(per, wper, c):
    x = c["pred_dist"].float().view(*c["fg_mask"].shape, 4, 16)
    R = (x.amax(-1) - x.amin(-1)).amax(-1).clamp(min=16.0)
    ulp = torch.exp2(torch.floor(torch.log2(R)) - 23)
    bound = 1e-5 * wper[..., 1].abs() + 4 * ulp * c["target_scores"].sum(-1) + 1e-30
    return float(((per[..., 1] - wper[..., 1]).abs() / bound).max())


def _same_bits(x, y):
    """Bit-equal, NaN payloads included."""
    iv = {torch.float32: torch.int32, torch.float16: torch.int16}[x.dtype]
    return x.dtype == y.dtype and torch.equal(x.view(iv), y.view(iv))


def _finite_rows(gb, wgb):
    """Anchors whose box gradient is finite in both; a non-finite one must be non-finite in both (the reference's fp16
    autocast gradient of a zero-height box is NaN: w1 / h1 overflows half)."""
    fk, fw = torch.isfinite(gb).all(-1), torch.isfinite(wgb).all(-1)
    assert torch.equal(fk, fw), "non-finite box gradients differ from the port's"
    return fw


def compare_with_port(ops, c, amp, rec, tag, got=None):
    """Kernel against the port on the same GPU, every bound of the module docstring; records the worst ratios."""
    li, ld, gd, gb, per = _kernel(ops, c, amp) if got is None else got
    wi, wd, wgd, wgb, wper = _port(c, amp)
    n_rows = c["fg_mask"].numel()
    tss = c["target_scores_sum"]
    m = {}
    m["ciou_mismatch"] = int((per[..., 0] != wper[..., 0]).sum())
    m["dfl"] = _dfl_ratio(per, wper, c)
    m["scalar_iou"] = scalar_ratio(li, per[..., 0], tss, n_rows)
    m["scalar_dfl"] = scalar_ratio(ld, per[..., 1], tss, n_rows)
    m["port_iou"] = abs(float(li) - float(wi)) / (1e-5 * abs(float(wi)) + 1e-30)
    m["port_dfl"] = abs(float(ld) - float(wd)) / (1e-5 * abs(float(wd)) + 1e-30)
    for k, v in m.items():
        rec(f"{tag}:{k}", v)
    ok = _finite_rows(gb, wgb)
    if amp:
        m["grad_box"], m["changed_box"] = half_grads_ratio(gb[ok], wgb[ok], 4, MAX_CHANGED_F16)
        m["grad_dist"], m["changed_dist"] = half_grads_ratio(gd, wgd, 16, MAX_CHANGED_F16)
    else:
        (vd, vb), (ed, eb) = grad_error_bound(**c, g_iou=GO[0], g_dfl=GO[1])
        m["grad_box"], m["grad_dist"] = grad_bound_ratio(gb, wgb, eb, 2), grad_bound_ratio(gd, wgd, ed, 2)
        m["f64_box"], m["f64_dist"] = grad_bound_ratio(gb, vb, eb, 1), grad_bound_ratio(gd, vd, ed, 1)
        del vd, vb, ed, eb
    for k in [k for k in m if k.startswith(("grad", "changed", "f64"))]:
        rec(f"{tag}:{k}", m[k])
    assert m["grad_box"] <= 1.0 and m["grad_dist"] <= 1.0, "gradients off the port's"
    assert m.get("f64_box", 0.0) <= 1.0 and m.get("f64_dist", 0.0) <= 1.0, "gradients off the float64 closed form"
    assert m["ciou_mismatch"] == 0, f"{m['ciou_mismatch']} per-anchor CIoU terms differ from the port's"
    assert m["dfl"] <= 1.0, "per-anchor DFL term"
    assert m["scalar_iou"] <= 1.0 and m["scalar_dfl"] <= 1.0, "scalars off the kernel's own per-anchor terms"
    assert m["port_iou"] <= 1.0 and m["port_dfl"] <= 1.0, "scalars off the port's"
    return li, ld, gd, gb, per


# ----------------------------------------------------------------------------- 1. box loss at scale
SHAPES = [(1, 75_776), (3, 25_259), (64, 8400), (16, 33_600)]  # one full grid pass; a second pass of one anchor; trainer; 1280


@pytest.mark.parametrize("fg", [0.04, 1.0])
@pytest.mark.parametrize("amp", [False, True], ids=["fp32", "autocast"])
@pytest.mark.parametrize("B,A", SHAPES, ids=["BA75776", "BA75777", "B64x8400", "B16x33600"])
def test_bbox_loss_at_scale_matches_port(ops, B, A, amp, fg, record_property):
    """B * A = 75 776 anchors fill the capped grid (1184 CTAs x 64 anchors) exactly once, 75 777 leave one anchor for a
    second pass, B=64 x 8400 makes 8 passes and 1184 partials for the last CTA; 4 % and 100 % foreground."""
    c = _cuda(flat_case(100 + B, B, A, fg=fg), torch.float16 if amp else torch.float32)
    compare_with_port(ops, c, amp, record_property, "scale")


def test_bbox_loss_trainer_shape_is_deterministic_graph_replayable_and_resets_its_ticket(ops):
    from cerberusdet_b200 import _lib

    B, A = 64, 8400
    c = _cuda(flat_case(201, B, A))
    a, b = _kernel(ops, c, False), _kernel(ops, c, False)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    # CUDA graph: forward + backward captured once, replayed twice on fresh inputs, equal to eager
    static = {k: v.clone() for k, v in c.items()}
    pd = static["pred_dist"].requires_grad_(True)
    pb = static["pred_bboxes"].requires_grad_(True)
    go = tuple(torch.tensor(g, device="cuda") for g in GO)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            li, ld = ops.bbox_loss(**static)
            torch.autograd.grad((li, ld), (pd, pb), go)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        li, ld = ops.bbox_loss(**static)
        gd, gb = torch.autograd.grad((li, ld), (pd, pb), go)
    for seed in (202, 203):
        fresh = _cuda(flat_case(seed, B, A))
        for k, v in fresh.items():
            static[k].detach().copy_(v)
        graph.replay()
        torch.cuda.synchronize()
        e = _kernel(ops, fresh, False)
        assert torch.equal(li, e[0]) and torch.equal(ld, e[1]) and torch.equal(gd, e[2]) and torch.equal(gb, e[3])
    # the C ABI on one workspace, launched twice: the last CTA leaves the ticket at 0, and poisoned partials are all
    # overwritten before they are read
    lib = _lib.load()
    ws_bytes = int(lib.cerb_bbox_loss_workspace_bytes(B, A))
    ws = torch.full((ws_bytes // 4,), float("nan"), device="cuda")
    ws.view(torch.int32)[:4] = 0
    out = torch.empty(2, device="cuda")
    for _ in range(2):
        rc = lib.cerb_bbox_loss_fwd(c["pred_dist"].data_ptr(), c["pred_bboxes"].data_ptr(), c["anchor_points"].data_ptr(),
                                    c["target_bboxes"].data_ptr(), c["target_scores"].data_ptr(), c["fg_mask"].data_ptr(),
                                    c["target_scores_sum"].data_ptr(), 1.0, B, A, c["target_scores"].shape[-1], 16,
                                    _lib.CERB_F32, out[0:].data_ptr(), out[1:].data_ptr(), None, ws.data_ptr(), ws_bytes,
                                    torch.cuda.current_stream().cuda_stream)
        _lib.check(rc)
        torch.cuda.synchronize()
        assert int(ws.view(torch.int32)[0]) == 0, "ticket not reset"
        assert torch.equal(out[0], a[0]) and torch.equal(out[1], a[1])


# ----------------------------------------------------------------------------- 1b. box loss at its numeric edges
def _edge_case(kind, amp):
    if kind.startswith("C"):
        return flat_case(300, 4, 2048, C=int(kind[1:]), fg=0.3)
    if kind == "logits":  # bins far below the maximum underflow in exp
        return flat_case(301, 4, 2048, fg=0.3, logit=3.0 * (12 if amp else 40))
    if kind == "near160":  # half's ulp is 0.125 in [128, 256)
        return flat_case(302, 4, 2048, fg=0.3, ap_lo=150.0)
    if kind == "dfl_edges":  # integer boxes: DFL targets exactly 0, on bin edges and past 14.99; corner ties
        pd, pb, ap, tb, ts, fg = (t.float() for t in _host_case(303, B=4, A=1024, ties=True))
        return dict(pred_dist=pd, pred_bboxes=pb, anchor_points=ap, target_bboxes=tb, target_scores=ts,
                    target_scores_sum=ts.sum().clamp(min=1), fg_mask=fg.bool())
    assert kind == "degenerate"
    c = flat_case(304, 4, 2048, fg=0.5)
    c["target_bboxes"] = c["target_bboxes"].half().float()  # so that a half prediction can equal its target
    tb, pb = c["target_bboxes"], c["pred_bboxes"]
    k = torch.arange(pb.shape[1]) % 4
    pb[:, k == 0, 2] = pb[:, k == 0, 0]  # zero width
    pb[:, k == 1, 3] = pb[:, k == 1, 1]  # zero height: w1 / h1 = w1 / eps
    pb[:, k == 2] = tb[:, k == 2]  # the target itself: v = 0
    pb[:, k == 3] += torch.tensor([40.0, 0.0, 40.0, 0.0])  # far away: iou = 0
    return c


@pytest.mark.parametrize("amp", [False, True], ids=["fp32", "autocast"])
@pytest.mark.parametrize("kind", ["C1", "C3", "C365", "logits", "near160", "dfl_edges", "degenerate"])
def test_bbox_loss_edge_inputs_match_port(ops, kind, amp, record_property):
    """Fewer than four classes (lanes of ``score_weight`` that sum nothing) and many; logits x40 (fp32) / x12 (fp16);
    coordinates near 160 grid units; DFL targets on 0, integer edges and past 14.99; degenerate predicted boxes."""
    c = _cuda(_edge_case(kind, amp), torch.float16 if amp else torch.float32)
    if kind == "degenerate":
        assert (c["pred_bboxes"] == c["target_bboxes"].to(c["pred_bboxes"].dtype)).all(-1)[c["fg_mask"]].any()
    compare_with_port(ops, c, amp, record_property, "edge")


@pytest.mark.parametrize("amp", [False, True], ids=["fp32", "autocast"])
def test_bbox_loss_tss_forms_and_misaligned_pred_dist_give_the_same_bits(ops, amp, record_property):
    """``target_scores_sum`` as a Python number, a CPU tensor and a CUDA tensor; ``pred_dist`` as a contiguous view at
    a 16-byte (fp32) / 8-byte (fp16) offset, which ``ops.bbox_loss`` clones to a 32-byte aligned row start."""
    c = _cuda(flat_case(400, 8, 4096, fg=0.2), torch.float16 if amp else torch.float32)
    ref = compare_with_port(ops, c, amp, record_property, "forms")
    tss = c["target_scores_sum"]
    for form in (float(tss), tss.cpu()):
        got = _kernel(ops, c, amp, tss=form)
        assert all(_same_bits(x, y) for x, y in zip(got, ref)), type(form)
    n = c["pred_dist"].numel()
    buf = torch.zeros(n + 8, dtype=c["pred_dist"].dtype, device="cuda")
    view = buf[4:4 + n].view_as(c["pred_dist"])
    view.copy_(c["pred_dist"])
    assert view.data_ptr() % 32 != 0 and view.is_contiguous()
    got = _kernel(ops, c, amp, pd=view.requires_grad_(True))
    assert all(_same_bits(x, y) for x, y in zip(got, ref))


# ----------------------------------------------------------------------------- 2. assigner at scale and at its limits
def _port_assign(c, nc, topk=10, slice_=8):
    """The port on the CPU, image slice by image slice (it materialises [B, G, topk, A]): the five outputs and the
    number of boxes claiming each anchor before the claims are resolved."""
    per_image = ("pd_scores", "pd_bboxes", "gt_labels", "gt_bboxes", "mask_gt")
    parts = []
    for s in range(0, c["pd_scores"].shape[0], slice_):
        sub = {k: (v[s:s + slice_] if k in per_image else v) for k, v in c.items()}
        out = rp.tal_assign_port(**sub, topk=topk, num_classes=nc, claims=True)
        parts.append(out[:5] + out[6:])
    return tuple(torch.cat(t) for t in zip(*parts))


def _assign(ops, c, nc, topk=10):
    """Kernel on the whole batch against the port: ``(got, want, claims)``."""
    got = ops.tal_assign(**{k: v.cuda() for k, v in c.items()}, topk=topk, num_classes=nc)
    *want, claims = _port_assign(c, nc, topk)
    torch.cuda.synchronize()
    return got, tuple(want), claims


@pytest.mark.parametrize("name,bs,level_hw,nc,G,dtype", [
    ("B64x8400", 64, LEVELS, 20, 30, torch.float16),                            # the trainer's batch
    ("A33600", 2, [(160, 160), (80, 80), (40, 40)], 20, 20, torch.float32),     # 1280 input
    ("G513", 2, [(32, 32), (16, 16), (8, 8)], 12, 513, torch.float32),          # a second pass of the 512-thread box loops
    ("G1024", 1, [(32, 32), (16, 16), (8, 8)], 12, 1024, torch.float16),        # the limit: shared memory of 1024 boxes
])
def test_tal_assign_at_scale_matches_port(ops, name, bs, level_hw, nc, G, dtype, record_property):
    """G in {513, 1024} on a 256 x 256 image (1344 anchors): boxes of 12-100 px, each anchor inside dozens of them, so
    most positives are claimed by several boxes and go through the argmax over all boxes."""
    c = rp.tal_case(500 + G, bs, level_hw, STRIDES, nc, G, score_dtype=dtype)
    got, want, claims = _assign(ops, c, nc)
    record_property(f"{name}:scores", assign_ratio(got, want))
    assert got[3].any()
    if G > 512:  # most positives are claimed by several boxes (cnt > 1 in the kernel)
        assert int((claims > 1).sum()) >= int(want[3].sum()) // 2


def test_tal_assign_rejects_more_than_1024_boxes_and_topk_over_16(ops):
    c = {k: v.cuda() for k, v in rp.tal_case(510, 1, [(8, 8), (4, 4), (2, 2)], STRIDES, 5, 1025).items()}
    with pytest.raises(ValueError, match="G=1025"):
        ops.tal_assign(**c, topk=10, num_classes=5)
    c = {k: v.cuda() for k, v in rp.tal_case(511, 1, [(8, 8), (4, 4), (2, 2)], STRIDES, 5, 4).items()}
    with pytest.raises(ValueError, match="topk=17"):
        ops.tal_assign(**c, topk=17, num_classes=5)


@pytest.mark.parametrize("topk", [1, 13, 16])
def test_tal_assign_topk_values_match_port(ops, topk, record_property):
    c = rp.tal_case(520 + topk, 4, [(40, 40), (20, 20), (10, 10)], STRIDES, 10, 16)
    got, want, _ = _assign(ops, c, 10, topk=topk)
    record_property(f"topk{topk}:scores", assign_ratio(got, want))


def test_tal_assign_interleaved_padding_and_special_boxes(ops, record_property):
    """Padded boxes (``mask_gt = 0``) between real ones; in image 0 two identical boxes (the tie goes to the first),
    a box between anchor centres, a zero-area box and a zero-width box, none of which may own an anchor."""
    nc, G = 10, 16
    c = rp.tal_case(530, 4, [(40, 40), (20, 20), (10, 10)], STRIDES, nc, G)
    perm = torch.randperm(G, generator=torch.Generator().manual_seed(531))
    for k in ("gt_labels", "gt_bboxes", "mask_gt"):
        c[k] = c[k][:, perm].contiguous()
    m = c["mask_gt"][..., 0]
    assert any(bool((m[b, :-1] < m[b, 1:]).any()) for b in range(4)), "a padded box should come before a real one"
    real = m[0].nonzero().flatten().tolist()
    i, j, e1, e2, e3 = real[:5]
    c["gt_bboxes"][0, j] = c["gt_bboxes"][0, i]
    c["gt_labels"][0, j] = c["gt_labels"][0, i]
    c["gt_bboxes"][0, e1] = torch.tensor([100.5, 100.5, 103.5, 103.5])  # no anchor centre of any level inside
    c["gt_bboxes"][0, e2] = torch.tensor([50.0, 50.0, 50.0, 50.0])
    c["gt_bboxes"][0, e3] = torch.tensor([60.0, 40.0, 60.0, 90.0])
    got, want, _ = _assign(ops, c, nc)
    record_property("special:scores", assign_ratio(got, want))
    fg, gidx = got[3][0].cpu(), got[4][0].cpu()
    assert (fg & (gidx == i)).any() and not (fg & (gidx == j)).any()
    for e in (e1, e2, e3):
        assert not (fg & (gidx == e)).any()


# ----------------------------------------------------------------------------- 3. the training chain
@pytest.mark.parametrize("amp", [False, True], ids=["fp32", "autocast"])
def test_training_chain_matches_the_ports(ops, amp, record_property):
    """Head logits -> bbox_decode -> assigner -> box loss -> backward to the logits, as ``Loss.__call__`` composes them
    (utils/loss.py:139-170), at B=16, 640: kernels against the same chain of ports.  The decodes' last bits differ by
    design (tol.check_bbox_decode: one half ulp of a corner under autocast), and the assignment is a discontinuous
    function of the boxes, so the port chain carries the kernel decode's box values forward and sends the gradient
    back through its own decode (``kernel_pb + (pb - pb.detach())``, exactly the kernel's values).  Assigner and loss then see the same inputs in
    both chains: assignments bit for bit, scalars within 1e-5, and the gradient of ``pred_dist`` meets its two sources,
    the DFL term and the CIoU term through each decode's backward."""
    B, nc = 16, 20
    dt = torch.float16 if amp else torch.float32
    c = rp.tal_case(600, B, LEVELS, STRIDES, nc, 20)
    g = torch.Generator().manual_seed(601)
    A = c["anc_points"].shape[0]
    dist = (torch.randn(B, A, 64, generator=g) * 3).to("cuda", dt)
    cls = (torch.randn(B, A, nc, generator=g) * 2 - 1).to("cuda", dt)
    anc, st = rp.anchor_grid(LEVELS, STRIDES, dt, "cuda")
    ap, st = anc.t().contiguous(), st.t().contiguous()  # [A, 2], [A, 1]
    gt = {k: c[k].cuda() for k in ("gt_labels", "gt_bboxes", "mask_gt")}

    def chain(decode, assign, loss, boxes=None):
        pd = dist.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
            pb = decode(ap, pd)
            if boxes is not None:
                pb = boxes + (pb - pb.detach())
            args = dict(pd_scores=cls.detach().sigmoid(), pd_bboxes=(pb.detach() * st).type(gt["gt_bboxes"].dtype),
                        anc_points=ap * st, **gt)
            out = assign(args)
            tb = out[1] / st
            tss = out[2].sum().clamp(min=1)
            li, ld = loss(pd, pb, ap, tb, out[2], tss, out[3])
        (gd,) = torch.autograd.grad((li, ld), (pd,), tuple(torch.tensor(v, device="cuda") for v in GO))
        return out, li.detach(), ld.detach(), gd, pb.detach()

    kout, ki, kd, kg, kpb = chain(ops.bbox_decode, lambda a: ops.tal_assign(**a, topk=10, num_classes=nc), ops.bbox_loss)

    def port_assign(a):
        cpu = {k: v.float().cpu() if k != "pd_scores" else v.cpu() for k, v in a.items()}
        return tuple(t.cuda() for t in _port_assign(cpu, nc)[:5])

    pout, pi, pdl, pg, ppb = chain(rp.bbox_decode_port, port_assign, lp.bbox_loss_port, boxes=kpb)
    assert torch.equal(ppb, kpb)
    record_property("chain:assign_scores", assign_ratio(kout, pout))
    for a, b, tag in ((ki, pi, "iou"), (kd, pdl, "dfl")):
        r = abs(float(a) - float(b)) / (1e-5 * abs(float(b)))
        record_property(f"chain:scalar_{tag}", r)
        assert r <= 1.0, tag
    r = _grads_close(kg, pg, 2e-2 if amp else 1e-4, 16, amp)
    record_property("chain:grad_logits", r)
