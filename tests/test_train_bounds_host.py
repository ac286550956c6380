"""The comparators of the training-loss scale tests (tests/test_gpu_train_scale.py), and proof on CPU tensors that each
of them rejects small errors of a correct result.  No kernel is launched here.

``scalar_ratio`` checks a loss scalar of ``ops.bbox_loss`` against the kernel's own per-anchor terms without depending
on the order in which the kernel adds them; ``kernel_order_scalar`` restates that order in float32 so that a correct
scalar can be made on the CPU.  ``half_grads_ratio`` adds a limit on the number of changed values to the per-element
bound of ``test_gpu_loss._grads_close``.  ``assign_ratio`` is the assigner's comparison: indices and masks exact."""
import math
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import bbox_loss_port as lp  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from test_gpu_loss import _grads_close  # noqa: E402
from test_loss_host import _host_case, bbox_loss_grad  # noqa: E402

U = 2.0**-24  # unit roundoff of float32
BL_THREADS, BL_MAX_CTAS = 256, 148 * 8  # bbox_loss.cu: forward CTA size and grid cap


# ----------------------------------------------------------------------------- inputs
def flat_case(seed, B, A, C=20, fg=0.04, ap_lo=2.0, ap_span=20.0, logit=3.0):
    """Inputs of ``BboxLoss.forward`` on a flat ``[A, 2]`` anchor set (the loss does not look at levels), built like
    ``test_loss_host._host_case``: target side distances uniform in [0, 14), predicted distances the targets' plus
    N(0, 1) clamped to the 15 bins, a foreground fraction ``fg``, one-hot target scores times a uniform norm, 16-bin
    logits N(0, logit^2).  float32 on the CPU; ``target_scores_sum`` is ``max(sum, 1)`` as a 0-d tensor."""
    g = torch.Generator().manual_seed(seed)
    ap = torch.rand(A, 2, generator=g) * ap_span + ap_lo
    lt = torch.rand(B, A, 4, generator=g) * 14
    tb = torch.cat((ap - lt[..., :2], ap + lt[..., 2:]), -1)
    d = (lt + torch.randn(B, A, 4, generator=g)).clamp(0, 15)
    pb = torch.cat((ap - d[..., :2], ap + d[..., 2:]), -1)
    fgm = torch.rand(B, A, generator=g) < fg
    lab = torch.randint(0, C, (B, A), generator=g)
    ts = torch.nn.functional.one_hot(lab, C).float() * torch.rand(B, A, 1, generator=g) * fgm[..., None]
    pd = torch.randn(B, A, 64, generator=g) * logit
    return dict(pred_dist=pd, pred_bboxes=pb, anchor_points=ap, target_bboxes=tb, target_scores=ts,
                target_scores_sum=ts.sum().clamp(min=1), fg_mask=fgm)


# ----------------------------------------------------------------------------- loss scalars
def fwd_ctas(n_rows):
    return min(max(-(-n_rows * 4 // BL_THREADS), 1), BL_MAX_CTAS)


def sum_depth(n_rows):
    """Depth ``d`` of the forward kernel's summation tree over ``n_rows = B * A`` anchors: the largest number of float32
    additions on the way from one per-anchor term to the scalar (bbox_loss.cu, ``bbox_loss_fwd_kernel``).

    - the grid-stride loop: each of the ``ctas * 256 / 4`` anchor slots of a pass adds its anchor's term to the
      thread's accumulator, serially over ``passes = ceil(n_rows / (ctas * 64))`` passes: ``passes`` additions;
    - ``block_sum2``: a 5-level shuffle tree over the 32 lanes of a warp (5), then thread 0 adds the 8 warp sums in
      order, starting from 0 (8);
    - the last CTA: thread ``i`` adds the partials ``i, i + 256, ...`` serially: ``ceil(ctas / 256)``;
    - ``block_sum2`` again: 5 + 8.

    ``d = passes + ceil(ctas / 256) + 26``: 39 at the trainer's B=64 x 8400 (8 passes, 1184 partials), 28 for one pass
    of at most 256 CTAs.  (Additions of an exact 0 -- the lanes of sides 1-3, background anchors -- count too; the
    bound only needs an upper limit.)"""
    ctas = fwd_ctas(n_rows)
    passes = max(-(-n_rows // (ctas * BL_THREADS // 4)), 1)
    return passes + 5 + 8 + -(-ctas // BL_THREADS) + 5 + 8


def scalar_ratio(loss, terms, tss, n_rows):
    """Error of ``loss * tss`` against the float64 sum ``S`` of the terms the kernel summed, over its bound.

    The kernel adds the float32 terms ``t_i`` in a tree of depth ``d`` (``sum_depth``) to ``S'``; then
    ``|S' - S| <= gamma_d * sum |t_i|`` with ``gamma_d = d u / (1 - d u)``, ``u = 2^-24``, in any order of the additions
    (Higham, Accuracy and Stability of Numerical Algorithms, 4.2).  ``loss = fl(S' / tss) = S' / tss * (1 + e)`` with
    ``|e| <= u``; ``loss * tss`` is exact in float64, so ``|loss * tss - S| <= gamma_d sum |t_i| + u / (1 - u) |loss * tss|``.
    ``tss`` is the float32 value the kernel divided by.  The ratio is <= 1 for every summation order of depth d."""
    t = terms.detach().double().cpu().flatten()
    S, A = float(t.sum()), float(t.abs().sum())
    d = sum_depth(n_rows)
    got = float(torch.as_tensor(loss).detach()) * float(np.float32(float(tss)))
    bound = d * U / (1 - d * U) * A + U / (1 - U) * abs(got)
    err = abs(got - S)
    return err / bound if bound > 0 else (0.0 if err == 0 else math.inf)


def assert_scalar_matches_terms(loss, terms, tss, n_rows):
    r = scalar_ratio(loss, terms, tss, n_rows)
    assert r <= 1.0, f"scalar off its own per-anchor terms by {r:.3g} x the bound"
    return r


def _block_sum(v):
    """block_sum2 of bbox_loss.cu on ``v [n, 256]`` float32: shuffle-down tree per warp, then the 8 warp sums in order."""
    v = v.reshape(v.shape[0], 8, 32)
    for o in (16, 8, 4, 2, 1):
        v = v + np.concatenate((v[..., o:], v[..., 32 - o:]), -1)  # out-of-range lanes read their own value
    s = np.zeros(v.shape[0], np.float32)
    for w in range(8):
        s = s + v[:, w, 0]
    return s


def kernel_order_scalar(terms, tss):
    """The forward kernel's own float32 reduction of one per-anchor column ``terms [B, A]`` (grid-stride passes, the
    CTA's tree, the last CTA's serial pass over the partials, the tree again), divided by ``tss`` in float32."""
    col = terms.detach().float().cpu().flatten().numpy()
    n = col.size
    ctas = fwd_ctas(n)
    per_pass = ctas * BL_THREADS // 4
    passes = max(-(-n // per_pass), 1)
    x = np.zeros(passes * per_pass, np.float32)
    x[:n] = col
    x = x.reshape(passes, ctas, 64)
    acc = np.zeros((ctas, 256), np.float32)
    for p in range(passes):
        acc[:, 0::4] = acc[:, 0::4] + x[p]  # side 0 of each anchor holds the terms; sides 1-3 add 0
    part = _block_sum(acc)
    k = -(-ctas // BL_THREADS)
    part = np.concatenate((part, np.zeros(k * BL_THREADS - ctas, np.float32))).reshape(k, BL_THREADS)
    tot = np.zeros((1, BL_THREADS), np.float32)
    for j in range(k):
        tot = tot + part[j]
    return torch.tensor(_block_sum(tot)[0] / np.float32(float(tss)))


# ----------------------------------------------------------------------------- gradients
ETA = 2.0**-126  # half the smallest float32 subnormal, in units of u (the kernels keep subnormals: no -ftz)


class _E:
    """A float64 value ``v`` with a first-order bound ``e`` of the error, in units of ``u = 2^-24``, that float32
    evaluation of the same operations in the same order accumulates.  Inputs and constants are float32 values (the
    kernels and the port see the same ones), so they start at ``e = 0``.  A rounded operation adds ``|v| + ETA``: float32
    rounds to ``v (1 + d) + n`` with ``|d| <= u`` and, below the normal range (bins whose ``exp`` underflows, their tiny
    products), ``|n| <= 2^-150 = ETA u``.  The operands' errors propagate through the operation's first derivatives.  ``e`` is large exactly where a value is a difference of
    larger terms, whatever the sign of the result."""

    def __init__(self, v, e=None):
        self.v = v
        self.e = torch.zeros_like(v) if e is None else e

    def __add__(self, o):
        v = self.v + o.v
        return _E(v, self.e + o.e + v.abs() + ETA)

    def __sub__(self, o):
        v = self.v - o.v
        return _E(v, self.e + o.e + v.abs() + ETA)

    def __mul__(self, o):
        v = self.v * o.v
        return _E(v, o.v.abs() * self.e + self.v.abs() * o.e + v.abs() + ETA)

    def __truediv__(self, o):
        v = self.v / o.v
        return _E(v, (self.e + v.abs() * o.e) / o.v.abs() + v.abs() + ETA)

    def __neg__(self):
        return _E(-self.v, self.e)

    def exact(self, c):  # times a power of two
        return _E(self.v * c, self.e * abs(c))


def _c(x, like):
    """A float32 constant, as the kernels and the port round it."""
    return _E(torch.full_like(like, float(np.float32(x))))


def _atan(x):  # libdevice atanf: within 2 ulp = 4 u |v|
    v = torch.atan(x.v)
    return _E(v, x.e / (1 + x.v * x.v) + 4 * v.abs() + ETA)


def _exp(x):  # expf: within 2 ulp
    v = torch.exp(x.v)
    return _E(v, v * x.e + 4 * v + ETA)


def _log(x):  # logf: within 1 ulp
    v = torch.log(x.v)
    return _E(v, x.e / x.v.abs() + 2 * v.abs() + ETA)


def _sel(cond, a, b):
    return _E(torch.where(cond, a.v, b.v), torch.where(cond, a.e, b.e))


def _fmin(a, b):
    return _sel(a.v < b.v, a, _sel(a.v > b.v, b, _E(a.v, torch.maximum(a.e, b.e))))


def _fmax(a, b):
    return _sel(a.v > b.v, a, _sel(a.v < b.v, b, _E(a.v, torch.maximum(a.e, b.e))))


def _paths(*ts):
    """A sum of gradient paths: in whatever order they are added, each of the n - 1 additions rounds a partial sum
    no larger than ``sum |t|``."""
    return _E(sum(t.v for t in ts), sum(t.e for t in ts) + (len(ts) - 1) * sum(t.v.abs() for t in ts))


def _pick(cond_lt, tie, g):  # autograd's share of minimum / maximum: all, half on a tie (exact), none
    z = _E(torch.zeros_like(g.v))
    return _sel(cond_lt, g, _sel(tie, g.exact(0.5), z))


def grad_error_bound(pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, target_scores_sum, fg_mask,
                     g_iou, g_dfl):
    """The closed-form gradient of ``bbox_loss`` in float64 (``test_loss_host.bbox_loss_grad``, restated op by op in
    the order of bbox_loss.cu's backward) and a first-order bound of the error of a float32 evaluation, both
    ``(dist [B, A, 64], boxes [B, A, 4])``, in units of ``u = 2^-24`` (``_E``).  Inputs are the float32 tensors; the DFL
    target ``bbox2dist`` is taken as float32 computes it, as kernels and port both do."""
    f64 = torch.float64
    p = [_E(t.double()) for t in pred_bboxes.unbind(-1)]
    t = [_E(x.double()) for x in target_bboxes.unbind(-1)]
    one = p[0].v
    eps, K = _c(1e-7, one), _c(4.0 / math.pi**2, one)
    w = _E(target_scores.sum(-1).double())  # one-hot row: exact
    tss = float(np.float32(float(target_scores_sum)))
    G = -((_c(g_iou, one) / _c(tss, one)) * w)
    # ciou_fwd
    w1, h1 = p[2] - p[0], (p[3] - p[1]) + eps
    w2, h2 = t[2] - t[0], (t[3] - t[1]) + eps
    ix, iy = _fmin(p[2], t[2]) - _fmax(p[0], t[0]), _fmin(p[3], t[3]) - _fmax(p[1], t[1])
    zero = _E(torch.zeros_like(one))
    cix, ciy = _sel(ix.v > 0, ix, zero), _sel(iy.v > 0, iy, zero)
    inter = cix * ciy
    uni = ((w1 * h1 + w2 * h2) - inter) + eps
    iou = inter / uni
    cw, ch = _fmax(p[2], t[2]) - _fmin(p[0], t[0]), _fmax(p[3], t[3]) - _fmin(p[1], t[1])
    c2 = (cw * cw + ch * ch) + eps
    dx, dy = ((t[0] + t[2]) - p[0]) - p[2], ((t[1] + t[3]) - p[1]) - p[3]
    rho2 = (dx * dx + dy * dy).exact(0.25)
    r1 = w1 / h1
    at = _atan(w2 / h2) - _atan(r1)
    v = K * (at * at)
    alpha = v / ((v - iou) + _c(1.0 + 1e-7, one))
    # ciou_bwd
    gS = -G
    g_union = (-G) * (iou / uni)
    g_inter = G / uni + (-g_union)
    g_ix, g_iy = _sel(ix.v >= 0, g_inter * ciy, zero), _sel(iy.v >= 0, g_inter * cix, zero)
    g_rho2 = gS / c2
    g_c2 = (-gS) * ((rho2 / c2) / c2)
    g_sq = g_rho2.exact(0.25)
    g_dx, g_dy = g_sq * dx.exact(2.0), g_sq * dy.exact(2.0)
    g_cw, g_ch = g_c2 * cw.exact(2.0), g_c2 * ch.exact(2.0)
    g_at = ((gS * alpha) * K) * at.exact(2.0)
    g_r1 = (-g_at) / (r1 * r1 + _c(1.0, one))
    gw_u, gw_r = g_union * h1, g_r1 / h1  # the two paths of w1 (the product w1 * h1, the ratio w1 / h1)
    gh_u, gh_r = g_union * w1, (-g_r1) * (r1 / h1)

    def lt(a, b):
        return a.v < b.v

    def gt(a, b):
        return a.v > b.v

    def eq(a, b):
        return a.v == b.v

    gb = [
        _paths(-gw_u, -gw_r, _pick(gt(p[0], t[0]), eq(p[0], t[0]), -g_ix), _pick(lt(p[0], t[0]), eq(p[0], t[0]), -g_cw), -g_dx),
        _paths(-gh_u, -gh_r, _pick(gt(p[1], t[1]), eq(p[1], t[1]), -g_iy), _pick(lt(p[1], t[1]), eq(p[1], t[1]), -g_ch), -g_dy),
        _paths(gw_u, gw_r, _pick(lt(p[2], t[2]), eq(p[2], t[2]), g_ix), _pick(gt(p[2], t[2]), eq(p[2], t[2]), g_cw), -g_dx),
        _paths(gh_u, gh_r, _pick(lt(p[3], t[3]), eq(p[3], t[3]), g_iy), _pick(gt(p[3], t[3]), eq(p[3], t[3]), g_ch), -g_dy)]
    # DFL: log_softmax of the 16 bins, then (softmax - onehot) of the two cross-entropies
    target = lp.bbox2dist(anchor_points.float(), target_bboxes.float(), 15).double()  # [B, A, 4]
    tl = target.floor()
    wl = _E(tl + 1 - target, (tl + 1 - target).abs() + ETA)
    wr = _c(1.0, target) - wl
    x = pred_dist.double().view(*pred_dist.shape[:2], 4, 16)
    d = _E(x - x.amax(-1, keepdim=True))
    d.e = d.v.abs() + ETA
    ex = _exp(d)
    s = _E(ex.v.sum(-1, keepdim=True), ex.e.sum(-1, keepdim=True) + 4 * ex.v.sum(-1, keepdim=True))  # 4-level tree
    ls = d - _log(s)
    pr = _exp(ls)
    onew = torch.ones_like(target)
    gq = ((_c(g_dfl, onew) / _c(tss, onew)) * _E(w.v[..., None].expand_as(target))).exact(0.25)
    gL, gR = (-(gq * wl)), (-(gq * wr))
    k = torch.arange(16, dtype=f64, device=target.device)
    oh_l, oh_r = (k == tl[..., None]).to(f64), (k == tl[..., None] + 1).to(f64)
    gLk, gRk = _E(gL.v[..., None].expand_as(x), gL.e[..., None].expand_as(x)), _E(gR.v[..., None].expand_as(x),
                                                                                  gR.e[..., None].expand_as(x))
    a = _E(oh_l * gLk.v, oh_l * gLk.e) - pr * gLk
    b = _E(oh_r * gRk.v, oh_r * gRk.e) - pr * gRk
    gd = a + b
    fg4 = fg_mask[..., None].to(pred_bboxes.device)
    zb = torch.zeros_like(pred_bboxes, dtype=f64)
    vb = torch.where(fg4, torch.stack([g.v for g in gb], -1), zb)
    eb = torch.where(fg4, torch.stack([g.e for g in gb], -1), zb)
    fgd = fg_mask[..., None, None]
    vd = torch.where(fgd, gd.v, 0.0).view_as(pred_dist)
    ed = torch.where(fgd, gd.e, 0.0).view_as(pred_dist)
    return (vd, vb), (ed, eb)


def grad_bound_ratio(got, want, err, n_evals):
    """Worst ``|got - want| / (2 n_evals u e)``: each float32 evaluation is within ``u e`` of the exact gradient to
    first order; the factor 2 covers the second-order terms and the few places where the port's autograd adds the same
    terms in another order.  ``n_evals`` = 1 against the float64 value, 2 between kernel and port."""
    g, w, e = got.double(), want.double(), err.double()
    assert torch.isfinite(g).all()
    bound = 2 * n_evals * U * e + 1e-300
    return float(((g - w).abs() / bound).max())


def assert_grads_within(got, want, err, n_evals):
    r = grad_bound_ratio(got, want, err, n_evals)
    assert r <= 1.0, f"gradient off by {r:.3g} x its path bound"
    return r


MAX_CHANGED_F16 = 0.05


def half_grads_ratio(got, want, group, max_changed):
    """fp16 gradients: ``_grads_close(got, want, 1e-3, group, half=True)`` per element, and at most a fraction
    ``max_changed`` of the values may differ from the port's at all.  The per-element bound admits one half ulp of the
    group's largest value anywhere, so alone it would not notice a rounding made in the wrong place on every value;
    the count does (the same rule as ``tol.check_bbox_decode``).  Returns ``(per-element ratio, changed fraction)``."""
    r = _grads_close(got, want, 1e-3, group, True)
    frac = float((got.cpu() != want.cpu()).float().mean())
    assert frac <= max_changed, f"{frac:.2%} of the fp16 gradient values differ from the port's (limit {max_changed:.0%})"
    return r, frac


# ----------------------------------------------------------------------------- assigner
def assign_ratio(got, want):
    """``ops.tal_assign`` against ``tal_assign_port``: labels, boxes, foreground mask and box index bit for bit, the
    normalised scores positive at the same places and within ``1e-5 (|want| + S) + 1e-9``, ``S`` the largest score of
    the same box in the same image.  The port runs on the CPU, whose powf / atanf differ from the GPU's in the last
    bits; a score is ``CIoU^6`` times the box's scale, and a small CIoU is a difference of larger terms, so its error
    scales with the box's best score rather than its own (crowded images with hundreds of boxes reach it)."""
    names = ("target_labels", "target_bboxes", "target_scores", "fg_mask", "target_gt_idx")
    r = 0.0
    for n, a, b in zip(names, got, want):
        a, b = a.cpu(), b.cpu()
        assert a.dtype == b.dtype and a.shape == b.shape, n
        if n == "target_scores":
            assert torch.equal(a > 0, b > 0), n
            v, gidx = b.sum(-1), want[4].cpu()
            S = torch.zeros(v.shape[0], int(gidx.max()) + 1).scatter_reduce(1, gidx, v, "amax").gather(1, gidx)
            r = float(((a - b).abs() / (1e-5 * (b.abs() + S[..., None]) + 1e-9)).max())
            assert r <= 1.0, f"{n}: {r:.3g} x the bound"
        else:
            assert torch.equal(a, b), f"{n}: {int((a != b).sum())} values differ"
    return r


# ----------------------------------------------------------------------------- the comparators reject small errors
FG64 = 21_504  # foreground anchors of the B=64 x 8400 case of test_gpu_train_scale (4 % of 537 600)


def _b64_terms():
    """Per-anchor terms with the B=64 foreground count, from the port on the CPU: a compact [1, FG64] column whose
    terms are those of the trainer's shape (the background's zeros add nothing to the sum or to its bound)."""
    c = flat_case(5, 1, FG64, fg=1.0)
    _, _, per = lp.bbox_loss_port(**c, terms=True)
    return per, c["target_scores_sum"]


def test_kernel_order_scalar_is_within_the_bound_and_depth_is_derived():
    assert sum_depth(64 * 8400) == 8 + 5 + 26 and fwd_ctas(64 * 8400) == BL_MAX_CTAS
    assert sum_depth(75_776) == 1 + 5 + 26 and sum_depth(75_777) == 2 + 5 + 26
    assert sum_depth(1) == 1 + 1 + 26
    per, tss = _b64_terms()
    for col in range(2):
        for n_rows in (FG64, 64 * 8400):  # the same terms spread over the trainer's grid: the deeper tree
            t = torch.zeros(n_rows)
            t[torch.linspace(0, n_rows - 1, FG64).long()] = per[0, :, col]
            assert_scalar_matches_terms(kernel_order_scalar(t, tss), t, tss, n_rows)
    z = torch.zeros(1, 100)
    assert scalar_ratio(torch.tensor(0.0), z, 1.0, 100) == 0.0
    assert scalar_ratio(torch.tensor(1e-30), z, 1.0, 100) > 1.0  # nothing to sum: exactly 0


def test_scalar_bound_rejects_a_missing_term_and_a_scaled_sum():
    per, tss = _b64_terms()
    n_rows = 64 * 8400
    d = sum_depth(n_rows)
    for col in range(2):
        t = per[0, :, col]
        good = kernel_order_scalar(t, tss)
        assert_scalar_matches_terms(good, t, tss, n_rows)
        k = int(t.argsort()[FG64 // 2])  # a typical (median) foreground term left out
        drop = t.clone()
        drop[k] = 0
        with pytest.raises(AssertionError):
            assert_scalar_matches_terms(kernel_order_scalar(drop, tss), t, tss, n_rows)
        with pytest.raises(AssertionError):
            assert_scalar_matches_terms(good * (1 + 4 * U * d), t, tss, n_rows)


def _port_grads(c):
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    li, ld = lp.bbox_loss_port(**dict(c, pred_dist=pd, pred_bboxes=pb))
    return torch.autograd.grad((li, ld), (pd, pb), (torch.tensor(0.7), torch.tensor(1.3)))


def _ties_case(seed, B, A):
    pd, pb, ap, tb, ts, fg = (t.float() for t in _host_case(seed, B=B, A=A, ties=True))
    return dict(pred_dist=pd, pred_bboxes=pb, anchor_points=ap, target_bboxes=tb, target_scores=ts,
                target_scores_sum=ts.sum().clamp(min=1), fg_mask=fg.bool())


@pytest.mark.parametrize("seed", [1, 2])
def test_path_bound_values_are_the_closed_form_gradient(seed):
    """``grad_error_bound``'s values are ``test_loss_host.bbox_loss_grad`` (checked against autograd in fp64 there), up
    to what the float32 constants (eps, 4 / pi^2) and the float32 DFL target change: relative 2^-24 each."""
    pd, pb, ap, tb, ts, fg = (t.float() for t in _host_case(seed))
    fg = fg.bool()
    tss = ts.sum().clamp(min=1)
    (vd, vb), (ed, eb) = grad_error_bound(pd, pb, ap, tb, ts, tss, fg, 0.7, 1.3)
    f = lambda t: t.double()  # noqa: E731
    wd, wb = bbox_loss_grad(f(pd), f(pb), f(ap), f(tb), f(ts), float(np.float32(float(tss))), fg,
                            float(np.float32(0.7)), float(np.float32(1.3)))
    for v, w in ((vd, wd), (vb, wb)):
        assert torch.allclose(v, w, rtol=1e-6, atol=1e-6 * float(w.abs().max()))
    assert (ed >= 0).all() and (eb >= 0).all()


@pytest.mark.parametrize("case", ["ties", "flat", "logits"])
def test_float32_port_gradient_is_within_the_path_bound(case):
    """The port in float32 (autograd) against the float64 closed form: inside the path bound, the rows whose paths
    cancel to ~1e-14 (a predicted box equal to its target, in the integer-tie case) and the bins whose softmax
    underflows (logits x40) included."""
    c = {"ties": lambda: _ties_case(303, 4, 1024), "flat": lambda: flat_case(11, 4, 4096, fg=0.5),
         "logits": lambda: flat_case(301, 4, 2048, fg=0.3, logit=120.0)}[case]()
    gd, gb = _port_grads(c)
    (vd, vb), (ed, eb) = grad_error_bound(**c, g_iou=0.7, g_dfl=1.3)
    if case == "ties":
        assert ((c["pred_bboxes"] == c["target_bboxes"]).all(-1) & c["fg_mask"]).any()
    assert_grads_within(gb, vb, eb, 1)
    assert_grads_within(gd, vd, ed, 1)


def test_fp32_gradient_bound_rejects_one_row_off_by_1e_4():
    c = flat_case(6, 2, 512, fg=0.5)
    gd, gb = _port_grads(c)
    (vd, vb), (ed, eb) = grad_error_bound(**c, g_iou=0.7, g_dfl=1.3)
    for g, v, e in ((gb, vb, eb), (gd, vd, ed)):
        assert grad_bound_ratio(g, g, e, 2) == 0.0
        assert_grads_within(g, v, e, 1)
        # a typical row: the foreground anchor whose largest value is largest against its path bound
        gr, vr, er = (t.flatten(0, 1) for t in (g, v, e))
        a = int(torch.where(c["fg_mask"].flatten(), (vr.abs().amax(-1) / er.amax(-1).clamp(min=1e-300)), -1.0).argmax())
        bad = gr.clone()
        bad[a] *= 1 + 1e-4
        with pytest.raises(AssertionError):
            assert_grads_within(bad.view_as(g), g, e, 2)
        with pytest.raises(AssertionError):
            _grads_close(bad.view_as(g), g, 1e-5, e.shape[-1], False)


def test_fp16_gradient_count_rejects_ulp_flips_on_20_percent_not_on_2():
    c = flat_case(7, 4, 2048, fg=1.0)
    pd = c["pred_dist"].clone().requires_grad_(True)
    pb = c["pred_bboxes"].clone().requires_grad_(True)
    li, ld = lp.bbox_loss_port(**dict(c, pred_dist=pd, pred_bboxes=pb))
    g32 = torch.autograd.grad((li, ld), (pd, pb), (torch.tensor(0.7), torch.tensor(1.3)))
    gen = torch.Generator().manual_seed(8)
    for g, group in zip(g32, (16, 4)):
        want = g.half()
        for frac, ok in ((0.02, True), (0.20, False)):
            flip = (torch.rand(want.shape, generator=gen) < frac) & (want != 0)
            got = torch.where(flip, (want.view(torch.int16) ^ 1).view(torch.float16), want)  # one ulp, last bit
            assert _grads_close(got, want, 1e-3, group, True) <= 1.0  # each flip alone is inside the per-element bound
            if ok:
                half_grads_ratio(got, want, group, MAX_CHANGED_F16)
            else:
                with pytest.raises(AssertionError):
                    half_grads_ratio(got, want, group, MAX_CHANGED_F16)


def test_assign_comparison_rejects_one_swapped_index():
    c = rp.tal_case(9, 2, [(20, 20), (10, 10), (5, 5)], [8, 16, 32], 7, 9)
    want = rp.tal_assign_port(**c, num_classes=7)[:5]
    assert assign_ratio(want, want) == 0.0
    gidx = want[4].clone()
    fg = want[3][0].nonzero().flatten()
    i = int(fg[0])
    j = int(next(k for k in fg.tolist() if gidx[0, k] != gidx[0, i]))
    gidx[0, i], gidx[0, j] = gidx[0, j].clone(), gidx[0, i].clone()
    with pytest.raises(AssertionError):
        assign_ratio(want[:4] + (gidx,), want)
    scores = want[2].clone()
    top = int(scores[0].sum(-1).argmax())  # the best score of its box: S = |want|
    scores[0, top] *= 1 + 1e-4
    with pytest.raises(AssertionError):
        assign_ratio((want[0], want[1], scores, want[3], want[4]), want)
