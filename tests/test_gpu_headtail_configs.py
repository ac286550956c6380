"""The fused head-tail kernel (``cerb_head_tail``, csrc/head_tail.cu) across its launch space, on inputs whose convolution
no summation order can change, compared BIT FOR BIT with a plain reference.

Exact inputs.  Activations are integers * 2^-3 in [-8, 8], weights integers * 2^-7 in [-16, 16], biases integers * 2^-6
in [-16, 16]: all exact in fp16, every product an integer multiple of u = 2^-10.  ``exact_case`` asserts for every
output channel that max|a| * sum|w| + |b| < 2^24 u, so every partial sum of every order (and ``acc + bias``) is an fp32
number: the fp32 accumulation is exact whatever order the tensor cores use.  The one rounding left is fp32 -> half of
the conv output, the same on both sides.  So the reference is the fp64 convolution, ``.half()``, then
``ops.decode_heads_split`` (itself pinned bit for bit to the reference port by test_gpu_parity), and the fused kernel
must equal it on every output element of every anchor, and its score summary must be the exact 8-anchor maximum.

Planted ties.  One input channel k* of each tower has all weights 2^-7, so the activation at k* moves every output of
that anchor by a whole number of units.  For a few anchors of image 0 the generator sets it so that one conv output
lies exactly halfway between two halves; round-to-nearest-even has to pick the same neighbour on both sides.

Launch configuration.  ``derive`` restates the host-side sizing of csrc/head_tail.cu (launch split, ring stage rows,
accumulator buffers, epilogue groups, ring depth) to name the configuration each case forces; a case id reads
``<what it covers>-<derived configuration>``.  The ring depth in the id is the one a device with the B200's 232448
bytes of opt-in shared memory gets; the tests that depend on it read the device's own value."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------------------- exact inputs
# (grid step, largest integer, standard deviation) per tensor kind; the weights' deviation is divided by sqrt(c)
EXACT = dict(a=(2.0**-3, 64, 2.5), w=(2.0**-7, 2048, 2.5), b=(2.0**-6, 1024, 1.5))
B200_SMEM_OPTIN = 232448


def _grid(gen, shape, step, imax, std, mean=0.0):
    """float64 tensor of integers * step, |integer| <= imax, drawn around mean with standard deviation std."""
    q = torch.round((torch.randn(shape, generator=gen, dtype=torch.float64) * std + mean) / step)
    return q.clamp_(-imax, imax) * step


def half_midpoint(x):
    """True where the float64 values x lie exactly halfway between two neighbouring fp16 numbers."""
    x = np.asarray(x, dtype=np.float64)
    h16 = x.astype(np.float16)
    h = h16.astype(np.float64)
    other = np.nextafter(h16, np.where(x > h, np.float16(np.inf), np.float16(-np.inf))).astype(np.float64)
    return (h != x) & (np.abs(x - h) == np.abs(other - x))


def _plant(a, w, b, n_of, p_list, kstar, step_a, step_w):
    """Set a[kstar, p] (activations [c, hw] of one image, float64) so that output n_of(p, S) of anchor p is an exact
    half midpoint.  w[:, kstar] == step_w, so a[kstar, p] = i * step_a moves every output of p by i units.  Returns
    [(n, p, value)]."""
    out = []
    steps = np.arange(-64, 65)
    steps = steps[np.argsort(np.abs(steps), kind="stable")]
    for p in p_list:
        a[kstar, p] = 0.0
        s_rest = (w @ a[:, p] + b).numpy()  # exact: every partial sum is on the grid and far below 2^53
        n = n_of(p, s_rest)
        cand = s_rest[n] + steps * step_a * step_w
        ok = half_midpoint(cand)
        if ok.any():
            i = int(steps[np.argmax(ok)])
            a[kstar, p] = i * step_a
            out.append((n, p, float(cand[np.argmax(ok)])))
    return out


def exact_case(B, tasks, levels, seed, grid=EXACT, plant=True, zero_feats=False):
    """Inputs of one ``ops.head_tail`` call on an exact grid: tasks = [(c2, c3, nc)], levels = [(H, W)].  Returns
    (host, plants): host = dict(box, cls, bw, bb, cw, cb) of per-task per-level float64 CPU tensors (weights
    [n, c, 1, 1]); plants = [(t, l, tower, n, p, value)] of the planted ties (image 0)."""
    gen = torch.Generator().manual_seed(seed)
    (sa, ia, da), (sw, iw, dw), (sb, ib, db) = grid["a"], grid["w"], grid["b"]
    assert sb >= sa * sw, "biases must lie on the products' grid"
    limit = 2.0**24 * sa * sw  # 2^24 grid units of a product
    host = dict(box=[], cls=[], bw=[], bb=[], cw=[], cb=[])
    plants = []
    for t, (c2, c3, nc) in enumerate(tasks):
        for k in host:
            host[k].append([])
        for l, (H, W) in enumerate(levels):
            hw = H * W
            per_tower = []
            for tower, c, n in (("box", c2, 64), ("cls", c3, nc)):
                x = torch.zeros(B, c, hw, dtype=torch.float64) if zero_feats else _grid(gen, (B, c, hw), sa, ia, da)
                wt = _grid(gen, (n, c), sw, iw, dw / c**0.5)
                bias = _grid(gen, (n,), sb, ib, db, mean=0.0 if tower == "box" else -4.0)
                if plant and not zero_feats:
                    kstar = c - 1
                    wt[:, kstar] = sw
                    ps = list(range(0, hw, max(1, hw // 16)))

                    def n_of(p, s, n=n, tower=tower):
                        if tower == "box":
                            order = [(p + j) % n for j in range(n)]
                            good = [m for m in order if abs(s[m]) >= 2]
                        else:  # a negative class logit: there a one-ulp logit change moves the score's half
                            order = [(p + j) % n for j in range(n)]
                            good = [m for m in order if -14 <= s[m] <= -2] or [m for m in order if abs(s[m]) >= 2]
                        return good[0] if good else order[0]

                    for n_, p, v in _plant(x[0], wt, bias, n_of, ps, kstar, sa, sw):
                        plants.append((t, l, tower, n_, p, v))
                # every partial sum of every summation order is bounded by this, so each one is an fp32 number
                assert float(x.abs().max()) * float(wt.abs().sum(1).max()) + float(bias.abs().max()) < limit, "inexact grid"
                per_tower.append((x.reshape(B, c, H, W), wt.reshape(n, c, 1, 1), bias))
            (xb, wb, bb), (xc, wc, bc) = per_tower
            for k, v in zip(("box", "bw", "bb", "cls", "cw", "cb"), (xb, wb, bb, xc, wc, bc)):
                host[k][t].append(v)
    return host, plants


def to_device(host):
    return {k: [[x.half().cuda() for x in lv] for lv in v] for k, v in host.items()}


def exact_raw(x, w, b):
    """[B, c, H, W] x [n, c, 1, 1] + b in fp64 on the GPU, rounded once to half (exact in fp32 first: one rounding)."""
    out = torch.empty((x.shape[0], w.shape[0]) + tuple(x.shape[2:]), dtype=torch.float16, device=x.device)
    w64, b64 = w.reshape(w.shape[0], -1).double(), b.double()
    for i in range(0, x.shape[0], 8):
        out[i : i + 8] = (torch.einsum("nc,bchw->bnhw", w64, x[i : i + 8].double()) + b64[None, :, None, None]).half()
    return out


def oracle(ops, d, strides):
    """fp64 convolution -> half -> decode_heads_split: y per task."""
    T, L = len(d["box"]), len(d["box"][0])
    box = [[exact_raw(d["box"][t][l], d["bw"][t][l], d["bb"][t][l]) for l in range(L)] for t in range(T)]
    cls = [[exact_raw(d["cls"][t][l], d["cw"][t][l], d["cb"][t][l]) for l in range(L)] for t in range(T)]
    return ops.decode_heads_split(box, cls, strides)


def run(ops, d, strides):
    return ops.head_tail(d["box"], d["cls"], d["bw"], d["bb"], d["cw"], d["cb"], strides)


def summary_of(ops, y):
    """The score summary remembered for y, without the row padding the kernel does not write."""
    sm = ops.find_summary(y)
    return None if sm is None else sm[..., : y.shape[2] // 8]


def assert_same(ys, want, what):
    for t, (y, w) in enumerate(zip(ys, want)):
        assert y.shape == w.shape and y.dtype == w.dtype
        if not torch.equal(y, w):
            bad = (y != w).nonzero()
            b, r, a = bad[0].tolist()
            raise AssertionError(f"{what}, task {t}: {bad.shape[0]} of {y.numel()} outputs differ; first at image {b} row {r} "
                                 f"anchor {a}: {y[b, r, a].item()} vs {w[b, r, a].item()}")


def assert_summary(ops, ys, want, what):
    """The summary the fused kernel left for y_t is the 8-anchor maximum of the EXPECTED y_t."""
    for t, (y, w) in enumerate(zip(ys, want)):
        sm = summary_of(ops, y)
        assert sm is not None, f"{what}, task {t}: no score summary"
        B, nc, A = w.shape[0], w.shape[1] - 4, w.shape[2]
        ref = w[:, 4:].reshape(B, nc, A // 8, 8).amax(dim=-1)
        assert torch.equal(sm, ref), f"{what}, task {t}: score summary is not the 8-anchor maximum of the expected y"


# ---------------------------------------------------------------------------------------------- launch configuration
def _stage_rows(c):
    return next(d for d in range(128, 15, -16) if c % d == 0)


def derive(tasks, L, smem_optin=B200_SMEM_OPTIN):
    """The host-side sizing of cerb_head_tail (csrc/head_tail.cu) for tasks = [(c2, c3, nc)] and L levels: one dict per
    launch with its tasks, accumulator buffers NB, epilogue groups, ring stage rows and ring depth S (< 2: CERB_ENOSPC)."""
    tpl = max(1, 12 // L)
    launches = []
    for t0 in range(0, len(tasks), tpl):
        part = tasks[t0 : t0 + tpl]
        ncp = [(nc + 15) // 16 * 16 for _, _, nc in part]
        buf_cols = 64 + max(ncp)
        stage_rows = max(max(_stage_rows(c2), _stage_rows(c3)) for c2, c3, _ in part)
        w2 = max((c2 + 63) // 64 * 64 * 128 for c2, _, _ in part)
        w3 = max((c3 + 63) // 64 * p * 128 for (_, c3, _), p in zip(part, ncp))
        fixed = w2 + w3 + 2 * (64 + 192) * 4 + (2 * 8 + 2 + 2 * 4 + 2) * 8 + 1024
        launches.append(dict(tasks=list(range(t0, t0 + len(part))), NB=min(4, 512 // buf_cols),
                             groups=1 if min(c2 + c3 for c2, c3, _ in part) >= 384 else 2,
                             rb=[(_stage_rows(c2), _stage_rows(c3)) for c2, c3, _ in part],
                             S=min(8, (smem_optin - fixed) // (stage_rows * 256))))
    return launches


def describe(tasks, L):
    ls = derive(tasks, L)
    rbs = sorted({r for lc in ls for pair in lc["rb"] for r in pair})
    return (f"{len(ls)}launch-NB{'/'.join(str(lc['NB']) for lc in ls)}-g{'/'.join(str(lc['groups']) for lc in ls)}"
            f"-rb{'/'.join(map(str, rbs))}-S{'/'.join(str(lc['S']) for lc in ls)}")


class Case:
    def __init__(self, name, B, tasks, levels, strides=None):
        self.name, self.B, self.tasks, self.levels = name, B, tasks, levels
        self.strides = strides or [8.0 * 2**l for l in range(len(levels))]
        shapes = "_".join(f"{h}x{w}" for h, w in levels)
        heads = "+".join(f"{c2}.{c3}.nc{nc}" for c2, c3, nc in tasks)
        self.id = f"{name}-B{B}-T{len(tasks)}L{len(levels)}-{shapes}-{heads}-{describe(tasks, len(levels))}"

    def seed(self):
        return sum(c2 * 7 + c3 * 3 + nc for c2, c3, nc in self.tasks) + self.B * 1000 + len(self.levels)


# Together: nc 1 8 9 17 64 65 96 97 176 177 192; c 16 (K < 64, one MMA per stage) 48 80 (K straddles a 64-block) 112
# 144 (rb 48) 176 (rb 16, 11 stages) 320; c2 + c3 = 368 / 384 / 400 (2 -> 1 epilogue groups); mixed widths in a launch;
# T x L = 5x3, 8x3 (2 launches), 4x4 (2), 8x4 (3), L = 1, L = 2; levels of <= 64 anchors (8x8, 1x8, 8x1: the second
# 64-anchor TMA box is out of range), 128 anchors exactly (8x16), 72 (9x8), non-square, W = 1; B = 1 with fewer tiles
# than SMs, odd B (3, 7), B = 16 at 640x640 (1072 tiles: every CTA loops).
NARROW = Case("narrow", 3, [(16, 16, 1), (48, 48, 9)], [(8, 8), (1, 8), (8, 1)])
V8X = Case("v8x", 2, [(80, 320, 20), (80, 320, 19), (80, 320, 12)], [(16, 16), (8, 8), (4, 4)])
T5 = Case("T5", 3, [(64, 64, 8), (64, 80, 17), (80, 64, 64), (64, 64, 65), (48, 64, 1)], [(9, 8), (4, 8), (2, 4)])
CASES = [
    NARROW,
    V8X,
    T5,
    Case("T8L3", 1, [(16, 16, 2), (32, 32, 3), (48, 48, 5), (64, 64, 7), (16, 64, 9), (64, 16, 11), (32, 48, 13), (48, 32, 15)],
         [(8, 16), (4, 8), (2, 4)]),
    Case("T4L4", 2, [(64, 64, 20), (64, 96, 33), (96, 64, 3), (64, 64, 80)], [(16, 8), (8, 8), (4, 4), (2, 4)]),
    Case("T8L4", 1, [(16, 32, 8), (32, 16, 9), (48, 48, 17), (64, 64, 1), (16, 16, 24), (32, 64, 40), (64, 32, 12), (48, 16, 4)],
         [(8, 8), (4, 4), (2, 4), (1, 8)]),
    Case("L1-nc96", 7, [(112, 112, 96)], [(12, 20)]),
    Case("L2-nc97", 1, [(144, 176, 97), (176, 144, 65)], [(10, 16), (5, 8)]),
    Case("mixed", 2, [(64, 80, 80), (64, 64, 20), (80, 320, 12)], [(16, 16), (8, 8), (4, 4)]),
    Case("nc64", 1, [(64, 128, 64)], [(8, 8), (4, 4), (2, 4)]),
    Case("nc65", 1, [(64, 128, 65)], [(8, 8), (4, 4), (2, 4)]),
    Case("nc176", 1, [(80, 384, 176)], [(8, 16), (4, 8)]),
    Case("nc177", 1, [(48, 64, 177)], [(8, 16), (4, 8)]),
    Case("nc192", 2, [(80, 320, 192)], [(16, 16), (8, 8), (4, 4)]),
    Case("sum368", 1, [(48, 320, 8)], [(8, 16), (4, 8)]),
    Case("sum384", 1, [(64, 320, 17)], [(8, 16), (4, 8)]),
    Case("persist640", 16, [(64, 64, 20)], [(80, 80), (40, 40), (20, 20)]),
]
_BY_ID = {c.id: c for c in CASES}


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    return o


_PREPARED = {}


def prepared(ops, case):
    """(device inputs, expected y per task, plants) of a case, built once per module."""
    if case.id not in _PREPARED:
        host, plants = exact_case(case.B, case.tasks, case.levels, case.seed())
        d = to_device(host)
        _PREPARED.clear()  # one case at a time on the device
        _PREPARED[case.id] = (d, oracle(ops, d, case.strides), plants)
    return _PREPARED[case.id]


@pytest.mark.parametrize("case_id", [c.id for c in CASES])
def test_exact_launch_space(ops, case_id):
    """Every output element of every anchor and the score summary equal the fp64 convolution + half + decode."""
    case = _BY_ID[case_id]
    d, want, plants = prepared(ops, case)
    ys = run(ops, d, case.strides)
    torch.cuda.synchronize()
    assert_same(ys, want, case.name)
    assert_summary(ops, ys, want, case.name)
    assert plants, "no tie was planted"


SCHEDULES = [(o, g, s) for o in (0, 1) for g in (1, 2) for s in (2, 3, None)]


@pytest.mark.parametrize("case_id", [NARROW.id, V8X.id, T5.id])
@pytest.mark.parametrize("order,groups,stages", SCHEDULES,
                         ids=[f"order{o}-groups{g}-stages{s or 'default'}" for o, g, s in SCHEDULES])
def test_schedule_knobs_give_the_same_bits(ops, knobs, case_id, order, groups, stages):
    """A CTA's arithmetic does not depend on the schedule: round-robin or chunked tiles, one or two epilogue groups, a
    2-, 3- or full-depth ring all give the default schedule's bits (y and summary), which equal the oracle."""
    case = _BY_ID[case_id]
    d, want, _ = prepared(ops, case)
    ys0 = run(ops, d, case.strides)
    sm0 = [summary_of(ops, y).clone() for y in ys0]
    knobs("ht_order", order)
    knobs("ht_groups", groups)
    if stages is not None:
        knobs("ht_stages", stages)
    ys = run(ops, d, case.strides)
    torch.cuda.synchronize()
    assert_same(ys, ys0, f"{case.name} order={order} groups={groups} stages={stages} vs the default schedule")
    for t, y in enumerate(ys):
        assert torch.equal(summary_of(ops, y), sm0[t]), f"task {t}: summary differs from the default schedule's"
    assert_same(ys, want, f"{case.name} order={order} groups={groups} stages={stages} vs the oracle")
    assert_summary(ops, ys, want, case.name)


@pytest.mark.parametrize("case_id", [c.id for c in CASES if c.name in ("v8x", "T5", "T8L3", "T4L4", "T8L4")])
def test_launch_split(ops, case_id):
    """T*L > 12 (task, level) rows go out in several launches of whole tasks: count the kernel launches."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    case = _BY_ID[case_id]
    d, want, _ = prepared(ops, case)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ys = run(ops, d, case.strides)
        torch.cuda.synchronize()
    n = sum(1 for e in prof.events() if e.device_type == DeviceType.CUDA and "head_tail_kernel" in e.name)
    assert n == len(derive(case.tasks, len(case.levels)))
    assert_same(ys, want, case.name)


@pytest.mark.parametrize("c2,c3,nc", [(80, 384, 176), (80, 384, 177), (80, 448, 192), (80, 320, 192)])
def test_shared_memory_sizing(ops, c2, c3, nc):
    """Weights + two ring stages must fit the device's opt-in shared memory: where they do the result is exact, where
    they do not the call fails with CERB_ENOSPC (inference then runs the heads unfused; see the test below)."""
    from cerberusdet_b200 import _lib

    smem = torch.cuda.get_device_properties(torch.cuda.current_device()).shared_memory_per_block_optin
    S = derive([(c2, c3, nc)], 2, smem)[0]["S"]
    print(f"opt-in shared memory {smem} B: c2={c2} c3={c3} nc={nc} -> S={S}")
    levels, strides = [(8, 16), (4, 8)], [8.0, 16.0]
    host, _ = exact_case(1, [(c2, c3, nc)], levels, seed=c3 + nc)
    d = to_device(host)
    if S < 2:
        with pytest.raises(_lib.CerbLibraryError, match="do not fit") as err:
            run(ops, d, strides)
        assert err.value.code == _lib.CERB_ENOSPC
        return
    ys = run(ops, d, strides)
    assert_same(ys, oracle(ops, d, strides), f"c3={c3} nc={nc}")


# ------------------------------------------------------------------------------------------- numeric edges of the epilogue
def test_half_overflow_matches_the_decode_of_the_same_raw(ops):
    """Conv outputs whose exact value rounds past 65504 (coarse grid: exact in fp32 up to 2^28), in box and class
    channels: inf / NaN in the same places as the decode of the same raw tensors, finite values equal."""
    grid = dict(a=(1.0, 8, 4.0), w=(16.0, 2047, 12000.0), b=(16.0, 2047, 1000.0))
    levels, strides = [(8, 16), (4, 8)], [8.0, 16.0]
    host, _ = exact_case(2, [(64, 64, 20), (48, 80, 9)], levels, seed=5, grid=grid, plant=False)
    d = to_device(host)
    ys, want = run(ops, d, strides), oracle(ops, d, strides)
    raw_inf = sum(int(torch.isinf(exact_raw(d["box"][0][l], d["bw"][0][l], d["bb"][0][l])).sum()) for l in range(2))
    assert raw_inf > 0, "no box logit overflowed"
    saw_nonfinite = False
    for t, (y, w) in enumerate(zip(ys, want)):
        assert torch.equal(torch.isnan(y), torch.isnan(w)), f"task {t}: NaN positions differ"
        assert torch.equal(torch.isposinf(y), torch.isposinf(w)) and torch.equal(torch.isneginf(y), torch.isneginf(w))
        fin = torch.isfinite(w)
        assert torch.equal(y[fin], w[fin]), f"task {t}: finite outputs differ"
        saw_nonfinite |= not bool(fin.all())
    assert saw_nonfinite, "the overflow case produced no non-finite output"


def test_saturated_scores(ops):
    """Class logits beyond +-24: sigmoid is exactly 1 or 0 in half; boxes stay on the exact grid."""
    levels, strides = [(8, 16), (4, 8)], [8.0, 16.0]
    host, _ = exact_case(2, [(64, 16, 12)], levels, seed=9, plant=False)
    gen = torch.Generator().manual_seed(10)
    for l in range(2):
        x = host["cls"][0][l]
        host["cls"][0][l] = torch.randint(-1, 2, x.shape, generator=gen).double()
        host["cw"][0][l] = torch.randint(-1, 2, (12, 16, 1, 1), generator=gen).double()
        sign = torch.randint(0, 2, (12,), generator=gen).double() * 2 - 1
        host["cb"][0][l] = sign * (40 + torch.randint(0, 40, (12,), generator=gen).double())  # |acc| <= 16
    d = to_device(host)
    ys, want = run(ops, d, strides), oracle(ops, d, strides)
    scores = ys[0][:, 4:]
    assert bool((scores == 0).any()) and bool((scores == 1).any()) and bool(((scores == 0) | (scores == 1)).all())
    assert_same(ys, want, "saturated")
    assert_summary(ops, ys, want, "saturated")


def test_zero_activations_decode_the_biases(ops):
    levels, strides = [(8, 8), (4, 8)], [8.0, 16.0]
    tasks = [(64, 64, 20), (80, 320, 9)]
    host, _ = exact_case(2, tasks, levels, seed=3, zero_feats=True)
    d = to_device(host)
    ys = run(ops, d, strides)
    box = [[b.half().cuda()[None, :, None, None].expand(2, 64, h, w).contiguous() for b, (h, w) in zip(host["bb"][t], levels)]
           for t in range(2)]
    cls = [[b.half().cuda()[None, :, None, None].expand(2, tasks[t][2], h, w).contiguous() for b, (h, w) in zip(host["cb"][t], levels)]
           for t in range(2)]
    want = ops.decode_heads_split(box, cls, strides)
    assert_same(ys, want, "zero activations")
    assert_summary(ops, ys, want, "zero activations")


def test_planted_ties_round_to_even_on_both_sides(ops):
    """The planted conv outputs are exact half midpoints: the reference's fp64 -> half conversion and the kernel's
    fp32 -> half conversion both round them to the even neighbour."""
    case = V8X
    d, want, plants = prepared(ops, case)
    assert len(plants) >= 50
    for t, l, tower, n, p, v in plants[:64]:
        x, w, b = (d["box"], d["bw"], d["bb"]) if tower == "box" else (d["cls"], d["cw"], d["cb"])
        raw = exact_raw(x[t][l][:1], w[t][l], b[t][l]).reshape(w[t][l].shape[0], -1)[n, p].item()
        assert half_midpoint(v) and float(np.float16(v)) == raw, (t, l, tower, n, p, v, raw)
        assert np.float16(raw).view(np.uint16) % 2 == 0  # the even neighbour
    ys = run(ops, d, case.strides)
    assert_same(ys, want, "planted ties")


def test_nms_on_the_fused_output(ops):
    """On a wide case NMS selects the same rows with and without the fused kernel's summary, and the rows NMS selects
    on the oracle's y."""
    case = V8X
    d, want, _ = prepared(ops, case)
    ys = run(ops, d, case.strides)
    kw = dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)
    d1, c1 = ops.nms_batched(ys, **kw)
    d2, c2 = ops.nms_batched(ys, use_summary=False, **kw)
    d3, c3 = ops.nms_batched(want, **kw)
    assert torch.equal(c1, c2) and torch.equal(d1, d2)
    assert torch.equal(c1, c3) and torch.equal(d1, d3)
    assert int(c1.min()) > 0


# ------------------------------------------------------------------------------------------------ the op as torch sees it
def _flat(d):
    return [[x for lv in d[k] for x in lv] for k in ("box", "cls", "bw", "bb", "cw", "cb")]


def test_opcheck_head_tail(ops):
    case = NARROW
    d, _, _ = prepared(ops, case)
    tests = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.cerb.head_tail.default, (*_flat(d), case.strides, len(case.tasks)), test_utils=tests)


def test_head_tail_under_torch_compile(ops):
    case = T5
    d, want, _ = prepared(ops, case)
    T = len(case.tasks)

    def fn(*args):
        return torch.ops.cerb.head_tail(*args, case.strides, T)

    eager = fn(*_flat(d))
    compiled = torch.compile(fn, backend="aot_eager", fullgraph=True)(*_flat(d))
    assert len(compiled) == 2 * T
    for a, b in zip(eager[:T], compiled[:T]):  # outputs, then summaries (compared without their row padding)
        assert torch.equal(a, b)
    for y, a, b in zip(eager[:T], eager[T:], compiled[T:]):
        assert torch.equal(a[..., : y.shape[2] // 8], b[..., : y.shape[2] // 8])
    assert_same(compiled[:T], want, "torch.compile")


@pytest.mark.parametrize("case_id", [NARROW.id, T5.id])
def test_head_tail_in_a_cuda_graph(ops, case_id):
    """Capture once, replay on fresh inputs copied into the static ones: the eager bits of those inputs (T5: two
    launches inside the capture)."""
    case = _BY_ID[case_id]
    static = to_device(exact_case(case.B, case.tasks, case.levels, case.seed() + 1)[0])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(ops, static, case.strides)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run(ops, static, case.strides)
    d, want, _ = prepared(ops, case)
    for k in static:
        for s_lv, f_lv in zip(static[k], d[k]):
            for s, f in zip(s_lv, f_lv):
                s.copy_(f)
    graph.replay()
    torch.cuda.synchronize()
    assert_same(out, run(ops, d, case.strides), "graph replay vs eager")
    assert_same(out, want, "graph replay vs oracle")


def _odd_offset(x):
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 16 != 0 and v.is_contiguous()
    return v


def _sliced(x):
    """The same values as a non-contiguous view (a channel slice of a wider tensor, or every other element)."""
    if x.dim() == 1:
        return torch.stack([x, torch.full_like(x, 7.0)], 1)[:, 0]
    wide = torch.cat([x, torch.full_like(x, 7.0)], 1)
    v = wide[:, : x.shape[1]]
    assert not v.is_contiguous()
    return v


@pytest.mark.parametrize("layout", ["channels_last", "odd_offset", "sliced", "weights_2d"])
def test_input_layouts_give_the_same_bits(ops, layout):
    case = Case("layout", 2, [(64, 80, 20), (48, 64, 9)], [(8, 16), (4, 8)])
    host, _ = exact_case(case.B, case.tasks, case.levels, case.seed())
    d = to_device(host)
    ys0 = run(ops, d, case.strides)
    feats = ("box", "cls")
    if layout == "channels_last":
        e = {k: [[x.to(memory_format=torch.channels_last) if k in feats else x for x in lv] for lv in v] for k, v in d.items()}
        assert not e["box"][0][0].is_contiguous()
    elif layout == "odd_offset":
        e = {k: [[_odd_offset(x) for x in lv] for lv in v] for k, v in d.items()}
    elif layout == "sliced":
        e = {k: [[_sliced(x) for x in lv] for lv in v] for k, v in d.items()}
    else:
        e = {k: [[x.reshape(x.shape[0], -1) if k in ("bw", "cw") else x for x in lv] for lv in v] for k, v in d.items()}
    ys = run(ops, e, case.strides)
    assert_same(ys, ys0, layout)
    assert_summary(ops, ys, ys0, layout)


def _tiny(T=1, L=1, nc=4, c2=64, c3=64, hw=(8, 8), dtype=torch.float16):
    z = lambda *s: torch.zeros(*s, dtype=dtype, device="cuda")  # noqa: E731
    return dict(box=[[z(1, c2, *hw) for _ in range(L)] for _ in range(T)], cls=[[z(1, c3, *hw) for _ in range(L)] for _ in range(T)],
                bw=[[z(64, c2, 1, 1) for _ in range(L)] for _ in range(T)], bb=[[z(64) for _ in range(L)] for _ in range(T)],
                cw=[[z(nc, c3, 1, 1) for _ in range(L)] for _ in range(T)], cb=[[z(nc) for _ in range(L)] for _ in range(T)])


@pytest.mark.parametrize("kw,exc,match", [
    (dict(nc=193), ValueError, r"nc\[0\]=193 outside \[1, 192\]"),
    (dict(c2=40), ValueError, "multiples of 16"),
    (dict(c3=24), ValueError, "multiples of 16"),
    (dict(hw=(3, 3)), ValueError, "must be a multiple of 8"),
    (dict(dtype=torch.float32), TypeError, "float16"),
    (dict(dtype=torch.bfloat16), TypeError, "float16"),
    (dict(T=9), ValueError, r"T=9 outside \[1, 8\]"),
    (dict(L=5), ValueError, r"L=5 outside \[1, 4\]"),
], ids=["nc193", "c2_40", "c3_24", "hw9", "fp32", "bf16", "T9", "L5"])
def test_head_tail_rejections(ops, kw, exc, match):
    d = _tiny(**kw)
    with pytest.raises(exc, match=match):
        run(ops, d, [8.0 * 2**l for l in range(kw.get("L", 1))])


# ---------------------------------------------------------------------- inference with a head the fused kernel cannot fit
class _Detect(torch.nn.Module):
    """Stand-in for the reference Detect (the attributes the drop-in reads); both towers end in conv3x3 -> conv1x1."""

    dynamic = False
    export = False
    shape = None

    def __init__(self, nc, ch, c2, c3):
        super().__init__()
        from cerberusdet_b200.synth import STRIDES

        self.nc, self.nl, self.reg_max, self.no = nc, len(ch), 16, nc + 64
        self.stride = torch.tensor(STRIDES)
        nn = torch.nn
        self.cv2 = nn.ModuleList(nn.Sequential(nn.Conv2d(c, c2, 3, padding=1), nn.Conv2d(c2, 64, 1)) for c in ch)
        self.cv3 = nn.ModuleList(nn.Sequential(nn.Conv2d(c, c3, 3, padding=1), nn.Conv2d(c3, nc, 1)) for c in ch)
        for s in self.cv3:
            nn.init.normal_(s[-1].weight, std=0.2)
            nn.init.constant_(s[-1].bias, -2.0)

    def forward(self, x):  # the oracle's restatement of the reference eval branch (CPU / training only here)
        from oracle import ref_port as rp

        for i in range(self.nl):
            x[i] = torch.cat((self.cv2[i](x[i]), self.cv3[i](x[i])), 1)
        if self.training:
            return x
        y = rp.decode_port(x, self.nc, [float(s) for s in self.stride])
        return y if self.export else (y, x)


class _TwoTask(torch.nn.Module):
    def __init__(self, heads):
        super().__init__()
        from cerberusdet_b200.synth import STRIDES

        self.stem = torch.nn.Conv2d(3, 16, 3, padding=1)
        self.heads = torch.nn.ModuleDict({k: _Detect(nc, (16, 16, 16), c2, c3) for k, (c2, c3, nc) in heads.items()})
        self.names = {k: [f"{k}{i}" for i in range(nc)] for k, (_, _, nc) in heads.items()}
        self.stride = torch.tensor(STRIDES)

    def forward(self, x):
        from cerberusdet_b200.synth import STRIDES

        f = self.stem(x)
        feats = [torch.nn.functional.avg_pool2d(f, int(s)) for s in STRIDES]
        return {t: h([z.clone() for z in feats]) for t, h in self.heads.items()}


@pytest.fixture()
def patched_detect():
    from cerberusdet_b200.detect import detect_forward

    _Detect._cerb_reference_forward = _Detect.forward
    orig = _Detect.forward
    _Detect.forward = detect_forward
    yield
    _Detect.forward = orig
    del _Detect._cerb_reference_forward


def test_inference_runs_heads_unfused_when_they_do_not_fit(ops, patched_detect):
    """Task b has c3 = 384 and nc = 180: detect.can_fuse_tail accepts it, but its weights and two ring stages do not
    fit shared memory.  predict must not raise; it runs the heads unfused from then on, with the unfused result."""
    from cerberusdet_b200 import detect
    from cerberusdet_b200.inference import CerberusDetInference

    torch.manual_seed(4)
    model = _TwoTask({"a": (64, 64, 20), "b": (80, 384, 180)}).cuda()
    fused = CerberusDetInference(model=model, device="cuda:0", conf_thres=0.001, iou_thres=0.45, half=True, img_size=128)
    plain = CerberusDetInference(model=model, device="cuda:0", conf_thres=0.001, iou_thres=0.45, half=True, img_size=128)
    fused.fuse_head_tail, plain.fuse_head_tail = True, False
    x = torch.rand(2, 3, 128, 128, device="cuda").half()
    with torch.no_grad():
        f = model.stem(x)
        feats = [torch.nn.functional.avg_pool2d(f, s) for s in (8, 16, 32)]
    assert all(detect.can_fuse_tail(h, feats) for h in model.heads.values())
    got = fused.predict(x, max_det=50)
    assert fused.fuse_head_tail is False
    want = plain.predict(x, max_det=50)
    assert got == want
    assert sum(len(r) for r in got) > 0
    assert fused.predict(x, max_det=50) == want
