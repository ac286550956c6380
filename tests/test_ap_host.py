"""CPU tests of the mAP statistics path (``cerb_ap_per_class``, ``ops.ap_per_class``, ``val_stats.ap_per_class``,
``install(metrics=True)``): the port against the reference's text, the numpy facts the kernels reproduce, the drop-in's
guard, the patch on stand-in modules and the C prototypes.  No kernel is launched here."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import ap_port  # noqa: E402


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_port_equals_reference_text_without_ties(seed):
    tp, conf, pred_cls, target_cls = ap_port.make_stats(30000, 12, seed=seed, unlabelled=2, unpredicted=2)
    conf = np.random.default_rng(seed).permutation(np.linspace(0.001, 1, conf.size, dtype=np.float32))  # tie-free
    assert np.unique(conf).size == conf.size
    names = {k: f"c{k}" for k in range(20)}
    want = ap_port.ap_per_class_verbatim(tp, conf, pred_cls, target_cls, names)
    got = ap_port.ap_per_class_port(tp, conf, pred_cls, target_cls, names)
    for a, b in zip(got, want):
        assert a.dtype == b.dtype and np.array_equal(a, b)


# ------------------------------------------------------------------- the numpy facts cerb_ap_per_class reproduces
def _interp(x, xp, fp, left=None, right=None):
    """np.interp restated: the last j with xp[j] <= x; left / right / exact knot; one rounding per operation."""
    left = fp[0] if left is None else left
    right = fp[-1] if right is None else right
    out = np.empty(len(x))
    for k, v in enumerate(x):
        j = int(np.searchsorted(xp, v, side="right")) - 1
        if j == -1:
            out[k] = left
        elif v > xp[-1]:
            out[k] = right
        elif j == len(xp) - 1 or xp[j] == v:
            out[k] = fp[j]
        else:
            slope = np.float64(fp[j + 1] - fp[j]) / np.float64(xp[j + 1] - xp[j])
            out[k] = np.float64(slope * np.float64(v - xp[j])) + fp[j]
    return out


def _trapz101(y):
    """np.trapz over linspace(0, 1, 101): numpy's pairwise sum of the 100 terms (8 accumulators over 0..95, a tree,
    then 96..99 in order)."""
    x = np.linspace(0, 1, 101)
    a = [np.float64(x[i + 1] - x[i]) * np.float64(y[i + 1] + y[i]) / 2.0 for i in range(100)]
    r = a[:8]
    for i in range(8, 96, 8):
        r = [r[k] + a[i + k] for k in range(8)]
    s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for i in range(96, 100):
        s += a[i]
    return s


def test_numpy_linspace_is_index_times_step():
    for n in (101, 1000):
        x = np.linspace(0, 1, n)
        want = np.arange(n) * (1.0 / (n - 1))
        want[-1] = 1.0
        assert np.array_equal(x, want)


def test_numpy_interp_is_last_knot_formula():
    rng = np.random.default_rng(0)
    for t in range(300):
        m = int(rng.integers(1, 40))
        xp = np.sort(np.round(rng.random(m), 1 + t % 3))  # rounding makes duplicate knots
        fp = rng.random(m)
        x = np.concatenate((rng.random(50), xp, [0.0, 1.0, -0.5, 1.5]))
        for lr in ((None, None), (0.0, None), (1.0, None)):
            assert np.array_equal(np.interp(x, xp, fp, *lr), _interp(x, xp, fp, *lr))
    # the curve interpolations of the kernels: x = -px against -conf (float32 knots)
    conf = np.sort(rng.random(500, dtype=np.float32).astype(np.float16).astype(np.float32))[::-1]
    px = np.linspace(0, 1, 1000)
    f = np.cumsum(rng.random(500) < 0.5) / 200.0
    assert np.array_equal(np.interp(-px, -conf, f, left=0), _interp(-px, -conf.astype(np.float64), f, left=0))


def test_numpy_trapz_sums_in_pairwise_order():
    rng = np.random.default_rng(1)
    x = np.linspace(0, 1, 101)
    for _ in range(2000):
        y = np.sort(rng.random(101))[::-1] * rng.random()
        assert ap_port._trapz(y, x) == _trapz101(y)


# ------------------------------------------------------------------------------------------ the C ABI, without a GPU
def test_ap_prototypes_match_header():
    from cerberusdet_b200 import _lib

    text = open(os.path.join(os.path.dirname(HERE), "include", "cerb_post.h")).read()
    lib = _lib.load()
    ctype = {"size_t": ctypes.c_size_t, "int": ctypes.c_int, "long": ctypes.c_long, "double": ctypes.c_double}
    for name in ("cerb_ap_workspace_bytes", "cerb_ap_per_class"):
        m = re.search(r"(\w+)\s+" + name + r"\(([^)]*)\);", text)
        assert m, name
        fn = getattr(lib, name)
        assert fn.restype is ctype[m.group(1)]
        params = [p.strip() for p in m.group(2).split(",")]
        assert len(params) == len(fn.argtypes), name
        for p, t in zip(params, fn.argtypes):
            if "*" in p:
                assert t is ctypes.c_void_p, (name, p)
            else:
                assert t is ctype[p.rsplit(" ", 1)[0]], (name, p)


def test_ap_abi_validation_without_gpu():
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    fake = ctypes.c_void_p(256)
    cls = (ctypes.c_float * 3)(0.0, 1.0, 2.0)
    nl = (ctypes.c_longlong * 3)(4, 5, 6)

    def call(n=10, K=10, classes=cls, n_labels=nl, nc=3):
        return lib.cerb_ap_per_class(fake, K, fake, fake, n, classes, n_labels, nc, 1e-16, fake, fake, fake, fake, 1 << 30, None)

    assert call(n=-1) == _lib.CERB_EINVAL and b"n=-1" in lib.cerb_last_error()
    assert call(n=1 << 31) == _lib.CERB_EINVAL
    assert call(K=0) == _lib.CERB_EINVAL and b"K=0" in lib.cerb_last_error()
    assert call(K=33) == _lib.CERB_EINVAL
    assert call(nc=-1) == _lib.CERB_EINVAL
    assert call(classes=(ctypes.c_float * 3)(0.0, 2.0, 1.0)) == _lib.CERB_EINVAL and b"ascending" in lib.cerb_last_error()
    assert call(classes=(ctypes.c_float * 3)(0.0, 1.0, 1.0)) == _lib.CERB_EINVAL  # duplicate
    assert call(classes=(ctypes.c_float * 3)(0.0, float("nan"), 2.0)) == _lib.CERB_EINVAL
    assert call(n_labels=(ctypes.c_longlong * 3)(1, -1, 1)) == _lib.CERB_EINVAL
    assert call(nc=0) == 0  # no class: nothing to compute, nothing launched
    assert lib.cerb_ap_workspace_bytes(-1, 10, 3) == 0 and lib.cerb_ap_workspace_bytes(10, 33, 3) == 0


def test_ops_ap_per_class_refuses_cpu_tensors():
    import torch

    from cerberusdet_b200 import ops

    with pytest.raises(TypeError):
        ops.ap_per_class(torch.zeros(4, 10, dtype=torch.bool), torch.zeros(4), torch.zeros(4), torch.zeros(2))


# ------------------------------------------------------------------------------------------------ the drop-in's guard
def _case(n=50):
    tp, conf, pred_cls, target_cls = ap_port.make_stats(n, 3, seed=5)
    return tp, conf, pred_cls, target_cls


@pytest.mark.parametrize("what", ["plot", "no_cuda", "tp_uint8", "nan_conf", "nan_target", "k33", "float64", "cpu_tensor",
                                  "unknown_kwarg"])
def test_guard_sends_off_path_calls_to_the_reference(what, monkeypatch):
    import torch

    from cerberusdet_b200 import val_stats

    calls = []

    def reference(*a, **k):
        calls.append((a, k))
        return "reference"

    tp, conf, pred_cls, target_cls = _case()
    kw = {"names": {0: "a"}}
    monkeypatch.setattr(torch.cuda, "is_available", lambda: what != "no_cuda")
    if what == "plot":
        kw["plot"] = True
    elif what == "tp_uint8":
        tp = tp.astype(np.uint8)
    elif what == "nan_conf":
        conf = conf.copy()
        conf[3] = np.nan
    elif what == "nan_target":
        target_cls = target_cls.copy()
        target_cls[0] = np.nan
    elif what == "k33":
        tp = np.concatenate((tp, tp, tp, tp[:, :3]), 1)
    elif what == "float64":
        conf = conf.astype(np.float64)
    elif what == "cpu_tensor":
        conf = torch.from_numpy(conf)
    elif what == "unknown_kwarg":
        kw["on_plot"] = None
    fn = val_stats.make_ap_per_class(reference)
    assert fn._cerb_reference is reference
    assert fn(tp, conf, pred_cls, target_cls, **kw) == "reference"
    assert len(calls) == 1 and calls[0][1] == kw


def test_guard_keeps_ordinary_stats_on_the_kernels(monkeypatch):
    import torch

    from cerberusdet_b200 import val_stats

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(val_stats, "ap_per_class", lambda *a, **k: "kernels")
    fn = val_stats.make_ap_per_class(lambda *a, **k: "reference")
    tp, conf, pred_cls, target_cls = _case()
    assert fn(tp, conf, pred_cls, target_cls, plot=False, names={}) == "kernels"
    assert fn(tp, conf.astype(np.float16), pred_cls, target_cls) == "kernels"  # half scores widen exactly


# ---------------------------------------------------------------------------- the patch, on stand-in reference modules
@pytest.fixture()
def stub_reference(monkeypatch):
    """The modules ``patch.install(metrics=True)`` touches, as stand-ins (the reference tree is not needed)."""
    mods = {}
    for name in ("cerberusdet", "cerberusdet.models", "cerberusdet.models.yolo", "cerberusdet.utils", "cerberusdet.utils.general",
                 "cerberusdet.utils.metrics", "cerberusdet.evaluation", "cerberusdet.other"):
        mods[name] = types.ModuleType(name)
        monkeypatch.setitem(sys.modules, name, mods[name])
    mods["cerberusdet.models.yolo"].Detect = type("Detect", (), {"forward": lambda self, x: x})
    mods["cerberusdet.utils.general"].non_max_suppression = lambda *a, **k: None

    def reference_ap_per_class(tp, conf, pred_cls, target_cls, plot=False, save_dir=None, names=(), eps=1e-16, prefix=""):
        return ap_port.ap_per_class_verbatim(tp, conf, pred_cls, target_cls, names, eps)

    mods["cerberusdet.utils.metrics"].ap_per_class = reference_ap_per_class
    mods["cerberusdet.evaluation"].ap_per_class = reference_ap_per_class  # `from ..utils.metrics import ap_per_class`
    mods["cerberusdet.other"].ap_per_class = lambda *a: None  # a different function of the same name stays
    from cerberusdet_b200 import patch

    patch.uninstall()
    yield mods
    patch.uninstall()
    if hasattr(mods["cerberusdet.models.yolo"].Detect, "_cerb_reference_forward"):
        del mods["cerberusdet.models.yolo"].Detect._cerb_reference_forward


def test_install_metrics_rebinds_ap_per_class(stub_reference, monkeypatch):
    import torch

    from cerberusdet_b200 import patch

    metrics, evaluation, other = (stub_reference[k] for k in ("cerberusdet.utils.metrics", "cerberusdet.evaluation", "cerberusdet.other"))
    original, other_fn = metrics.ap_per_class, other.ap_per_class
    info = patch.install(metrics=True)
    assert "cerberusdet.utils.metrics.ap_per_class" in info["patched"] and "cerberusdet.evaluation.ap_per_class" in info["patched"]
    assert metrics.ap_per_class is evaluation.ap_per_class and metrics.ap_per_class._cerb_reference is original
    assert other.ap_per_class is other_fn
    assert patch.install(metrics=True) == {"already": ["installed"]}  # idempotent
    # off the kernels' path (here: plot=True; without a GPU: everything) the reference's own function, bit for bit
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    tp, conf, pred_cls, target_cls = _case(400)
    got = metrics.ap_per_class(tp, conf, pred_cls, target_cls, names={0: "a", 1: "b", 2: "c"})
    want = ap_port.ap_per_class_verbatim(tp, conf, pred_cls, target_cls, {0: "a", 1: "b", 2: "c"})
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    patch.uninstall()
    assert metrics.ap_per_class is original and evaluation.ap_per_class is original
    # composes with the other switches
    info = patch.install(val=False)
    assert not any("ap_per_class" in p for p in info["patched"])
    info = patch.install(metrics=True)
    assert sorted(info["patched"]) == ["cerberusdet.evaluation.ap_per_class", "cerberusdet.utils.metrics.ap_per_class"]
