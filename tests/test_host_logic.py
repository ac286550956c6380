"""CPU tests of the host-side pieces: C-ABI exports, drop-in surfaces, cross-task tail, sharding
(world_size-2 gloo).  No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_import import reference_available  # noqa: E402

REF = reference_available()  # /root/reference in the build container, oracle/_ref (oracle/make_ref.py) on the GPU box


def test_shared_library_exports_every_declared_symbol():
    from cerberusdet_b200 import _lib

    header = open(os.path.join(ROOT, "include", "cerb_post.h")).read()
    declared = set(re.findall(r"\b(cerb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no prototypes found in include/cerb_post.h"
    lib = _lib.load()
    for sym in sorted(declared):
        assert getattr(lib, sym) is not None, sym
    assert declared == set(_lib.EXPORTS)
    assert lib.cerb_version() >= 100
    assert lib.cerb_last_error() is not None


def test_argument_validation_without_gpu():
    """Bad arguments are rejected on the host before any CUDA call."""
    from cerberusdet_b200 import _lib

    lib = _lib.load()
    vp = ctypes.c_void_p
    rc = lib.cerb_nms(_lib.ptr_array([0]), _lib.int_array([5]), 1, 1, 10, 7, 0.25, 0.45, None, 0, 0, 0, 300, 30000,
                      7680.0, None, None, None, None, 0, None)
    assert rc == _lib.CERB_EINVAL and b"dtype" in lib.cerb_last_error()
    # more than 1024 rows per image need the workspace form (nothing is dereferenced before the check fails)
    fake = ctypes.c_void_p(256)
    rc = lib.cerb_cross_task(fake, fake, 3, 2, 400, _lib.int_array([0, 20, 39]), 0.8, None, fake, fake, None)
    assert rc == _lib.CERB_ENOSPC and b"workspace" in lib.cerb_last_error()
    assert lib.cerb_cross_task_workspace_bytes(3, 2, 300) == 0 and lib.cerb_cross_task_workspace_bytes(3, 2, 400) > 2 * 1200 * 38 * 4
    # thread-local test knobs: unknown names are refused, known ones set and reset
    assert lib.cerb_debug_set(b"no_such_knob", 1) == _lib.CERB_EINVAL and b"unknown knob" in lib.cerb_last_error()
    assert lib.cerb_debug_set(b"nms_minb", 1) == 0 and lib.cerb_debug_reset() == 0
    rc = lib.cerb_nms(_lib.ptr_array([0]), _lib.int_array([5]), 1, 1, 10, 0, 1.5, 0.45, None, 0, 0, 0, 300, 30000,
                      7680.0, None, None, None, None, 0, None)
    assert rc == _lib.CERB_EINVAL and lib.cerb_last_error().startswith(b"Invalid Confidence threshold")
    with pytest.raises(AssertionError):
        _lib.check(rc)
    assert lib.cerb_debug_set_chunking(5, 1) == _lib.CERB_EINVAL
    assert lib.cerb_debug_set_chunking(0, 0) == 0
    assert lib.cerb_summary_row_len(8400, 0) == 1056 and lib.cerb_summary_row_len(8400, 1) == 2100
    assert lib.cerb_summary_row_len(8401, 0) == 0
    # training-time decode: reg_max other than 16 and a row count that is not a multiple of A are refused
    rc = lib.cerb_bbox_decode_fwd(None, None, 100, 10, 8, 0, None, None)
    assert rc == _lib.CERB_EINVAL and b"reg_max" in lib.cerb_last_error()
    rc = lib.cerb_bbox_decode_fwd(None, None, 101, 10, 16, 1, None, None)
    assert rc == _lib.CERB_EINVAL and b"multiple" in lib.cerb_last_error()
    assert lib.cerb_bbox_decode_fwd(None, None, 0, 0, 16, 1, None, None) == 0  # empty batch: nothing to launch
    rc = lib.cerb_bbox_decode_bwd(None, None, 10, 16, 5, None, None)
    assert rc == _lib.CERB_EINVAL and b"dtype" in lib.cerb_last_error()
    rc = lib.cerb_decode_split(_lib.ptr_array([0]), None, _lib.int_array([5]), 1, 1, 1, _lib.int_array([2]), _lib.int_array([2]),
                               _lib.float_array([8.0]), 0, _lib.ptr_array([0]), None, None, None)
    assert rc == _lib.CERB_EINVAL and b"null" in lib.cerb_last_error()
    # round-2 entry points: head-tail fusion, delivery, TAL assigner
    one = _lib.ptr_array([256])
    ia = _lib.int_array
    rc = lib.cerb_head_tail(one, one, one, one, one, one, ia([64]), ia([64]), ia([4]), 1, 1, 1, ia([8]), ia([8]), _lib.float_array([8.0]),
                            _lib.CERB_F32, one, None, None, None)
    assert rc == _lib.CERB_EINVAL and b"fp16 only" in lib.cerb_last_error()
    rc = lib.cerb_head_tail(one, one, one, one, one, one, ia([64]), ia([64]), ia([4]), 1, 1, 0, ia([8]), ia([8]), _lib.float_array([8.0]),
                            _lib.CERB_F16, one, None, None, None)
    assert rc == _lib.CERB_EINVAL and b"B=0" in lib.cerb_last_error()
    rc = lib.cerb_deliver_push(fake, ctypes.c_void_p(260), 64, fake, fake, fake, fake, None)
    assert rc == _lib.CERB_EINVAL and b"16-byte" in lib.cerb_last_error()
    rc = lib.cerb_deliver_push(fake, fake, 62, fake, fake, fake, fake, None)
    assert rc == _lib.CERB_EINVAL and b"multiple of 4" in lib.cerb_last_error()
    rc = lib.cerb_deliver_collect(fake, _lib.ptr_array([None, 256]), fake, 17, 0, None)
    assert rc == _lib.CERB_EINVAL and b"at most 16 ranks" in lib.cerb_last_error()
    rc = lib.cerb_deliver_collect(fake, _lib.ptr_array([None, None]), fake, 2, 0, None)
    assert rc == _lib.CERB_EINVAL and b"ack_remote[1]" in lib.cerb_last_error()
    dv = _lib.Delivery()
    dv.push_src, dv.push_dst, dv.push_words = 256, 512, 64  # a push without protocol words
    rc = lib.cerb_nms_deliver(_lib.ptr_array([256]), ia([5]), 1, 1, 16, 0, 0.25, 0.45, None, 0, 0, 0, 300, 30000, 7680.0, None, fake, fake,
                              None, 0, ctypes.byref(dv), None)
    assert rc == _lib.CERB_EINVAL and b"protocol words" in lib.cerb_last_error()
    rc = lib.cerb_nms_deliver(_lib.ptr_array([256]), ia([5]), 1, 1, 16, 0, 0.25, 0.45, None, 0, 0, 0, 300, 30000, 7680.0, None, fake, fake,
                              None, 0, None, None)
    assert rc == _lib.CERB_EINVAL and b"null delivery" in lib.cerb_last_error()
    assert lib.cerb_tal_workspace_bytes(64, 8400, 20, 10) == (64 * 20 * 10 + 64 * 8400 * 3 + 64 * 20 * 2) * 4
    rc = lib.cerb_tal_assign(fake, fake, fake, fake, fake, fake, 2, 100, 5, 0, 10, 0.5, 6.0, 1e-9, 1, fake, fake, fake, fake, fake, fake, 1 << 20, None)
    assert rc == _lib.CERB_EINVAL and b"G=0" in lib.cerb_last_error()
    rc = lib.cerb_tal_assign(fake, fake, fake, fake, fake, fake, 2, 100, 5, 3, 17, 0.5, 6.0, 1e-9, 1, fake, fake, fake, fake, fake, fake, 1 << 20, None)
    assert rc == _lib.CERB_EINVAL and b"topk=17" in lib.cerb_last_error()
    rc = lib.cerb_tal_assign(fake, fake, fake, fake, fake, fake, 2, 100, 5, 3, 10, 0.5, 6.0, 1e-9, 1, fake, fake, fake, fake, fake, fake, 16, None)
    assert rc == _lib.CERB_ENOSPC and b"workspace" in lib.cerb_last_error()


def test_ops_refuse_cpu_tensors():
    from cerberusdet_b200 import ops
    from cerberusdet_b200.nms import non_max_suppression

    with pytest.raises(TypeError):
        non_max_suppression(torch.zeros(1, 6, 8))
    with pytest.raises(TypeError):
        ops.decode_heads([[torch.zeros(1, 69, 2, 2)]], [8.0])
    with pytest.raises(AssertionError):
        non_max_suppression(torch.zeros(1, 6, 8), conf_thres=2.0)
    with pytest.raises(TypeError):
        ops.decode_heads_split([[torch.zeros(1, 64, 2, 2)]], [[torch.zeros(1, 5, 2, 2)]], [8.0])
    with pytest.raises(TypeError):
        ops.bbox_decode(torch.zeros(4, 2), torch.zeros(1, 4, 64))


def test_nms_statistics_takes_the_keywords_of_nms_batched():
    import inspect

    from cerberusdet_b200 import ops

    defaults = lambda fn: {k: p.default for k, p in inspect.signature(fn).parameters.items() if k not in ("out", "deliver")}  # noqa: E731
    assert defaults(ops.nms_statistics) == defaults(ops.nms_batched)
    preds = [torch.zeros(1, 9, 8)]
    with pytest.raises(TypeError, match="iou_thresh"):  # a misspelt keyword is an error, not the default threshold
        ops.nms_statistics(preds, iou_thresh=0.5)
    with pytest.raises(AssertionError, match="Invalid IoU"):  # the reference's assert, as in nms_batched
        ops.nms_statistics(preds, iou_thres=1.5)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the arm the driver runs first) on the host cores: one bounded step, one JSON line."""
    import json
    import subprocess
    import sys

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["value"] > 0
    # the reference's own code when its tree is there (/root/reference here, oracle/_ref on the GPU box), else the port
    assert line["cpu_baseline"]["kind"] == ("reference" if REF else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["config"]["workload"].startswith("BASELINE config 3")


def test_shard_ranges_cover_the_batch():
    from cerberusdet_b200.shard import shard_range, shard_sizes

    for n in (0, 1, 7, 64, 513):
        for w in (1, 2, 3, 8):
            got = [i for r in range(w) for i in shard_range(n, r, w)]
            assert got == list(range(n))
            assert sum(shard_sizes(n, w)) == n and max(shard_sizes(n, w)) - min(shard_sizes(n, w)) <= 1


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from cerberusdet_b200.shard import gather_detections, shard_range
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=world)
N, T, MD = 7, 3, 5                                   # 7 images over 2 ranks: 4 + 3 (ragged)
g = torch.Generator().manual_seed(0)
full_d = torch.rand(T, N, MD, 6, generator=g); full_c = torch.randint(0, MD + 1, (T, N), generator=g, dtype=torch.int32)
mine = shard_range(N, rank, world)
d, c = gather_detections(full_d[:, mine.start:mine.stop].contiguous(), full_c[:, mine.start:mine.stop].contiguous(), dst=0, n_images=N)
if rank == 0:
    assert torch.equal(d, full_d) and torch.equal(c, full_c), "gathered shards differ from the 1-rank result"
    print("GATHER_OK")
else:
    assert d is None and c is None
dist.destroy_process_group()
"""


def test_gather_detections_two_ranks_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, port=29611))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GATHER_OK" in outs[0]


# ------------------------------------------------------------------ cross-task tail vs the reference
def _random_dets(gen, n, ncls_total, clustered=True):
    k = 6
    centres = torch.rand(k, 2, generator=gen) * 500 + 50
    pick = torch.randint(0, k, (n,), generator=gen)
    c = centres[pick] + torch.randn(n, 2, generator=gen) * (4 if clustered else 80)
    wh = 60 + torch.rand(n, 2, generator=gen) * 40
    det = torch.cat((c - wh / 2, c + wh / 2, torch.rand(n, 1, generator=gen),
                     torch.randint(0, ncls_total, (n, 1), generator=gen).float()), 1)
    return det


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_cross_task_tail_matches_reference():
    from cerberusdet_b200 import cross_task as ct
    from oracle.ref_import import load_reference

    ref = load_reference()
    names = {"voc": [f"v{i}" for i in range(20)], "animals": [f"a{i}" for i in range(19)], "tableware": [f"t{i}" for i in range(12)]}
    maps, all_names = ct.category_maps(names)
    assert len(all_names) == 51 and maps["animals"][0] == 20 and maps["tableware"][11] == 50
    gen = torch.Generator().manual_seed(4)
    for trial in range(12):
        det = _random_dets(gen, int(torch.randint(0, 60, (1,), generator=gen)), 51, clustered=trial % 3 != 0)
        for thr in (0.8, 0.5, 0.2):
            want = ref.general.nms_between_tasks(det.clone(), maps, thr)
            got = ct.suppress_between_tasks(det.clone(), maps, thr)
            assert got.shape == want.shape and torch.equal(got, want), (trial, thr)
        if det.shape[0]:
            for shp in ((480, 640), (1080, 1920), (333, 500)):
                a = ref.general.scale_boxes((640, 640), det[:, :4].clone(), shp)
                b = ct.rescale_boxes((640, 640), det[:, :4].clone(), shp)
                assert torch.equal(a, b)
            i1 = ref.general.box_iou(det[:7, :4], det[3:, :4])
            assert torch.equal(i1, ct.pairwise_iou(det[:7, :4], det[3:, :4]))


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_patch_install_rebinds_and_restores():
    from cerberusdet_b200 import patch
    from oracle.ref_import import load_reference

    ref = load_reference()
    orig_fwd, orig_nms = ref.yolo.Detect.forward, ref.general.non_max_suppression
    info = patch.install()
    try:
        assert "cerberusdet.models.yolo.Detect.forward" in info["patched"]
        assert ref.yolo.Detect.forward is not orig_fwd and ref.general.non_max_suppression is not orig_nms
        # non-CUDA tensors still run the reference's own code: identical results
        pred = torch.rand(2, 9, 200)
        a = ref.general.non_max_suppression(pred, 0.25, 0.45)
        b = orig_nms(pred, 0.25, 0.45)
        assert all(torch.equal(x, y) for x, y in zip(a, b))
        m = ref.yolo.Detect(nc=5, ch=(16, 16, 16))
        m.stride = torch.tensor([8.0, 16.0, 32.0])
        m.eval()
        feats = [torch.randn(1, 16, 8, 8), torch.randn(1, 16, 4, 4), torch.randn(1, 16, 2, 2)]
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            y1, _ = m([f.clone() for f in feats])
            y0, _ = orig_fwd(m, [f.clone() for f in feats])
        assert torch.equal(y1, y0)
        assert type(m).__name__ == "Detect" and type(m).__module__ == "cerberusdet.models.yolo"  # class kept for pickles
    finally:
        patch.uninstall()
    assert ref.yolo.Detect.forward is orig_fwd and ref.general.non_max_suppression is orig_nms


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_patch_install_train_rebinds_bbox_decode_and_keeps_cpu_results():
    import types

    from cerberusdet_b200 import patch
    from oracle.ref_import import load_reference

    load_reference()
    import cerberusdet.utils.loss as loss_mod

    orig = loss_mod.Loss.bbox_decode
    info = patch.install(train=True)
    try:
        assert "cerberusdet.utils.loss.Loss.bbox_decode" in info["patched"] and loss_mod.Loss.bbox_decode is not orig
        me = types.SimpleNamespace(use_dfl=True, proj=torch.arange(16, dtype=torch.float))
        ap, pred = torch.rand(30, 2) * 8, torch.randn(2, 30, 64)
        assert torch.equal(loss_mod.Loss.bbox_decode(me, ap, pred), orig(me, ap, pred))  # CPU: the reference's own code
    finally:
        patch.uninstall()
    assert loss_mod.Loss.bbox_decode is orig


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_patched_inference_class_keeps_cpu_models_working(tmp_path, monkeypatch):
    """ADVICE r1: after install() a device='cpu' CerberusDetInference must still work (the reference's own NMS runs)."""
    import copy
    import warnings

    from cerberusdet_b200 import patch
    from oracle.ref_import import REFERENCE_ROOT, load_reference

    monkeypatch.setenv("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD", "1")  # attempt_load unpickles whole modules (torch >= 2.6)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", os.environ.get("CUDA_VISIBLE_DEVICES", ""))  # select_device('cpu') rewrites it
    load_reference()
    import cerberusdet.cerberusdet_inference as inf_mod
    import cerberusdet.models.cerberus as cerb_mod

    patch.uninstall()

    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        # a narrow copy of the config keeps the CPU forward fast
        import yaml

        with open(os.path.join(REFERENCE_ROOT, "cerberusdet/models/yolov8x_voc_obj365.yaml")) as f:
            cfg = yaml.safe_load(f)
        cfg["width_multiple"], cfg["depth_multiple"] = 0.125, 0.33
        model = cerb_mod.CerberusDet(task_ids=["voc", "objects365_animals"], nc=[20, 19], cfg=cfg, ch=3, verbose=False)
        model.sequential_split(copy.deepcopy(model.yaml["cerber"]), "cpu")
        for m in model.modules():
            if type(m).__name__ == "Detect":
                for seq in m.cv3:
                    seq[-1].bias.data.fill_(-2.0)
        model.names = {"voc": [f"voc{i}" for i in range(20)], "objects365_animals": [f"ani{i}" for i in range(19)]}
        path = os.path.join(str(tmp_path), "small.pt")
        torch.save({"model": model}, path)
        img = torch.rand(1, 3, 128, 128)
        ref_eng = inf_mod.CerberusDetInference(path, device="cpu", conf_thres=0.1, img_size=128)
        want = ref_eng.predict(img)
        patch.install(import_all=True)
        eng = inf_mod.CerberusDetInference(path, device="cpu", conf_thres=0.1, img_size=128)
        got = eng.predict(img)
    assert type(eng).__module__ == "cerberusdet_b200.inference"
    assert got == want and len(want[0]) > 0
    patch.uninstall()
    assert inf_mod.CerberusDetInference is not type(eng)


_WORKER2 = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from cerberusdet_b200.shard import DetectionGatherer
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=world)
T, BL, MD = 3, 4, 5
g = torch.Generator().manual_seed(1)
full_d = torch.rand(T, world * BL, MD, 6, generator=g); full_c = torch.randint(0, MD + 1, (T, world * BL), generator=g, dtype=torch.int32)
gat = DetectionGatherer(T, BL, MD, "cpu", dst=0)
for rep in range(3):                                   # buffers are reused across batches
    d, c = gat.out
    d.copy_(full_d[:, rank * BL:(rank + 1) * BL] + rep); c.copy_(full_c[:, rank * BL:(rank + 1) * BL])
    gat.launch()
    D, C = gat.result()
    if rank == 0:
        assert torch.equal(D, full_d + rep) and torch.equal(C, full_c)
    else:
        assert D is None and C is None
# the per-batch delivery interface the streaming engine drives (CPU: always the gather flavour), several batches per slot
from cerberusdet_b200.shard import make_delivery, GatherDelivery
deliv = make_delivery(T, BL, MD, "cpu", dst=0)
assert isinstance(deliv, GatherDelivery) and len(deliv.outs) == 2
for step in range(5):
    slot = step & 1
    deliv.before_write(slot)
    d, c = deliv.outs[slot]
    d.copy_(full_d[:, rank * BL:(rank + 1) * BL] * (step + 1)); c.copy_(full_c[:, rank * BL:(rank + 1) * BL])
    deliv.after_write(slot)
deliv.drain()
D, C = deliv.result(0)  # slot 0 holds step 4
if rank == 0:
    assert torch.equal(D, full_d * 5) and torch.equal(C, full_c)
    D1, _ = deliv.result(1)
    assert torch.equal(D1, full_d * 4)
    print("GATHERER_OK")
dist.destroy_process_group()
"""


def test_detection_gatherer_two_ranks_gloo(tmp_path):
    script = tmp_path / "worker2.py"
    script.write_text(_WORKER2.format(root=ROOT, port=29612))
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=120)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GATHERER_OK" in outs[0]


def _val_case(g, M, N, ncls=4):
    c = torch.rand(M, 2, generator=g) * 300 + 50
    wh = 40 + torch.rand(M, 2, generator=g) * 80
    lab = torch.cat((torch.randint(0, ncls, (M, 1), generator=g).float(), c - wh / 2, c + wh / 2), 1)
    if M and N:
        pick = torch.randint(0, M, (N,), generator=g)
        dc = c[pick] + torch.randn(N, 2, generator=g) * 8
        dwh = wh[pick] * (1 + 0.15 * torch.randn(N, 2, generator=g)).clamp_min(0.2)
        dcls = torch.where(torch.rand(N, generator=g) < 0.8, lab[pick, 0], torch.randint(0, ncls, (N,), generator=g).float())
    else:
        dc = torch.rand(N, 2, generator=g) * 300
        dwh = torch.rand(N, 2, generator=g) * 50 + 10
        dcls = torch.randint(0, ncls, (N,), generator=g).float()
    conf = torch.rand(N, 1, generator=g).sort(0, descending=True).values
    det = torch.cat((dc - dwh / 2, dc + dwh / 2, conf, dcls[:, None]), 1)
    return det, lab


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_val_matching_matches_reference_process_batch():
    """val_stats.match_predictions == the reference's process_batch (cerberusdet/val.py:32-54)."""
    from oracle.ref_import import load_reference

    load_reference()
    import cerberusdet.val as ref_val

    from cerberusdet_b200.val_stats import match_predictions

    g = torch.Generator().manual_seed(0)
    iouv = torch.linspace(0.5, 0.95, 10)
    for trial in range(120):
        M = int(torch.randint(1, 25, (1,), generator=g))
        N = int(torch.randint(1, 60, (1,), generator=g))
        det, lab = _val_case(g, M, N)
        assert torch.equal(ref_val.process_batch(det, lab, iouv), match_predictions(det, lab, iouv)), trial


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_batched_rescale_equals_reference_scale_boxes_on_cpu():
    """The rescale half of val_stats.validation_batch_statistics (SURVEY 8f-2) against the reference's own scale_boxes, with
    and without ratio_pad, bit for bit on CPU tensors (true division there; the GPU test pins the CUDA reciprocal form)."""
    from oracle.ref_import import load_reference

    load_reference()
    from cerberusdet.utils.general import scale_boxes

    from cerberusdet_b200 import val_stats

    ori = [(480, 640), (720, 1280), (333, 500), (640, 640)]
    g = torch.Generator().manual_seed(5)
    for with_rp in (True, False):
        rp = []
        for (h0, w0) in ori:
            r = min(384 / h0, 640 / w0)
            rp.append(((r, r), ((640 - w0 * r) / 2, (384 - h0 * r) / 2)) if with_rp else None)
        boxes = torch.rand(len(ori), 40, 4, generator=g) * 700 - 30  # some outside the image: clip_boxes matters
        cols = val_stats._scale_params((384, 640), ori, rp, torch.device("cpu"))
        got = val_stats._scale_boxes_batched(boxes, *cols)
        for i in range(len(ori)):
            want = boxes[i].clone()
            scale_boxes((384, 640), want, ori[i], ratio_pad=rp[i])
            assert torch.equal(got[i], want)


@pytest.mark.parametrize("role", ["writer", "dst"])
@pytest.mark.parametrize("side", ["piggyback", "branch3", "after"])
def test_pipeline_delivery_bookkeeping(role, side, monkeypatch):
    """Which batch is pushed / collected at which step (pipeline.PostHeadPipeline.step / flush with an in-graph delivery),
    without a GPU: the graphs are replaced by recorders.  For every run length, on both sides of the delivery: every batch
    is pushed (collected) exactly once, in order, into the slot of its parity; a batch is pushed no earlier than the step
    after its NMS launch and before the NMS launch that overwrites its staging slot; it is collected no earlier than one
    step after it was pushed; instrumented steps and the stand-alone placements change none of that."""
    from types import SimpleNamespace

    from cerberusdet_b200 import pipeline

    monkeypatch.setattr(pipeline, "_SIDE", side)
    log = []

    class G:
        def __init__(self, what, slot=None):
            self.what, self.slot = what, slot

        def replay(self):
            log.append((self.what, self.slot, pipe.k))

    def make(n_steps, timed_at):
        p = object.__new__(pipeline.PostHeadPipeline)
        p.overlap, p.k, p.pending = True, 0, None
        p.delivery = SimpleNamespace(rank=1 if role == "writer" else 0, dst=0, direct=False)
        p._g_first = [G("first", s) for s in (0, 1)]
        p._g_step = [G("plain", s) for s in (0, 1)]
        p._g_full = [G("full", s) for s in (0, 1)]
        p._g_flush = [G("flush", s) for s in (0, 1)]
        p._g_flush_full = [G("flush_full", s) for s in (0, 1)]
        p._g_push = [G("push", s) if role == "writer" else None for s in (0, 1)]
        p._g_collect = [G("collect", s) if role == "dst" else None for s in (0, 1)]
        p.timed = [(G("timed_side" if (k >= 3 and side == "piggyback") else "timed", k & 1), None) for k in timed_at]
        p.timed_parity = [k & 1 for k in timed_at]
        p.timed_has_side = [k >= 3 and side == "piggyback" for k in timed_at]
        return p

    for n_steps in (1, 2, 3, 4, 5, 8, 9):
        for timed_at in ([], [1], [2, 3], [1, 2, 3, 4, 5, 6, 7]):
            timed_at = [k for k in timed_at if k < n_steps]
            log.clear()
            pipe = make(n_steps, timed_at)
            slot_of = {k: i for i, k in enumerate(timed_at)}
            for k in range(n_steps):
                pipe.step(timed=slot_of.get(k))
            pipe.flush()
            # expand the log into delivery events (batch, at_step); a graph that carries the side work does it for batch
            # k-2 (push) / k-3 (collect) of the step k it belongs to; the flush's launch is NMS launch n-1 = "step n"
            events = []
            in_flush = False
            for what, slot, k_after in log:
                in_flush = in_flush or what in ("flush", "flush_full")
                k = n_steps if in_flush else k_after - 1  # (step() has already advanced the counter when it replays)
                if what in ("full", "timed_side", "flush_full"):
                    step = k if what != "flush_full" else n_steps
                    batch = step - 2 if role == "writer" else step - 3
                    assert batch >= 0 and slot == (step & 1 if what != "flush_full" else (n_steps - 1) & 1)
                    events.append((batch, step))
                elif what in ("push", "collect"):
                    events.append((None, k, slot))
            # stand-alone kernels are logged with their slot only: recover their batch from the order
            batches, nxt = [], 0
            for e in events:
                if e[0] is None:
                    assert e[2] == nxt & 1, f"{role} {side} n={n_steps} timed={timed_at}: slot {e[2]} for batch {nxt}"
                    batches.append((nxt, e[1]))
                else:
                    assert e[0] == nxt, f"{role} {side} n={n_steps} timed={timed_at}: batch {e[0]} where {nxt} was due"
                    batches.append(e)
                nxt += 1
            assert [b for b, _ in batches] == list(range(n_steps)), f"{role} {side} n={n_steps} timed={timed_at}: {batches}"
            for b, at in batches:
                if role == "writer":  # beside step b+2 (its NMS launch was step b+1; launch b+2, at step b+3, reuses the staging) or in the flush
                    assert at == b + 2 or (at == n_steps and b >= n_steps - 2), (b, at, n_steps)
                else:                 # one step after the writers pushed it, or in the flush
                    assert at == b + 3 or (at == n_steps and b >= n_steps - 3), (b, at, n_steps)


@pytest.mark.skipif(not REF, reason="needs the reference tree (/root/reference or oracle/_ref)")
def test_can_fuse_tail_preconditions_on_the_real_detect():
    """detect.can_fuse_tail mirrors cerb_head_tail's preconditions on the reference's own Detect module (no GPU needed):
    half tensors, both towers ending in a biased 1x1 nn.Conv2d with a multiple-of-16 input width, every H*W a multiple of
    8, nc <= 192 -- and FusedHeads hands out exactly the last convolutions' parameters."""
    from oracle.ref_import import load_reference

    ref = load_reference()
    from cerberusdet_b200 import detect

    head = ref.yolo.Detect(nc=20, ch=(64, 128, 256)).half()
    x640 = [torch.zeros(1, c, 80 >> i, 80 >> i, dtype=torch.float16) for i, c in enumerate((64, 128, 256))]
    assert detect.can_fuse_tail(head, x640)
    assert not detect.can_fuse_tail(head, [t.float() for t in x640])                       # fp32 activations
    x320 = [torch.zeros(1, c, 40 >> i, 40 >> i, dtype=torch.float16) for i, c in enumerate((64, 128, 256))]
    assert not detect.can_fuse_tail(head, x320)                                           # P5 is 10x10: H*W % 8 != 0
    assert not detect.can_fuse_tail(ref.yolo.Detect(nc=20, ch=(64, 128, 256)), x640)      # fp32 weights
    wide = ref.yolo.Detect(nc=365, ch=(64, 128, 256)).half()
    assert not detect.can_fuse_tail(wide, x640)                                           # nc > 192
    fused = detect.FusedHeads([t for t in x640], [t for t in x640], head)
    bw, bb, cw, cb = fused.weights()
    assert bw[0] is head.cv2[0][-1].weight and cb[2] is head.cv3[2][-1].bias and tuple(cw[1].shape) == (20, head.cv3[1][-1].in_channels, 1, 1)
    assert tuple(bw[0].shape)[0] == 64 and head.cv2[0][-1].in_channels % 16 == 0
