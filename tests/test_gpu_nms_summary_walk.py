"""The NMS kernel's summary-guided scans at the edges of their block-wide loops: pass 1 (the score summary) and pass 2
(the listed score vectors) issue their loads unconditionally with the index clamped to the last valid entry, so the
tails matter -- a summary shorter than one block, one that is not a multiple of the block, a pass 2 over more than one
block of listed vectors, and chunks small enough that a segment takes many of them.  The summary-guided result must
equal the summary-free kernel path and the oracle, bit for bit."""
import pytest
import torch

from cerberusdet_b200.synth import STRIDES, synth_heads

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from cerberusdet_b200 import _lib, ops as o

    _lib.load()
    yield o
    _lib.load().cerb_debug_set_chunking(0, 0)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float32])
# 168 anchors: the whole summary is a fraction of one block; 1680 and 33600: several blocks with a partial last one
@pytest.mark.parametrize("imgsz", [(128, 64), (320, 256), (1280, 1280)])
# default: one chunk per segment; (64, 40): many chunks; (4096, 3000): thousands of listed vectors in one pass 2
@pytest.mark.parametrize("chunking", [None, (64, 40), (4096, 3000)])
@pytest.mark.parametrize("kw", [
    dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300),
    dict(conf_thres=0.0, iou_thres=0.45, max_det=100),
    dict(conf_thres=0.01, iou_thres=0.5, classes=[0, 5, 11], multi_label=True, max_det=40),
])
def test_summary_walk_tails(ops, dtype, imgsz, chunking, kw):
    from cerberusdet_b200 import _lib
    from oracle import ref_port as rp

    ncs = [20, 12]
    bsz = 1 if imgsz[0] > 1000 else 2
    heads = synth_heads(range(bsz), ncs, imgsz, dtype, "planted", cfg=11)
    ys = ops.decode_heads([[x.cuda() for x in lv] for lv in heads], STRIDES)
    assert all(ops.find_summary(y) is not None for y in ys)
    if chunking is not None:
        assert _lib.load().cerb_debug_set_chunking(*chunking) == 0
    try:
        dets, counts = ops.nms_batched(ys, **kw)
        d0, c0 = ops.nms_batched(ys, use_summary=False, **kw)
    finally:
        _lib.load().cerb_debug_set_chunking(0, 0)
    assert torch.equal(c0, counts) and torch.equal(d0, dets)
    ch = counts.cpu()
    for t in range(len(ncs)):
        want = rp.nms_port(ys[t].cpu(), greedy="c", **kw)
        for b in range(bsz):
            assert torch.equal(dets[t, b, : ch[t, b]].cpu(), want[b]), (t, b)
