"""bfloat16 on the post-head path, host side (no GPU): the bf16 facts the kernels reproduce, pinned against torch on the
CPU (tests/test_gpu_bf16.py pins them again on the GPU); the reference port running end to end in bf16; the dtype
gates of the C ABI and of ``ops``; the parser of tools/sass_identity.py on a recorded ``cuobjdump -sass`` sample."""
import ctypes
import os
import sys

import pytest
import torch

from cerberusdet_b200 import _lib, ops
from cerberusdet_b200.synth import STRIDES, level_shapes, synth_heads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16 = torch.bfloat16


# ------------------------------------------------------------------ fact 1: anchors are not exact in bf16
def test_bf16_anchor_centres_round_above_128():
    ac = torch.arange(160, dtype=BF16) + 0.5  # make_anchors (utils/tal.py:188-189), P3 of a 1280 x 1280 input
    exact = torch.arange(160, dtype=torch.float64) + 0.5
    assert ac[128].item() == 128.0 and ac[129].item() == 130.0  # 128.5 -> 128, 129.5 -> 130: ties to even
    assert int((ac.double() != exact).sum()) == 32  # every k + 0.5 with k >= 128 rounds
    assert bool((ac[:128].double() == exact[:128]).all())
    # at 640 x 640 the largest anchor is 79.5: nothing rounds
    for h, w in level_shapes((640, 640), STRIDES):
        assert bool(((torch.arange(w, dtype=BF16) + 0.5).double() == torch.arange(w, dtype=torch.float64) + 0.5).all())
    # the port's anchor grid (what the kernels are compared against) carries the same rounding
    from oracle import ref_port as rp

    anchors, _ = rp.anchor_grid(level_shapes((1280, 1280), STRIDES), STRIDES, BF16)
    assert anchors.dtype == BF16 and anchors[0, 128].item() == 128.0 and anchors[0, 129].item() == 130.0


# ------------------------------------------------------------------ fact 2: conf_thres is rounded to bf16 before the compare
@pytest.mark.parametrize("conf,rounded", [(0.001, 0.0009994506835937500), (0.3, 0.30078125), (0.45, 0.44921875),
                                          (0.6, 0.6015625), (0.25, 0.25)])
def test_bf16_threshold_rounding(conf, rounded):
    assert torch.tensor(conf, dtype=torch.float32).to(BF16).item() == rounded  # double -> float -> bf16
    s = torch.tensor([rounded], dtype=BF16)
    assert not bool((s > conf).item())  # the score equal to bf16(conf) does not pass
    above = torch.tensor([rounded], dtype=BF16).nextafter(torch.tensor([1.0], dtype=BF16))
    assert bool((above > conf).item())


def test_bf16_elementwise_equals_rounded_fp32():
    """Fact 3 on the CPU: an add / sub / mul of two bf16 values computed in fp32 and rounded once to bf16 (what ATen does)
    equals the correctly rounded exact result (fp32 has >= 2 * 8 + 2 significant bits)."""
    g = torch.Generator().manual_seed(5)
    a = (torch.randn(200000, generator=g) * 64).to(BF16)
    b = (torch.randn(200000, generator=g) * 4).to(BF16)
    for op in (torch.add, torch.sub, torch.mul):
        got = op(a, b)
        exact = op(a.double(), b.double()).to(torch.float32)  # exact in double, one rounding to fp32 on the way is fine
        assert torch.equal(got, exact.to(BF16))


# ------------------------------------------------------------------ the reference port in bf16
def test_ref_port_end_to_end_in_bf16():
    from oracle import ref_port as rp

    heads = synth_heads(range(2), [20], (256, 192), BF16, "planted", cfg=3)[0]
    y = rp.decode_port(heads, 20, STRIDES)
    assert y.dtype == BF16 and tuple(y.shape) == (2, 24, sum(h * w for h, w in level_shapes((256, 192), STRIDES)))
    y32 = rp.decode_port([x.float() for x in heads], 20, STRIDES)
    # boxes: a few bf16 ulps of the corner (grid units) times the stride; scores: one rounding to bf16
    assert torch.allclose(y[:, :4].float(), y32[:, :4], rtol=2 ** -7, atol=2 * 0.25 * 32)
    assert torch.allclose(y[:, 4:].float(), y32[:, 4:], rtol=2 ** -8, atol=0)
    for kw in (dict(conf_thres=0.001, iou_thres=0.6, multi_label=True), dict(conf_thres=0.25, iou_thres=0.45)):
        rows = rp.nms_port(y, greedy="c", **kw)
        assert len(rows) == 2 and any(r.shape[0] for r in rows)
        for r in rows:
            assert r.dtype == torch.float32  # the cat at general.py:444-449 promotes the bf16 rows
            assert torch.equal(r[:, :5].to(BF16).float(), r[:, :5])  # boxes and scores are bf16 values
            assert bool((r[:, 4] > torch.tensor(kw["conf_thres"]).to(BF16).float()).all())
    pd = torch.randn(2, 50, 64, generator=torch.Generator().manual_seed(1)).to(BF16).requires_grad_()
    anchors = torch.rand(50, 2).mul(40).to(BF16)
    out = rp.bbox_decode_port(anchors, pd)
    assert out.dtype == BF16
    out.float().sum().backward()
    assert pd.grad.dtype == BF16 and torch.isfinite(pd.grad.float()).all()


# ------------------------------------------------------------------ dtype gates
def test_abi_takes_bf16_only_where_heads_are_read():
    lib = _lib.load()
    ia, fa = _lib.int_array, _lib.float_array
    assert _lib.CERB_BF16 == 2
    assert lib.cerb_summary_row_len(8400, _lib.CERB_BF16) == lib.cerb_summary_row_len(8400, _lib.CERB_F16) == 1056
    assert lib.cerb_summary_row_len(8400, 3) == 0
    one = _lib.ptr_array([256])
    # B = 0: accepted, nothing launched
    for code, want in ((_lib.CERB_BF16, 0), (3, _lib.CERB_EINVAL)):
        assert lib.cerb_decode(one, ia([5]), 1, 1, 0, ia([8]), ia([8]), fa([8.0]), code, one, None, None, None) == want
        assert lib.cerb_decode_split(one, one, ia([5]), 1, 1, 0, ia([8]), ia([8]), fa([8.0]), code, one, None, None, None) == want
        assert lib.cerb_nms(one, ia([5]), 1, 0, 64, code, 0.25, 0.45, None, 0, 0, 0, 300, 30000, 7680.0, None, None, None,
                            None, 0, None) == want
        assert lib.cerb_bbox_decode_fwd(None, None, 0, 0, 16, code, None, None) == want
        assert lib.cerb_bbox_decode_bwd(None, None, 0, 16, code, None, None) == want
    assert lib.cerb_decode_nms(one, ia([5]), 1, 1, 0, ia([8]), ia([8]), fa([8.0]), _lib.CERB_BF16, one, None, 0.25, 0.45,
                               None, 0, 0, 0, 300, 30000, 7680.0, None, None, None, 0, None) == 0
    # every other entry point keeps rejecting it
    rc = lib.cerb_head_tail(one, one, one, one, one, one, ia([64]), ia([64]), ia([4]), 1, 1, 1, ia([8]), ia([8]), fa([8.0]),
                            _lib.CERB_BF16, one, None, None, None)
    assert rc == _lib.CERB_EINVAL and b"fp16 only" in lib.cerb_last_error()
    src = _lib.ptr_array([256])
    rc = lib.cerb_letterbox(src, ia([4]), ia([4]), (ctypes.c_long * 1)(12), ia([4]), ia([4]), ia([0]), ia([0]), 1, 4, 4,
                            _lib.CERB_BF16, ctypes.c_void_p(256), None)
    assert rc == _lib.CERB_EINVAL and b"dtype" in lib.cerb_last_error()


def test_ops_dtype_code_is_not_widened_for_everyone():
    t = torch.empty(1, dtype=BF16)
    assert ops._dtype_code(t, head=True) == _lib.CERB_BF16
    with pytest.raises(TypeError):
        ops._dtype_code(t)  # letterbox, head_tail, bbox_loss, tal_assign, ap_per_class
    assert BF16 not in ops._DTYPES


# ------------------------------------------------------------------ tools/sass_identity.py
SAMPLE_OLD = """
Fatbin elf code:
================
arch = sm_100a
identifier = decode.cu

	code for sm_100a
		Function : _Z13decode_kernelIfLi1EEv12DecodeParams
	.headerflags	@"EF_CUDA_SM100 EF_CUDA_VIRTUAL_SM(EF_CUDA_SM100)"
        /*0000*/                   LDC R1, c[0x0][0x37c] ;                                             /* 0x0000df00ff017b82 */
                                                                                                       /* 0x000e300000000800 */
        /*0010*/                   S2R R0, SR_CTAID.X ;                                                /* 0x0000000000007919 */
                                                                                                       /* 0x000e220000002500 */
        /*0020*/                   EXIT ;                                                              /* 0x000000000000794d */
                                                                                                       /* 0x000fea0003800000 */
		..........

		Function : _ZN41_GLOBAL__N__a1b2c3d4_15_ap_per_class_cu_0123abcd10ap_kernelEv
	.headerflags	@"EF_CUDA_SM100 EF_CUDA_VIRTUAL_SM(EF_CUDA_SM100)"
        /*0000*/                   EXIT ;                                                              /* 0x000000000000794d */
                                                                                                       /* 0x000fea0003800000 */
		Function : _Z4gonev
        /*0000*/                   EXIT ;                                                              /* 0x000000000000794d */
                                                                                                       /* 0x000fea0003800000 */
"""


def _sass_tool():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import sass_identity
    finally:
        sys.path.pop(0)
    return sass_identity


def test_sass_identity_parser_on_recorded_sample():
    si = _sass_tool()
    old = si.parse_sass(SAMPLE_OLD)
    assert set(old) == {"_Z13decode_kernelIfLi1EEv12DecodeParams", "_ZN41_GLOBAL__N__<anon>10ap_kernelEv", "_Z4gonev"}
    assert old["_Z13decode_kernelIfLi1EEv12DecodeParams"] == [
        ("LDC R1, c[0x0][0x37c]", "0x0000df00ff017b82:0x000e300000000800"),
        ("S2R R0, SR_CTAID.X", "0x0000000000007919:0x000e220000002500"),
        ("EXIT", "0x000000000000794d:0x000fea0003800000"),
    ]
    # the new build: one instruction's control bits changed, the anonymous-namespace hash moved, a kernel was removed and
    # one was added
    new_text = (SAMPLE_OLD.replace("0x000e220000002500", "0x000e240000002500")
                .replace("a1b2c3d4_15_ap_per_class_cu_0123abcd", "ffff0000_15_ap_per_class_cu_9999ffff")
                .replace("_Z4gonev", "_Z5addedv"))
    same, diff, missing, added = si.compare(old, si.parse_sass(new_text))
    assert same == ["_ZN41_GLOBAL__N__<anon>10ap_kernelEv"]
    assert diff == ["_Z13decode_kernelIfLi1EEv12DecodeParams"]
    assert missing == ["_Z4gonev"] and added == ["_Z5addedv"]
    assert si.compare(old, si.parse_sass(SAMPLE_OLD)) == (sorted(old), [], [], [])
    text = si.report(same, diff, missing, added)
    assert text.startswith("identical: 1  differing: 1  missing: 1  new: 1")
