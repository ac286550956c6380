"""Phase breakdown of nms_kernel (thread 0 of every block, averaged) using the -DNMS_PROFILE build.
Build: CERB_OUT=cerberusdet_b200/libcerb_post_prof.so sh cerberusdet_b200/csrc/build.sh -DNMS_PROFILE
Run:   CERB_LIB=cerberusdet_b200/libcerb_post_prof.so python tools/nms_phases.py cfg2 cfg3"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cerberusdet_b200 import _lib, ops
from cerberusdet_b200.synth import STRIDES, synth_heads
from kbench import CFG
names = ["setup", "hist", "collect", "sort", "A gather", "B prev+kept", "C pairwise", "D fixpoint", "E append", "rest"]
lib = _lib.load()
buf = (ctypes.c_ulonglong * 24)()
for name in sys.argv[1:] or ["cfg2", "cfg3"]:
    c = CFG[name]
    heads = synth_heads(range(c["B"]), c["ncs"], c["imgsz"], c["dtype"], c.get("regime", "iid"), cfg=3)
    ys = ops.decode_heads([[x.cuda() for x in lv] for lv in heads], STRIDES)
    ops.nms_batched(ys, **c["kw"]); lib.cerb_debug_read_profile(buf, 1)
    for _ in range(10): ops.nms_batched(ys, **c["kw"])
    lib.cerb_debug_read_profile(buf, 1)
    runs = buf[10]; tot = sum(buf[i] for i in range(10))
    print(f"{name}: cycles per block {tot/runs:.0f} (~{tot/runs/1.965e3:.1f} us @1.965GHz), consumed per block {buf[11]/runs:.0f}, blocks {runs}")
    for i, n in enumerate(names):
        print(f"   {n:14s} {buf[i]/runs:9.0f} cyc  {100*buf[i]/tot:5.1f}%")
    print("   fixpoint rounds per block:", buf[15] / runs)
    print(f"   collect sub-steps (cycles per block): pass 1 {buf[12]/runs:.0f}, wait {buf[13]/runs:.0f}, pass 2 {buf[14]/runs:.0f}")
    print(f"   chunks per block {buf[16]/runs:.3f}, tiles per block {buf[17]/runs:.3f}, vectors listed per block {buf[18]/runs:.0f}, "
          f"plain-scan chunks {buf[19]}, exact-histogram rebuilds {buf[20]}")
    print(f"   fixpoint: settle iterations per warp-round {buf[21]/max(buf[15]*16,1):.2f}, settle cycles per warp-round {buf[22]/max(buf[15]*16,1):.0f}")
