"""Micro-benchmark of the fused conv-module tail (cfb_op_dw_pw2) against the two kernels it replaces, on the cfg2
shape (32 x 500 x 512) by default.  L2-warm back-to-back launches, CUDA events on the launching stream."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
from gpu_util import ptr, stream, DT
from conformer_nemo_b200 import _lib

lib = _lib.load_library()
B, T, d = [int(v) for v in (sys.argv[1:4] if len(sys.argv) >= 4 else (32, 500, 512))]
reps = 1 if "--once" in sys.argv else 50
g = torch.randn(B, T, d, device="cuda").to(torch.bfloat16)
t32 = torch.randn(32, d, device="cuda") / 5.5
W2 = (torch.randn(d, d, device="cuda") / d ** 0.5).to(torch.bfloat16)
b2 = torch.randn(d, device="cuda") * 0.1
x = torch.zeros(B, T, d, device="cuda")
c = torch.empty_like(g)
taps = t32[:31].contiguous(); bias = t32[31].contiguous()

def fused():
    assert lib.cfb_op_dw_pw2(ptr(g), ptr(t32), ptr(W2), ptr(b2), ptr(x), B, T, d, stream()) == 0
def split():
    assert lib.cfb_op_depthwise(ptr(g), ptr(taps), ptr(bias), ptr(c), _lib.CFB_BF16, B, T, d, 31, stream()) == 0
    assert lib.cfb_op_gemm(1, _lib.EPI_RESID, ptr(c), d, ptr(W2), d, ptr(b2), None, B * T, d, d, ptr(x), d, _lib.CFB_F32,
                           1.0, None, 1, 0, None, stream()) == 0

def timeit(fn, name):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    print(f"{name:28s} {us:8.1f} us   ({B * T * d * 10 / us / 1e3:.0f} GB/s of g + x traffic)")
timeit(fused, "fused dw+pw2")
if "--once" not in sys.argv:
    timeit(split, "depthwise, then pw2 GEMM")
