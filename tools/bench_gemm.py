"""Micro-benchmark of the tcgen05 GEMM family on the cfg2 layer shapes (M = 16000)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
from gpu_util import ptr, stream
from conformer_nemo_b200 import _lib

lib = _lib.load_library()
M = 16000
CFG4 = len(sys.argv) > 1 and sys.argv[1] == "cfg4"   # python tools/bench_gemm.py cfg4: the Medium shapes (d = 256, 256 x 100 frames)
EPI = dict(LINEAR=0, SWISH=1, RELU=2, RESID=3, QKV=4, GLU=5)
CASES = [("linear1+swish", "SWISH", 2048, 512, "bf16"), ("linear2", "RESID", 512, 2048, "f32"),
         ("qkv", "QKV", 1536, 512, "bf16"), ("linear_out", "RESID", 512, 512, "f32"),
         ("pw1+glu", "GLU", 1024, 512, "bf16"), ("plain bf16 N512", "LINEAR", 512, 512, "bf16"),
         ("plain bf16 N2048", "LINEAR", 2048, 512, "bf16"), ("plain f32 N512 K2048", "LINEAR", 512, 2048, "f32")]
CASES.append(("conv0 as GEMM (M=1.28M)", "RELU", 512, 24, "bf16"))
if CFG4:
    M = 25600
    CASES = [("linear1+swish", "SWISH", 1024, 256, "bf16"), ("linear2", "RESID", 256, 1024, "f32"), ("qkv", "QKV", 768, 256, "bf16"),
             ("linear_out", "RESID", 256, 256, "f32"), ("pw1+glu", "GLU", 512, 256, "bf16"), ("plain bf16 N1024", "LINEAR", 1024, 256, "bf16")]
M0 = M
for name, epi, N, K, od in CASES:
    M = 1280000 if K == 24 else M0
    A = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
    W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
    bias = torch.randn(N, device="cuda")
    ncols = {"QKV": N + (256 if CFG4 else 512), "GLU": N // 2}.get(epi, N)
    out = torch.zeros(M, ncols, device="cuda", dtype=torch.bfloat16 if od == "bf16" else torch.float32)
    lens = torch.full((M // 100 if CFG4 else 32,), 100 if CFG4 else 500, dtype=torch.int32, device="cuda")
    def run():
        rc = lib.cfb_op_gemm(1, EPI[epi], ptr(A), K, ptr(W), K, ptr(bias), ptr(bias), M, N, K, ptr(out), ncols,
                             _lib.CFB_BF16 if od == "bf16" else _lib.CFB_F32, 0.5, ptr(lens) if epi == "GLU" else None,
                             100 if CFG4 else 500, (256 if CFG4 else 512) if epi == "QKV" else 0, None, stream())
        assert rc == 0, _lib.last_error(None)
    for _ in range(3): run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n): run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    print(f"{name:24s} N={N:5d} K={K:5d}: {ms * 1e3:7.1f} us  {2.0 * M * N * K / ms / 1e9:7.0f} TFLOP/s")
