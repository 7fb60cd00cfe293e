"""Small-M GEMMs (one group of an 8-GPU share: ~1000 token rows) timed under CUDA-graph replay of a dependent chain, so the
number is the kernel's latency in a chain and not the host's launch rate."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
from gpu_util import ptr
from conformer_nemo_b200 import _lib

lib = _lib.load_library()
for M in (1059, 2118, 3176):
    for name, epi, N, K in (("linear2 (resid)", 3, 512, 2048), ("linear_out (resid)", 3, 512, 512), ("plain bf16", 0, 512, 512)):
        A = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
        W = (torch.randn(N, K, device="cuda") / K ** 0.5).bfloat16()
        bias = torch.randn(N, device="cuda")
        out = torch.zeros(M, N, device="cuda", dtype=torch.float32 if epi == 3 else torch.bfloat16)
        s = torch.cuda.Stream()
        def run(stream):
            rc = lib.cfb_op_gemm(1, epi, ptr(A), K, ptr(W), K, ptr(bias), None, M, N, K, ptr(out), N,
                                 _lib.CFB_F32 if epi == 3 else _lib.CFB_BF16, 0.5, None, 1, 0, None, ctypes.c_void_p(stream))
            assert rc == 0, _lib.last_error(None)
        with torch.cuda.stream(s):
            for _ in range(3): run(s.cuda_stream)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                for _ in range(20): run(torch.cuda.current_stream().cuda_stream)
            g.replay(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10): g.replay()
            e1.record(); torch.cuda.synchronize()
        print(f"M={M:5d} {name:20s} N={N} K={K:4d}: {e0.elapsed_time(e1) / 200 * 1e3:6.2f} us per launch in a chain")
