"""Micro-benchmark of the fused rel-pos attention kernel alone (cfg2 layer shape by default)."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
from gpu_util import op_attention, ptr, stream
from conformer_nemo_b200 import _lib

B, T, H, dk = [int(v) for v in (sys.argv[1:5] if len(sys.argv) > 4 else (32, 500, 8, 64))]
Dp = H * 64
torch.manual_seed(0)
qkv = (torch.randn(B * T, 4 * Dp, device="cuda") * 0.5).bfloat16()
pos = (torch.randn(2 * T - 1, Dp, device="cuda") * 0.5).bfloat16()
ctx = torch.empty(B * T, Dp, device="cuda", dtype=torch.bfloat16)
lens = torch.full((B,), T, dtype=torch.int32, device="cuda")
lib = _lib.load_library()
def run():
    rc = lib.cfb_op_rel_attention(1, ptr(qkv), ptr(pos), pos.stride(0), ptr(ctx), ptr(lens), B, T, H, dk, 64, stream())
    assert rc == 0
for _ in range(3): run()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 20
e0.record()
for _ in range(n): run()
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / n
fl = 6.0 * B * T * T * H * dk
print(f"B={B} T={T} H={H}: {ms*1e3:.1f} us  {fl/ms/1e9:.1f} TFLOP/s")


# quick numerics check against torch (fp32 math on the bf16 inputs), full lengths
import math
q = qkv.float().view(B, T, 4, H, 64)
qu, qv, k, v = [q[:, :, j].permute(0, 2, 1, 3) for j in range(4)]
pp = pos.float().view(2 * T - 1, H, 64).permute(1, 0, 2)
if B * H * T * T <= 64 * 1024 * 1024:
    ac = qu @ k.transpose(-1, -2)
    bd = qv @ pp.transpose(-1, -2).unsqueeze(0)
    bd = torch.nn.functional.pad(bd, (1, 0)).view(B, H, -1, T)[:, :, 1:].view(B, H, T, 2 * T - 1)[..., :T]
    want = (torch.softmax((ac + bd) / math.sqrt(dk), -1) @ v).permute(0, 2, 1, 3).reshape(B * T, Dp)
    diff = (ctx.float() - want).abs()
    print(f"max_abs {float(diff.max()):.4e} rel_l2 {float(diff.norm() / want.norm()):.4e}")
