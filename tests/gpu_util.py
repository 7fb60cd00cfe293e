"""Helpers for the -m gpu tests: thin wrappers that call the kernel-level C-ABI entry points (include/cfb.h) on torch
device tensors, and error metrics."""
import ctypes

import torch

from conformer_nemo_b200 import _lib

DT = {torch.float32: _lib.CFB_F32, torch.bfloat16: _lib.CFB_BF16}


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def op_gemm(use_tc, epi, A, W, bias=None, bias2=None, out=None, alpha=1.0, lens=None, frames_per_seq=1, qkv_dp=0):
    """A (M,K), W (N,K); out preallocated.  Returns out."""
    lib = _lib.load_library()
    M, K = A.shape
    N = W.shape[0]
    scratch = None if use_tc else torch.empty(M * N, dtype=torch.float32, device=A.device)
    rc = lib.cfb_op_gemm(int(use_tc), epi, ptr(A), A.stride(0), ptr(W), W.stride(0), ptr(bias), ptr(bias2), M, N, K,
                         ptr(out), out.stride(0), DT[out.dtype], float(alpha), ptr(lens), frames_per_seq, qkv_dp,
                         ptr(scratch), stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out


def expected_instance(M, N, K, mode=None, sms=148):
    """The tensor-core kernel launch_gemm_tc (gemm_tc.cu) picks for an (M, N, K) problem with 16-byte aligned operand
    strides: ("tc", BN, STAGES) for gemm_tc_kernel<BN, STAGES, ...>, ("tc2",) for the CTA-pair gemm_tc2_kernel.
    mode is CFB_GEMM_2CTA as a string ("0" never pairs, "1" pairs whenever gemm_tc2_supported, None: the default)."""
    m_tiles = -(-M // 128)
    small_m = N % 256 == 0 and 2 * m_tiles * (N // 256) <= sms
    if not small_m:
        flag = int(mode) if mode is not None else -1
        tc2_supported = N % 256 == 0 and K % 8 == 0 and M > 128
        if flag != 0 and tc2_supported and (flag == 1 or (K <= 1024 and N >= 1536)):
            return ("tc2",)
    if N % 256 == 0 and not small_m:
        return ("tc", 256, 4 if -(-K // 64) >= 16 else 3)
    return ("tc", 128, 5)


def tiles_per_cta(M, N, inst, sms=148):
    """Most output tiles one CTA (one CTA pair for "tc2") of the persistent grid works through."""
    if inst[0] == "tc2":
        tiles, workers = -(-M // 256) * (N // 256), sms // 2
    else:
        tiles, workers = -(-M // 128) * -(-N // inst[1]), sms
    return -(-tiles // min(tiles, workers))


def op_layernorm(x, gamma, beta, out, lens=None, frames_per_seq=1):
    lib = _lib.load_library()
    rows, d = x.shape
    rc = lib.cfb_op_layernorm(ptr(x), ptr(gamma), ptr(beta), ptr(out), DT[out.dtype], rows, d, ptr(lens),
                              frames_per_seq, stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out


def op_layernorm_dual(x, g1, b1, out1, g2, b2, out2):
    """out1 = LN(x; g1, b1) fp32 (may be x itself), out2 = LN(out1; g2, b2) bf16 (cfb_op_layernorm_dual)."""
    lib = _lib.load_library()
    rows, d = x.shape
    rc = lib.cfb_op_layernorm_dual(ptr(x), ptr(g1), ptr(b1), ptr(out1), ptr(g2), ptr(b2), ptr(out2), rows, d, stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out1, out2


def op_depthwise(x, taps, bias, out):
    """taps given as (d, ksize) like the reference's depthwise_conv.weight; the kernel wants them tap-major."""
    lib = _lib.load_library()
    B, T, d = x.shape
    taps_km = taps.t().contiguous()
    rc = lib.cfb_op_depthwise(ptr(x), ptr(taps_km), ptr(bias), ptr(out), DT[x.dtype], B, T, d, taps.shape[1], stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out


def op_attention(use_tc, qkv, pos, ctx, lens, B, T, H, dk, dkp=64):
    lib = _lib.load_library()
    rc = lib.cfb_op_rel_attention(int(use_tc), ptr(qkv), ptr(pos), pos.stride(0), ptr(ctx), ptr(lens), B, T, H, dk,
                                  dkp, stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return ctx


def op_lengths(lengths, B, T_full, n_stages=2):
    lib = _lib.load_library()
    out = torch.empty(B, dtype=torch.int32, device="cuda")
    rc = lib.cfb_op_lengths(ptr(lengths), ptr(out), B, T_full, n_stages, stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out


def err_stats(got, want):
    got = got.double()
    want = want.double()
    diff = (got - want).abs()
    rel_l2 = float(diff.norm() / want.norm().clamp_min(1e-30))
    return dict(max_abs=float(diff.max()), rel_l2=rel_l2, nan=int(torch.isnan(got).sum()),
                argmax=tuple(int(v) for v in torch.unravel_index(diff.argmax(), diff.shape)))


def describe_mismatch(got, want, tol):
    """Row / column pattern of the mismatching elements (helps to tell descriptor bugs from epilogue bugs)."""
    bad = (got.double() - want.double()).abs() > tol
    if bad.dim() != 2 or not bad.any():
        return ""
    rows = bad.any(1).nonzero().flatten().tolist()
    cols = bad.any(0).nonzero().flatten().tolist()
    return f" bad rows {rows[:12]}..({len(rows)}) bad cols {cols[:12]}..({len(cols)}) frac {float(bad.float().mean()):.4f}"


def op_dw_pw2(g, taps, bias, W2, bias2, x):
    """Fused conv-module tail (cfb_op_dw_pw2).  g (B,T,d) bf16; taps (d, ksize) like depthwise_conv.weight with the
    BatchNorm already folded; bias (d); W2 (d,d) bf16; bias2 (d); x (B,T,d) fp32 updated in place."""
    lib = _lib.load_library()
    B, T, d = g.shape
    k = taps.shape[1]
    t32 = torch.zeros(32, d, dtype=torch.float32, device=g.device)
    sh = 15 - (k - 1) // 2
    t32[sh:sh + k] = taps.t()
    t32[31] = bias
    rc = lib.cfb_op_dw_pw2(ptr(g), ptr(t32), ptr(W2), ptr(bias2), ptr(x), B, T, d, stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return x
