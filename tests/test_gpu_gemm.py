"""GPU: tcgen05 GEMM (+ every fused epilogue) against torch fp32 and against the CUDA-core validation kernel,
called through the C ABI (cfb_op_gemm)."""
import pytest
import torch

from conformer_nemo_b200 import _lib
from gpu_util import describe_mismatch, err_stats, expected_instance, op_gemm, ptr, stream

pytestmark = pytest.mark.gpu


def _mk(M, N, K, seed=0, ints=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if ints:  # small integers: every product and partial sum is exact in bf16 x bf16 -> fp32
        A = torch.randint(-3, 4, (M, K), generator=g, device="cuda").float()
        W = torch.randint(-3, 4, (N, K), generator=g, device="cuda").float()
    else:
        A = torch.randn(M, K, generator=g, device="cuda")
        W = torch.randn(N, K, generator=g, device="cuda") / K ** 0.5
    return A, W


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (128, 128, 256), (256, 256, 128), (300, 192, 176), (77, 64, 64),
                                   (1000, 1024, 512), (640, 2048, 512), (130, 704, 176)])
def test_tc_linear_exact_on_integers(M, N, K):
    A, W = _mk(M, N, K, ints=True)
    want = A @ W.t()
    out = torch.full((M, N), float("nan"), device="cuda")
    op_gemm(True, _lib.EPI_LINEAR, A.bfloat16(), W.bfloat16(), out=out)
    st = err_stats(out, want)
    assert st["nan"] == 0 and st["max_abs"] == 0.0, f"{st}{describe_mismatch(out, want, 0.0)}"


@pytest.mark.parametrize("use_tc", [False, True])
@pytest.mark.parametrize("M,N,K", [(300, 192, 176), (513, 512, 512),
                                   # pre_encode.out: K = F2 * C (F2 = 20 at 80 mel bins; 21 at 81, 11 at 41)
                                   (406, 256, 5120), (300, 176, 3696), (77, 64, 168), (1000, 512, 10240)])
def test_linear_bias(use_tc, M, N, K):
    A, W = _mk(M, N, K, seed=1)
    bias = torch.randn(N, device="cuda")
    if use_tc:
        Ab, Wb = A.bfloat16(), W.bfloat16()
        want = Ab.float() @ Wb.float().t() + bias
        out = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
        op_gemm(True, _lib.EPI_LINEAR, Ab, Wb, bias=bias, out=out)
        st = err_stats(out.float(), want)
        assert st["nan"] == 0 and st["rel_l2"] < 4e-3, st
        # fp32 output (as pre_encode.out writes the residual stream): K products and the bias summed in fp32 are off by
        # at most K * 2^-24 * sum |a w| (+ |bias|) from the exact sum of the bf16 operands
        out32 = torch.full((M, N), float("nan"), device="cuda")
        op_gemm(True, _lib.EPI_LINEAR, Ab, Wb, bias=bias, out=out32)
        a64, w64 = Ab.double(), Wb.double()
        want64 = a64 @ w64.t() + bias.double()
        bound = K * 2.0 ** -24 * (a64.abs() @ w64.abs().t() + bias.double().abs())
        bad = (out32.double() - want64).abs() > bound
        assert not torch.isnan(out32).any() and not bad.any(), f"{int(bad.sum())} elements out of bound, first {bad.nonzero()[:4].tolist()}"
    else:
        want = A @ W.t() + bias
        out = torch.zeros(M, N, device="cuda")
        op_gemm(False, _lib.EPI_LINEAR, A, W, bias=bias, out=out)
        st = err_stats(out, want)
        assert st["nan"] == 0 and st["max_abs"] < 1e-4, st


@pytest.mark.parametrize("use_tc", [False, True])
def test_swish_relu(use_tc):
    M, N, K = 260, 704, 176
    A, W = _mk(M, N, K, seed=2)
    bias = torch.randn(N, device="cuda") * 0.5
    dt = torch.bfloat16 if use_tc else torch.float32
    Ai, Wi = A.to(dt), W.to(dt)
    z = Ai.float() @ Wi.float().t() + bias
    for epi, fn in ((_lib.EPI_SWISH, torch.nn.functional.silu), (_lib.EPI_RELU, torch.relu)):
        out = torch.zeros(M, N, device="cuda", dtype=dt)
        op_gemm(use_tc, epi, Ai, Wi, bias=bias, out=out)
        st = err_stats(out.float(), fn(z))
        assert st["nan"] == 0 and st["rel_l2"] < (5e-3 if use_tc else 1e-5), (epi, st)


@pytest.mark.parametrize("use_tc", [False, True])
def test_residual(use_tc):
    M, N, K = 200, 176, 704
    A, W = _mk(M, N, K, seed=3)
    bias = torch.randn(N, device="cuda")
    dt = torch.bfloat16 if use_tc else torch.float32
    Ai, Wi = A.to(dt), W.to(dt)
    resid = torch.randn(M, N, device="cuda")
    want = resid + 0.5 * (Ai.float() @ Wi.float().t() + bias)
    out = resid.clone()
    op_gemm(use_tc, _lib.EPI_RESID, Ai, Wi, bias=bias, out=out, alpha=0.5)
    st = err_stats(out, want)
    assert st["nan"] == 0 and st["max_abs"] < (2e-4 if use_tc else 1e-4), st


@pytest.mark.parametrize("use_tc", [False, True])
def test_qkv_epilogue(use_tc):
    M, K, Dp = 150, 176, 256
    N = 3 * Dp
    A, W = _mk(M, N, K, seed=4)
    bias = torch.randn(N, device="cuda")
    bias2 = torch.randn(Dp, device="cuda")
    dt = torch.bfloat16 if use_tc else torch.float32
    Ai, Wi = A.to(dt), W.to(dt)
    z = Ai.float() @ Wi.float().t()
    want = torch.cat([z[:, :Dp] + bias[:Dp], z[:, :Dp] + bias2, z[:, Dp:] + bias[Dp:]], dim=1)
    out = torch.zeros(M, 4 * Dp, device="cuda", dtype=dt)
    op_gemm(use_tc, _lib.EPI_QKV, Ai, Wi, bias=bias, bias2=bias2, out=out, qkv_dp=Dp)
    st = err_stats(out.float(), want)
    assert st["nan"] == 0 and st["rel_l2"] < (4e-3 if use_tc else 1e-5), st


@pytest.mark.parametrize("use_tc", [False, True])
def test_glu_mask_epilogue(use_tc):
    B, T, d, K = 3, 50, 176, 176
    M, N = B * T, 2 * d
    A, W = _mk(M, N, K, seed=5)
    bias = torch.randn(N, device="cuda")
    lens = torch.tensor([50, 31, 0], dtype=torch.int32, device="cuda")
    dt = torch.bfloat16 if use_tc else torch.float32
    Ai, Wi = A.to(dt), W.to(dt)
    z = Ai.float() @ Wi.float().t() + bias  # reference channel order: [a (d) | gate (d)]
    want = z[:, :d] * torch.sigmoid(z[:, d:])
    valid = (torch.arange(T, device="cuda")[None, :] < lens[:, None]).reshape(M, 1)
    want = want * valid
    # interleave rows the way cfb_finalize_weights does: groups of 32 accumulator columns = [16 a | 16 gate]
    cols = torch.arange(N, device="cuda")
    grp, j = cols // 32, cols % 32
    src = torch.where(j < 16, grp * 16 + j, d + grp * 16 + (j - 16))
    out = torch.full((M, d), float("nan"), device="cuda", dtype=dt)
    op_gemm(use_tc, _lib.EPI_GLU, Ai, Wi[src].contiguous(), bias=bias[src].contiguous(), out=out, lens=lens,
            frames_per_seq=T)
    st = err_stats(out.float(), want)
    assert st["nan"] == 0 and st["rel_l2"] < (5e-3 if use_tc else 1e-5), st


def test_tc_matches_simt_on_bf16_inputs():
    M, N, K = 384, 512, 2048
    A, W = _mk(M, N, K, seed=6)
    Ab, Wb = A.bfloat16(), W.bfloat16()
    o_tc = torch.zeros(M, N, device="cuda")
    o_ref = torch.zeros(M, N, device="cuda")
    op_gemm(True, _lib.EPI_LINEAR, Ab, Wb, out=o_tc)
    op_gemm(False, _lib.EPI_LINEAR, Ab.float(), Wb.float(), out=o_ref)
    st = err_stats(o_tc, o_ref)
    assert st["nan"] == 0 and st["max_abs"] < 1e-4, st


@pytest.mark.parametrize("epi", ["LINEAR", "SWISH", "RESID", "QKV", "GLU"])
@pytest.mark.parametrize("M,N,K", [(4999, 2048, 512), (9900, 512, 176), (16000, 2048, 512), (19999, 1536, 512),
                                   (19999, 2048, 512), (5000, 768, 2048), (20100, 1024, 2000), (20100, 768, 2000)])
def test_cta_pair_kernel_is_bit_identical_to_the_single_cta_kernel(epi, M, N, K, monkeypatch):
    """gemm_tc2.cu (cta_group::2, 256 x 256 tiles per CTA pair) against gemm_tc.cu's 256-wide kernel on the same
    operands: same k-block order and the same epilogue arithmetic -> identical bits, including M tails where the last
    pair's second CTA owns a few rows (4999, 9900, 5000, 20100), none (16000) or the first one only part of its rows
    (19999).  CFB_GEMM_2CTA forces either kernel (the default picks by shape)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    single, pair = expected_instance(M, N, K, "0", sms), expected_instance(M, N, K, "1", sms)
    assert single[:2] == ("tc", 256) and pair == ("tc2",), (single, pair)
    A, W = _mk(M, N, K, seed=5)
    A, W = A.bfloat16(), W.bfloat16()
    bias = torch.randn(N, device="cuda") * 0.3
    frames = 50
    kw = {}
    if epi == "QKV":
        if N % 3:
            pytest.skip("QKV needs N = 3 * Dp")
        dp = N // 3
        kw = dict(bias2=torch.randn(dp, device="cuda") * 0.3, qkv_dp=dp)
        ncols, dt = N + dp, torch.bfloat16
    elif epi == "GLU":
        kw = dict(lens=torch.randint(0, frames + 1, ((M + frames - 1) // frames,), device="cuda", dtype=torch.int32),
                  frames_per_seq=frames)
        ncols, dt = N // 2, torch.bfloat16
    elif epi == "RESID":
        kw = dict(alpha=0.5)
        ncols, dt = N, torch.float32
    else:
        ncols, dt = N, torch.bfloat16
    outs = []
    for mode in ("0", "1", "1"):  # the pair kernel twice: run-to-run repeatability
        monkeypatch.setenv("CFB_GEMM_2CTA", mode)
        gen = torch.Generator(device="cuda").manual_seed(9)
        out = torch.randn(M, ncols, device="cuda", generator=gen).to(dt) if epi == "RESID" else torch.full(
            (M, ncols), float("nan"), device="cuda", dtype=dt)
        op_gemm(True, getattr(_lib, "EPI_" + epi), A, W, bias=bias, out=out, **kw)
        outs.append(out)
    assert int(torch.isnan(outs[0].float()).sum()) == 0
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2]), err_stats(outs[1].float(), outs[0].float())


CFB_ERR_INVALID_ARG, CFB_ERR_UNSUPPORTED = 1, 2


# (use_tc, epilogue, N, out dtype, out columns, ldo, qkv_dp, status): combinations no GEMM kernel can write
REFUSED = {
    "tc-swish-f32": (1, _lib.EPI_SWISH, 256, torch.float32, 256, 256, 0, CFB_ERR_UNSUPPORTED),
    "tc-relu-f32": (1, _lib.EPI_RELU, 256, torch.float32, 256, 256, 0, CFB_ERR_UNSUPPORTED),
    "tc-qkv-f32": (1, _lib.EPI_QKV, 192, torch.float32, 256, 256, 64, CFB_ERR_UNSUPPORTED),
    "tc-glu-f32": (1, _lib.EPI_GLU, 256, torch.float32, 128, 128, 0, CFB_ERR_UNSUPPORTED),
    "tc-resid-bf16": (1, _lib.EPI_RESID, 256, torch.bfloat16, 256, 256, 0, CFB_ERR_UNSUPPORTED),
    "simt-resid-bf16": (0, _lib.EPI_RESID, 256, torch.bfloat16, 256, 256, 0, CFB_ERR_UNSUPPORTED),
    "tc-linear-f16": (1, _lib.EPI_LINEAR, 256, torch.float16, 256, 256, 0, CFB_ERR_UNSUPPORTED),
    "tc-qkv-dp-96": (1, _lib.EPI_QKV, 288, torch.bfloat16, 384, 384, 96, CFB_ERR_INVALID_ARG),
    "simt-qkv-dp-96": (0, _lib.EPI_QKV, 288, torch.float32, 384, 384, 96, CFB_ERR_INVALID_ARG),
    "tc-qkv-dp-0": (1, _lib.EPI_QKV, 192, torch.bfloat16, 256, 256, 0, CFB_ERR_INVALID_ARG),
    "tc-qkv-n-not-3dp": (1, _lib.EPI_QKV, 256, torch.bfloat16, 320, 320, 64, CFB_ERR_INVALID_ARG),
    "tc-glu-n-200": (1, _lib.EPI_GLU, 200, torch.bfloat16, 104, 104, 0, CFB_ERR_INVALID_ARG),
    "simt-glu-n-200": (0, _lib.EPI_GLU, 200, torch.float32, 104, 104, 0, CFB_ERR_INVALID_ARG),
    "tc-linear-ldo": (1, _lib.EPI_LINEAR, 256, torch.bfloat16, 256, 248, 0, CFB_ERR_INVALID_ARG),
    "tc-qkv-ldo": (1, _lib.EPI_QKV, 192, torch.bfloat16, 256, 192, 64, CFB_ERR_INVALID_ARG),
    "simt-glu-ldo": (0, _lib.EPI_GLU, 256, torch.float32, 128, 120, 0, CFB_ERR_INVALID_ARG),
    "tc-unknown-epilogue": (1, 6, 256, torch.bfloat16, 256, 256, 0, CFB_ERR_INVALID_ARG),
}


@pytest.mark.parametrize("case", list(REFUSED))
def test_op_gemm_refuses_outputs_its_kernels_cannot_write(case):
    """cfb_op_gemm returns an error before it enqueues anything: `out` (a sentinel) is left as it was."""
    use_tc, epi, N, dt, cols, ldo, qkv_dp, status = REFUSED[case]
    M, K = 64, 64
    A, W = _mk(M, N, K, seed=7)
    if use_tc:
        A, W = A.bfloat16(), W.bfloat16()
    bias = torch.zeros(N, device="cuda")
    bias2 = torch.zeros(max(qkv_dp, 1), device="cuda")
    out = torch.full((M, cols), 7.0, device="cuda", dtype=dt)
    keep = out.clone()
    scratch = torch.zeros(M * N, device="cuda")
    lib = _lib.load_library()
    dtype = {torch.float32: _lib.CFB_F32, torch.bfloat16: _lib.CFB_BF16, torch.float16: _lib.CFB_F16}[dt]
    rc = lib.cfb_op_gemm(use_tc, epi, ptr(A), A.stride(0), ptr(W), W.stride(0), ptr(bias), ptr(bias2), M, N, K, ptr(out),
                         ldo, dtype, 1.0, None, 1, qkv_dp, ptr(scratch), stream())
    torch.cuda.synchronize()
    assert rc == status, (rc, _lib.last_error(None))
    assert "op_gemm" in _lib.last_error(None)
    assert torch.equal(out, keep)
