"""GPU: memory-bound kernels against torch fp32 references, through the C ABI."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import err_stats, op_depthwise, op_layernorm, op_layernorm_dual, op_lengths

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("d", [64, 176, 256, 512, 1024])
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.bfloat16])
def test_layernorm(d, out_dtype):
    torch.manual_seed(d)
    rows = 333
    x = torch.randn(rows, d, device="cuda") * 3 + 1.5
    g = torch.randn(d, device="cuda")
    b = torch.randn(d, device="cuda")
    want = F.layer_norm(x, (d,), g, b, 1e-5)
    out = torch.full((rows, d), float("nan"), device="cuda", dtype=out_dtype)
    op_layernorm(x, g, b, out)
    st = err_stats(out.float(), want)
    assert st["nan"] == 0
    assert st["max_abs"] < (2e-5 if out_dtype == torch.float32 else 5e-2) and st["rel_l2"] < (1e-6 if out_dtype == torch.float32 else 4e-3), st


def test_layernorm_in_place_and_masked():
    torch.manual_seed(0)
    B, T, d = 3, 21, 176
    x = torch.randn(B * T, d, device="cuda")
    g, b = torch.randn(d, device="cuda"), torch.randn(d, device="cuda")
    lens = torch.tensor([21, 9, 0], dtype=torch.int32, device="cuda")
    want = F.layer_norm(x, (d,), g, b, 1e-5)
    valid = (torch.arange(T, device="cuda")[None] < lens[:, None]).reshape(-1, 1)
    y = x.clone()
    op_layernorm(y, g, b, y)  # in place (norm_out of the inner layers)
    assert err_stats(y, want)["max_abs"] < 2e-5
    out = torch.full_like(x, float("nan"))
    op_layernorm(x, g, b, out, lens=lens, frames_per_seq=T)
    assert err_stats(out, want * valid)["max_abs"] < 2e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,T,d,k", [(2, 50, 176, 31), (3, 130, 512, 31), (1, 7, 64, 31), (2, 64, 256, 9)])
def test_depthwise_bn_swish(dtype, B, T, d, k):
    torch.manual_seed(T)
    x = torch.randn(B, T, d, device="cuda").to(dtype)
    taps = torch.randn(d, k, device="cuda") / k ** 0.5
    bias = torch.randn(d, device="cuda") * 0.1
    want = F.silu(F.conv1d(x.float().transpose(1, 2), taps.unsqueeze(1), bias, padding=(k - 1) // 2, groups=d)).transpose(1, 2)
    out = torch.full((B, T, d), float("nan"), device="cuda", dtype=dtype)
    op_depthwise(x, taps, bias, out)
    st = err_stats(out.float(), want)
    assert st["nan"] == 0 and st["max_abs"] < (2e-5 if dtype == torch.float32 else 3e-2), st


def test_lengths_bit_exact_against_reference_golden():
    z = np.load(os.path.join(GOLDEN, "lengths.npz"))
    lengths = torch.from_numpy(z["lengths"]).cuda()
    for rep in (1, 2, 3):
        got = op_lengths(lengths, lengths.numel(), 0, rep)
        assert got.dtype == torch.int32
        assert np.array_equal(got.cpu().numpy(), z[f"rep{rep}"]), rep
    # length=None: every row is T_full
    got = op_lengths(None, 5, 2001, 2)
    assert got.tolist() == [501] * 5


def _bf16_ulp(got, want):
    _, e = torch.frexp(torch.maximum(got.abs(), want.abs()))
    return torch.ldexp(torch.ones_like(got), e - 8)


@pytest.mark.parametrize("d", [16, 64, 144, 176, 256, 512, 1024])
@pytest.mark.parametrize("offset,scale", [(0.0, 1.0), (1e3, 0.1)])
def test_layernorm_dual_in_place_against_fp64(d, offset, scale):
    """norm_out + the next layer's norm_feed_forward1 in one kernel, in place as the engine runs it (out1 == x), against
    LN2(LN1(x)) in fp64.  A large common offset (mean 1e3, std 0.1) is where a plain fp32 sum of the row loses the
    mean (~1e-3 at the output); the kernel sums x - x[0] instead."""
    torch.manual_seed(d)
    rows = 333  # not a multiple of the 8 rows of a block
    x = torch.randn(rows, d, device="cuda", dtype=torch.float64) * scale + offset
    x = x.float()
    g1, b1 = torch.randn(d, device="cuda"), torch.randn(d, device="cuda")
    g2, b2 = torch.randn(d, device="cuda"), torch.randn(d, device="cuda")

    def ln64(v, g, b):
        v = v.double()
        m = v.mean(-1, keepdim=True)
        return (v - m) / torch.sqrt(((v - m) ** 2).mean(-1, keepdim=True) + 1e-5) * g.double() + b.double()

    want1 = ln64(x, g1, b1)
    want2 = ln64(want1, g2, b2)
    y = x.clone()
    out2 = torch.full((rows, d), float("nan"), device="cuda", dtype=torch.bfloat16)
    op_layernorm_dual(y, g1, b1, y, g2, b2, out2)
    assert float((y.double() - want1).abs().max()) < 2e-5
    o2 = out2.double()
    assert not torch.isnan(o2).any()
    assert torch.all((o2 - want2).abs() <= _bf16_ulp(o2, want2) + 2e-5)
    # Against cfb_op_layernorm applied twice: the same formula, but not the same bits.  The dual kernel gives lane l the
    # float4 columns l, l + 32, ... and sums x - x[0]; layernorm_kernel gives it the pairs 2l, 2l + 1, 2l + 64, ... and
    # sums x itself, so the two reductions round differently.  Without the offset both meet the same fp64 bound.
    if offset == 0.0:
        t1 = torch.empty_like(x)
        t2 = torch.empty(rows, d, device="cuda", dtype=torch.bfloat16)
        op_layernorm(x, g1, b1, t1)
        op_layernorm(t1, g2, b2, t2)
        assert float((t1.double() - want1).abs().max()) < 2e-5
        assert torch.all((t2.double() - want2).abs() <= _bf16_ulp(t2.double(), want2) + 2e-5)
