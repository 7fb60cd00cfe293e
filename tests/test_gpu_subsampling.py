"""GPU: the stages in front of (and around) the first Conformer layer, each against a float64 CPU restatement whose input
is the device's own input to that stage, so every stage is judged by its own rounding only.

Stages: the first strided conv (y1), the implicit-GEMM second conv (y2), the sinusoid table (pe), the per-layer
linear_pos projections in their head packing (pos, fp16 on the bf16 path), the attention of the last layer (ctx) and
the final norm_out (encoded).  Buffers are read with ConformerEncoder.debug_buffer after a dense forward with B <= 7
(from B = 8 on, cfb_forward splits a bf16 batch into two half-batch plans and cfb_debug_buffer refuses it).

Tolerances are bounds, not measurements: u = 2^-24 is the fp32 unit roundoff, S the same sum taken over magnitudes
(so the fp32 accumulation of n terms is off by at most n * u * S), and a rounded output may move by one ulp of its
format.  A wrong tap, row, plane or tile is an O(1) error at that element and cannot hide under them.

Layouts (engine.cu, elementwise.cu):
  y1  [B][plane][Th][Fh][C], plane = (t1 & 1) * 2 + (f1 & 1), row t1 >> 1, column f1 >> 1; positions t1 >= T1 or
      f1 >= F1 are padding and hold exact zeros
  y2  [B][T2][F2][C]
  pe  (2T' - 1, d), row k = relative position T' - 1 - k, even columns sin, odd columns cos
  pos (2T' - 1, L * Dp), layer l at column l * Dp, head h at l * Dp + h * 64 ... + dk - 1, lanes dk ... 63 zero
"""
import math

import pytest
import torch
import torch.nn.functional as F

import conformer_nemo_b200 as cn
from oracle import conformer_oracle as oc
from test_gpu_attention import torch_reference

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def ulp(v, mant_bits):
    """Spacing of a format with `mant_bits` stored mantissa bits at |v| (0 where v == 0)."""
    _, e = torch.frexp(v.abs())
    return torch.where(v == 0, torch.zeros_like(v), torch.ldexp(torch.ones_like(v), e - 1 - mant_bits))


def bf16_ulp(got, want):
    return ulp(torch.maximum(got.abs(), want.abs()), 7)


def f32_ulp(got, want):
    return ulp(torch.maximum(got.abs(), want.abs()), 23)


def assert_within(got, want, tol, what):
    got, want = got.double(), want.double()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert not torch.isnan(got).any() and not torch.isinf(got).any(), what
    bad = (got - want).abs() > tol
    if bad.any():
        idx = [tuple(int(i) for i in r) for r in bad.nonzero()[:8]]
        worst = tuple(int(i) for i in torch.unravel_index(((got - want).abs() / tol.clamp_min(1e-300)).argmax(), got.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound, first at {idx}; worst "
                             f"{worst}: got {float(got[worst])} want {float(want[worst])} tol {float(tol[worst])}")


def conv3x3s2(x, w, b=None):
    """(B, Cin, T, F) float64 -> (B, Cout, ceil(T/2), ceil(F/2)): the reference's Conv2d(k=3, s=2, p=1), kh along time."""
    return F.conv2d(x, w, b, stride=2, padding=1)


def planes_to_dense(y1, B, Th, Fh, C):
    """[B][plane][Th][Fh][C] -> (B, C, 2 Th, 2 Fh) with t1 = 2 * row + (plane >> 1), f1 = 2 * col + (plane & 1)."""
    return y1.view(B, 2, 2, Th, Fh, C).permute(0, 5, 3, 1, 4, 2).reshape(B, C, 2 * Th, 2 * Fh)


def layer_norm64(x, g, b):
    x = x.double()
    m = x.mean(-1, keepdim=True)
    v = ((x - m) ** 2).mean(-1, keepdim=True)
    return (x - m) / torch.sqrt(v + 1e-5) * g.double() + b.double()


def conv_out(n):
    return (n - 1) // 2 + 1


class Run:
    """One dense forward and its intermediates, copied to the host."""

    def __init__(self, feat_in, C, d, H, L, T, lens, feat_dtype, precision, seed, feat_out=-1):
        self.cfg = oc.EncoderConfig(feat_in=feat_in, n_layers=L, d_model=d, n_heads=H, subsampling_conv_channels=C,
                                    feat_out=feat_out)
        self.sd = oc.random_state_dict(self.cfg, seed)
        self.B, self.T, self.F = len(lens), T, feat_in
        self.C = self.cfg.conv_channels
        self.d, self.H, self.L, self.dk = d, H, L, d // H
        self.T1, self.F1 = conv_out(T), conv_out(feat_in)
        self.T2, self.F2 = conv_out(self.T1), conv_out(self.F1)
        self.Th, self.Fh = (self.T1 + 1) // 2, (self.F1 + 1) // 2
        self.P = 2 * self.T2 - 1
        self.Dp = H * 64
        g = torch.Generator().manual_seed(seed + 1000)
        # non-zero features everywhere, also behind every length: the convolutions run over the padded batch
        self.x = (torch.randn(self.B, feat_in, T, generator=g) * 2.0).to(feat_dtype)
        self.lens = torch.tensor(lens, dtype=torch.int64)
        enc = cn.ConformerEncoder(feat_in=feat_in, n_layers=L, d_model=d, n_heads=H, subsampling_conv_channels=C,
                                  feat_out=feat_out, precision=precision)
        missing, unexpected = enc.load_state_dict(self.sd, strict=False)
        assert not unexpected and all("num_batches_tracked" in m for m in missing), (missing, unexpected)
        enc = enc.cuda().eval()
        enc.packed = False
        y, ylen = enc(audio_signal=self.x.cuda(), length=self.lens.cuda())
        torch.cuda.synchronize()
        self.y, self.ylen = y.transpose(1, 2).cpu(), ylen.cpu()
        self.bf16 = precision == "bf16"
        adt = torch.bfloat16 if self.bf16 else torch.float32
        buf = lambda name, dt: enc.debug_buffer(self.B, T, name).view(dt).cpu()  # noqa: E731
        self.y1 = buf("y1", adt).double().view(self.B, 4, self.Th, self.Fh, self.C)
        self.y2 = buf("y2", adt).double().view(self.B, self.T2, self.F2, self.C)
        self.pe = buf("pe", adt).double().view(self.P, d)
        self.pos = buf("pos", torch.float16 if self.bf16 else torch.float32).double().view(self.P, L * self.Dp)
        self.qkv = buf("qkv", adt).double().view(self.B, self.T2, 4, H, 64)
        self.ctx = buf("ctx", adt).double().view(self.B, self.T2, H, 64)
        self.xs = buf("x", torch.float32).double().view(self.B, self.T2, d)
        self.div_term = torch.exp(torch.arange(0, d, 2, dtype=torch.float32) * -(math.log(10000.0) / d))
        del enc


def check_y1(r):
    x = r.x.float().transpose(1, 2).unsqueeze(1)  # (B, 1, T, F)
    w = r.sd["pre_encode.conv.0.weight"].float()
    b = r.sd["pre_encode.conv.0.bias"].float()
    dense = planes_to_dense(r.y1, r.B, r.Th, r.Fh, r.C)
    pad = torch.ones_like(dense, dtype=torch.bool)
    pad[:, :, :r.T1, :r.F1] = False
    assert torch.all(dense[pad] == 0), "y1: a padding position of the planes is not 0"
    got = dense[:, :, :r.T1, :r.F1]
    if r.bf16:
        # the GEMM operands of conv0_im2col_kernel / cfb_finalize_weights: features split hi + lo, weights rounded, bias
        # split hi + lo; 24 products summed in fp32, the result rounded to bf16
        hi = x.bfloat16().float()
        lo = (x - hi).bfloat16().float()
        xs = hi.double() + lo.double()
        wb = w.bfloat16().double()
        bh = b.bfloat16().float()
        bl = (b - bh).bfloat16().double()
        want = torch.relu(conv3x3s2(xs, wb, bh.double() + bl))
        S = conv3x3s2(hi.double().abs() + lo.double().abs(), wb.abs(), bh.double().abs() + bl.abs())
        assert_within(got, want, bf16_ulp(got, want) + 24 * U * S, "y1 vs its bf16 operands")
        # only the nine weights are rounded: against the conv with fp32 weights the error is the weights' rounding
        # (bf16 keeps 8 significant bits: 2^-8 relative), the output's rounding (half a bf16 ulp) and < 2^-16 S for the
        # hi + lo split and the fp32 sum
        want32 = torch.relu(conv3x3s2(x.double(), w.double(), b.double()))
        S32 = conv3x3s2(x.double().abs(), w.double().abs(), b.double().abs())
        assert_within(got, want32, (2.0 ** -8 + 2.0 ** -16) * S32 + 0.5 * bf16_ulp(got, want32), "y1 vs the fp32-weight conv")
    else:
        # subsample_first_kernel: bias + nine fp32 FMAs
        want = torch.relu(conv3x3s2(x.double(), w.double(), b.double()))
        S = conv3x3s2(x.double().abs(), w.double().abs(), b.double().abs())
        assert_within(got, want, 9 * U * S, "y1 (fp32 path)")


def check_y2(r):
    y1 = planes_to_dense(r.y1, r.B, r.Th, r.Fh, r.C)[:, :, :r.T1, :r.F1]
    w = r.sd["pre_encode.conv.2.weight"].float()
    b = r.sd["pre_encode.conv.2.bias"].double()
    w = (w.bfloat16() if r.bf16 else w).double()
    want = torch.relu(conv3x3s2(y1, w, b)).permute(0, 2, 3, 1)  # (B, T2, F2, C)
    S = conv3x3s2(y1.abs(), w.abs(), b.abs()).permute(0, 2, 3, 1)
    tol = 9 * r.C * U * S
    if r.bf16:
        tol = tol + bf16_ulp(r.y2, want)
    assert_within(r.y2, want, tol, "y2 from the device y1")


def check_pe(r):
    positions = torch.arange(r.T2 - 1, -r.T2, -1, dtype=torch.float32).unsqueeze(1)
    ang = positions * r.div_term  # fp32 product, as the kernel's __fmul_rn
    want = torch.stack([torch.sin(ang), torch.cos(ang)], dim=-1).reshape(r.P, r.d).double()
    tol = bf16_ulp(r.pe, want) if r.bf16 else 4 * f32_ulp(r.pe, want)
    assert_within(r.pe, want, tol, "pe")


def check_pos(r):
    got = r.pos.view(r.P, r.L, r.H, 64)
    assert torch.all(got[..., r.dk:] == 0), "pos: a padding lane is not 0"
    for l in range(r.L):
        w = r.sd[f"layers.{l}.self_attn.linear_pos.weight"].bfloat16().double()
        want = (r.pe @ w.t()).view(r.P, r.H, r.dk)
        S = (r.pe.abs() @ w.abs().t()).view(r.P, r.H, r.dk)
        g = got[:, l, :, :r.dk]
        # bf16 GEMM output, then bf16 -> fp16 in place: exact except below fp16's normal range (spacing 2^-24)
        assert_within(g, want, bf16_ulp(g, want) + r.d * U * S + 2.0 ** -25, f"pos layer {l}")


def check_ctx(r):
    parts = [r.qkv[:, :, i, :, :r.dk].permute(0, 2, 1, 3) for i in range(4)]  # (B, H, T', dk)
    l = r.L - 1
    p = r.pos[:, l * r.Dp:(l + 1) * r.Dp].view(r.P, r.H, -1)[..., :r.dk].permute(1, 0, 2)
    lens = r.ylen.long()
    want = torch_reference(*parts, p, lens)  # (B, T', H, dk)
    got = r.ctx[..., :r.dk]
    for b, n in enumerate(lens.tolist()):
        assert torch.all(r.ctx[b, n:] == 0), f"ctx: row >= encoded_len of utterance {b} is not 0"
    diff = (got - want).abs()
    rel = float(diff.norm() / want.norm().clamp_min(1e-30))
    assert rel < 1.5e-2 and float(diff.max()) < 6e-2, (rel, float(diff.max()))


def check_encoded(r):
    l = r.L - 1
    want = layer_norm64(r.xs, r.sd[f"layers.{l}.norm_out.weight"], r.sd[f"layers.{l}.norm_out.bias"])
    valid = (torch.arange(r.T2)[None, :] < r.ylen[:, None].long())[..., None]
    want = want * valid
    assert torch.all(r.y[~valid.expand_as(r.y)] == 0), "encoded: a frame >= encoded_len is not 0"
    assert_within(r.y, want, torch.full_like(want, 2e-5), "encoded from the device x")


# feat_in, C (-1 = d_model), d_model, heads, layers, T, lengths, feature dtype.  feat_in 81 / 41 are odd (the
# padded column of the odd-f1 plane, a partial 4-bin output tile of the second conv), 359 is the largest the first
# conv's shared-memory patch holds; C 8 / 24 / 72 leave one partial 64-channel chunk per tap; T 1 ... 5 give odd and
# even T1; lengths include 0.
CASES = [
    (80, -1, 64, 4, 2, 203, [203, 150, 0], torch.float32),
    (64, 8, 64, 2, 1, 33, [33, 17, 1], torch.bfloat16),
    (128, 24, 96, 2, 2, 8, [8, 5, 0, 3], torch.float32),
    (81, 72, 80, 2, 1, 1037, [1037, 500], torch.float32),
    (41, 176, 176, 4, 2, 5, [5, 4, 1], torch.bfloat16),
    (359, 24, 48, 1, 1, 203, [203, 99], torch.float32),
    (81, 8, 64, 16, 2, 1, [1, 0], torch.float32),
    (41, 72, 144, 4, 1, 2, [2, 1, 2], torch.float32),
    (359, 8, 64, 2, 1, 3, [3, 2, 0], torch.bfloat16),
    (80, 176, 176, 4, 1, 4, [4, 3], torch.float32),
    (81, -1, 64, 1, 2, 33, [33, 0, 7, 32, 1, 20, 33], torch.float32),
    (41, 24, 64, 4, 1, 1037, [900, 1037], torch.bfloat16),
]
IDS = [f"F{c[0]}-C{c[1]}-d{c[2]}h{c[3]}L{c[4]}-T{c[5]}-B{len(c[6])}-{str(c[7])[6:]}" for c in CASES]


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_bf16_path_stage_by_stage(case):
    r = Run(*case, precision="bf16", seed=11)
    check_y1(r)
    check_y2(r)
    check_pe(r)
    check_pos(r)
    check_ctx(r)
    check_encoded(r)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_fp32_validation_path_stage_by_stage(case):
    """subsample_first_kernel, im2col_kernel + the CUDA-core GEMM and the fp32 table: the path the long-form bf16 test
    (test_full_size_cfg5_*) is compared against."""
    r = Run(*case, precision="fp32_validate", seed=12)
    check_y1(r)
    check_y2(r)
    check_pe(r)
    check_encoded(r)


@pytest.mark.parametrize("precision", ["bf16", "fp32_validate"])
def test_long_form_positional_table(precision):
    """T = 30000 (T' = 7500): the table's arguments reach ~7500 rad, where a reduced-range sine would be far off."""
    r = Run(80, -1, 64, 4, 1, 30000, [30000], torch.float32, precision=precision, seed=13)
    check_pe(r)
    if r.bf16:
        check_pos(r)
