"""GPU: the body of a Conformer layer module by module, each stage against a float64 CPU restatement whose input is the
device's own input to that stage, the way test_gpu_subsampling.py checks the front end.

One live module per forward.  The engine reuses its buffers, so after a forward most intermediates of a layer are gone.
A module's residual writer (feed_forward{1,2}.linear2, self_attn.linear_out, conv.pointwise_conv2) with zero weight
and bias adds exactly +0 to the fp32 stream, while everything upstream of it still runs.  With the same weights and
features:
  R0      all four writers of the layer zeroed: x holds x_in, the layer's input, and every module ran on exactly x_in.
          qkv (from LN_att(x_in)), ctx, g (from LN_conv(x_in)), c (unfused tail only), a = LN_ff2(x_in) and h (from a)
          survive.  On a one-layer encoder x_in is pre_encode.out's x0 (from the surviving y2).
  R_att / R_conv / R_ff2
          only that writer live: x = x_in + the module's update, computed from that forward's own ctx, c or h.
          R_conv runs with CFB_FUSED_TAIL=0 and, where dw_pw_supported(d), again with =2: both x must be identical.
  R_ff1'  only FF2 live, with feed_forward1.* and norm_feed_forward1.* copied into FF2's keys.
  R_ff1   only FF1 live.  Both run the same arithmetic on x_in, so x must be bit-identical: FF1's weight slot, packing and
          0.5 factor are then checked as tightly as FF2's.  On the bf16 path at layer l > 0 FF1's LayerNorm is computed
          by layernorm_dual inside the previous norm_out (other summation order), so there FF1's update is instead checked
          against float64 through two unknown bf16 operands (see operand()): a weaker check.
On a two-layer encoder layer 0 is fully live and the runs zero layer 1's writers: layer 1 reads its own pos columns
(l * Dp) and weights.  B <= 7 throughout (cfb_debug_buffer refuses half-batches).

Bounds are derived, not measured: u = 2^-24 is the fp32 unit roundoff, S the same sum taken over magnitudes, a K-term
fp32 accumulation is off by at most K u S (any order), and a bf16 output is rounded to nearest (half an ulp; see
test_gpu_gemm_fp64.py).  tanh.approx.f32 has a maximum relative error of 2^-10.987 (PTX ISA, tanh); the bf16 path's
sigmoid is 0.5 + 0.5 tanh.approx(x/2) and its swish h + h tanh.approx(h), h = x/2; the validation path uses expf.
  pre_encode.out  x0 = y2 W^T + b with W = bf16(fp32(W_sd sqrt(d))) with K permuted (c, f) -> (f, c): K u S + the bias
                  add; against the unrounded weights (2^-8 + (K + 8) u) S
  a               LN_ff2(x_in): the fp32 LayerNorm bound ln_ref() + half a bf16 ulp
  h               swish(a W1^T + b1): K u S through the swish slope (<= 1.1) + 0.5 |v| 2^-10.987 + 2u |h| + half an ulp
  qkv             [q+u | q+v | k | v], head h at h dkp, lanes dk..dkp-1 exactly 0: K u S + u |bq + pos_bias| (the host
                  sums bq + u, bq + v in fp32) + half an ulp, with the LN operand's uncertainty (operand())
  ctx             check_ctx (test_gpu_subsampling.py): the attention is covered elsewhere, here it is linear_out's input
  g               value * sigmoid(gate) from the state dict's pointwise_conv1 rows (not the GLU interleave): both K u S
                  with the LN operand's uncertainty, sigmoid' <= 1/4, 2^-10.987 / 2, 2u |g|, half an ulp; frames >=
                  encoded_len exactly 0
  c               swish(depthwise conv of the device's g with the state dict's taps, bias and BatchNorm running stats,
                  eps 1e-5, zero padding at both ends of each sequence), every frame: (ks + 2) u S (fp32 FMA chain and
                  the fp32 rounding of the folded taps and bias), the swish bound, half an ulp
  x (updates)     x_in + alpha (acc + b), alpha 1 or 0.5, every row: alpha K u S + 2u |update| + one fp32 ulp of x
The LN-fed GEMMs (qkv, g, FF1 at l > 0) read a bf16 operand that no longer exists.  Its float64 value y and the fp32
LayerNorm bound e bracket it: bf16(y - e) <= operand <= bf16(y + e) (rounding is monotonic).  Where the two agree the
operand is known exactly; only where they differ does |W| |hi - lo| enter the tolerance.  A blanket one-ulp allowance
per operand (~2^-8 S) would be as large as one wrong K term at d = 512.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import conformer_nemo_b200 as cn
from oracle import conformer_oracle as oc
from test_gpu_subsampling import U, assert_within, bf16_ulp, check_ctx, f32_ulp

pytestmark = pytest.mark.gpu

TANH_APPROX = 2.0 ** -10.987  # maximum relative error of tanh.approx.f32 (PTX ISA); |tanh| <= 1, so also absolute
WRITERS = ("feed_forward1.linear2", "self_attn.linear_out", "conv.pointwise_conv2", "feed_forward2.linear2")


def half_bf16_ulp(got, want):
    return 0.5 * bf16_ulp(got, want)


def ln_ref(x, g, b):
    """float64 LayerNorm (eps 1e-5) of the fp32 rows x, and a bound on the error of the fp32 kernels' value of it
    (layernorm_kernel, the second half of layernorm_dual_kernel): first order in u, for any summation order.
      mean:    (d - 1) u sum|x| / d for the sum, u each for 1/d and the product: dm = (d + 1) u mean|x|
      x - m:   dm + u |x - m|
      rstd:    the sum of squares (d + 3) u relative (+ dm^2 / var from the centring), 1/d, the product and + eps 3u;
               the square root halves that, sqrt and the division add 2u: rho
      y:       (x - m) rstd rounded, fma with gamma and beta rounded
    The factor 1 + 2^-10 covers the second-order terms."""
    x, g, b = x.double(), g.double(), b.double()
    d = x.shape[-1]
    xc = x - x.mean(-1, keepdim=True)
    r = 1.0 / torch.sqrt((xc * xc).mean(-1, keepdim=True) + 1e-5)
    z = xc * r
    y = z * g + b
    dm = (d + 1) * U * x.abs().mean(-1, keepdim=True)
    rho = ((d + 6) * U + (dm * r) ** 2) / 2 + 2 * U
    e = g.abs() * (r * (dm + 2 * U * xc.abs()) + z.abs() * (rho + 3 * U)) + U * y.abs()
    return y, e * (1 + 2.0 ** -10)


def operand(y, e, bf16):
    """The GEMM operand the device rounded from an fp32 value within y +- e, as (value, uncertainty).  bf16: rounding is
    monotonic, so bf16(y - e) <= operand <= bf16(y + e); where the two agree the operand is known exactly, elsewhere it
    is off from bf16(y) by at most hi - lo.  fp32: the value itself, within e."""
    if not bf16:
        return y, e
    lo, hi = (y - e).bfloat16().double(), (y + e).bfloat16().double()
    return y.bfloat16().double(), hi - lo


def linear(A, dA, W, b, K=None, eb=0.0):
    """A W^T + b and the bound on the device's fp32 value of it: the operand's uncertainty dA through |W|, K u S of the
    fp32 accumulation (K: the GEMM's K, padding included), the bias's own uncertainty eb, the bias add's rounding."""
    K = A.shape[-1] if K is None else K
    Wt = W.t()
    v = A @ Wt + b
    e = dA @ Wt.abs() + K * U * ((A.abs() + dA) @ Wt.abs()) + eb
    return v, e + U * (v.abs() + e)


def swish_ref(v, e, fast):
    """swish of a value within v +- e: slope <= 1.1; fast h + h tanh.approx(h): 0.5 |v| 2^-10.987 and 2u |f|; accurate
    x / (1 + expf(-x)): 2^-21 |f| (test_gpu_gemm_fp64.reference)."""
    f = v * torch.sigmoid(v)
    return f, 1.1 * e + (0.5 * v.abs() * TANH_APPROX if fast else 0.0) + (2.0 ** -23 if fast else 2.0 ** -21) * f.abs()


def glu_ref(a, ea, gt, eg, fast):
    """a sigmoid(gate): sigmoid' <= 1/4; fast 0.5 + 0.5 tanh.approx(gate / 2): 2^-10.987 / 2; 2u |f| (accurate: 2^-21)."""
    s = torch.sigmoid(gt)
    f = a * s
    rnd = 2.0 ** -23 if fast else 2.0 ** -21
    return f, ea * s + a.abs() * (eg / 4 + (TANH_APPROX / 2 if fast else 0.0)) + ea * eg / 4 + rnd * f.abs()


class Forward:
    """The buffers of one dense forward, copied to the host (the attributes check_ctx reads included)."""

    def __init__(self, case, sd, fused, monkeypatch):
        c = case
        monkeypatch.setenv("CFB_FUSED_TAIL", "2" if fused else "0")
        missing, unexpected = c.enc.load_state_dict(sd, strict=False)
        assert not unexpected and all("num_batches_tracked" in m for m in missing), (missing, unexpected)
        _, ylen = c.enc(audio_signal=c.feats.cuda(), length=c.lens.cuda())
        torch.cuda.synchronize()
        self.ylen = ylen.cpu()
        self.L, self.H, self.dk, self.Dp, self.P = c.L, c.H, c.dk, c.Dp, 2 * c.T2 - 1
        adt = torch.bfloat16 if c.bf16 else torch.float32
        buf = lambda name, dt: c.enc.debug_buffer(c.B, c.T, name).view(dt).cpu().double()  # noqa: E731
        self.x = buf("x", torch.float32).view(c.N, c.d)
        self.y2 = buf("y2", adt).view(c.N, c.F2 * c.C)
        self.a = buf("a", adt).view(c.N, c.d)
        self.h = buf("h", adt).view(c.N, c.dff)
        self.qkv = buf("qkv", adt).view(c.B, c.T2, 4, c.H, c.dkp)
        self.ctx = buf("ctx", adt).view(c.B, c.T2, c.H, c.dkp)
        self.g = buf("g", adt).view(c.B, c.T2, c.d)
        self.c = buf("c", adt).view(c.B, c.T2, c.d)
        self.pos = buf("pos", torch.float16 if c.bf16 else torch.float32).view(self.P, c.L * c.Dp)


class Case:
    def __init__(self, feat_in, d, H, ks, ff, T, lens, L, xscaling, precision, seed):
        self.cfg = oc.EncoderConfig(feat_in=feat_in, n_layers=L, d_model=d, n_heads=H, conv_kernel_size=ks,
                                    ff_expansion_factor=ff, xscaling=xscaling)
        self.sd = oc.random_state_dict(self.cfg, seed)
        self.d, self.H, self.ks, self.dff, self.L, self.l, self.xscaling = d, H, ks, d * ff, L, L - 1, xscaling
        self.dk = d // H
        self.dkp = 64 if self.dk <= 64 else 128  # as cfb_create: every head padded to its attention kernel's width
        self.Dp = H * self.dkp
        self.C = self.cfg.conv_channels
        self.F2 = oc.subsampled_extent(feat_in, 2)
        self.B, self.T, self.T2 = len(lens), T, oc.subsampled_extent(T, 2)
        self.N = self.B * self.T2
        self.bf16 = precision == "bf16"
        g = torch.Generator().manual_seed(seed + 1000)
        # non-zero features everywhere, also behind every length: the padded frames are computed from defined inputs
        self.feats = torch.randn(self.B, feat_in, T, generator=g) * 2.0
        self.lens = torch.tensor(lens, dtype=torch.int64)
        self.enc = cn.ConformerEncoder(feat_in=feat_in, n_layers=L, d_model=d, n_heads=H, conv_kernel_size=ks,
                                       ff_expansion_factor=ff, xscaling=xscaling, precision=precision).cuda().eval()
        self.enc.packed = False

    def key(self, name):
        return f"layers.{self.l}.{name}"

    def w(self, name):
        """The device's GEMM operand of a weight matrix of this layer: bf16-rounded on the bf16 path."""
        t = self.sd[self.key(name)].float()
        t = t.reshape(t.shape[0], -1)
        return (t.bfloat16() if self.bf16 else t).double()

    def vec(self, name):
        return self.sd[self.key(name)].double()

    def weights(self, live=(), ff1_into_ff2=False):
        """The state dict with every residual writer of layer l zeroed except those in `live`."""
        sd = dict(self.sd)
        for m in WRITERS:
            if m not in live:
                for p in ("weight", "bias"):
                    sd[self.key(f"{m}.{p}")] = torch.zeros_like(self.sd[self.key(f"{m}.{p}")])
        if ff1_into_ff2:
            for p in ("linear1.weight", "linear1.bias", "linear2.weight", "linear2.bias"):
                sd[self.key(f"feed_forward2.{p}")] = self.sd[self.key(f"feed_forward1.{p}")]
            for p in ("weight", "bias"):
                sd[self.key(f"norm_feed_forward2.{p}")] = self.sd[self.key(f"norm_feed_forward1.{p}")]
        return sd

    def rounded(self, got, want, tol):
        """tol plus the rounding of the stored value: half an ulp of a bf16 output, nothing more for fp32."""
        return tol + half_bf16_ulp(got, want) if self.bf16 else tol

    # ---------------------------------------------------------------------------------------------- stages
    def check_pre_encode(self, r):
        ow = self.sd["pre_encode.out.weight"].float().view(self.d, self.C, self.F2).permute(0, 2, 1).reshape(self.d, -1)
        ob = self.sd["pre_encode.out.bias"].float()
        xs = torch.tensor(float(self.d)).sqrt() if self.xscaling else torch.tensor(1.0)  # sqrtf(d): fp32
        W = ow * xs  # the host's fold: fp32 products, then the bf16 rounding of the matrix
        W = (W.bfloat16() if self.bf16 else W).double()
        want, tol = linear(r.y2, torch.zeros_like(r.y2), W, (ob * xs).double())
        assert_within(r.x, want, tol, "pre_encode.out (x0) from the device y2, folded weights restated")
        # against the reference weights: bf16 keeps 8 significant bits (2^-8 relative), xscale and the fold 2u
        s64 = math.sqrt(self.d) if self.xscaling else 1.0
        W64, b64 = ow.double() * s64, ob.double() * s64
        want = r.y2 @ W64.t() + b64
        S = r.y2.abs() @ W64.abs().t() + b64.abs()
        K = r.y2.shape[1]
        assert_within(r.x, want, ((2.0 ** -8 if self.bf16 else 0.0) + (K + 8) * U) * S, "pre_encode.out vs the reference weights")

    def check_a(self, r, x_in, norm):
        want, e = ln_ref(x_in, self.vec(f"{norm}.weight"), self.vec(f"{norm}.bias"))
        assert_within(r.a, want, self.rounded(r.a, want, e), f"a = {norm}(x_in)")

    def check_h(self, r, ff):
        v, e = linear(r.a, torch.zeros_like(r.a), self.w(f"{ff}.linear1.weight"), self.vec(f"{ff}.linear1.bias"))
        want, e = swish_ref(v, e, self.bf16)
        assert_within(r.h, want, self.rounded(r.h, want, e), f"h = swish({ff}.linear1(a))")

    def ln_operand(self, x_in, norm):
        y, e = ln_ref(x_in, self.vec(f"{norm}.weight"), self.vec(f"{norm}.bias"))
        return operand(y, e, self.bf16)

    def check_qkv(self, r, x_in):
        A, dA = self.ln_operand(x_in, "norm_self_att")
        pu, pv = self.vec("self_attn.pos_bias_u").flatten(), self.vec("self_attn.pos_bias_v").flatten()
        bq = self.vec("self_attn.linear_q.bias")
        parts = [linear(A, dA, self.w("self_attn.linear_q.weight"), bq + pu, eb=U * (bq + pu).abs()),
                 linear(A, dA, self.w("self_attn.linear_q.weight"), bq + pv, eb=U * (bq + pv).abs()),
                 linear(A, dA, self.w("self_attn.linear_k.weight"), self.vec("self_attn.linear_k.bias")),
                 linear(A, dA, self.w("self_attn.linear_v.weight"), self.vec("self_attn.linear_v.bias"))]
        got = r.qkv.view(self.N, 4, self.H, self.dkp)
        assert torch.all(got[..., self.dk:] == 0), "qkv: a padding lane dk..dkp-1 of a head is not 0"
        for i, (name, (want, e)) in enumerate(zip(("q+u", "q+v", "k", "v"), parts)):
            g = got[:, i, :, :self.dk].reshape(self.N, self.d)
            assert_within(g, want, self.rounded(g, want, e), f"qkv part {i} ({name}) from norm_self_att(x_in)")

    def check_g(self, r, x_in):
        A, dA = self.ln_operand(x_in, "norm_conv")
        W = self.w("conv.pointwise_conv1.weight")
        b = self.vec("conv.pointwise_conv1.bias")
        d = self.d
        va, ea = linear(A, dA, W[:d], b[:d])
        vg, eg = linear(A, dA, W[d:], b[d:])
        want, e = glu_ref(va, ea, vg, eg, self.bf16)
        valid = (torch.arange(self.T2)[None, :] < r.ylen[:, None].long()).reshape(self.N)
        got = r.g.view(self.N, d)
        assert torch.all(got[~valid] == 0), "g: a frame >= encoded_len is not 0"
        assert_within(got[valid], want[valid], self.rounded(got[valid], want[valid], e[valid]),
                      "g = GLU(pointwise_conv1(norm_conv(x_in)))")

    def check_c(self, r):
        s = self.vec("conv.batch_norm.weight") / torch.sqrt(self.vec("conv.batch_norm.running_var") + 1e-5)
        taps = self.vec("conv.depthwise_conv.weight")[:, 0, :] * s[:, None]
        bias = (self.vec("conv.depthwise_conv.bias") - self.vec("conv.batch_norm.running_mean")) * s + self.vec("conv.batch_norm.bias")
        gt = r.g.transpose(1, 2)  # (B, d, T')
        pad = (self.ks - 1) // 2
        v = F.conv1d(gt, taps.unsqueeze(1), bias, padding=pad, groups=self.d).transpose(1, 2)
        S = F.conv1d(gt.abs(), taps.abs().unsqueeze(1), bias.abs(), padding=pad, groups=self.d).transpose(1, 2)
        want, e = swish_ref(v, (self.ks + 2) * U * S, self.bf16)
        assert_within(r.c, want, self.rounded(r.c, want, e), "c = swish(BN(depthwise_conv(g)))")

    def check_update(self, x, x_in, A, dA, W, b, alpha, K, what):
        v, e = linear(A, dA, W, b, K=K)
        inc = alpha * v
        want = x_in + inc
        assert_within(x, want, alpha * e + 2 * U * inc.abs() + f32_ulp(x, want), what)

    def check_ctx(self, r):
        check_ctx(r)


CASES = [  # feat_in, d_model, heads, conv_kernel_size, ff_expansion_factor, T, lengths, layers, xscaling
    (80, 64, 4, 31, 4, 515, [515, 300, 1], 1, True),      # T' = 129: one frame past a 128-frame tail tile; dk 16
    (80, 176, 4, 9, 4, 203, [203, 150, 0], 1, True),      # d % 64 != 0 (unfused only); dk 44 -> 64; runtime-K taps
    (80, 320, 5, 31, 2, 1021, [1021, 520], 1, True),      # fused tail with bnc = 160; T' = 256
    (80, 448, 7, 3, 4, 263, [263, 100], 1, False),        # bnc = 224; taps32 shift 14; no xscaling
    (80, 512, 4, 31, 4, 517, [517, 260, 9], 1, True),     # dk = 128: attention_tc128 inside a layer
    (80, 256, 4, 1, 8, 129, [129, 64], 2, True),          # kernel size 1; ff 8; the checks on layer 1
]
IDS = [f"d{c[1]}h{c[2]}k{c[3]}ff{c[4]}-T{c[5]}-B{len(c[6])}-L{c[7]}{'' if c[8] else '-noxscale'}" for c in CASES]
VALIDATION = [CASES[i] for i in (1, 2, 5)]
VALIDATION_IDS = [IDS[i] for i in (1, 2, 5)]


def run_layer(case, monkeypatch):
    c = case
    errors = []

    def check(fn, *args):
        try:
            fn(*args)
        except AssertionError as ex:
            errors.append(str(ex))

    r0 = Forward(c, c.weights(), False, monkeypatch)
    x_in = r0.x
    if c.L == 1:
        check(c.check_pre_encode, r0)
    check(c.check_a, r0, x_in, "norm_feed_forward2")
    check(c.check_h, r0, "feed_forward2")
    check(c.check_qkv, r0, x_in)
    check(c.check_ctx, r0)
    check(c.check_g, r0, x_in)
    check(c.check_c, r0)

    r = Forward(c, c.weights(live=("self_attn.linear_out",)), False, monkeypatch)
    ctx = r.ctx[..., :c.dk].reshape(c.N, c.d)
    check(c.check_update, r.x, x_in, ctx, torch.zeros_like(ctx), c.w("self_attn.linear_out.weight"),
          c.vec("self_attn.linear_out.bias"), 1.0, c.Dp, "x after linear_out (from the device ctx)")

    r = Forward(c, c.weights(live=("conv.pointwise_conv2",)), False, monkeypatch)
    cc = r.c.view(c.N, c.d)
    check(c.check_update, r.x, x_in, cc, torch.zeros_like(cc), c.w("conv.pointwise_conv2.weight"),
          c.vec("conv.pointwise_conv2.bias"), 1.0, c.d, "x after pointwise_conv2 (from the device c)")
    if c.bf16 and c.d % 64 == 0 and c.d <= 512:  # dw_pw_supported
        fused = Forward(c, c.weights(live=("conv.pointwise_conv2",)), True, monkeypatch)
        if not torch.equal(fused.x, r.x):
            bad = (fused.x != r.x).nonzero()
            errors.append(f"x after the fused conv tail differs from the two-kernel tail at {bad.shape[0]} elements, "
                          f"first {bad[:8].tolist()}")

    r = Forward(c, c.weights(live=("feed_forward2.linear2",)), False, monkeypatch)
    check(c.check_update, r.x, x_in, r.h, torch.zeros_like(r.h), c.w("feed_forward2.linear2.weight"),
          c.vec("feed_forward2.linear2.bias"), 0.5, c.dff, "x after feed_forward2 (from the device h)")

    # FF1's weights through FF2's slot: the stages checked as FF2's above
    rp = Forward(c, c.weights(live=("feed_forward2.linear2",), ff1_into_ff2=True), False, monkeypatch)
    check(c.check_a, rp, x_in, "norm_feed_forward1")
    check(c.check_h, rp, "feed_forward1")
    check(c.check_update, rp.x, x_in, rp.h, torch.zeros_like(rp.h), c.w("feed_forward1.linear2.weight"),
          c.vec("feed_forward1.linear2.bias"), 0.5, c.dff, "x after feed_forward1's weights in FF2's slot")

    r = Forward(c, c.weights(live=("feed_forward1.linear2",)), False, monkeypatch)
    if c.bf16 and c.l > 0:
        # FF1's operand came from layernorm_dual: two bf16 operands (its LayerNorm output and h) are unknown
        A, dA = c.ln_operand(x_in, "norm_feed_forward1")
        v, e = linear(A, dA, c.w("feed_forward1.linear1.weight"), c.vec("feed_forward1.linear1.bias"))
        hv, dh = operand(*swish_ref(v, e, True), True)
        check(c.check_update, r.x, x_in, hv, dh, c.w("feed_forward1.linear2.weight"), c.vec("feed_forward1.linear2.bias"),
              0.5, c.dff, "x after feed_forward1 (layer > 0, from layernorm_dual's operand)")
    elif not torch.equal(r.x, rp.x):
        bad = (r.x != rp.x).nonzero()
        errors.append(f"x after feed_forward1 differs from FF1's weights run in FF2's slot at {bad.shape[0]} elements, "
                      f"first {bad[:8].tolist()}")
    assert not errors, "\n".join(errors)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_bf16_layer_stage_by_stage(case, monkeypatch):
    run_layer(Case(*case, precision="bf16", seed=31), monkeypatch)


@pytest.mark.parametrize("case", VALIDATION, ids=VALIDATION_IDS)
def test_fp32_validation_layer_stage_by_stage(case, monkeypatch):
    """The fp32 CUDA-core path the bf16 path is compared against: fp32 activations and weights, accurate expf."""
    run_layer(Case(*case, precision="fp32_validate", seed=32), monkeypatch)
