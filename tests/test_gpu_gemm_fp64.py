"""GEMM kernels (cfb_op_gemm) against float64, element by element: every tcgen05 kernel instance -- gemm_tc_kernel
<128, 5>, <256, 3>, <256, 4> and the CTA-pair gemm_tc2_kernel -- with every fused epilogue, at shapes that give each
persistent CTA several tiles, with M / N / K tails, padded strides and masked rows; and the CUDA-core validation kernel
under the same bounds.

Operands are bf16 values, so every product is exact in float64 and the reference is the exact sum.  The per-element
bound is the fp32 accumulation error K 2^-24 sum|a w| (the tcgen05 accumulation order is not documented; this bound is
the one test_gpu_gemm.test_linear_bias has held up to K = 10240), carried through the epilogue's arithmetic (fp32
rounding, the slope of the activation, the error of tanh.approx.f32: 2^-10.987 by the PTX ISA), plus half a bf16 ulp
where the output is bf16 (round to nearest even).  Which kernel runs is pinned per case: the profiler's kernel name
must be the one gpu_util.expected_instance (a copy of launch_gemm_tc's choice) names."""
import json
import os
import re
import subprocess
import sys
import zlib

import pytest
import torch

from conformer_nemo_b200 import _lib
from gpu_util import expected_instance, op_gemm, tiles_per_cta

U = 2.0 ** -24          # fp32 unit roundoff
TANH_APPROX = 2.0 ** -10.987
ALPHA = 0.5             # residual scale (the feed-forward modules' 0.5)
SENTINEL = 12345.0      # residual-stream guard value: must survive

# Epilogue variants: (cfb epilogue, tensor-core output dtype, rows masked by lens).  The validation kernel runs each
# with an fp32 output.
VARIANTS = {
    "LINEAR_bf16": (_lib.EPI_LINEAR, torch.bfloat16, False),
    "LINEAR_f32": (_lib.EPI_LINEAR, torch.float32, False),
    "LINEAR_lens": (_lib.EPI_LINEAR, torch.float32, True),
    "SWISH": (_lib.EPI_SWISH, torch.bfloat16, False),
    "SWISH_lens": (_lib.EPI_SWISH, torch.bfloat16, True),
    "RELU": (_lib.EPI_RELU, torch.bfloat16, False),
    "RESID": (_lib.EPI_RESID, torch.float32, False),
    "QKV": (_lib.EPI_QKV, torch.bfloat16, False),
    "GLU": (_lib.EPI_GLU, torch.bfloat16, True),
}
ALL = ("LINEAR_bf16", "LINEAR_f32", "LINEAR_lens", "SWISH", "SWISH_lens", "RELU", "RESID", "GLU")
NO_GLU = tuple(v for v in ALL if v != "GLU")  # GLU needs N % 32 == 0
KERNELS = {"128x5": ("tc", 128, 5), "256x3": ("tc", 256, 3), "256x4": ("tc", 256, 4), "pair": ("tc2",)}

# (kernel, M, N, K, CFB_GEMM_2CTA, variants)
SHAPES = [
    ("128x5", 30000, 704, 176, None, ALL),           # 10 tiles per CTA, N tail (704 = 5.5 x 128), K tail (2.75 k-blocks)
    ("128x5", 30000, 352, 176, None, ("GLU",)),
    ("128x5", 30000, 384, 176, None, ("QKV",)),
    ("128x5", 1, 256, 8, None, ALL),                 # one row, one k-block mostly zero fill
    ("128x5", 1, 192, 8, None, ("QKV",)),
    ("128x5", 127, 200, 40, None, NO_GLU),           # bf16 box tail: 200 = 3 x 64 + 8
    ("256x3", 20000, 1024, 176, None, ALL),
    ("256x3", 20000, 768, 960, None, ("QKV",)),      # 15 k-blocks: the last 3-stage K
    ("256x4", 20000, 1024, 1000, None, ALL),         # 16 k-blocks: the first 4-stage K
    ("256x4", 20000, 768, 2000, None, ("QKV",)),
    ("pair", 19999, 2048, 512, None, ALL),           # the last pair's first CTA holds the M tail, its second none
    ("pair", 19999, 1536, 512, None, ("QKV",)),
    ("pair", 20100, 1024, 2000, "1", ALL),           # the last pair's second CTA partly filled
    ("pair", 20100, 768, 2000, "1", ("QKV",)),
    # cfg 2 (d_model 512, 8 heads, 17 layers, ~16000 frames a step) as the encoder calls them
    ("pair", 16000, 1536, 512, None, ("QKV",)),         # linear_qkv
    ("pair", 16000, 2048, 512, None, ("SWISH",)),       # feed_forward.linear1
    ("256x4", 16000, 512, 2048, None, ("RESID",)),      # feed_forward.linear2
    ("256x3", 16000, 512, 512, None, ("RESID",)),       # linear_out
    ("256x3", 16000, 1024, 512, None, ("GLU",)),        # pointwise_conv1
    ("pair", 999, 8704, 512, None, ("LINEAR_bf16",)),   # linear_pos of all 17 layers at once (2T - 1 = 999)
    ("256x4", 16000, 512, 5120, None, ("LINEAR_f32",)),  # pre_encode.out
]
CASES = [pytest.param(kern, M, N, K, mode, v, id=f"{kern}-{M}x{N}x{K}{'-2cta' if mode else ''}-{v}")
         for kern, M, N, K, mode, vs in SHAPES for v in vs]
# one multi-tile case per kernel is run three times: the bits must not change
REPEAT = {(30000, 704, 176), (20000, 1024, 176), (20000, 1024, 1000), (19999, 2048, 512)}

# small shapes for the CUDA-core validation kernel: (M, N, K, variants)
SIMT_SHAPES = [(1, 256, 8, ALL[1:]), (127, 200, 40, NO_GLU[1:]), (257, 704, 176, ALL[1:]), (1, 192, 8, ("QKV",)),
               (257, 384, 176, ("QKV",))]
SIMT_CASES = [pytest.param(M, N, K, v, id=f"{M}x{N}x{K}-{v}") for M, N, K, vs in SIMT_SHAPES for v in vs]


def instance_key(inst, variant):
    epi, dt, _ = VARIANTS[variant]
    return inst + (epi, dt == torch.float32)


# ------------------------------------------------------------------------------------------------------ CPU (no GPU)
def test_case_grid_reaches_every_instance_with_several_tiles_per_cta():
    """The grid runs all 28 non-conv instantiations (4 kernels x LINEAR bf16 / fp32, SWISH, RELU, RESID, QKV, GLU), each
    in at least one case where a CTA (a CTA pair) works through more than 2 tiles: the TMEM accumulator's double
    buffer wraps its phase, the staging boxes and the shared-memory bias buffer are reused across tiles."""
    most = {}
    for kern, M, N, K, mode, vs in SHAPES:
        inst = expected_instance(M, N, K, mode, 148)
        assert inst == KERNELS[kern], (kern, M, N, K, mode, inst)
        for v in vs:
            key = instance_key(inst, v)
            most[key] = max(most.get(key, 0), tiles_per_cta(M, N, inst, 148))
    combos = {(_lib.EPI_LINEAR, False), (_lib.EPI_LINEAR, True), (_lib.EPI_SWISH, False), (_lib.EPI_RELU, False),
              (_lib.EPI_RESID, True), (_lib.EPI_QKV, False), (_lib.EPI_GLU, False)}
    assert set(most) == {k + c for k in KERNELS.values() for c in combos}
    assert len(most) == 28
    few = {k: t for k, t in most.items() if t <= 2}
    assert not few, few


def test_instance_mirror_follows_the_dispatch_rules():
    """Spot checks of gpu_util.expected_instance on the rules of launch_gemm_tc: the small-M rule comes before
    CFB_GEMM_2CTA, the pair default is K <= 1024 and N >= 1536, and 256-wide tiles switch to 4 stages at 16 k-blocks."""
    assert expected_instance(1000, 1024, 512) == ("tc", 128, 5)        # 2 * 8 * 4 <= 148
    assert expected_instance(1000, 1024, 512, "1") == ("tc", 128, 5)   # small M wins over the forced pair
    assert expected_instance(16000, 2048, 512) == ("tc2",)
    assert expected_instance(16000, 2048, 512, "0") == ("tc", 256, 3)
    assert expected_instance(16000, 1024, 512) == ("tc", 256, 3)       # N < 1536
    assert expected_instance(16000, 2048, 1088) == ("tc", 256, 4)      # K > 1024, 17 k-blocks
    assert expected_instance(16000, 2048, 1088, "1") == ("tc2",)
    assert expected_instance(128, 19200, 512, "1") == ("tc", 256, 3)   # not small (2 * 75 > 148), but pairs need M > 128
    assert expected_instance(30000, 704, 176, "1") == ("tc", 128, 5)   # N % 256 != 0
    assert expected_instance(20000, 1024, 960) == ("tc", 256, 3)
    assert expected_instance(20000, 1024, 1000) == ("tc", 256, 4)


# ------------------------------------------------------------------------------------------------------ references
def half_ulp_bf16(x):
    """Half a bf16 ulp of |x| (8 significant bits): 2^(e - 9) for x in [2^(e-1), 2^e); 0 at 0."""
    _, e = torch.frexp(x)
    return torch.where(x > 0, torch.exp2((e - 9).double()), torch.zeros_like(x))


def glu_columns(N, device):
    """Accumulator columns of output column c in the [16 a | 16 gate] interleave cfb_finalize_weights builds."""
    c = torch.arange(N // 2, device=device)
    a = (c // 16) * 32 + c % 16
    return a, a + 16


def reference(variant, acc, e_acc, bias, bias2, x0, fast):
    """float64 value of the epilogue output and the bound on the kernel's error in front of the final bf16 rounding.
    acc: the exact A W^T, e_acc: the bound on the fp32 accumulation error.  fast: tanh.approx.f32 (the tensor-core
    instances); else accurate expf, whose 2 ulp plus the add and the division stay within 2^-21 of the result."""
    epi = VARIANTS[variant][0]
    b = bias.double()
    rnd = 2.0 ** -23 if fast else 2.0 ** -21
    if epi == _lib.EPI_QKV:
        dp = acc.shape[1] // 3
        v = torch.cat([acc[:, :dp], acc[:, :dp], acc[:, dp:]], 1) + torch.cat([b[:dp], bias2.double(), b[dp:]])
        e = torch.cat([e_acc[:, :dp], e_acc[:, :dp], e_acc[:, dp:]], 1)
        return v, e + U * (v.abs() + e)
    if epi == _lib.EPI_RESID:  # x + fmaf(alpha, acc, alpha * b), added in fp32
        inc = ALPHA * (acc + b)
        want = x0.double() + inc
        return want, ALPHA * e_acc + U * ((ALPHA * b).abs() + inc.abs() + want.abs())
    v = acc + b
    e_v = e_acc + U * (v.abs() + e_acc)  # acc + bias rounded to fp32
    if epi == _lib.EPI_LINEAR:
        return v, e_v
    if epi == _lib.EPI_RELU:
        return v.clamp_min(0.0), e_v
    if epi == _lib.EPI_SWISH:  # fast: h + h tanh(h), h = v / 2; silu' <= 1.1
        f = v * torch.sigmoid(v)
        return f, 1.1 * e_v + (0.5 * v.abs() * TANH_APPROX if fast else 0.0) + rnd * f.abs()
    ai, gi = glu_columns(acc.shape[1], acc.device)  # GLU, fast: a (1/2 + 1/2 tanh(g / 2)); sigmoid' <= 1/4
    a, g, ea, eg = v[:, ai], v[:, gi], e_v[:, ai], e_v[:, gi]
    s = torch.sigmoid(g)
    f = a * s
    return f, ea * s + a.abs() * (eg / 4 + (TANH_APPROX / 2 if fast else 0.0)) + ea * eg / 4 + rnd * f.abs()


def out_columns(variant, N):
    epi = VARIANTS[variant][0]
    return N + N // 3 if epi == _lib.EPI_QKV else N // 2 if epi == _lib.EPI_GLU else N


def make_inputs(M, N, K, variant, op_dtype, strided, seed):
    """bf16-valued operands (held in op_dtype), A and W optionally column slices of wider tensors (lda = ldw = K + 64)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    pad = 64 if strided else 0
    A = torch.randn(M, K + pad, generator=g, device="cuda").bfloat16().to(op_dtype)[:, :K]
    W = (torch.randn(N, K + pad, generator=g, device="cuda") / K ** 0.5).bfloat16().to(op_dtype)[:, :K]
    kw = dict(bias=torch.randn(N, generator=g, device="cuda") * 0.5)
    epi, _, masked = VARIANTS[variant]
    if epi == _lib.EPI_QKV:
        kw.update(bias2=torch.randn(N // 3, generator=g, device="cuda") * 0.5, qkv_dp=N // 3)
    if epi == _lib.EPI_RESID:
        kw.update(alpha=ALPHA)
    valid = None
    if masked:  # frames_per_seq does not divide 128; lens: a partial first sequence, an empty one, a full one, random
        F = 333 if M > 333 else max(1, (M + 2) // 3)
        n_seq = -(-M // F)
        lens = torch.randint(0, F + 1, (n_seq,), generator=g, device="cuda", dtype=torch.int32)
        lens[0] = F * 3 // 10
        lens[1:2] = 0
        lens[2:3] = F
        rows = torch.arange(M, device="cuda")
        valid = (rows % F) < lens[rows // F]
        kw.update(lens=lens, frames_per_seq=F)
    x0 = torch.randn(M, N, generator=g, device="cuda") if epi == _lib.EPI_RESID else None
    return A, W, kw, x0, valid


def guarded_out(M, cols, dt, x0):
    """out as a view into a larger buffer (ldo = cols + 64, 3 rows more) filled with NaN (the residual stream: a
    sentinel); x0 is the residual stream's initial value."""
    big = torch.full((M + 3, cols + 64), SENTINEL if x0 is not None else float("nan"), device="cuda", dtype=dt)
    if x0 is not None:
        big[:M, :cols] = x0
    return big, big[:M, :cols]


def bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def check_against_reference(got, variant, A, W, kw, x0, valid, fast):
    M, K = A.shape
    a64, w64 = A.double(), W.double()
    acc = a64 @ w64.t()
    e_acc = K * U * (a64.abs() @ w64.abs().t())
    want, bound = reference(variant, acc, e_acc, kw["bias"], kw.get("bias2"), x0, fast)
    g = got.double()
    assert torch.isfinite(g).all(), f"{int((~torch.isfinite(g)).sum())} non-finite elements, first {(~torch.isfinite(g)).nonzero()[:4].tolist()}"
    if valid is not None:  # masked rows are exactly 0
        nz = (g[~valid] != 0).any(1)
        assert not nz.any(), f"{int(nz.sum())} masked rows not zero, first {(~valid).nonzero().flatten()[nz.nonzero().flatten()[:4]].tolist()}"
        want, bound, g = want[valid], bound[valid], g[valid]
    if got.dtype == torch.bfloat16:
        bound = bound + half_ulp_bf16(torch.maximum(g.abs(), want.abs()))
    err = (g - want).abs()
    bad = err > bound
    if bad.any():
        ratio = err / bound.clamp_min(1e-300)
        i = int(ratio.argmax())
        r, c = divmod(i, ratio.shape[1])
        pytest.fail(f"{int(bad.sum())} of {bad.numel()} elements out of bound; worst |err|/bound {float(ratio.max()):.3f} at "
                    f"(valid row {r}, col {c}): got {float(g[r, c])!r} want {float(want[r, c])!r} bound {float(bound[r, c]):.3e}")


def check_guards(big, M, cols, resid):
    for name, region in (("guard columns", big[:M, cols:]), ("guard rows", big[M:])):
        untouched = (region == SENTINEL) if resid else torch.isnan(region)
        assert untouched.all(), f"{name}: {int((~untouched).sum())} elements written, first {(~untouched).nonzero()[:4].tolist()}"


KNAME = re.compile(r"gemm_tc_kernel<(\d+),(\d+),(\d+),(\w+),|gemm_tc2_kernel<(\d+),(\w+)>")


def launched_gemms(prof):
    """(kernel, [BN, STAGES,] epilogue, fp32 output) of every tensor-core GEMM in a profiler trace."""
    out = set()
    for e in prof.events():
        m = KNAME.search(e.name.replace(" ", ""))
        if m and m.group(1):
            out.add(("tc", int(m.group(1)), int(m.group(2)), int(m.group(3)), m.group(4) == "float"))
        elif m:
            out.add(("tc2", int(m.group(5)), m.group(6) == "float"))
    return out


def trace_cases():
    """Runs every case once, each in a profiler session of its own, and returns the GEMM kernels each one launched."""
    traced = {}
    for p in CASES:
        kern, M, N, K, mode, variant = p.values
        if mode is None:
            os.environ.pop("CFB_GEMM_2CTA", None)
        else:
            os.environ["CFB_GEMM_2CTA"] = mode
        epi, dt, _ = VARIANTS[variant]
        A, W, kw, x0, _ = make_inputs(M, N, K, variant, torch.bfloat16, False, 0)
        _, out = guarded_out(M, out_columns(variant, N), dt, x0)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            op_gemm(True, epi, A, W, out=out, **kw)
        traced[p.id] = sorted(launched_gemms(prof))
    return traced


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("kern,M,N,K,mode,variant", CASES)
def test_tensor_core_gemm_against_float64(kern, M, N, K, mode, variant, monkeypatch):
    if mode is None:
        monkeypatch.delenv("CFB_GEMM_2CTA", raising=False)
    else:
        monkeypatch.setenv("CFB_GEMM_2CTA", mode)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    inst = expected_instance(M, N, K, mode, sms)
    assert inst == KERNELS[kern], f"on {sms} SMs this shape runs {inst}, not the {kern} kernel the case is for"
    epi, dt, _ = VARIANTS[variant]
    seed = zlib.crc32(f"{M}x{N}x{K}-{variant}".encode())
    A, W, kw, x0, valid = make_inputs(M, N, K, variant, torch.bfloat16, variant == "RELU", seed)
    cols = out_columns(variant, N)
    big, out = guarded_out(M, cols, dt, x0)
    op_gemm(True, epi, A, W, out=out, **kw)
    check_guards(big, M, cols, x0 is not None)
    check_against_reference(out, variant, A, W, kw, x0, valid, fast=True)
    if M > 128:  # the first tile row again as an M = 128 problem, one tile per CTA of the 128-wide kernel
        assert expected_instance(128, N, K, mode, sms) == ("tc", 128, 5)
        _, out128 = guarded_out(128, cols, dt, None if x0 is None else x0[:128])
        op_gemm(True, epi, A[:128], W, out=out128, **kw)
        assert torch.equal(bits(out128), bits(out[:128])), "first 128 rows differ from the M = 128 run"
    if (M, N, K) in REPEAT:
        for _ in range(2):
            _, again = guarded_out(M, cols, dt, x0)
            op_gemm(True, epi, A, W, out=again, **kw)
            assert torch.equal(bits(again), bits(out)), "a repeated run changed bits"


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,variant", SIMT_CASES)
def test_validation_kernel_against_float64(M, N, K, variant):
    """The CUDA-core kernel the tensor-core path is validated against: fp32 operands holding bf16 values, fp32 output,
    accurate expf in the activations."""
    epi = VARIANTS[variant][0]
    A, W, kw, x0, valid = make_inputs(M, N, K, variant, torch.float32, variant == "RELU", zlib.crc32(f"simt-{M}x{N}x{K}-{variant}".encode()))
    cols = out_columns(variant, N)
    big, out = guarded_out(M, cols, torch.float32, x0)
    op_gemm(False, epi, A, W, out=out, **kw)
    check_guards(big, M, cols, x0 is not None)
    check_against_reference(out, variant, A, W, kw, x0, valid, fast=False)


@pytest.mark.gpu
def test_each_case_runs_the_kernel_the_mirror_names():
    """The kernel every case of test_tensor_core_gemm_against_float64 launches, by its name in a profiler trace, is the
    instance gpu_util.expected_instance names, so a change of launch_gemm_tc's choice cannot silently drop coverage.
    The traces are taken in a fresh process: in a process that has already run a profiler session and much untraced
    work since, later sessions were seen to come back without the kernel records."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.dirname(here), here, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__)], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    traced = json.loads(r.stdout.strip().splitlines()[-1])
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    wrong = {}
    for p in CASES:
        kern, M, N, K, mode, variant = p.values
        want = [list(instance_key(expected_instance(M, N, K, mode, sms), variant))]
        if traced[p.id] != want:
            wrong[p.id] = (traced[p.id], want)
    assert not wrong, wrong


if __name__ == "__main__":
    print(json.dumps(trace_cases()))
