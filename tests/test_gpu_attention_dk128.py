"""Attention heads wider than 64 (64 < dk <= 128, padded to 128 columns; csrc/attention_tc128.cu).

Kernel level through cfb_op_rel_attention against the torch restatement of the reference (test_gpu_attention.py), and
encoder level against the oracle for the shapes this opens up: d_model / n_heads = 1024 / 8, 512 / 4, 640 / 8, 768 / 8.
The two host tests at the end need no GPU."""
import ctypes

import pytest
import torch

import conformer_nemo_b200 as cn
from conformer_nemo_b200 import _lib
from oracle import conformer_oracle as oc

CFB_ERR_INVALID_ARG, CFB_ERR_UNSUPPORTED = 1, 2
DKP = 128


def make_case(B, T, H, dk, lens, seed, dtype, scale=1.0):
    """qkv (B T, 4 H 128) = [q+u | q+v | k | v], pos (2T-1, 2 H 128) with this layer's columns in the second half (the
    first half is a poison value), every head padded from dk to 128 columns with zeros; and the reference result."""
    from test_gpu_attention import torch_reference

    g = torch.Generator(device="cuda").manual_seed(seed)
    Dp = H * DKP
    parts = [(torch.randn(B, H, T, dk, generator=g, device="cuda") * scale).to(dtype).float() for _ in range(4)]
    p = (torch.randn(H, 2 * T - 1, dk, generator=g, device="cuda") * scale).to(dtype).float()
    qkv = torch.zeros(B * T, 4 * Dp, device="cuda")
    for i, t in enumerate(parts):
        blk = torch.zeros(B, T, H, DKP, device="cuda")
        blk[..., :dk] = t.permute(0, 2, 1, 3)
        qkv[:, i * Dp:(i + 1) * Dp] = blk.reshape(B * T, Dp)
    pos = torch.full((2 * T - 1, 2 * Dp), 7.0, device="cuda")
    pblk = torch.zeros(2 * T - 1, H, DKP, device="cuda")
    pblk[..., :dk] = p.permute(1, 0, 2)
    pos[:, Dp:] = pblk.reshape(2 * T - 1, Dp)
    lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
    return qkv, pos[:, Dp:], lens_t, torch_reference(*parts, p, lens_t), Dp


def run(use_tc, qkv, pos, lens_t, B, T, H, dk, dkp=DKP):
    """cfb_op_rel_attention into a NaN-filled context buffer; returns (rc, ctx)."""
    lib = _lib.load_library()
    dt = torch.bfloat16 if use_tc else torch.float32
    ctx = torch.full((B * T, H * dkp), float("nan"), device="cuda", dtype=dt)
    rc = lib.cfb_op_rel_attention(int(use_tc), ctypes.c_void_p(qkv.data_ptr()), ctypes.c_void_p(pos.data_ptr()),
                                  pos.stride(0), ctypes.c_void_p(ctx.data_ptr()), ctypes.c_void_p(lens_t.data_ptr()), B, T,
                                  H, dk, dkp, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, ctx


def err_stats(got, want):
    diff = (got.double() - want.double()).abs()
    return dict(max_abs=float(diff.max()), rel_l2=float(diff.norm() / want.double().norm().clamp_min(1e-30)),
                nan=int(torch.isnan(got).sum()))


def check_zeros(ctx, B, T, H, dk, lens):
    got = ctx.float().view(B, T, H, DKP)
    assert torch.all(got[..., dk:] == 0), "pad columns dk..127 must be exact zeros"
    for b, n in enumerate(lens):
        assert torch.all(got[b, n:] == 0), f"query rows past len[{b}] = {n} must be exact zeros"


T_GRID = [1, 21, 64, 65, 128, 129, 333, 700, 1100]  # key-tile edges, one tile, T on both sides of 512
DK_GRID = [66, 80, 96, 128]


def lengths_for(T, idx):
    """Three sequences: full, a tile edge, and 0 or 1 frames."""
    edge = [64, 65, 128, 129][idx % 4]
    return [T, min(T, edge), idx % 2]


@pytest.mark.gpu
@pytest.mark.parametrize("dk", DK_GRID)
@pytest.mark.parametrize("T", T_GRID)
def test_tc128_attention_matches_reference(T, dk):
    idx = T_GRID.index(T) + DK_GRID.index(dk)
    lens = lengths_for(T, idx)
    B, H = len(lens), 2
    qkv, pos, lens_t, want, Dp = make_case(B, T, H, dk, lens, 100 + idx, torch.bfloat16)
    rc, ctx = run(True, qkv.bfloat16(), pos.bfloat16(), lens_t, B, T, H, dk)
    assert rc == 0, _lib.last_error(None)
    st = err_stats(ctx.float().view(B, T, H, DKP)[..., :dk], want)
    # bf16 probabilities and bf16 output rounding: ~3 significant digits (the dk-64 kernel's bound)
    assert st["nan"] == 0 and st["rel_l2"] < 1.5e-2 and st["max_abs"] < 6e-2, st
    check_zeros(ctx, B, T, H, dk, lens)
    # the same launch again gives the same bits
    rc2, ctx2 = run(True, qkv.bfloat16(), pos.bfloat16(), lens_t, B, T, H, dk)
    assert rc2 == 0 and torch.equal(ctx, ctx2)


@pytest.mark.gpu
@pytest.mark.parametrize("dk", [66, 96])
def test_tc128_pad_columns_are_zero_whatever_v_holds(dk):
    """The kernel writes the pad columns dk..127 of ctx as zeros itself (linear_out reads them): with non-zero values in
    the pad columns of V, where P V would carry them through, the pad columns of ctx are still exact zeros and the head
    columns are unchanged."""
    B, T, H, lens = 2, 200, 2, [200, 77]
    qkv, pos, lens_t, want, Dp = make_case(B, T, H, dk, lens, 7, torch.bfloat16)
    rc, clean = run(True, qkv.bfloat16(), pos.bfloat16(), lens_t, B, T, H, dk)
    assert rc == 0, _lib.last_error(None)
    v = qkv[:, 3 * Dp:].view(B * T, H, DKP)
    v[..., dk:] = 3.0 + torch.randn_like(v[..., dk:])
    rc, ctx = run(True, qkv.bfloat16(), pos.bfloat16(), lens_t, B, T, H, dk)
    assert rc == 0, _lib.last_error(None)
    check_zeros(ctx, B, T, H, dk, lens)
    assert torch.equal(ctx, clean)


@pytest.mark.gpu
@pytest.mark.parametrize("dk", [66, 128])
@pytest.mark.parametrize("T", [21, 129, 333])
def test_simt_attention_at_dkp_128_matches_reference(T, dk):
    lens = lengths_for(T, T)
    B, H = len(lens), 2
    qkv, pos, lens_t, want, Dp = make_case(B, T, H, dk, lens, 200 + T, torch.float32)
    rc, ctx = run(False, qkv, pos, lens_t, B, T, H, dk)
    assert rc == 0, _lib.last_error(None)
    st = err_stats(ctx.view(B, T, H, DKP)[..., :dk], want)
    assert st["nan"] == 0 and st["max_abs"] < 2e-5, st
    check_zeros(ctx, B, T, H, dk, lens)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [4.0, 16.0, 40.0])
def test_tc128_position_term_has_headroom(scale):
    """The position term runs on fp16 operands into an fp16 accumulator with (q + v) / 16, summing 128 products per score:
    operands 4 ... 40 times larger than a normalised layer produces must stay finite and keep selecting the keys the fp32
    reference selects (the criterion of the dk-64 test)."""
    B, T, H, dk, lens = 2, 160, 2, 128, [160, 97]
    qkv, pos, lens_t, want, Dp = make_case(B, T, H, dk, lens, 5, torch.bfloat16, scale=scale)
    rc, ctx = run(True, qkv.bfloat16(), pos.bfloat16(), lens_t, B, T, H, dk)
    assert rc == 0, _lib.last_error(None)
    got = ctx.float().view(B, T, H, DKP)
    assert not torch.isnan(got).any() and not torch.isinf(got).any()
    for b, n in enumerate(lens):
        assert torch.all(got[b, n:] == 0)
        diff = (got[b, :n, :, :dk] - want[b, :n]).abs().amax(-1)
        ok = diff <= 0.02 * scale + 1e-3
        assert ok.float().mean().item() >= 0.97, (scale, b, ok.float().mean().item(), float(diff.max()))


# ---------------------------------------------------------------------------------------------------- encoder level
def build(cfg, sd, precision):
    enc = cn.ConformerEncoder(feat_in=cfg.feat_in, n_layers=cfg.n_layers, d_model=cfg.d_model, n_heads=cfg.n_heads,
                              precision=precision)
    missing, unexpected = enc.load_state_dict(sd, strict=False)
    assert not unexpected and all("num_batches_tracked" in m for m in missing), (missing, unexpected)
    return enc.cuda().eval()


def compare(got, want, enc_len):
    m = (torch.arange(want.shape[2])[None, :] < enc_len.cpu()[:, None].long())[:, None, :].expand_as(want)
    g, w = got.double()[m], want.double()[m]
    return dict(rel_l2=float((g - w).norm() / w.norm()), max_abs=float((g - w).abs().max()), nan=int(torch.isnan(got).sum()))


def zeros_behind(y, ylen):
    for b, n in enumerate(ylen.tolist()):
        assert n >= y.shape[2] or float(y[b, :, n:].abs().max()) == 0.0, (b, n)


# d_model, n_heads (dk), layers, T, lengths
WIDE = [
    (1024, 8, 2, 301, [301, 250, 1, 0]),
    (512, 4, 2, 513, [513, 300, 0, 5]),
    (640, 8, 1, 260, [260, 1, 199]),
    (768, 8, 1, 400, [400, 257, 0]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("row", WIDE, ids=[f"d{r[0]}h{r[1]}L{r[2]}" for r in WIDE])
def test_wide_heads_encoder_against_oracle(row):
    d, heads, layers, t, lens = row
    cfg = oc.EncoderConfig(feat_in=80, n_layers=layers, d_model=d, n_heads=heads)
    sd = oc.random_state_dict(cfg, 300 + d)
    x, length = oc.synthetic_batch(len(lens), 80, t, lens, seed=310 + d)
    g = torch.Generator().manual_seed(d)
    for b, n in enumerate(lens):  # non-zero features behind every utterance
        x[b, :, n:] = torch.randn(80, t - n, generator=g)
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    xd, ld = x.cuda(), length.cuda()
    for prec in ("fp32_validate", "bf16"):
        enc = build(cfg, sd, prec)
        enc.packed = False
        y, ylen = enc(audio_signal=xd, length=ld)
        torch.cuda.synchronize()
        assert torch.equal(ylen.cpu(), want_len), (prec, ylen, want_len)
        st = compare(y.cpu(), want, ylen)
        if prec == "fp32_validate":
            assert st["nan"] == 0 and st["rel_l2"] < 1e-4 and st["max_abs"] < 1e-4 * max(1.0, float(want.abs().max())), st
        else:
            assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
        zeros_behind(y, ylen)
    # bf16: the packed layout (attention over the tile table) equals the dense one bit for bit
    yd = y.clone()
    enc.packed = True
    yp, ylp = enc(audio_signal=xd, length=ld, length_host=lens)
    torch.cuda.synchronize()
    assert torch.equal(ylp, ylen)
    for b in range(len(lens)):
        n = int(ylen[b])
        assert torch.equal(yd[b, :, :n], yp[b, :, :n]), (b, float((yd[b, :, :n] - yp[b, :, :n]).abs().max()))
    zeros_behind(yp, ylp)
    # and CUDA-graph replay equals the eager launches bit for bit
    enc.packed = False
    enc.enable_cuda_graphs(True)
    for _ in range(2):  # capture, then replay
        yg, lg = enc(audio_signal=xd, length=ld)
        torch.cuda.synchronize()
        assert torch.equal(lg, ylen) and torch.equal(yg, yd)
    enc.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_xlarge_depth_against_oracle():
    """d_model 1024, 8 heads of 128, 24 layers, bf16."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=24, d_model=1024, n_heads=8)
    sd = oc.random_state_dict(cfg, 400)
    x, length = oc.synthetic_batch(2, 80, 1000, [1000, 613], seed=401)
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    enc = build(cfg, sd, "bf16")
    y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
    torch.cuda.synchronize()
    assert torch.equal(ylen.cpu(), want_len)
    st = compare(y.cpu(), want, ylen)
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    zeros_behind(y, ylen)


@pytest.mark.gpu
def test_xlarge_full_batch_runs_and_matches_oracle_on_a_sub_batch():
    """ConformerEncoder(feat_in=80, n_layers=24, d_model=1024, n_heads=8) on 32 x 20 s in bf16; two utterances of the
    batch against the oracle (utterances are independent given the padded extent)."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=24, d_model=1024, n_heads=8)
    sd = oc.random_state_dict(cfg, 410)
    B, T = 32, 2000
    g = torch.Generator().manual_seed(411)
    lens = torch.randint(200, T + 1, (B,), generator=g).tolist()
    lens[0], lens[3] = T, 777
    x, length = oc.synthetic_batch(B, 80, T, lens, seed=412)
    enc = build(cfg, sd, "bf16")
    y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
    torch.cuda.synchronize()
    assert y.shape == (B, 1024, 500) and int(torch.isnan(y).sum()) == 0
    want_len = torch.tensor([((n + 1) // 2 + 1) // 2 for n in lens], dtype=torch.int32)
    assert torch.equal(ylen.cpu(), want_len)
    zeros_behind(y, ylen)
    sub = [0, 3]
    want, wl = oc.encoder_forward(sd, cfg, x[sub], length[sub])
    assert torch.equal(ylen[sub].cpu(), wl)
    st = compare(y[sub].cpu(), want, ylen[sub])
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st


# ---------------------------------------------------------------------------------------------------- host (no GPU)
def test_tensor_core_attention_rejects_unsupported_head_padding():
    """The tensor-core path of cfb_op_rel_attention takes dkp 64 or 128 with 1 <= dk <= dkp; anything else is an argument
    error before anything is launched (so no device is needed to check it)."""
    lib = _lib.load_library()
    for dk, dkp in ((96, 96), (130, 128), (65, 64), (0, 128), (64, 256)):
        rc = lib.cfb_op_rel_attention(1, None, None, 0, None, None, 1, 16, 1, dk, dkp, None)
        assert rc == CFB_ERR_INVALID_ARG, (dk, dkp, rc)
        assert "dkp 64 or 128" in _lib.last_error(None)


def test_create_accepts_heads_up_to_128_wide():
    lib = _lib.load_library()
    cfg = _lib.CfbConfig(feat_in=80, n_layers=1, d_model=1024, feat_out=-1, subsampling_factor=4,
                         subsampling_conv_channels=-1, ff_expansion_factor=4, n_heads=4, conv_kernel_size=31,
                         xscaling=1, precision=0)
    handle = ctypes.c_void_p()
    assert lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle)) == CFB_ERR_UNSUPPORTED  # dk 256
    assert "head dimension > 128" in _lib.last_error(None)
    cfg.d_model, cfg.n_heads = 1008, 16  # dk 63: odd head widths stay rejected
    assert lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle)) == CFB_ERR_UNSUPPORTED
    assert "even" in _lib.last_error(None)
    cfg.d_model, cfg.n_heads = 1024, 8  # dk 128: past the configuration checks
    rc = lib.cfb_create(ctypes.byref(cfg), 0, ctypes.byref(handle))
    if torch.cuda.is_available():
        assert rc == 0 and handle.value, _lib.last_error(None)
        lib.cfb_destroy(handle)
    else:
        assert rc != 0 and not handle.value
        assert "no CPU fallback" in _lib.last_error(None)
