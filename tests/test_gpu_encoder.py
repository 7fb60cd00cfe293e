"""GPU: end-to-end parity of the CUDA encoder (through conformer_nemo_b200.ConformerEncoder -> ctypes -> libcfb.so)
against the oracle and the committed reference golden vectors.

Tolerances (BASELINE.json north_star): encoded_len bit-exact; on valid frames rel-L2 <= 1e-2 and max-abs <= 5e-2 in
bf16, <= 1e-4 in the fp32 validation mode; CTC greedy argmax agreement >= 99 %.
"""
import glob
import json
import os

import numpy as np
import pytest
import torch

import conformer_nemo_b200 as cn
from oracle import conformer_oracle as oc

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")) if "lengths" not in p and not os.path.basename(p).startswith(("ctc_head_", "ctc_collapse", "frontend_", "rnnt_")))


def load_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    cfg = oc.EncoderConfig(**meta["config"])
    stored = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    sd = stored if stored else oc.random_state_dict(cfg, meta["weight_seed"])
    return z, cfg, sd


def build(cfg: oc.EncoderConfig, sd, precision):
    enc = cn.ConformerEncoder(feat_in=cfg.feat_in, n_layers=cfg.n_layers, d_model=cfg.d_model, feat_out=cfg.feat_out,
                              subsampling_conv_channels=cfg.subsampling_conv_channels,
                              ff_expansion_factor=cfg.ff_expansion_factor, n_heads=cfg.n_heads, xscaling=cfg.xscaling,
                              conv_kernel_size=cfg.conv_kernel_size, untie_biases=cfg.untie_biases, precision=precision)
    missing, unexpected = enc.load_state_dict(sd, strict=False)
    assert not unexpected and all("num_batches_tracked" in m for m in missing), (missing, unexpected)
    return enc.cuda().eval()


def valid_mask(enc_len, t_out):
    return (torch.arange(t_out)[None, :] < enc_len.cpu()[:, None].long())


def compare(got, want, enc_len):
    """got/want (B, D, T') on cpu; metrics over valid frames only (SURVEY 4.7)."""
    m = valid_mask(enc_len, want.shape[2])[:, None, :].expand_as(want)
    g, w = got.double()[m], want.double()[m]
    return dict(rel_l2=float((g - w).norm() / w.norm()), max_abs=float((g - w).abs().max()),
                nan=int(torch.isnan(got).sum()))


def ctc_agreement(got, want, enc_len, seed=0, vocab=129):
    """ConvASRDecoder-equivalent 1x1 conv head (conv_asr.py:437-444) applied in fp32 to both outputs."""
    gen = torch.Generator().manual_seed(seed)
    d = want.shape[1]
    bound = (6.0 / (d + vocab)) ** 0.5  # xavier_uniform
    w = (torch.rand(vocab, d, generator=gen) * 2 - 1) * bound
    a = torch.einsum("vd,bdt->bvt", w, got.float()).argmax(1)
    b = torch.einsum("vd,bdt->bvt", w, want.float()).argmax(1)
    m = valid_mask(enc_len, want.shape[2])
    return float((a == b)[m].float().mean())


@pytest.mark.parametrize("name", CASES)
def test_fp32_validation_mode_matches_reference_golden(name):
    z, cfg, sd = load_case(name)
    enc = build(cfg, sd, "fp32_validate")
    x = torch.from_numpy(z["audio_signal"]).cuda()
    length = torch.from_numpy(z["length"]).cuda() if bool(z["has_length"]) else None
    y, ylen = enc(audio_signal=x, length=length)
    torch.cuda.synchronize()
    assert ylen.dtype == torch.int32 and np.array_equal(ylen.cpu().numpy(), z["encoded_len"])
    assert tuple(y.shape) == z["encoded"].shape and not y.is_contiguous() and y.transpose(1, 2).is_contiguous()
    st = compare(y.cpu(), torch.from_numpy(z["encoded"]), ylen)
    assert st["nan"] == 0 and st["rel_l2"] < 1e-4 and st["max_abs"] < 1e-4 * max(1.0, float(np.abs(z["encoded"]).max())), st
    # frames beyond encoded_len are written as zeros
    m = valid_mask(ylen, y.shape[2])[:, None, :].expand_as(y)
    assert torch.all(y.cpu()[~m] == 0)


@pytest.mark.parametrize("name", CASES)
def test_bf16_tensor_core_path_matches_reference_golden(name):
    z, cfg, sd = load_case(name)
    enc = build(cfg, sd, "bf16")
    x = torch.from_numpy(z["audio_signal"]).cuda()
    length = torch.from_numpy(z["length"]).cuda() if bool(z["has_length"]) else None
    y, ylen = enc(audio_signal=x, length=length)
    torch.cuda.synchronize()
    assert np.array_equal(ylen.cpu().numpy(), z["encoded_len"])
    want = torch.from_numpy(z["encoded"])
    st = compare(y.cpu(), want, ylen)
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    assert enc.last_launch_count() > 0


def test_intermediates_tc_vs_validation_single_layer():
    """Stage-by-stage comparison of the two CUDA paths on a 1-layer model (localises a faulty kernel)."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=1, d_model=176, n_heads=4)
    sd = oc.random_state_dict(cfg, 21)
    x, length = oc.synthetic_batch(2, 80, 203, [203, 150], seed=5)
    outs = {}
    for prec in ("fp32_validate", "bf16"):
        enc = build(cfg, sd, prec)
        enc(audio_signal=x.cuda(), length=length.cuda())
        torch.cuda.synchronize()
        dt = torch.float32 if prec == "fp32_validate" else torch.bfloat16
        # the bf16 path keeps the positional projections as fp16: the attention kernels' position-term MMA takes fp16 operands
        dts = {n: (torch.float16 if n == "pos" and prec == "bf16" else dt) for n in ("y1", "y2", "pe", "pos", "qkv", "ctx", "g", "c", "h")}
        outs[prec] = {n: enc.debug_buffer(2, 203, n).clone().view(d_).float().cpu() for n, d_ in dts.items()}
    report = {}
    for n in outs["bf16"]:
        a, b = outs["bf16"][n].double(), outs["fp32_validate"][n].double()
        report[n] = float((a - b).norm() / b.norm().clamp_min(1e-30))
    assert all(v < 2e-2 for v in report.values()), report


def test_large_config_mixed_lengths_against_oracle():
    """Conformer-L shaped layers (d=512, H=8, dk=64), 3 layers, mixed lengths incl. a very short row; oracle on CPU."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=3, d_model=512, n_heads=8)
    sd = oc.random_state_dict(cfg, 31)
    x, length = oc.synthetic_batch(4, 80, 1037, [1037, 640, 333, 9], seed=7)
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    for prec, tol_l2, tol_abs in (("fp32_validate", 1e-4, 1e-3), ("bf16", 1e-2, 5e-2)):
        enc = build(cfg, sd, prec)
        y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
        torch.cuda.synchronize()
        assert torch.equal(ylen.cpu(), want_len)
        st = compare(y.cpu(), want, ylen)
        assert st["nan"] == 0 and st["rel_l2"] <= tol_l2 and st["max_abs"] <= tol_abs, (prec, st)
        agree = ctc_agreement(y.cpu(), want, ylen)
        assert agree >= 0.99, (prec, agree)


def test_bf16_input_and_output_dtypes_and_repeatability():
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 41)
    x, length = oc.synthetic_batch(3, 80, 400, [400, 399, 120], seed=9)
    enc = build(cfg, sd, "bf16")
    y1, l1 = enc(audio_signal=x.cuda(), length=length.cuda())
    y2, l2 = enc(audio_signal=x.cuda(), length=length.cuda())
    torch.cuda.synchronize()
    assert torch.equal(y1, y2) and torch.equal(l1, l2)  # deterministic: no atomics, fixed schedule
    y3, _ = enc(audio_signal=x.cuda(), length=length.cuda(), out_dtype=torch.bfloat16)
    assert y3.dtype == torch.bfloat16
    assert float((y3.float() - y1).abs().max()) < 4e-2
    # int32 lengths are accepted like the reference accepts any integer dtype
    y4, l4 = enc(audio_signal=x.cuda(), length=length.int().cuda())
    assert torch.equal(l4, l1) and torch.equal(y4, y1)
    # different batch shape on the same handle (workspace regrows)
    xb, lb = oc.synthetic_batch(5, 80, 777, [777, 700, 512, 300, 41], seed=10)
    wb, wl = oc.encoder_forward(sd, cfg, xb, lb)
    yb, ylb = enc(audio_signal=xb.cuda(), length=lb.cuda())
    assert torch.equal(ylb.cpu(), wl)
    st = compare(yb.cpu(), wb, ylb)
    assert st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st


def test_cuda_graph_capture_of_forward():
    """cfb_forward is enqueue-only (no allocation / sync), so the whole forward can be captured in a CUDA graph."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 51)
    x, length = oc.synthetic_batch(2, 80, 320, [320, 200], seed=11)
    enc = build(cfg, sd, "bf16")
    xs, ls = x.cuda(), length.cuda()
    y_ref, _ = enc(audio_signal=xs, length=ls)  # warm-up: allocates workspace, packs weights
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y_cap, len_cap = enc(audio_signal=xs, length=ls)
    xs.copy_(torch.roll(x, 1, 0).cuda())
    ls.copy_(torch.roll(length, 1, 0).cuda())
    graph.replay()
    torch.cuda.synchronize()
    y_new, len_new = enc(audio_signal=xs, length=ls)
    torch.cuda.synchronize()
    assert torch.equal(len_cap, len_new)
    assert float((y_cap - y_new).abs().max()) == 0.0
    assert float((y_cap - y_ref).abs().max()) > 0.0


def test_enable_cuda_graphs_matches_eager_and_tracks_shapes():
    """ConformerEncoder.enable_cuda_graphs(): one captured graph per input shape, replayed on later calls; results
    are bit-identical to the eager launches, including length=None and a second shape."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 52)
    enc = build(cfg, sd, "bf16")
    cases = []
    for seed, (b, t, lens) in enumerate([(2, 320, [320, 200]), (2, 320, [100, 320]), (3, 200, [200, 150, 9])]):
        x, length = oc.synthetic_batch(b, 80, t, lens, seed=20 + seed)
        cases.append((x.cuda(), length.cuda()))
    eager = [tuple(v.clone() for v in enc(audio_signal=x, length=l)) for x, l in cases]
    eager_none = enc(audio_signal=cases[0][0], length=None)[0].clone()
    enc.enable_cuda_graphs(True)
    for rep in range(2):  # first pass captures, second pass replays
        for (x, l), (y0, l0) in zip(cases, eager):
            y, ylen = enc(audio_signal=x, length=l)
            torch.cuda.synchronize()
            assert torch.equal(ylen, l0)
            assert float((y - y0).abs().max()) == 0.0
        y, _ = enc(audio_signal=cases[0][0], length=None)
        assert float((y - eager_none).abs().max()) == 0.0
    assert len(enc._graphs) == 3
    enc.enable_cuda_graphs(False)
    y, _ = enc(audio_signal=cases[0][0], length=cases[0][1])
    assert float((y - eager[0][0]).abs().max()) == 0.0


def test_two_stream_micro_batching_is_bit_identical_to_separate_halves():
    """B >= 8: cfb_forward runs the batch as two half-batches on two streams (fork / join).  Utterances are independent
    and both halves see the same padded extent T, so the result must equal running the halves as separate calls bit
    for bit, encoded_len included -- eagerly and under graph replay."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 53)
    lens = [400, 333, 17, 256, 399, 1, 120, 64, 400, 250, 77]
    x, length = oc.synthetic_batch(len(lens), 80, 400, lens, seed=31)
    enc = build(cfg, sd, "bf16")
    xs, ls = x.cuda(), length.cuda()
    y, ylen = enc(audio_signal=xs, length=ls)
    torch.cuda.synchronize()
    b0 = (len(lens) + 1) // 2
    ya, la = (t.clone() for t in enc(audio_signal=xs[:b0].contiguous(), length=ls[:b0].contiguous()))  # B < 8: one stream
    yb, lb = (t.clone() for t in enc(audio_signal=xs[b0:].contiguous(), length=ls[b0:].contiguous()))
    torch.cuda.synchronize()
    assert torch.equal(ylen, torch.cat([la, lb]))
    assert float((y - torch.cat([ya, yb])).abs().max()) == 0.0
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    assert torch.equal(ylen.cpu(), want_len)
    st = compare(y.cpu(), want, ylen)
    assert st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    enc.enable_cuda_graphs(True)
    for _ in range(2):
        yg, lg = enc(audio_signal=xs, length=ls)
        torch.cuda.synchronize()
        assert torch.equal(lg, ylen) and float((yg - y).abs().max()) == 0.0


@pytest.mark.parametrize("seed", [0, 1, 2, 3, 4, 5])
def test_random_shapes_and_lengths_against_oracle(seed):
    """Seeded sweep over the shapes the kernels special-case: d_model 176 / 256 / 512 (head dims 44 / 64 / 32), batch
    sizes on both sides of the micro-batching threshold, T not a multiple of anything, utterances from 1 frame to full
    length, subsampling_conv_channels != d_model, feat_out projection."""
    rnd = np.random.RandomState(100 + seed)
    d_model, heads = [(176, 4), (256, 4), (512, 8), (256, 8), (512, 16), (176, 4)][seed]
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=d_model, n_heads=heads,
                           subsampling_conv_channels=[-1, 64, -1, 128, -1, 176][seed],
                           feat_out=[-1, -1, 320, -1, -1, 128][seed])
    sd = oc.random_state_dict(cfg, 60 + seed)
    b = int(rnd.choice([1, 3, 8, 11]))
    t = int(rnd.randint(9, 700))
    lens = [int(v) for v in rnd.randint(1, t + 1, size=b)]
    lens[int(rnd.randint(0, b))] = t
    x, length = oc.synthetic_batch(b, 80, t, lens, seed=70 + seed)
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    enc = build(cfg, sd, "bf16")
    y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
    torch.cuda.synchronize()
    assert torch.equal(ylen.cpu(), want_len), (lens, ylen, want_len)
    st = compare(y.cpu(), want, ylen)
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, (st, cfg, b, t, lens)
    for row, n in enumerate(want_len.tolist()):  # frames past encoded_len are written as zeros
        assert float(y[row, :, n:].abs().max()) == 0.0 if n < y.shape[2] else True


@pytest.mark.parametrize("name", ["large_d512", "char_d256", "tiny_d64"])
def test_fused_conv_tail_is_bit_identical_to_the_two_kernel_path(name, monkeypatch):
    """csrc/conv_tail.cu (depth-wise conv + pointwise_conv2 + residual in one kernel) is chosen by an occupancy
    heuristic; CFB_FUSED_TAIL=2 forces it, =0 forbids it.  Same arithmetic in the same order: identical bits, and
    both stay inside the golden tolerance."""
    z, cfg, sd = load_case(name)
    enc = build(cfg, sd, "bf16")
    x = torch.from_numpy(z["audio_signal"]).cuda()
    length = torch.from_numpy(z["length"]).cuda() if bool(z["has_length"]) else None
    monkeypatch.setenv("CFB_FUSED_TAIL", "2")
    y_fused, ylen = enc(audio_signal=x, length=length)
    n_fused = enc.last_launch_count()
    torch.cuda.synchronize()
    y_fused = y_fused.clone()
    monkeypatch.delenv("CFB_FUSED_TAIL")
    y_auto, _ = enc(audio_signal=x, length=length)
    n_auto = enc.last_launch_count()
    torch.cuda.synchronize()
    assert n_fused == n_auto - cfg.n_layers, (n_fused, n_auto)  # one launch fewer per layer (tiny batches: auto = split)
    assert torch.equal(y_fused, y_auto)
    st = compare(y_fused.float().cpu(), torch.from_numpy(z["encoded"]), ylen)
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st


def test_full_size_cfg2_properties_and_oracle_sample():
    """BASELINE.json configs[1] at its full size (Conformer-L: d_model 512, 17 layers, 8 heads; 32 utterances x 2000
    frames), mixed lengths.  Size-independent properties of the path -- utterances are independent given the padded
    extent -- are checked BITWISE on the whole batch (product configuration: two-stream micro-batches, fused conv tail,
    CTA-pair GEMMs, persistent attention), and two utterances are compared with the CPU oracle at full depth."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    sd = oc.random_state_dict(cfg, 5)
    B, T = 32, 2000
    g = torch.Generator().manual_seed(17)
    lens = torch.randint(200, T + 1, (B,), generator=g).tolist()
    lens[0], lens[3] = T, 777
    x, length = oc.synthetic_batch(B, 80, T, lens, seed=11)
    enc = build(cfg, sd, "bf16")
    xd, ld = x.cuda(), length.cuda()
    y, ylen = enc(audio_signal=xd, length=ld)
    y = y.clone()
    ylen = ylen.clone()
    torch.cuda.synchronize()
    assert int(torch.isnan(y).sum()) == 0
    # (1) encoded_len: (L + 1) // 2 twice, int32 (subsampling.py:272-282)
    want_len = torch.tensor([((n + 1) // 2 + 1) // 2 for n in lens], dtype=torch.int32)
    assert ylen.dtype == torch.int32 and torch.equal(ylen.cpu(), want_len)
    # (2) frames past encoded_len are zeros
    for b in (0, 3, 7):
        assert torch.all(y[b, :, int(want_len[b]):] == 0)
    # (3) permuting the utterances permutes the result, bit for bit (rows change micro-batch half and tile position)
    perm = torch.randperm(B, generator=g)
    yp, lp = enc(audio_signal=xd[perm.cuda()].contiguous(), length=ld[perm.cuda()].contiguous())
    assert torch.equal(lp.cpu(), want_len[perm]) and torch.equal(yp, y[perm.cuda()])
    # (4) an utterance's result does not depend on what the other utterances contain
    x2 = xd.clone()
    x2[5] = torch.flip(x2[5], dims=[0])
    y2, _ = enc(audio_signal=x2, length=ld)
    keep = [b for b in range(B) if b != 5]
    assert torch.equal(y2[keep], y[keep]) and not torch.equal(y2[5], y[5])
    # (5) ... nor on the batch size: the same two utterances alone (same padded extent T)
    ys, ls = enc(audio_signal=xd[[0, 3]].contiguous(), length=ld[[0, 3]].contiguous())
    ys = ys.clone()
    assert torch.equal(ys, y[[0, 3]])
    # (6) and those two against the CPU oracle at full depth
    want, wl = oc.encoder_forward(sd, cfg, x[[0, 3]], length[[0, 3]])
    assert torch.equal(ls.cpu(), wl)
    st = compare(ys.cpu(), want, ls)
    assert st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    assert ctc_agreement(ys.cpu(), want, ls) >= 0.99


def test_full_size_cfg4_properties_and_oracle_sample():
    """BASELINE.json configs[3] at full size (Conformer-CTC Medium: d_model 256, 18 layers, 4 heads; 256 x 400 frames):
    permutation equivariance bit for bit and 24 utterances against the CPU oracle."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=18, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 6)
    B, T = 256, 400
    g = torch.Generator().manual_seed(23)
    lens = torch.randint(40, T + 1, (B,), generator=g).tolist()
    lens[0], lens[1], lens[2] = T, 333, 41
    x, length = oc.synthetic_batch(B, 80, T, lens, seed=12)
    enc = build(cfg, sd, "bf16")
    y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
    y, ylen = y.clone(), ylen.clone()
    perm = torch.randperm(B, generator=g).cuda()
    yp, lp = enc(audio_signal=x.cuda()[perm].contiguous(), length=length.cuda()[perm].contiguous())
    assert torch.equal(lp, ylen[perm]) and torch.equal(yp, y[perm])
    n = 24  # ~1500 valid frames: one frame is < 0.1 % of the agreement statistic
    want, wl = oc.encoder_forward(sd, cfg, x[:n], length[:n])
    assert torch.equal(ylen[:n].cpu(), wl)
    st = compare(y[:n].cpu(), want, ylen[:n])
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    # a random-init 129-class head has many near-ties, and which frames flip depends on the head: over six heads the agreement
    # of this batch spreads over 0.989 ... 0.998 (the same with every build measured), so the statistic is their mean
    agree = [ctc_agreement(y[:n].cpu(), want, ylen[:n], seed=s) for s in range(6)]
    assert sum(agree) / len(agree) >= 0.99 and min(agree) >= 0.985, (agree, st)


def test_full_size_cfg5_long_form_bf16_against_fp32_validation_path():
    """BASELINE.json configs[4] at full size (1 x 5 min = 30000 frames, T' = 7500, Conformer-L): the CPU oracle needs
    minutes there, so the bf16 product path is compared with the library's fp32 CUDA-core validation path (itself
    pinned to 1e-4 against the reference at the sizes the oracle handles), plus encoded_len and repeatability."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    sd = oc.random_state_dict(cfg, 7)
    x, length = oc.synthetic_batch(1, 80, 30000, [29991], seed=13)
    enc = build(cfg, sd, "bf16")
    y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
    y = y.clone()
    assert ylen.tolist() == [((29991 + 1) // 2 + 1) // 2] and y.shape == (1, 512, 7500)
    y2, _ = enc(audio_signal=x.cuda(), length=length.cuda())
    assert torch.equal(y2, y)
    del enc
    ref = build(cfg, sd, "fp32_validate")
    w, wl = ref(audio_signal=x.cuda(), length=length.cuda())
    torch.cuda.synchronize()
    assert torch.equal(wl, ylen)
    st = compare(y.cpu(), w.cpu(), ylen)
    assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
    assert ctc_agreement(y.cpu(), w.cpu(), ylen) >= 0.99


def test_forward_many_runs_sub_batches_concurrently_and_bit_identically():
    """ConformerEncoder.forward_many: the sub-batches of a rank on side streams (graphs with private workspaces) give
    bit-identical results to running them one after the other, including two sub-batches of the same shape."""
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    sd = oc.random_state_dict(cfg, 53)
    enc = build(cfg, sd, "bf16")
    batches = []
    for seed, (b, t, lens) in enumerate([(3, 400, [400, 391, 350]), (2, 240, [240, 201]), (5, 120, [120, 99, 80, 64, 7]),
                                         (2, 240, [222, 240]), (1, 640, [640])]):
        x, length = oc.synthetic_batch(b, 80, t, lens, seed=30 + seed)
        batches.append((x.cuda(), length.cuda()))
    want = [tuple(o.clone() for o in enc(audio_signal=x, length=ln)) for x, ln in batches]
    enc.enable_cuda_graphs(True, max_shapes=8, private_workspaces=True)
    for _ in range(3):  # first pass captures, later passes replay
        got = enc.forward_many(batches, n_streams=3)
        torch.cuda.synchronize()
        assert len(got) == len(want)
        for (y, yl), (w, wl) in zip(got, want):
            assert torch.equal(yl, wl) and float((y - w).abs().max()) == 0.0
    workspaces = {e[5].data_ptr() for e in enc._graphs.values()}
    assert len(workspaces) == len(enc._graphs) == 4  # one private workspace per captured shape


def test_profile_report_from_eager_brackets_and_from_graph_nodes():
    """cfb_set_profiling brackets every launch with CUDA events; captured in a graph the brackets become event-record nodes
    that every replay re-records (what bench.py's per-kernel table is read from).  Both forms list the same launches, the
    calibration bracket around nothing included, and leave the result untouched."""
    z, cfg, sd = load_case("tiny_d64")
    enc = build(cfg, sd, "bf16")
    x = torch.from_numpy(z["audio_signal"]).cuda()
    length = torch.from_numpy(z["length"]).cuda()
    y0, _ = enc(audio_signal=x, length=length)
    y0 = y0.clone()
    enc.set_profiling(True)
    y1, _ = enc(audio_signal=x, length=length)
    eager = enc.profile_report()
    assert "(empty bracket)" in eager and eager["(empty bracket)"][0] == 1
    for label in ("subsample conv 2", "linear1+swish", "linear2", "rel-pos attention", "norm_out"):
        assert label in eager and eager[label][1] > 0.0, (label, eager)
    assert eager["linear2"][0] == 2 * cfg.n_layers and eager["rel-pos attention"][0] == cfg.n_layers
    assert torch.equal(y1, y0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        enc.set_profiling(True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            y2, _ = enc(audio_signal=x, length=length)
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
        nodes = enc.profile_report()
    enc.set_profiling(False)
    assert {k: v[0] for k, v in nodes.items()} == {k: v[0] for k, v in eager.items()}
    assert all(v[1] > 0.0 for v in nodes.values())
    assert torch.equal(y2, y0)


# The configuration surface cfb_create accepts beyond the shipped recipes: any feat_in <= 359 (odd ones pad the
# odd-f1 plane and leave a partial output tile in the second conv), subsampling channels C that leave a partial 64-channel
# chunk, head dimensions 48 / 40 / 36 / 4, d_model 1024 (LayerNorm at its widest, no fused conv tail, d_ff 4096), odd
# kernel sizes down to 1, ff_expansion_factor 1 and 3, and feat_out below and above d_model.
# feat_in, C, d_model, heads, layers, conv_kernel_size, ff_expansion_factor, feat_out, T, lengths
SURFACE = [
    (64, 8, 80, 2, 2, 31, 4, -1, 203, [203, 150]),
    (128, 24, 144, 4, 1, 3, 1, -1, 160, [160, 97, 0]),
    (81, 72, 48, 1, 2, 1, 3, -1, 333, [333, 1, 200]),
    (41, -1, 64, 16, 2, 31, 4, 8, 120, [120, 77]),
    (359, 8, 64, 4, 1, 31, 4, -1, 99, [99, 64, 33]),
    (80, 72, 1024, 16, 1, 31, 4, -1, 140, [140, 101]),
    (81, 24, 176, 4, 1, 3, 3, 640, 257, [257, 190, 2]),
    (41, 8, 96, 2, 2, 1, 1, -1, 400, [400, 311]),
]


@pytest.mark.parametrize("row", SURFACE, ids=[f"F{r[0]}-C{r[1]}-d{r[2]}h{r[3]}L{r[4]}-k{r[5]}-ff{r[6]}-out{r[7]}" for r in SURFACE])
def test_accepted_configuration_surface_against_oracle(row):
    feat_in, C, d, heads, layers, ks, ff, feat_out, t, lens = row
    cfg = oc.EncoderConfig(feat_in=feat_in, n_layers=layers, d_model=d, n_heads=heads, subsampling_conv_channels=C,
                           conv_kernel_size=ks, ff_expansion_factor=ff, feat_out=feat_out)
    sd = oc.random_state_dict(cfg, 80 + feat_in)
    x, length = oc.synthetic_batch(len(lens), feat_in, t, lens, seed=90 + feat_in)
    g = torch.Generator().manual_seed(feat_in)
    for b, n in enumerate(lens):  # non-zero features behind every utterance: the convolutions run over the padded batch
        x[b, :, n:] = torch.randn(feat_in, t - n, generator=g)
    want, want_len = oc.encoder_forward(sd, cfg, x, length)
    for prec in ("fp32_validate", "bf16"):
        enc = build(cfg, sd, prec)
        enc.packed = False
        y, ylen = enc(audio_signal=x.cuda(), length=length.cuda())
        torch.cuda.synchronize()
        assert torch.equal(ylen.cpu(), want_len), (prec, ylen, want_len)
        st = compare(y.cpu(), want, ylen)
        if prec == "fp32_validate":
            assert st["nan"] == 0 and st["rel_l2"] < 1e-4 and st["max_abs"] < 1e-4 * max(1.0, float(want.abs().max())), st
        else:
            assert st["nan"] == 0 and st["rel_l2"] <= 1e-2 and st["max_abs"] <= 5e-2, st
        m = valid_mask(ylen, y.shape[2])[:, None, :].expand_as(y)
        assert torch.all(y.cpu()[~m] == 0)
    if feat_out > 0 and feat_out != d:
        return  # out_proj runs dense batches only
    yd = y.clone()
    enc.packed = True
    yp, ylp = enc(audio_signal=x.cuda(), length=length.cuda(), length_host=lens)
    torch.cuda.synchronize()
    assert torch.equal(ylp, ylen)
    for b in range(len(lens)):
        n = int(ylen[b])
        assert torch.equal(yd[b, :, :n], yp[b, :, :n]), (b, float((yd[b, :, :n] - yp[b, :, :n]).abs().max()))
        assert n == yp.shape[2] or float(yp[b, :, n:].abs().max()) == 0.0
