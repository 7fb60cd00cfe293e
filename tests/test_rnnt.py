"""Transducer greedy decode (SURVEY.md 8(f) rank 4): oracle vs the reference's golden vectors and the host-side surface on
the CPU; the persistent CUDA decode (through cfb_op_rnnt_greedy) against the golden vectors and the oracle on the GPU."""
import glob
import os

import numpy as np
import pytest
import torch

import conformer_nemo_b200 as cn
from oracle import rnnt_oracle as ro

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "rnnt_*.npz")))


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    e, p, j, v = (int(a) for a in z["dims"])
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(e, p, j, v, int(z["weight_seed"]), float(z["blank_bias"]))
    checksum = float(sum(w.double().sum() for w in list(dec_sd.values()) + list(joint_sd.values())))
    assert abs(checksum - float(z["weight_checksum"])) < 1e-6
    ms = int(z["max_symbols"])
    return dict(dims=(e, p, j, v), dec_sd=dec_sd, joint_sd=joint_sd, x=torch.from_numpy(z["encoder_output"]),
                lens=torch.from_numpy(z["encoded_lengths"]), max_symbols=None if ms < 0 else ms,
                activation=str(z["activation"]), n=z["n_tokens"], tokens=z["tokens"], timesteps=z["timesteps"],
                scores=z["scores"], h=z["h"], c=z["c"])


def build_modules(dims, dec_sd, joint_sd, activation, max_symbols, device=None):
    e, p, j, v = dims
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=p, pred_rnn_layers=1, dropout=0.1), vocab_size=v)
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=e, pred_hidden=p, joint_hidden=j, activation=activation, dropout=0.1),
                         num_classes=v)
    dec.load_state_dict(dec_sd, strict=True)
    joint.load_state_dict(joint_sd, strict=True)
    if device is not None:
        dec, joint = dec.to(device), joint.to(device)
    return dec, joint, cn.GreedyBatchedRNNTInfer(dec, joint, blank_index=v, max_symbols_per_step=max_symbols)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    g = load(name)
    res = ro.rnnt_greedy_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["max_symbols"], g["activation"], True)
    for b, r in enumerate(res):
        n = int(g["n"][b])
        assert r.tokens == g["tokens"][b, :n].tolist()          # bit-exact: integer work
        assert r.timesteps == g["timesteps"][b, :n].tolist()
        assert abs(r.score - float(g["scores"][b])) <= 1e-4 * max(1.0, abs(float(g["scores"][b])))
        assert float((r.h - torch.from_numpy(g["h"][b])).abs().max()) <= 2e-6
        assert float((r.c - torch.from_numpy(g["c"][b])).abs().max()) <= 2e-6


def test_oracle_matches_live_reference_when_mounted():
    from oracle import reference_loader as rl

    if not rl.reference_available():
        pytest.skip("reference tree not mounted")
    import warnings

    dec_cls, joint_cls, greedy_cls = rl.load_reference_rnnt_classes()
    dims = (40, 48, 44, 25)
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=11, blank_bias=0.7)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dec = dec_cls(prednet=dict(pred_hidden=48, pred_rnn_layers=1, dropout=0.1), vocab_size=25)
    joint = joint_cls(jointnet=dict(encoder_hidden=40, pred_hidden=48, joint_hidden=44, activation="relu", dropout=0.1),
                      num_classes=25)
    dec.load_state_dict(dec_sd, strict=True)
    joint.load_state_dict(joint_sd, strict=True)
    x = torch.randn(4, 40, 30, generator=torch.Generator().manual_seed(5))
    lens = torch.tensor([30, 21, 30, 2])
    (hyps,) = greedy_cls(dec, joint, blank_index=25, max_symbols_per_step=4)(encoder_output=x, encoded_lengths=lens)
    res = ro.rnnt_greedy_decode(x, lens, dec_sd, joint_sd, 4, "relu", True)
    for h, r in zip(hyps, res):
        assert h.y_sequence.tolist() == r.tokens and list(h.timestep) == r.timesteps
        assert abs(h.score - r.score) <= 1e-4


def test_sample_level_greedy_of_the_reference_gives_the_batched_hypotheses():
    """decoding.strategy = greedy (one utterance at a time, rnnt_greedy_decoding.py:262-355) and greedy_batch agree on
    tokens, timesteps and scores -- the premise of serving both through the one batched kernel."""
    from oracle import reference_loader as rl

    if not rl.reference_available():
        pytest.skip("reference tree not mounted")
    import warnings

    dec_cls, joint_cls, batched_cls = rl.load_reference_rnnt_classes()
    sample_cls = rl.load_reference_sample_greedy_class()
    g = load("rnnt_tiny")
    e, p, j, v = g["dims"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dec = dec_cls(prednet=dict(pred_hidden=p, pred_rnn_layers=1, dropout=0.1), vocab_size=v)
    joint = joint_cls(jointnet=dict(encoder_hidden=e, pred_hidden=p, joint_hidden=j, activation=g["activation"], dropout=0.1),
                      num_classes=v)
    dec.load_state_dict(g["dec_sd"], strict=True)
    joint.load_state_dict(g["joint_sd"], strict=True)
    (a,) = sample_cls(dec, joint, blank_index=v, max_symbols_per_step=g["max_symbols"])(encoder_output=g["x"],
                                                                                      encoded_lengths=g["lens"])
    for b, h in enumerate(a):
        n = int(g["n"][b])
        assert h.y_sequence.tolist() == g["tokens"][b, :n].tolist() and list(h.timestep) == g["timesteps"][b, :n].tolist()
        assert abs(h.score - float(g["scores"][b])) <= 1e-3
        assert (h.dec_state is None) == (n == 0)


@pytest.mark.parametrize("name", CASES)
def test_one_utterance_at_a_time_gives_the_reference_batched_golden(name):
    """The premise of test_sample_level_greedy_of_the_reference_gives_the_batched_hypotheses without the reference tree:
    decoding each utterance alone (decoding.strategy = greedy) reproduces the reference's stored greedy_batch
    hypotheses -- tokens and timesteps exactly, scores to fp32 rounding."""
    g = load(name)
    for b in range(g["x"].shape[0]):
        (r,) = ro.rnnt_greedy_decode(g["x"][b:b + 1], g["lens"][b:b + 1], g["dec_sd"], g["joint_sd"], g["max_symbols"],
                                     g["activation"], True)
        n = int(g["n"][b])
        assert r.tokens == g["tokens"][b, :n].tolist() and r.timesteps == g["timesteps"][b, :n].tolist(), b
        assert abs(r.score - float(g["scores"][b])) <= 1e-4 * max(1.0, abs(float(g["scores"][b]))), b


def test_oracle_per_utterance_independence():
    g = load("rnnt_bpe128")
    full = ro.rnnt_greedy_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["max_symbols"], g["activation"], False)
    for b in (0, 4, 8):
        alone = ro.rnnt_greedy_decode(g["x"][b:b + 1], g["lens"][b:b + 1], g["dec_sd"], g["joint_sd"], g["max_symbols"],
                                      g["activation"], False)[0]
        assert alone.tokens == full[b].tokens and alone.timesteps == full[b].timesteps


def test_module_surface_and_errors():
    dec, joint, greedy = build_modules((48, 64, 56, 30), *ro.random_rnnt_state_dicts(48, 64, 56, 30, 0), "relu", 5)
    assert list(dec.state_dict()) == ["prediction.embed.weight", "prediction.dec_rnn.lstm.weight_ih_l0",
                                      "prediction.dec_rnn.lstm.weight_hh_l0", "prediction.dec_rnn.lstm.bias_ih_l0",
                                      "prediction.dec_rnn.lstm.bias_hh_l0"]
    assert list(joint.state_dict()) == ["pred.weight", "pred.bias", "enc.weight", "enc.bias", "joint_net.2.weight",
                                        "joint_net.2.bias"]
    assert joint.num_classes_with_blank == 31 and dec.blank_idx == 30
    with pytest.raises(ValueError):  # rnnt.py:1023-1024
        cn.RNNTJoint(jointnet=dict(encoder_hidden=48, pred_hidden=64, joint_hidden=56, activation="gelu"), num_classes=30)
    with pytest.raises(ValueError):  # rnnt.py:754-755
        cn.RNNTJoint(jointnet=dict(encoder_hidden=48, pred_hidden=64, joint_hidden=56, activation="relu"), num_classes=30,
                     fuse_loss_wer=True)
    with pytest.raises(NotImplementedError):
        cn.RNNTDecoder(prednet=dict(pred_hidden=64, pred_rnn_layers=2), vocab_size=30)
    with pytest.raises(ValueError):
        cn.GreedyBatchedRNNTInfer(dec, joint, blank_index=0)
    with pytest.raises(RuntimeError):  # no CPU path
        greedy(encoder_output=torch.zeros(1, 48, 4), encoded_lengths=torch.tensor([4]))
    with pytest.raises(NotImplementedError):  # rnnt_greedy_decoding.py:461-462
        greedy(encoder_output=torch.zeros(1, 48, 4), encoded_lengths=torch.tensor([4]), partial_hypotheses=[])


# ---------------------------------------------------------------------------------------------------------------- GPU

def _decode_gpu(greedy, x, lens):
    (hyps,) = greedy(encoder_output=x.cuda(), encoded_lengths=lens.cuda())
    return hyps


TIES = {"n": 0}  # utterances accepted at an oracle arg-max tie in this session (printed by the summary test)


def _compare(hyps, want, score_tol=2e-4, state_tol=2e-5):
    """tokens / timesteps exact; scores and states to fp32 rounding.  `want`: list of oracle results."""
    bad = []
    for b, (h, r) in enumerate(zip(hyps, want)):
        div = ro.first_divergence(h.y_sequence.tolist(), list(h.timestep), r)
        if div is not None:
            # Not a failure only if the oracle itself is undecided AT THE DECISION THAT DIFFERS (blank or symbol): its top-1 /
            # top-2 joint outputs there are within fp32 summation-order noise (the oracle's arithmetic depends on the host
            # CPU's BLAS kernels, the kernel's does not), after which an autoregressive decode continues differently.
            if div[1] < 2e-6:
                TIES["n"] += 1
                print(f"[rnnt tie] utterance {b}: decision {div[0]} differs at an oracle margin of {div[1]:.2e}")
            else:
                bad.append(b)
            continue
        assert abs(h.score - r.score) <= score_tol * max(1.0, abs(r.score)), (b, h.score, r.score)
        if h.dec_state is not None:
            assert float((h.dec_state[0][0] - r.h).abs().max()) <= state_tol
            assert float((h.dec_state[1][0] - r.c).abs().max()) <= state_tol
    return bad


def test_first_divergence_judges_the_decision_that_differs():
    """ADVICE r1: the tie allowance must look at the oracle's margin of the decision that differs, blanks included."""
    r = ro.RNNTGreedyResult(tokens=[5, 7], timesteps=[0, 2], length=3, max_symbols=2, blank=9)
    # oracle decisions: (0,0,5) (0,1,blank) (1,0,blank) (2,0,7) (2,1,blank)
    r.decision_margins = [1.0, 1e-7, 0.5, 3e-7, 0.25]
    assert ro.decisions(r.tokens, r.timesteps, 3, 2, 9) == [(0, 0, 5), (0, 1, 9), (1, 0, 9), (2, 0, 7), (2, 1, 9)]
    assert ro.first_divergence([5, 7], [0, 2], r) is None
    assert ro.first_divergence([5, 4, 7], [0, 0, 2], r) == (1, 1e-7)   # a symbol where the oracle chose blank: its blank margin
    assert ro.first_divergence([5], [0], r) == (3, 3e-7)               # a blank where the oracle emitted
    assert ro.first_divergence([5, 7], [0, 1], r) == (2, 0.5)          # same tokens, other frame: a REAL difference
    assert ro.first_divergence([6, 7], [0, 2], r) == (0, 1.0)
    # two symbols at a frame with max_symbols = 2: no blank decision follows them
    assert ro.decisions([1, 2], [0, 0], 1, 2, 9) == [(0, 0, 1), (0, 1, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_gpu_matches_reference_golden(name):
    g = load(name)
    _, _, greedy = build_modules(g["dims"], g["dec_sd"], g["joint_sd"], g["activation"], g["max_symbols"], "cuda")
    hyps = _decode_gpu(greedy, g["x"], g["lens"])
    for b, h in enumerate(hyps):
        n = int(g["n"][b])
        assert h.y_sequence.dtype == torch.int64
        assert h.y_sequence.tolist() == g["tokens"][b, :n].tolist()      # the reference's own tokens, bit-exact
        assert list(h.timestep) == g["timesteps"][b, :n].tolist()
        assert int(h.length) == int(g["lens"][b])
        if n:
            assert float((h.dec_state[0][0] - torch.from_numpy(g["h"][b])).abs().max()) <= 2e-5
            assert float((h.dec_state[1][0] - torch.from_numpy(g["c"][b])).abs().max()) <= 2e-5
    # scores: the reference log-normalises on the CPU only (rnnt_greedy_decoding.py:181-183); the CUDA branch sums raw logits
    raw = ro.rnnt_greedy_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["max_symbols"], g["activation"], False)
    assert _compare(hyps, raw) == []


@pytest.mark.gpu
@pytest.mark.parametrize("dims,B,T,max_symbols,blank_bias,seed", [
    ((512, 640, 640, 1024), 6, 90, 30, 1.05, 21),      # the Conformer-Transducer sizes (configs/conformer_transducer_bpe.yaml)
    ((256, 320, 320, 128), 11, 70, 5, 1.2, 22),
    ((176, 320, 320, 28), 7, 64, 10, 1.3, 23),        # char vocabulary: fewer joint rows than CTAs
])
def test_gpu_matches_oracle_seeded(dims, B, T, max_symbols, blank_bias, seed):
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=seed, blank_bias=blank_bias)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, dims[0], T, generator=gen)
    lens = torch.randint(1, T + 1, (B,), generator=gen)
    lens[0] = T
    _, _, greedy = build_modules(dims, dec_sd, joint_sd, "relu", max_symbols, "cuda")
    hyps = _decode_gpu(greedy, x, lens)
    want = ro.rnnt_greedy_decode(x, lens, dec_sd, joint_sd, max_symbols, "relu", False)
    assert sum(len(r.tokens) for r in want) > B  # the case does emit
    assert _compare(hyps, want) == []


@pytest.mark.gpu
def test_gpu_bf16_encoder_output_and_token_buffer_growth():
    dims = (64, 96, 80, 128)
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=31, blank_bias=0.6)
    x = torch.randn(5, 64, 48, generator=torch.Generator().manual_seed(31)).bfloat16()
    lens = torch.tensor([48, 40, 33, 48, 7])
    _, _, greedy = build_modules(dims, dec_sd, joint_sd, "relu", 12, "cuda")
    want = ro.rnnt_greedy_decode(x.float(), lens, dec_sd, joint_sd, 12, "relu", False)
    assert _compare(_decode_gpu(greedy, x, lens), want) == []
    # a token buffer that is too small is detected (flag) and the decode repeated with room for every symbol
    out = greedy.decode_arrays(x.cuda(), lens.cuda(), max_tokens=3)
    assert int(out["flags"].cpu()) == 1
    assert out["n_tokens"].cpu().tolist() == [len(r.tokens) for r in want]


@pytest.mark.gpu
def test_gpu_full_size_properties():
    """BASELINE cfg 3 sizes (transducer-large decoder on 32 x T' = 500 frames): decoding an utterance alone, in another
    batch order or in a batch of more than 128 utterances (several launches) gives bit-identical hypotheses; lengths bound
    the timesteps; at most max_symbols per frame."""
    dims = (512, 640, 640, 1024)
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=41, blank_bias=1.2)
    gen = torch.Generator().manual_seed(41)
    B, T = 32, 500
    x = torch.randn(B, 512, T, generator=gen)
    lens = torch.randint(50, T + 1, (B,), generator=gen)
    lens[3] = T
    _, _, greedy = build_modules(dims, dec_sd, joint_sd, "relu", 30, "cuda")
    hyps = _decode_gpu(greedy, x, lens)
    key = lambda h: (h.y_sequence.tolist(), list(h.timestep), h.score)
    perm = torch.randperm(B, generator=gen)
    hp = _decode_gpu(greedy, x[perm], lens[perm])
    for i, src in enumerate(perm.tolist()):
        assert key(hp[i])[:2] == key(hyps[src])[:2]
    for b in (0, 3, 17):
        assert key(_decode_gpu(greedy, x[b:b + 1], lens[b:b + 1])[0])[:2] == key(hyps[b])[:2]
    for b, h in enumerate(hyps):
        ts = np.asarray(h.timestep)
        if len(ts):
            assert ts.max() < int(lens[b]) and (np.diff(ts) >= 0).all() and np.bincount(ts).max() <= 30
    assert sum(len(h.timestep) for h in hyps) > 20 * B
    # oracle on a sample of utterances at the full sizes
    want = ro.rnnt_greedy_decode(x[:3], lens[:3], dec_sd, joint_sd, 30, "relu", False)
    assert _compare(hyps[:3], want) == []
    # > 128 utterances: the host entry point splits the batch into launches of 128
    reps = 9
    big = _decode_gpu(greedy, x[:, :, :60].repeat(reps, 1, 1), torch.clamp(lens, max=60).repeat(reps))
    for i in range(B, reps * B):
        assert key(big[i])[:2] == key(big[i % B])[:2]


@pytest.mark.gpu
def test_gpu_transducer_pipeline_waveform_to_hypotheses():
    """The whole transducer inference path on the device: collation service -> log-mel kernels -> encoder kernels ->
    greedy decode kernel; the decode is checked against the oracle fed with the SAME encoder output, the lengths against
    the encoder's."""
    from oracle import conformer_oracle as oc
    from oracle import frontend_oracle as fo

    x, lengths = fo.synthetic_waveforms(5, 32000, [32000, 20000, 9000, 32000, 16000], seed=7)
    svc = cn.CollationService([int(v) for v in lengths], lambda i: (x[i, :int(lengths[i])], torch.zeros(0, dtype=torch.int64)),
                              max_batch=8, bucket_frames=400, device="cuda")
    pre = cn.AudioToMelSpectrogramPreprocessor(sample_rate=16000, normalize="per_feature", window_size=0.025,
                                               window_stride=0.01, window="hann", features=80, n_fft=512, dither=0.0,
                                               pad_to=0).cuda()
    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    enc.load_state_dict(oc.random_state_dict(cfg, 4), strict=False)
    enc = enc.cuda().eval()
    dims = (256, 320, 320, 128)
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=51, blank_bias=0.4)
    _, _, greedy = build_modules(dims, dec_sd, joint_sd, "relu", 10, "cuda")
    seen = 0
    for batch in svc:
        svc.wait(batch)
        feats, flen = pre(input_signal=batch.audio_signal, length=batch.audio_lengths)
        # the service knows the lengths on the host: ragged sub-batches take the packed forward, which must equal the dense one
        enc.packed = False
        dense, dense_len = enc(audio_signal=feats, length=flen)
        dense = dense.clone()
        enc.packed = "auto"
        assert batch.feature_lengths_host() == flen.cpu().tolist()
        encoded, elen = enc(audio_signal=feats, length=flen, length_host=batch.feature_lengths_host())
        assert torch.equal(elen, dense_len)
        for row, n in enumerate(elen.cpu().tolist()):
            assert torch.equal(encoded[row, :, :n], dense[row, :, :n])
        (hyps,) = greedy(encoder_output=encoded, encoded_lengths=elen)
        want = ro.rnnt_greedy_decode(encoded.float().cpu(), elen.cpu(), dec_sd, joint_sd, 10, "relu", False)
        assert _compare(hyps, want) == []
        for h, n in zip(hyps, elen.cpu().tolist()):
            assert int(h.length) == n and (len(h.timestep) == 0 or max(h.timestep) < n)
        seen += len(hyps)
    assert seen == 5


_CLUSTER_SCRIPT = r"""
import os, sys, torch
sys.path.insert(0, os.environ["CFB_TEST_ROOT"])
sys.path.insert(0, os.path.join(os.environ["CFB_TEST_ROOT"], "tests"))
import test_rnnt as t
from oracle import rnnt_oracle as ro
dims = (512, 640, 640, 1024)
dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=61, blank_bias=1.1)
gen = torch.Generator().manual_seed(61)
x = torch.randn(7, 512, 120, generator=gen)
lens = torch.tensor([120, 97, 120, 64, 33, 2, 120])
_, _, greedy = t.build_modules(dims, dec_sd, joint_sd, "relu", 30, "cuda")
want = ro.rnnt_greedy_decode(x, lens, dec_sd, joint_sd, 30, "relu", False)
assert sum(len(r.tokens) for r in want) > 20
os.environ["CFB_RNNT_CLUSTER"] = "0"
assert t._compare(t._decode_gpu(greedy, x, lens), want) == []
os.environ["CFB_RNNT_CLUSTER"] = "1"
assert t._compare(t._decode_gpu(greedy, x, lens), want) == []
g = t.load("rnnt_bpe128")  # sizes where some ranks of a cluster own no row
_, _, greedy = t.build_modules(g["dims"], g["dec_sd"], g["joint_sd"], g["activation"], g["max_symbols"], "cuda")
raw = ro.rnnt_greedy_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["max_symbols"], g["activation"], False)
assert t._compare(t._decode_gpu(greedy, g["x"], g["lens"]), raw) == []
print("CLUSTER_VARIANT_OK")
"""


@pytest.mark.gpu
def test_gpu_both_kernel_variants_match_oracle():
    """The default kernel, wherever the sizes and the device allow it, splits the weights over K inside clusters of 4 CTAs
    and adds the partial sums through distributed shared memory (rnnt_greedy_c4_kernel); CFB_RNNT_CLUSTER=0 forces the
    row-partitioned one (rnnt_greedy_kernel).  Same hypotheses as the oracle from both.  Runs in a child process: tools that intercept launches
    (Nsight Compute) abort a process on a cooperative cluster launch, which must not take the test session with it."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CFB_TEST_ROOT=root)
    r = subprocess.run([sys.executable, "-c", _CLUSTER_SCRIPT], capture_output=True, text=True, env=env, timeout=600)
    if r.returncode != 0 and "Traceback" not in r.stderr:  # killed from outside, not a Python failure of the checks above
        pytest.skip("cooperative cluster launch not available in this environment: " + r.stderr[-300:])
    assert r.returncode == 0 and "CLUSTER_VARIANT_OK" in r.stdout, r.stderr[-2000:]


@pytest.mark.gpu
def test_gpu_sample_level_strategy_wrapper():
    g = load("rnnt_tiny")
    dec, joint, batched = build_modules(g["dims"], g["dec_sd"], g["joint_sd"], g["activation"], g["max_symbols"], "cuda")
    single = cn.GreedyRNNTInfer(dec, joint, blank_index=g["dims"][3], max_symbols_per_step=g["max_symbols"])
    a, b = _decode_gpu(single, g["x"], g["lens"]), _decode_gpu(batched, g["x"], g["lens"])
    for i, (ha, hb) in enumerate(zip(a, b)):
        n = int(g["n"][i])
        assert ha.y_sequence.tolist() == hb.y_sequence.tolist() == g["tokens"][i, :n].tolist()
        assert list(ha.timestep) == g["timesteps"][i, :n].tolist() and ha.score == hb.score
        assert (ha.dec_state is None) == (n == 0) and (ha.last_token == (g["tokens"][i, n - 1] if n else None))
