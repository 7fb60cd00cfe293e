"""Transducer beam search (decoding.strategy = beam, search_type = default; beam_size 1 = greedy_search): the oracle
against the stored n-best lists and its own invariants, the host-side surface on the CPU; the persistent CUDA search
(cfb_op_rnnt_beam through BeamRNNTInfer) against the stored lists and the oracle on the GPU."""
import glob
import os

import numpy as np
import pytest
import torch

import conformer_nemo_b200 as cn
from oracle import rnnt_beam_oracle as bo

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "rnnt_beam")
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz")))
TIE_MARGIN = 1e-5  # below this oracle decision margin a different result is reported, not failed


def load(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    e, p, j, v = (int(a) for a in z["dims"])
    dec_sd, joint_sd = bo.random_beam_state_dicts(e, p, j, v, int(z["weight_seed"]), float(z["blank_bias"]), float(z["sharpness"]))
    checksum = float(sum(w.double().sum() for w in list(dec_sd.values()) + list(joint_sd.values())))
    assert abs(checksum - float(z["weight_checksum"])) < 1e-6
    lists = []
    for b in range(len(z["counts"])):
        lists.append([(float(z["scores"][b, r]), z["tokens"][b, r, :z["lengths"][b, r]].tolist(),
                       z["timesteps"][b, r, :z["lengths"][b, r]].tolist()) for r in range(int(z["counts"][b]))])
    return dict(dims=(e, p, j, v), dec_sd=dec_sd, joint_sd=joint_sd, x=torch.from_numpy(z["encoder_output"]),
                lens=torch.from_numpy(z["encoded_lengths"]), beam=int(z["beam_size"]), score_norm=bool(z["score_norm"]),
                activation=str(z["activation"]), temperature=float(z["temperature"]), lists=lists, source=str(z["source"]))


def build(dims, dec_sd, joint_sd, activation, device=None, **kw):
    e, p, j, v = dims
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=p, pred_rnn_layers=1, dropout=0.1), vocab_size=v)
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=e, pred_hidden=p, joint_hidden=j, activation=activation, dropout=0.1),
                         num_classes=v)
    dec.load_state_dict(dec_sd, strict=True)
    joint.load_state_dict(joint_sd, strict=True)
    if device is not None:
        dec, joint = dec.to(device), joint.to(device)
    return cn.BeamRNNTInfer(dec, joint, **kw)


def _same_lists(got, want_lists, tol=1e-6):
    assert len(got) == len(want_lists)
    for g, w in zip(got, want_lists):
        assert [(y, ts) for _, y, ts in g] == [(y, ts) for _, y, ts in w]
        for (sg, _, _), (sw, _, _) in zip(g, w):
            assert abs(sg - sw) <= tol * max(1.0, abs(sw)), (sg, sw)


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_golden(name):
    g = load(name)
    res = bo.rnnt_beam_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["beam"], g["activation"], g["score_norm"],
                              g["temperature"])
    _same_lists([[(h.score, h.y, h.timestep) for h in r.nbest] for r in res], g["lists"])


def test_goldens_cover_the_issue_grid():
    gs = [load(n) for n in CASES]
    assert {g["beam"] for g in gs} >= {1, 2, 4, 8}
    assert {g["score_norm"] for g in gs} == {True, False}
    assert {g["activation"] for g in gs} >= {"relu", "tanh"}
    assert any(g["temperature"] != 1.0 for g in gs)
    assert any(bo.beam_widths(g["beam"], g["dims"][3])[1] < g["beam"] or g["beam"] > g["dims"][3] for g in gs)
    lens = {int(v) for g in gs for v in g["lens"]}
    assert 0 in lens and 1 in lens


def test_oracle_matches_live_reference_when_mounted():
    from oracle import reference_loader as rl

    if not rl.reference_available():
        pytest.skip("reference tree not mounted")
    import warnings

    dec_cls, joint_cls, _ = rl.load_reference_rnnt_classes()
    beam_cls = bo.load_reference_beam_class()
    dims = (40, 48, 44, 25)
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=11, blank_bias=1.0, sharpness=5.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dec = dec_cls(prednet=dict(pred_hidden=48, pred_rnn_layers=1, dropout=0.1), vocab_size=25)
    joint = joint_cls(jointnet=dict(encoder_hidden=40, pred_hidden=48, joint_hidden=44, activation="relu", dropout=0.1),
                      num_classes=25)
    dec.load_state_dict(dec_sd, strict=True)
    joint.load_state_dict(joint_sd, strict=True)
    x = torch.randn(3, 40, 12, generator=torch.Generator().manual_seed(5))
    lens = torch.tensor([12, 5, 1])
    for beam, norm in ((1, True), (3, True), (4, False)):
        (nb,) = beam_cls(dec, joint, beam_size=beam, score_norm=norm, return_best_hypothesis=False)(encoder_output=x,
                                                                                                   encoded_lengths=lens)
        res = bo.rnnt_beam_decode(x, lens, dec_sd, joint_sd, beam, "relu", norm)
        got = [[(float(h.score), [int(t) for t in h.y_sequence], [int(t) for t in h.timestep]) for h in n.n_best_hypotheses]
               for n in nb]
        _same_lists(got, [[(h.score, h.y, h.timestep) for h in r.nbest] for r in res], tol=1e-5)


def test_constructor_surface_and_errors():
    dims = (48, 64, 56, 30)
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=0)
    with pytest.raises(ValueError):
        build(dims, dec_sd, joint_sd, "relu", beam_size=0)
    for st in ("tsd", "alsd", "maes", "nsc"):
        with pytest.raises(NotImplementedError):
            build(dims, dec_sd, joint_sd, "relu", beam_size=4, search_type=st)
    with pytest.raises(NotImplementedError):
        build(dims, dec_sd, joint_sd, "relu", beam_size=4, search_type="unknown")
    with pytest.raises(NotImplementedError):
        build(dims, dec_sd, joint_sd, "relu", beam_size=4, language_model={"path": "lm.bin"})
    with pytest.raises(NotImplementedError):
        build(dims, dec_sd, joint_sd, "relu", beam_size=4, ngram_lm_model="lm.arpa")
    with pytest.raises(NotImplementedError):
        build(dims, dec_sd, joint_sd, "relu", beam_size=4, preserve_alignments=True)
    beam = build(dims, dec_sd, joint_sd, "relu", beam_size=4)
    assert beam.widths() == (4, 4) and beam.blank == 30 and beam.score_norm and beam.return_best_hypothesis
    assert build(dims, dec_sd, joint_sd, "relu", beam_size=64).widths() == (31, 30)
    with pytest.raises(RuntimeError):  # no CPU path
        beam(encoder_output=torch.zeros(1, 48, 4), encoded_lengths=torch.tensor([4]))
    with pytest.raises(NotImplementedError):
        beam(encoder_output=torch.zeros(1, 48, 4), encoded_lengths=torch.tensor([4]), partial_hypotheses=[])
    assert cn.NBestHypotheses([]).n_best_hypotheses == []


@pytest.mark.parametrize("beam,score_norm", [(2, True), (4, False), (8, True)])
def test_oracle_invariants(beam, score_norm):
    dims = (32, 40, 48, 20)
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=9, blank_bias=1.0, sharpness=5.0)
    x = torch.randn(3, 32, 9, generator=torch.Generator().manual_seed(9))
    res = bo.rnnt_beam_decode(x, torch.tensor([9, 0, 4]), dec_sd, joint_sd, beam, "relu", score_norm)
    key = (lambda h: h.score / len(h.y)) if score_norm else (lambda h: h.score)
    for r in res:
        keys = [key(h) for h in r.nbest]
        assert keys == sorted(keys, reverse=True)
        assert len(r.nbest) >= min(beam, 1 if r.length == 0 else beam)
        for h in r.nbest:
            assert h.y[0] == dims[3] and h.timestep[0] == -1 and len(h.y) == len(h.timestep)
            assert all(a <= b for a, b in zip(h.timestep, h.timestep[1:])) and (len(h.y) == 1 or h.timestep[-1] < r.length)
            assert h.score <= 0.0
    # encoded_len == 0: the initial hypothesis
    (h,) = res[1].nbest
    assert h.y == [dims[3]] and h.timestep == [-1] and h.score == 0.0 and float(h.h.abs().max()) == 0.0
    # scores never increase along a hypothesis: every prefix decoded over fewer frames scores no lower than the full path
    full = res[0]
    for t in range(1, 9):
        part = bo.rnnt_beam_decode(x[:1, :, :t], torch.tensor([t]), dec_sd, joint_sd, beam, "relu", score_norm)[0]
        assert max(h.score for h in part.nbest) >= max(h.score for h in full.nbest) - 1e-12


# ---------------------------------------------------------------------------------------------------------------- GPU

TIES = {"n": 0}


def _lists(hyps):
    return [[(h.score, h.y_sequence.tolist(), list(h.timestep)) for h in nb.n_best_hypotheses] for nb in hyps]


def _compare(hyps, want, score_tol=1e-5, state_tol=2e-5):
    """n-best lists equal to the oracle's (order, labels, frames exactly; scores and states to fp32 rounding), except
    where the oracle's smallest decision margin is within fp32 summation noise: then the difference is reported."""
    bad = []
    for b, (nb, r) in enumerate(zip(hyps, want)):
        got = nb.n_best_hypotheses
        div = bo.first_difference([(h.y_sequence.tolist(), list(h.timestep)) for h in got], r)
        if div is not None:
            if r.min_margin < TIE_MARGIN:
                TIES["n"] += 1
                print(f"[beam tie] utterance {b}: first difference at rank {div[0]} ({div[1]}); oracle margin {r.min_margin:.2e}")
            else:
                bad.append((b, div, r.min_margin))
            continue
        for h, w in zip(got, r.nbest):
            assert abs(h.score - w.score) <= score_tol * max(1.0, abs(w.score)), (b, h.score, w.score)
            if w.h is not None:
                assert float((h.dec_state[0].view(-1) - w.h).abs().max()) <= state_tol
                assert float((h.dec_state[1].view(-1) - w.c).abs().max()) <= state_tol
            else:
                assert h.dec_state is None
    return bad


def _decode(beam, x, lens):
    (hyps,) = beam(encoder_output=x.cuda(), encoded_lengths=lens.cuda())
    return hyps


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_gpu_matches_golden(name):
    g = load(name)
    beam = build(g["dims"], g["dec_sd"], g["joint_sd"], g["activation"], "cuda", beam_size=g["beam"], score_norm=g["score_norm"],
                 softmax_temperature=g["temperature"], return_best_hypothesis=False)
    hyps = _decode(beam, g["x"], g["lens"])
    want = bo.rnnt_beam_decode(g["x"], g["lens"], g["dec_sd"], g["joint_sd"], g["beam"], g["activation"], g["score_norm"],
                               g["temperature"])
    assert _compare(hyps, want) == []
    for b, (nb, lst) in enumerate(zip(hyps, g["lists"])):
        if want[b].min_margin >= TIE_MARGIN:
            assert [(y, ts) for _, y, ts in _lists([nb])[0]] == [(y, ts) for _, y, ts in lst]
        for h in nb.n_best_hypotheses:
            assert h.y_sequence.dtype == torch.int64 and int(h.length) == int(g["lens"][b])
    best = build(g["dims"], g["dec_sd"], g["joint_sd"], g["activation"], "cuda", beam_size=g["beam"],
                 score_norm=g["score_norm"], softmax_temperature=g["temperature"])
    for h, nb in zip(_decode(best, g["x"], g["lens"]), hyps):  # return_best_hypothesis: the head of the n-best list
        assert h.y_sequence.tolist() == nb.n_best_hypotheses[0].y_sequence.tolist() and h.score == nb.n_best_hypotheses[0].score


SEEDED = [  # dims, B, T, beam, score_norm, temperature, dtype, seed
    ((512, 640, 640, 1024), 4, 24, 4, True, 1.0, "fp32", 21),   # the Conformer-Transducer sizes
    ((512, 640, 640, 1024), 3, 20, 8, False, 1.0, "bf16", 22),
    ((256, 320, 320, 128), 6, 30, 1, True, 1.0, "fp32", 23),    # BPE-128, greedy_search
    ((256, 320, 320, 128), 6, 30, 2, False, 1.0, "fp32", 24),
    ((256, 320, 320, 128), 5, 30, 8, True, 1.3, "bf16", 25),
    ((176, 320, 320, 28), 6, 30, 4, True, 1.0, "fp32", 26),     # char vocabulary: fewer output rows than CTAs
    ((176, 320, 320, 28), 5, 30, 2, True, 0.8, "fp32", 27),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dims,B,T,beam_size,score_norm,temperature,dtype,seed", SEEDED)
def test_gpu_matches_oracle_seeded(dims, B, T, beam_size, score_norm, temperature, dtype, seed):
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=seed, blank_bias=2.5, sharpness=5.0)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, dims[0], T, generator=gen)
    if dtype == "bf16":
        x = x.bfloat16()
    lens = torch.randint(2, T + 1, (B,), generator=gen)
    lens[0], lens[1] = T, 1
    if B > 3:
        lens[2] = 0
    beam = build(dims, dec_sd, joint_sd, "relu", "cuda", beam_size=beam_size, score_norm=score_norm,
                 softmax_temperature=temperature, return_best_hypothesis=False)
    want = bo.rnnt_beam_decode(x.float(), lens, dec_sd, joint_sd, beam_size, "relu", score_norm, temperature)
    assert sum(len(h.y) - (beam_size > 1) for r in want for h in r.nbest) > 0  # the case does emit
    assert _compare(_decode(beam, x, lens), want) == []


def _key(hyps):
    return [[(h.score, h.y_sequence.tolist(), list(h.timestep)) for h in nb.n_best_hypotheses] for nb in hyps]


@pytest.mark.gpu
def test_gpu_determinism_and_capacity_retry():
    """Same bits for a batch-order permutation, an utterance alone, a second run and a batch of more than one launch;
    capacities that are too small set the flag and the retry returns what large capacities give."""
    dims = (256, 320, 320, 128)
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=31, blank_bias=1.0, sharpness=5.0)
    gen = torch.Generator().manual_seed(31)
    B, T = 12, 40
    x = torch.randn(B, 256, T, generator=gen)
    lens = torch.randint(1, T + 1, (B,), generator=gen)
    lens[0] = T
    beam = build(dims, dec_sd, joint_sd, "relu", "cuda", beam_size=4, return_best_hypothesis=False)
    ref = _key(_decode(beam, x, lens))
    assert _key(_decode(beam, x, lens)) == ref
    perm = torch.randperm(B, generator=gen)
    hp = _key(_decode(beam, x[perm], lens[perm]))
    for i, src in enumerate(perm.tolist()):
        assert hp[i] == ref[src]
    for b in (0, 5):
        assert _key(_decode(beam, x[b:b + 1], lens[b:b + 1]))[0] == ref[b]
    reps = 12  # 144 utterances: more than one launch holds
    big = _key(_decode(beam, x.repeat(reps, 1, 1), lens.repeat(reps)))
    assert all(big[i] == ref[i % B] for i in range(B * reps))
    # deliberately small capacities: the kernel flags, the wrapper grows them and decodes again
    small = dict(max_expansions=2, max_hyps=8, max_nodes=16, max_states=4, max_len=3)
    out = beam.decode_arrays(x.cuda(), lens.cuda(), small)
    assert int(out["flags"].cpu()) & 1
    orig = beam.default_caps
    beam.default_caps = lambda t: dict(small)
    try:
        assert _key(_decode(beam, x, lens)) == ref
    finally:
        beam.default_caps = orig


@pytest.mark.gpu
def test_gpu_encoder_output_beam_decoded():
    """Chain: the GPU encoder's output on a small config, beam-decoded, against the oracle on that same output."""
    from oracle import conformer_oracle as oc

    cfg = oc.EncoderConfig(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=2, d_model=256, n_heads=4)
    enc.load_state_dict(oc.random_state_dict(cfg, 4), strict=False)
    enc = enc.cuda().eval()
    feats = torch.randn(3, 80, 160, generator=torch.Generator().manual_seed(8)).cuda()
    flen = torch.tensor([160, 121, 64]).cuda()
    encoded, elen = enc(audio_signal=feats, length=flen)
    dims = (256, 320, 320, 128)
    dec_sd, joint_sd = bo.random_beam_state_dicts(*dims, seed=51, blank_bias=1.0, sharpness=5.0)
    beam = build(dims, dec_sd, joint_sd, "relu", "cuda", beam_size=4, return_best_hypothesis=False)
    hyps = _decode(beam, encoded, elen)
    want = bo.rnnt_beam_decode(encoded.float().cpu(), elen.cpu(), dec_sd, joint_sd, 4, "relu", True)
    assert _compare(hyps, want) == []
    for nb, n in zip(hyps, elen.cpu().tolist()):
        assert all(int(h.length) == n and max(h.timestep) < n for h in nb.n_best_hypotheses)
