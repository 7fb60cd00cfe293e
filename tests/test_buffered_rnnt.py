"""Buffered long-audio transducer inference (BatchedFrameASRRNNT, streaming_utils.py): the oracle's middle-token slice
and merge on hand-sized cases, the device merge against the oracle's, a file alone and among others in the oracle, and the
argument checks on the CPU; on the GPU the decode of every window against the transducer oracle run on the device's own
encoder output, the merge against the oracle's merge of the device's decodes, the whole pipeline against the oracle
pipeline, bit-identical results alone / among other files / with any windows_per_forward, and the token-capacity regrowth."""
import types

import numpy as np
import pytest
import torch

import conformer_nemo_b200 as cn
from conformer_nemo_b200.buffered import merge_middle_tokens
from oracle import buffered_oracle as bo
from oracle import buffered_rnnt_oracle as bro
from oracle import conformer_oracle as oc
from oracle import rnnt_oracle as ro
from test_buffered import PRE, STRIDE_SECS, Tokenizer, _pre, fake_featurize, nemo_chunking, synthetic_files

LW = 100  # encoder frames of a 4.0 s window (400 feature frames, subsampling 4)


def make_model(d_model=256, n_layers=2, n_heads=4, pred=320, vocab=128, blank_bias=1.0, max_symbols=10, seed=0,
               device="cpu"):
    cfg = oc.EncoderConfig(feat_in=80, n_layers=n_layers, d_model=d_model, n_heads=n_heads)
    enc_sd = oc.random_state_dict(cfg, seed)
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(d_model, pred, pred, vocab, seed + 1, blank_bias)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=n_layers, d_model=d_model, n_heads=n_heads)
    enc.load_state_dict(enc_sd, strict=False)
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=pred, pred_rnn_layers=1, dropout=0.1), vocab_size=vocab)
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=d_model, pred_hidden=pred, joint_hidden=pred, activation="relu",
                                       dropout=0.1), num_classes=vocab)
    dec.load_state_dict(dec_sd)
    joint.load_state_dict(joint_sd)
    decoding = {"strategy": "greedy_batch", "greedy": {} if max_symbols is None else {"max_symbols": max_symbols}}
    model = types.SimpleNamespace(_cfg={"sample_rate": 16000, "preprocessor": dict(PRE), "decoding": decoding},
                                  encoder=enc.to(device).eval(), decoder=dec.to(device), joint=joint.to(device),
                                  tokenizer=Tokenizer())
    return model, (cfg, enc_sd, dec_sd, joint_sd, max_symbols)


def oracle_from_decodes(decodes, blank, max_symbols, n_frames=LW):
    """The oracle's BatchedFrameASRRNNT with its per-window decodes given: (tokens, timesteps) per window per file."""
    asr = bro.BatchedFrameASRRNNT(None, None, 80, 0.01, 16000, blank_id=blank, batch_size=len(decodes))
    asr.all_alignments = [[bro.alignments_from_decode(t, s, n_frames, max_symbols, blank) for t, s in d] for d in decodes]
    asr.frame_bufferer.signal_end_index = [len(d) for d in decodes]
    asr.infer_logits = lambda: None
    return asr


# ---------------------------------------------------------------------------------------------------------------- CPU

# two windows of 8 frames, blank 9: (tokens, timesteps)
W0 = ([1, 2, 3, 4, 5, 6], [0, 2, 4, 4, 5, 7])
W1 = ([6, 7, 7, 8], [1, 4, 5, 7])


@pytest.mark.parametrize("tpc,delay,want", [
    (2, 3, [3, 4, 5, 7, 7]),         # offset 1: frames [8 - 1 - 3, + 2) = [4, 6)
    (3, 8, [1, 2, 6]),               # delay == Lw: offset 0, frames [0, 3)
    (10, 3, [3, 4, 5, 6, 7, 7, 8]),  # [4, 14) clipped at Lw like a Python slice
    (1, 0, [6, 8]),                  # delay 0: the last frame only
])
def test_oracle_slice_rule(tpc, delay, want):
    asr = oracle_from_decodes([[W0, W1]], 9, None, n_frames=8)
    assert asr.transcribe(tpc, delay) == [want]
    assert asr.unmerged == [want]
    # the device merge (tensor ops, here on the CPU) with the same bounds
    offset = 0 if delay == 8 else 1
    lo = 8 - offset - delay
    cap = 6
    tok = torch.tensor([W0[0], W1[0] + [0, 0]], dtype=torch.int32)
    ts = torch.tensor([W0[1], W1[1] + [-5, -5]], dtype=torch.int32)  # entries past n_tokens are never read
    merged, n = merge_middle_tokens(tok, ts, torch.tensor([6, 4], dtype=torch.int32), torch.tensor([0]), torch.tensor([2]),
                                    2, cap, lo, min(lo + tpc, 8), 8)
    assert merged[0, :int(n[0])].tolist() == want


def test_merge_is_a_plain_concatenation():
    """A token kept at the end of one window and again at the start of the next survives twice (no collapse)."""
    w0 = ([4, 5], [2, 5])
    w1 = ([5, 3], [4, 6])
    asr = oracle_from_decodes([[w0, w1]], 9, 2, n_frames=8)
    assert asr.transcribe(2, 3) == [[5, 5]]


def test_device_merge_equals_the_oracle_merge_on_random_decodes():
    """merge_middle_tokens (the device merge, run here on CPU tensors) against the oracle's transcribe, for ragged files,
    a window that emits nothing, overflowed rows (n_tokens > cap) clipped, and every slice shape."""
    g = np.random.default_rng(5)
    n_win = [3, 1, 7, 2]
    cap = 40
    rows = []
    for _ in range(sum(n_win)):
        n = int(g.integers(0, cap + 1))
        ts = np.sort(g.integers(0, LW, n))
        rows.append((g.integers(0, 30, n).tolist(), ts.tolist()))
    rows[4] = ([], [])
    first = np.concatenate([[0], np.cumsum(n_win[:-1])])
    decodes = [[rows[w] for w in range(first[f], first[f] + n_win[f])] for f in range(len(n_win))]
    tok = torch.zeros(len(rows), cap, dtype=torch.int32)
    ts = torch.full((len(rows), cap), 7, dtype=torch.int32)
    for w, (t, s) in enumerate(rows):
        tok[w, :len(t)] = torch.tensor(t, dtype=torch.int32)
        ts[w, :len(s)] = torch.tensor(s, dtype=torch.int32)
    counts = torch.tensor([len(t) for t, _ in rows], dtype=torch.int32)
    model, _ = make_model(d_model=64, n_heads=2, pred=64, vocab=30)
    asr = cn.BatchedFrameASRRNNT(model, batch_size=4)
    for tpc, delay in ((40, 70), (200, 10), (1, 0), (7, LW), (3, LW - 1)):
        lo, hi = asr._slice(tpc, delay)
        merged, n = merge_middle_tokens(tok, ts, counts, torch.from_numpy(first), torch.tensor(n_win), max(n_win), cap,
                                        lo, hi, LW)
        want = oracle_from_decodes(decodes, 30, None).transcribe(tpc, delay)
        assert [merged[f, :int(n[f])].tolist() for f in range(len(n_win))] == want, (tpc, delay)


def test_batched_bufferer_windows_equal_the_single_file_windows():
    """Each file keeps its own W-wide buffer in BatchedFeatureFrameBufferer: its windows are those FeatureFrameBufferer
    gives for the file alone (the files end at different steps)."""
    xs = [np.random.default_rng(n).standard_normal((3, n)).astype(np.float32) for n in (1003, 350, 7)]
    buf = bro.BatchedFeatureFrameBufferer(3, 0.01, 1.6, len(xs), 4.0)
    for i, x in enumerate(xs):
        buf.set_frame_reader(bo.AudioFeatureIterator(np.zeros(10, np.float32), 1.6, fake_featurize(x), 0.01), i)
    got = [[] for _ in xs]
    while True:
        batch = buf.get_buffers_batch()
        if not batch:
            break
        for i, b in enumerate(batch):
            if not buf.signal_end[i]:
                got[i].append(np.asarray(b)[0])
    for i, x in enumerate(xs):
        want = bo.file_windows(np.zeros(10, np.float32), fake_featurize(x), 3, 0.01, 1.6, 4.0)
        assert buf.signal_end_index[i] == len(want) == x.shape[1] // 160 + 1
        assert np.array_equal(np.stack(got[i]), want), i


def oracle_pipeline(parts, audios, tpc, delay):
    cfg, enc_sd, dec_sd, joint_sd, max_symbols = parts
    pre = _pre(normalize=None)
    model = bro.rnnt_model(enc_sd, cfg, dec_sd, joint_sd, max_symbols)
    asr = bro.BatchedFrameASRRNNT(bo.raw_featurizer(pre.featurizer.window, pre.featurizer.fb[0]), model, 80, 0.01, 16000,
                                 blank_id=dec_sd["prediction.embed.weight"].shape[0] - 1, batch_size=len(audios))
    asr.read_audio_file(audios, delay, STRIDE_SECS)
    return asr, asr.transcribe(tpc, delay)


def test_oracle_file_gives_the_same_ids_alone_and_batched():
    _, parts = make_model(d_model=64, n_heads=2, pred=64, vocab=30, blank_bias=0.3, max_symbols=4, seed=2)
    audios = synthetic_files([2.0, 1.0, 3.3], seed=9)
    batched, ids = oracle_pipeline(parts, audios, 40, 70)
    assert sum(len(i) for i in ids) > 0
    for f in range(3):
        alone, (want,) = oracle_pipeline(parts, audios[f:f + 1], 40, 70)
        assert ids[f] == want
        assert len(batched.all_preds[f]) == len(alone.all_preds[0])
        assert all(np.array_equal(a, b) for a, b in zip(batched.all_preds[f], alone.all_preds[0]))


def test_arguments_are_refused():
    model, _ = make_model(d_model=64, n_heads=2, pred=64, vocab=30)
    asr = cn.BatchedFrameASRRNNT(model, batch_size=2)
    assert (asr.window_tokens, asr.blank_id, asr.max_symbols, asr.initial_capacity) == (LW, 30, 10, 10 * LW)
    with pytest.raises(ValueError):
        asr.read_audio_file([np.zeros(100, np.float32)], 70, STRIDE_SECS)          # batch_size files, not one
    with pytest.raises(NotImplementedError):
        asr.read_audio_file(["/data/a.wav", "/data/b.wav"], 70, STRIDE_SECS)       # audio decoding stays with the caller
    with pytest.raises(NotImplementedError):
        asr.read_audio_file("/data/a.wav", 70, STRIDE_SECS)
    asr.read_audio_file([np.zeros(100, np.float32)] * 2, 70, STRIDE_SECS)
    with pytest.raises(ValueError):
        asr.transcribe(40, LW + 1)                                                # lo < 0: Python would index from the end
    with pytest.raises(ValueError):
        asr.transcribe(0, 70)
    with pytest.raises(ValueError):
        asr.transcribe(40, -1)
    assert asr._slice(40, LW) == (0, 40) and asr._slice(40, LW - 1) == (0, 40) and asr._slice(5, 0) == (LW - 1, LW)
    with pytest.raises(NotImplementedError):
        cn.BatchedFrameASRRNNT(model, stateful_decoding=True)
    for bad in (dict(decoder=torch.nn.Linear(2, 2)), dict(joint=torch.nn.Linear(2, 2)), dict(encoder=torch.nn.Linear(2, 2))):
        with pytest.raises(TypeError):
            cn.BatchedFrameASRRNNT(types.SimpleNamespace(**{**vars(model), **bad}))
    with pytest.raises(ValueError):
        cn.BatchedFrameASRRNNT(model, frame_len=0.155)
    with pytest.raises(ValueError):
        cn.BatchedFrameASRRNNT(model, batch_size=0)
    with pytest.raises(ValueError):
        cn.BatchedFrameASRRNNT(types.SimpleNamespace(**{**vars(model), "_cfg": {**model._cfg, "decoding": {
            "greedy": {"max_symbols": 0}}}}))
    no_limit = types.SimpleNamespace(**{**vars(model), "_cfg": {"sample_rate": 16000, "preprocessor": dict(PRE)}})
    asr = cn.BatchedFrameASRRNNT(no_limit)
    assert asr.max_symbols is None and asr.greedy.max_symbols is None and asr.initial_capacity == 4 * LW + 64
    assert cn.buffered_rnnt_transcribe(model, [], 1.6, 4.0, 40, 70, STRIDE_SECS) == []


def test_oracle_matches_live_reference_when_mounted():
    from oracle import reference_loader as rl

    if not rl.reference_available():
        pytest.skip("reference tree not mounted")
    su = bo.load_reference_streaming_utils()
    xs = [np.random.default_rng(n).standard_normal((80, n)).astype(np.float32) for n in (1003, 350)]

    class RawPreprocessor:  # what AudioFeatureIterator calls: preprocessor(input_signal=, length=) and ._cfg
        _cfg = {"window_stride": 0.01}

        def __init__(self, x):
            self.x = x

        def __call__(self, input_signal, length):
            return torch.from_numpy(self.x)[None], torch.tensor([self.x.shape[1]])

    model = types.SimpleNamespace(preprocessor=types.SimpleNamespace(log=True), _cfg=types.SimpleNamespace(
        sample_rate=16000, preprocessor=types.SimpleNamespace(window_stride=0.01, features=80)))
    ref = su.BatchedFeatureFrameBufferer(asr_model=model, frame_len=1.6, batch_size=2, total_buffer=4.0)
    mine = bro.BatchedFeatureFrameBufferer(80, 0.01, 1.6, 2, 4.0)
    for i, x in enumerate(xs):
        ref.set_frame_reader(su.AudioFeatureIterator(np.zeros(1000, np.float32), 1.6, RawPreprocessor(x), "cpu"), i)
        mine.set_frame_reader(bo.AudioFeatureIterator(np.zeros(1000, np.float32), 1.6, fake_featurize(x), 0.01), i)
    while True:
        a, b = ref.get_buffers_batch(), mine.get_buffers_batch()
        assert len(a) == len(b)
        if not a:
            break
        for i in range(2):
            assert np.array_equal(np.asarray(a[i]), np.asarray(b[i]))
    assert list(ref.signal_end_index) == list(mine.signal_end_index)
    # the merge, on fixed alignments
    tok = types.SimpleNamespace(ids_to_tokens=lambda ids: [str(i) for i in ids], ids_to_text=lambda ids: list(ids))
    mine = oracle_from_decodes([[W0, W1], [W1]], 9, None, n_frames=8)
    live = su.BatchedFrameASRRNNT.__new__(su.BatchedFrameASRRNNT)
    live.asr_model = types.SimpleNamespace(tokenizer=tok)
    live.tokenizer, live.blank_id, live.batch_size = tok, 9, 2
    live.all_alignments = mine.all_alignments
    live.frame_bufferer = types.SimpleNamespace(get_buffers_batch=lambda: [], signal_end_index=[2, 1])
    for tpc, delay in ((2, 3), (3, 8), (10, 3), (1, 0)):
        assert live.transcribe(tpc, delay) == mine.transcribe(tpc, delay)


# ---------------------------------------------------------------------------------------------------------------- GPU

BLANK_BIAS = 1.2  # the random weights then emit about 0.13 symbols per encoder frame of the d_model-256 encoder


def _decode(asr, audios, tpc, delay):
    return asr.decode(audios, int(delay * STRIDE_SECS * 16000), tpc, delay)


def _windows_encoded(asr, audios, delay):
    """The device's own encoder output of every window (fp32 on the host) and the windows per file."""
    wavs = [torch.from_numpy(a) for a in audios]
    dev = torch.device("cuda")
    with torch.no_grad():
        windows, first, n_win = asr._windows(wavs, int(delay * STRIDE_SECS * 16000), dev, None)
        enc = torch.cat([asr.encoder(audio_signal=windows[i:i + 64])[0].float().cpu() for i in range(0, windows.shape[0], 64)])
    return enc, n_win


def _divergences(decodes, want):
    """Windows whose decode differs from the oracle's beyond an oracle arg-max tie (margin < 2e-6, tests/test_rnnt.py)."""
    bad, ties = [], 0
    for w, ((tokens, steps), r) in enumerate(zip(decodes, want)):
        div = ro.first_divergence(tokens.tolist(), steps.tolist(), r)
        if div is not None:
            if div[1] < 2e-6:
                ties += 1
            else:
                bad.append((w, div))
    return bad, ties


@pytest.mark.gpu
def test_gpu_decode_of_every_window_matches_the_oracle_on_the_same_encoder_output():
    model, (_, _, dec_sd, joint_sd, ms) = make_model(device="cuda", blank_bias=BLANK_BIAS)
    tpc, delay = nemo_chunking()
    audios = synthetic_files([3.3, 7.1, 1.0, 20.0], seed=4)
    asr = cn.BatchedFrameASRRNNT(model, batch_size=4)
    _, decodes = _decode(asr, audios, tpc, delay)
    enc, n_win = _windows_encoded(asr, audios, delay)
    assert [len(d) for d in decodes] == n_win
    flat = [d for per_file in decodes for d in per_file]
    want = ro.rnnt_greedy_decode(enc, torch.full((enc.shape[0],), LW), dec_sd, joint_sd, ms, "relu", False)
    emitted = sum(len(t) for t, _ in flat)
    print(f"[buffered rnnt] {len(flat)} windows, {emitted / (len(flat) * LW):.3f} symbols per encoder frame")
    assert emitted > len(flat)
    bad, ties = _divergences(flat, want)
    assert bad == [], bad[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("tpc,delay", [(40, 70), (200, 10), (1, 0), (30, LW)])
def test_gpu_merge_equals_the_oracle_merge_of_the_device_decodes(tpc, delay):
    model, _ = make_model(device="cuda", blank_bias=BLANK_BIAS)
    audios = synthetic_files([2.0, 5.5, 9.0], seed=6)
    ids, decodes = _decode(cn.BatchedFrameASRRNNT(model, batch_size=3), audios, tpc, delay)
    assert sum(len(t) for d in decodes for t, _ in d) > 10
    assert ids == oracle_from_decodes(decodes, 128, 10).transcribe(tpc, delay)


@pytest.mark.gpu
def test_gpu_end_to_end_against_the_oracle_pipeline():
    """Every window's decode against the oracle pipeline's (oracle front end, windows, encoder and decode): the share of
    windows whose tokens and timesteps are equal, over >= 200 windows; the merged ids of the device's decodes equal the
    oracle's merge of them."""
    model, parts = make_model(device="cuda", blank_bias=BLANK_BIAS)
    tpc, delay = nemo_chunking()
    audios = synthetic_files([3.3, 7.1, 1.0, 300.0], seed=4)
    asr = cn.BatchedFrameASRRNNT(model, batch_size=4)
    ids, decodes = _decode(asr, audios, tpc, delay)
    ref, _ = oracle_pipeline(parts, audios, tpc, delay)
    equal = total = 0
    for f in range(4):
        assert len(decodes[f]) == len(ref.all_preds[f])
        for (tokens, steps), want_tokens, want_steps in zip(decodes[f], ref.all_preds[f], ref.all_timestamps[f]):
            equal += int(tokens.tolist() == want_tokens.tolist() and steps.tolist() == list(want_steps))
            total += 1
    print(f"[buffered rnnt] end to end: {equal} of {total} windows ({equal / total:.4f}) decode as the oracle pipeline's")
    assert ids == oracle_from_decodes(decodes, 128, 10).transcribe(tpc, delay)
    assert total >= 200 and equal / total >= 0.95, equal / total


@pytest.mark.gpu
def test_gpu_a_file_gives_the_same_bits_alone_among_others_and_with_any_windows_per_forward():
    model, _ = make_model(device="cuda", blank_bias=BLANK_BIAS)
    tpc, delay = nemo_chunking()
    audios = synthetic_files([4.0, 11.3, 0.5, 6.2], seed=8)
    alone_ids, alone = _decode(cn.BatchedFrameASRRNNT(model, batch_size=1), audios[1:2], tpc, delay)
    same = lambda a, b: len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
                                                 for x, y in zip(a, b))
    assert sum(len(t) for t, _ in alone[0]) > 0
    for wpf, graphs in ((1, False), (7, True), (256, False), (256, True)):
        model.encoder.enable_cuda_graphs(graphs)
        asr = cn.BatchedFrameASRRNNT(model, batch_size=4, windows_per_forward=wpf)
        ids, dec = _decode(asr, audios, tpc, delay)
        assert ids[1] == alone_ids[0] and same(dec[1], alone[0]), (wpf, graphs)
        ids, dec = _decode(asr, audios[::-1], tpc, delay)
        assert ids[2] == alone_ids[0] and same(dec[2], alone[0]), (wpf, graphs)
    model.encoder.enable_cuda_graphs(False)


@pytest.mark.gpu
def test_gpu_token_capacity_regrowth_equals_one_large_decode():
    """The windows that emit more tokens than the first capacity are encoded and decoded again with room for all of them;
    the result equals a decode whose first capacity holds every window.  The first capacity is that of max_symbols None
    (4 Lw + 64), lowered to 2 tokens here, on the symbol-limited model of the other tests: with these random weights and no
    symbol limit a decode either runs away (4096 symbols at one frame at blank bias 0.8, 1.2, 1.3 and 1.4) or emits
    nothing (1.5), so no bias makes a window pass 4 Lw + 64 tokens and end.  The regrowth does not depend on the limit."""
    no_limit, _ = make_model(device="cuda", blank_bias=BLANK_BIAS, max_symbols=None)
    assert cn.BatchedFrameASRRNNT(no_limit).initial_capacity == 4 * LW + 64
    model, _ = make_model(device="cuda", blank_bias=BLANK_BIAS)
    audios = synthetic_files([3.0, 6.5, 12.0], seed=12)
    small = cn.BatchedFrameASRRNNT(model, batch_size=3)
    small.initial_capacity = 2
    ids, decodes = _decode(small, audios, 40, 70)
    counts = [len(t) for d in decodes for t, _ in d]
    print(f"[buffered rnnt] regrowth: {sum(c > 2 for c in counts)} of {len(counts)} windows outgrew 2 tokens, "
          f"up to {max(counts)}")
    assert any(c > 2 for c in counts) and any(c <= 2 for c in counts)
    big = cn.BatchedFrameASRRNNT(model, batch_size=3)
    ids2, decodes2 = _decode(big, audios, 40, 70)
    assert ids2 == ids
    for d, e in zip(decodes, decodes2):
        assert len(d) == len(e) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) for x, y in zip(d, e))
    assert ids == oracle_from_decodes(decodes, 128, 10).transcribe(40, 70)


@pytest.mark.gpu
def test_gpu_class_equals_the_function():
    model, _ = make_model(device="cuda", blank_bias=BLANK_BIAS)
    tpc, delay = nemo_chunking()
    audios = synthetic_files([2.5, 8.0, 4.4], seed=10)
    asr = cn.BatchedFrameASRRNNT(model, batch_size=3)
    asr.read_audio_file(audios, delay, STRIDE_SECS)
    texts = asr.transcribe(tpc, delay)
    ids = cn.buffered_rnnt_transcribe(model, audios, 1.6, 4.0, tpc, delay, STRIDE_SECS)
    assert texts == [Tokenizer().ids_to_text(i) for i in ids] and asr.unmerged == ids
    assert [len(p) for p in asr.all_preds] == [len(d) for d in _decode(asr, audios, tpc, delay)[1]]
