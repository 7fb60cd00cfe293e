"""Buffered long-audio CTC inference (FrameBatchASR, streaming_utils.py:455-684): the oracle's restatement against the
closed form and hand-sized cases, argument checks and the normalize=None front end on the CPU; on the GPU the raw
log-mel kernel, the window kernel (cfb_op_feature_buffers) against float64, and the whole pipeline against the oracle
pipeline, including bit-identical results for a file alone, among other files and with any batch_size."""
import math
import types

import numpy as np
import pytest
import torch

import conformer_nemo_b200 as cn
from oracle import buffered_oracle as bo
from oracle import conformer_oracle as oc
from oracle import ctc_head_oracle as ho
from oracle import frontend_oracle as fo

PRE = dict(_target_="nemo.collections.asr.modules.AudioToMelSpectrogramPreprocessor", sample_rate=16000,
           window_size=0.025, window_stride=0.01, window="hann", normalize="per_feature", n_fft=512, features=80,
           dither=1e-5, pad_to=16)  # conformer_ctc_bpe.yaml model.preprocessor
STRIDE_SECS = 0.01 * 4  # model_stride_in_secs = window_stride * subsampling_factor
Z = -16.635


def nemo_chunking(frame_len=1.6, total_buffer=4.0):
    """tokens_per_chunk and delay as NeMo's buffered CTC script computes them."""
    tokens_per_chunk = math.ceil(frame_len / STRIDE_SECS)
    delay = math.ceil((frame_len + (total_buffer - frame_len) / 2) / STRIDE_SECS)
    return tokens_per_chunk, delay


class Tokenizer:
    def ids_to_text(self, ids):
        return " ".join(str(i) for i in ids)


def make_model(d_model=256, n_layers=2, n_heads=4, vocab=128, seed=0, device="cpu"):
    cfg = oc.EncoderConfig(feat_in=80, n_layers=n_layers, d_model=d_model, n_heads=n_heads)
    enc_sd = oc.random_state_dict(cfg, seed)
    head_sd = ho.random_head_state_dict(d_model, vocab, seed + 1)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=n_layers, d_model=d_model, n_heads=n_heads)
    enc.load_state_dict(enc_sd, strict=False)
    dec = cn.ConvASRDecoder(feat_in=d_model, num_classes=vocab)
    dec.load_state_dict(head_sd)
    model = types.SimpleNamespace(_cfg={"sample_rate": 16000, "preprocessor": dict(PRE)}, encoder=enc.to(device).eval(),
                                  decoder=dec.to(device), tokenizer=Tokenizer())
    return model, (cfg, enc_sd, head_sd)


# ---------------------------------------------------------------------------------------------------------------- CPU

def closed_form_windows(x: np.ndarray, n: int, fl: int, W: int) -> np.ndarray:
    """The restatement of DESIGN section 15: window k column j is frame s = (k+1) fl - W + j: Z for s < 0, x[:, s] for s < n, 0 after;
    n // fl + 1 windows; rows normalised with the population std + 1e-5 (float64)."""
    out = []
    for k in range(n // fl + 1):
        w = np.zeros((x.shape[0], W))
        for j in range(W):
            s = (k + 1) * fl - W + j
            w[:, j] = Z if s < 0 else (x[:, s] if s < n else 0.0)
        out.append((w - w.mean(1, keepdims=True)) / (w.std(1, keepdims=True) + 1e-5))
    return np.stack(out)


def fake_featurize(x):
    """A featurizer that hands the iterator fixed features: (1, F, n) and seq_len n."""
    return lambda signal, length: (torch.from_numpy(x)[None], torch.tensor([x.shape[1]]))


@pytest.mark.parametrize("n,fl,W", [(7, 16, 40),     # shorter than one chunk
                                    (64, 16, 40),    # n a multiple of fl: the last chunk is all zeros
                                    (161, 16, 40),   # W not a multiple of fl (160 / 400 scaled down)
                                    (50, 16, 16),    # fl == W
                                    (1003, 160, 400)])
def test_oracle_windows_are_the_closed_form(n, fl, W):
    x = np.random.default_rng(n).standard_normal((3, n))
    got = bo.file_windows(np.zeros(10, np.float32), fake_featurize(x), 3, 0.01, fl * 0.01, W * 0.01, dtype=np.float64)
    want = closed_form_windows(x, n, fl, W)
    assert got.shape == (n // fl + 1, 3, W) == want.shape
    assert np.abs(got - want).max() <= 1e-6  # the last chunk is float32 in the reference
    if n % fl == 0:  # the extra chunk: the last window ends in fl zero columns
        raw = bo.FeatureFrameBufferer(3, 0.01, fl * 0.01, 4, W * 0.01, dtype=np.float64)
        raw.set_frame_reader(bo.AudioFeatureIterator(np.zeros(10, np.float32), fl * 0.01, fake_featurize(x), 0.01))
        frames = [f for f in raw.frame_reader]
        assert len(frames) == n // fl + 1 and not np.any(np.asarray(frames[-1]))


def test_oracle_merge_slices_and_collapses():
    asr = bo.FrameBatchASR(None, None, 3, 0.01, 16000, blank_id=5)
    asr.all_preds = [np.array([0, 1, 1, 5, 2, 2, 3, 5]), np.array([2, 5, 5, 3, 3, 4, 4, 1])]
    asr.infer_logits = lambda: None
    # Lw = 8, delay 3: decoded[4:4 + tpc]; tokens_per_chunk past the end is clipped like a Python slice
    assert asr.transcribe(2, 3) == [2, 3, 4]
    assert asr.unmerged == [2, 2, 3, 4]
    assert asr.transcribe(10, 3) == [2, 3, 3, 4, 1]  # a blank between two 3s keeps both


def test_arguments_the_reference_gets_wrong_are_refused():
    model, _ = make_model()
    with pytest.raises(ValueError):
        cn.FrameBatchASR(model, frame_len=0.155)            # 15.5 feature frames
    with pytest.raises(ValueError):
        cn.FrameBatchASR(model, total_buffer=0.3333)
    with pytest.raises(ValueError):
        cn.FrameBatchASR(model, frame_len=4.0, total_buffer=1.6)  # fl > W
    with pytest.raises(ValueError):
        cn.FrameBatchASR(model, batch_size=0)
    asr = cn.FrameBatchASR(model, frame_len=1.6, total_buffer=4.0)
    assert (asr.n_frame_len, asr.n_buffer_len, asr.window_tokens, asr.blank_id) == (160, 400, 100, 128)
    asr.read_audio_file(np.zeros(16000, np.float32), 70, STRIDE_SECS)
    with pytest.raises(ValueError):
        asr.transcribe(40, 100)                              # Lw - 1 - delay < 0: Python would index from the end
    with pytest.raises(ValueError):
        asr.transcribe(0, 70)
    with pytest.raises(NotImplementedError):
        asr.read_audio_file("/data/a.wav", 70, STRIDE_SECS)  # audio decoding stays with the caller
    with pytest.raises(ValueError):
        cn.buffered_ctc_transcribe(model, [np.zeros(100, np.float32)], 1.6, 4.0, 40, -1, STRIDE_SECS)
    with pytest.raises(TypeError):
        cn.FrameBatchASR(types.SimpleNamespace(_cfg=model._cfg, encoder=torch.nn.Linear(2, 2), decoder=model.decoder))
    assert cn.buffered_ctc_transcribe(model, [], 1.6, 4.0, 40, 70, STRIDE_SECS) == []


def test_preprocessor_accepts_normalize_none():
    for value in (None, "None"):
        p = cn.AudioToMelSpectrogramPreprocessor(**{**{k: v for k, v in PRE.items() if k != "_target_"}, "normalize": value})
        assert p.normalize is None
    for value in ("all_features", "per_utterance"):
        with pytest.raises(NotImplementedError):
            cn.AudioToMelSpectrogramPreprocessor(**{**{k: v for k, v in PRE.items() if k != "_target_"}, "normalize": value})


def test_oracle_matches_live_reference_when_mounted():
    from oracle import reference_loader as rl

    if not rl.reference_available():
        pytest.skip("reference tree not mounted")
    su = bo.load_reference_streaming_utils()
    x = np.random.default_rng(3).standard_normal((80, 1003)).astype(np.float32)
    feats = torch.from_numpy(x)[None]

    class RawPreprocessor:  # what AudioFeatureIterator calls: preprocessor(input_signal=, length=) and ._cfg
        _cfg = {"window_stride": 0.01}

        def __call__(self, input_signal, length):
            return feats, torch.tensor([x.shape[1]])

    model = types.SimpleNamespace(preprocessor=types.SimpleNamespace(log=True), _cfg=types.SimpleNamespace(
        sample_rate=16000, preprocessor=types.SimpleNamespace(window_stride=0.01, features=80)))
    ref = su.FeatureFrameBufferer(asr_model=model, frame_len=1.6, batch_size=4, total_buffer=4.0)
    ref.set_frame_reader(su.AudioFeatureIterator(np.zeros(1000, np.float32), 1.6, RawPreprocessor(), "cpu"))
    want = []
    while True:
        batch = ref.get_buffers_batch()
        if not batch:
            break
        want += batch
    got = bo.file_windows(np.zeros(1000, np.float32), fake_featurize(x), 80, 0.01, 1.6, 4.0)
    assert np.array_equal(np.stack(want), got)
    asr = su.FrameBatchASR.__new__(su.FrameBatchASR)  # the merge, on fixed predictions
    asr.blank_id, asr.tokenizer = 5, types.SimpleNamespace(ids_to_text=lambda ids: list(ids))
    asr.frame_bufferer = types.SimpleNamespace(get_buffers_batch=lambda: [])
    asr.all_preds = [np.array([0, 1, 1, 5, 2, 2, 3, 5]), np.array([2, 5, 5, 3, 3, 4, 4, 1])]
    mine = bo.FrameBatchASR(None, None, 3, 0.01, 16000, blank_id=5)
    mine.all_preds, mine.infer_logits = asr.all_preds, (lambda: None)
    for tpc, delay in ((2, 3), (10, 3), (3, 0)):
        assert asr.transcribe(tpc, delay) == mine.transcribe(tpc, delay)


# ---------------------------------------------------------------------------------------------------------------- GPU

def _pre(**kw):
    args = {k: v for k, v in PRE.items() if k != "_target_"}
    args.update(pad_to=0, dither=0.0)
    args.update(kw)
    return cn.AudioToMelSpectrogramPreprocessor(**args)


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,lens", [(4, 80000, [80000, 51234, 16000, 401]), (1, 320000, [320000])])
def test_raw_logmel_kernel_matches_oracle(B, L, lens):
    x, lengths = fo.synthetic_waveforms(B, L, lens, seed=L % 89)
    p = _pre(normalize=None)
    want, wl = bo.raw_filterbank_features(x, lengths, p.featurizer.window, p.featurizer.fb[0])
    y, yl = p.cuda()(input_signal=x.cuda(), length=lengths.cuda())
    torch.cuda.synchronize()
    assert torch.equal(yl.cpu(), wl) and y.shape == want.shape
    d = (y.cpu().double() - want.double()).abs()
    # raw log-mel values (std ~ 2 - 4 per row): the front end's 2e-3 on unit-variance features, scaled back
    assert int(torch.isnan(y).sum()) == 0 and float(d.max()) <= 1e-2 and float(d.norm() / want.double().norm()) <= 2e-4
    for b, n in enumerate(wl.tolist()):
        assert torch.all(y[b, :, n:] == 0)
    # the normalising entry point on the same input is the raw one followed by the per-feature statistics
    yn, _ = _pre(normalize="per_feature").cuda()(input_signal=x.cuda(), length=lengths.cuda())
    for b, n in enumerate(wl.tolist()):
        r = y[b, :, :n].double()
        ref = (r - r.mean(1, keepdim=True)) / (r.std(1, keepdim=True) + 1e-5)
        assert float((yn[b, :, :n].double() - ref).abs().max()) <= 1e-3


@pytest.mark.gpu
def test_raw_logmel_one_frame_is_not_an_error():
    p = _pre(normalize="None").cuda()
    y, yl = p(input_signal=torch.randn(2, 2000, device="cuda"), length=torch.tensor([2000, 100], device="cuda"))
    torch.cuda.synchronize()
    assert yl.tolist() == [13, 1] and torch.all(y[1, :, 1:] == 0)


def feature_buffers(feats, seq_len, n_win, fl, W):
    from gpu_util import ptr, stream
    from conformer_nemo_b200 import _lib

    first = torch.tensor(np.concatenate([[0], np.cumsum(n_win[:-1])]), dtype=torch.int32, device="cuda")
    out = torch.empty(int(sum(n_win)), feats.shape[1], W, device="cuda")
    rc = _lib.load_library().cfb_op_feature_buffers(ptr(feats), feats.shape[0], feats.shape[1], feats.shape[2],
                                                    ptr(seq_len), ptr(first), out.shape[0], fl, W, ptr(out), stream())
    assert rc == 0, _lib.last_error(None)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("fl,W", [(160, 400), (16, 40), (50, 50), (300, 1100)])  # W > 1024: the three-pass form
def test_window_kernel_matches_float64_oracle(fl, W):
    """Ragged multi-file batches, one file of five minutes (30001 frames) included."""
    g = torch.Generator().manual_seed(fl)
    lens = [30001, 7, 2 * fl, 1003, W + 1] if fl == 160 else [7, 2 * fl, 311, W + 1, 3 * fl + 5]
    T = max(lens) + 3
    feats = torch.randn(len(lens), 80, T, generator=g) * 3 - 8
    n_win = [n // fl + 1 for n in lens]
    got = feature_buffers(feats.cuda(), torch.tensor(lens).cuda(), n_win, fl, W).cpu()
    w0 = 0
    for f, n in enumerate(lens):
        x = feats[f, :, :n].double().numpy()
        want = bo.file_windows(np.zeros(10, np.float32), fake_featurize(x), 80, 0.01, fl * 0.01, W * 0.01, dtype=np.float64)
        assert want.shape[0] == n_win[f]
        assert float(np.abs(got[w0:w0 + n_win[f]].double().numpy() - want).max()) <= 2e-4, f
        w0 += n_win[f]
    # the output of one file does not depend on the other files of the call
    alone = feature_buffers(feats[3:4].cuda(), torch.tensor(lens[3:4]).cuda(), n_win[3:4], fl, W)
    k = sum(n_win[:3])
    assert torch.equal(alone.cpu(), got[k:k + n_win[3]])


def synthetic_files(seconds, seed):
    lens = [int(s * 16000) for s in seconds]
    x, _ = fo.synthetic_waveforms(len(lens), max(lens), lens, seed=seed)
    return [x[i, :n].numpy() for i, n in enumerate(lens)]


def oracle_pipeline(model_parts, audio, tokens_per_chunk, delay, pad_delay=None):
    cfg, enc_sd, head_sd = model_parts
    pre = _pre(normalize=None)
    asr = bo.FrameBatchASR(bo.raw_featurizer(pre.featurizer.window, pre.featurizer.fb[0]),
                           bo.ctc_model(enc_sd, cfg, head_sd), 80, 0.01, 16000, blank_id=128)
    asr.read_audio_file(audio, delay if pad_delay is None else pad_delay, STRIDE_SECS)
    return asr, asr.transcribe(tokens_per_chunk, delay)


@pytest.mark.gpu
def test_end_to_end_against_the_oracle_pipeline():
    """Per-window arg-max agreement >= 99 % with the oracle model (the project's CTC criterion); the merge of the GPU's own
    predictions equals the oracle's merge of them exactly."""
    model, parts = make_model(device="cuda")
    tpc, delay = nemo_chunking()
    assert (tpc, delay) == (40, 70)
    audios = synthetic_files([3.3, 7.1, 1.0], seed=4)
    ids, preds = cn.FrameBatchASR(model).decode(audios, int(delay * STRIDE_SECS * 16000), tpc, delay)
    agree = total = 0
    for f, audio in enumerate(audios):
        ref, want_ids = oracle_pipeline(parts, audio, tpc, delay)
        assert len(preds[f]) == len(ref.all_preds)
        for p, q in zip(preds[f], ref.all_preds):
            agree += int((torch.from_numpy(p) == torch.from_numpy(q)).sum())
            total += q.size
        ref.all_preds, ref.infer_logits = preds[f], (lambda: None)
        assert ids[f] == ref.transcribe(tpc, delay)
    assert total >= 1000 and agree / total >= 0.99, agree / total


@pytest.mark.gpu
@pytest.mark.parametrize("tpc,delay", [(40, 70), (200, 10), (1, 0)])
def test_merge_equals_the_oracle_merge_and_short_pads(tpc, delay):
    """Slices clipped at Lw, delay 0 (no pad: every file's front end runs on its own) and a single-token slice."""
    model, _ = make_model(device="cuda", seed=3)
    audios = synthetic_files([2.0, 5.5], seed=6)
    asr = cn.FrameBatchASR(model)
    ids, preds = asr.decode(audios, int(delay * STRIDE_SECS * 16000), tpc, delay)
    for f in range(2):
        ref = bo.FrameBatchASR(None, None, 80, 0.01, 16000, blank_id=128)
        ref.all_preds, ref.infer_logits = preds[f], (lambda: None)
        assert ids[f] == ref.transcribe(tpc, delay)
    asr.read_audio_file(audios[1], delay, STRIDE_SECS)
    assert asr.transcribe(tpc, delay) == Tokenizer().ids_to_text(ids[1])
    assert len(asr.all_preds) == len(preds[1]) and all(np.array_equal(a, b) for a, b in zip(asr.all_preds, preds[1]))


@pytest.mark.gpu
def test_a_file_gives_the_same_bits_alone_among_others_and_with_any_batch_size():
    model, _ = make_model(device="cuda", seed=7)
    tpc, delay = nemo_chunking()
    audios = synthetic_files([4.0, 11.3, 0.5, 6.2], seed=8)
    asr = cn.FrameBatchASR(model, batch_size=4)
    asr.read_audio_file(audios[1], delay, STRIDE_SECS)
    text = asr.transcribe(tpc, delay)
    alone = [p.copy() for p in asr.all_preds]
    for bs, graphs in ((1, False), (4, False), (7, True), (64, False), (64, True)):
        model.encoder.enable_cuda_graphs(graphs)
        ids = cn.buffered_ctc_transcribe(model, audios, 1.6, 4.0, tpc, delay, STRIDE_SECS, batch_size=bs)
        _, preds = cn.FrameBatchASR(model, batch_size=bs).decode(audios[::-1], int(delay * STRIDE_SECS * 16000), tpc, delay)
        assert Tokenizer().ids_to_text(ids[1]) == text, bs
        assert all(np.array_equal(a, b) for a, b in zip(preds[2], alone)) and len(preds[2]) == len(alone), bs
    model.encoder.enable_cuda_graphs(False)
