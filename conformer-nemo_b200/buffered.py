"""Buffered long-audio CTC inference on the B200: drop-in for the reference's ``FrameBatchASR``
(nemo/collections/asr/parts/utils/streaming_utils.py:455-684: ``AudioFeatureIterator``, ``FeatureFrameBufferer``,
``FrameBatchASR``), restated in oracle/buffered_oracle.py.

A long recording is not run through one full-context forward.  Its raw log-mel features (no normalisation) are cut into
``frame_len`` chunks; every chunk becomes the right edge of a ``total_buffer`` window, normalised on its own statistics;
every window goes through the encoder and the CTC head; from each window's greedy predictions the ``tokens_per_chunk``
that end ``delay`` frames before the window's end are kept, concatenated over the file and collapsed.

Here all of it stays on the device, for many files at once: one raw log-mel call (``cfb_op_logmel_raw``), one window
kernel (``cfb_op_feature_buffers``), the encoder in chunks of ``batch_size`` windows, the head's arg-max, a gather of the
kept slices and the existing collapse kernel (``cfb_op_ctc_collapse``).  The host reads the ids once, at the end.
"""
from __future__ import annotations

import ctypes
import os
from collections.abc import Mapping
from typing import List, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .ctc_head import ConvASRDecoder, ctc_collapse_device
from .encoder import ConformerEncoder
from .preprocessor import AudioToMelSpectrogramPreprocessor


def _field(obj, name):
    return obj[name] if isinstance(obj, Mapping) else getattr(obj, name)


def _frames(seconds: float, stride: float, what: str) -> int:
    """Feature frames in ``seconds``.  The reference truncates ``seconds / stride`` with int(); a ratio that is not whole
    (within 1e-6) makes its chunk boundaries drift on long files, so it is refused here."""
    ratio = seconds / stride
    n = int(round(ratio))
    if n < 1 or abs(ratio - n) > 1e-6:
        raise ValueError(f"{what} / window_stride = {ratio!r} is not a positive whole number of feature frames")
    return n


class FrameBatchASR:
    """``FrameBatchASR(asr_model, frame_len=1.6, total_buffer=4.0, batch_size=4)`` as in the reference.

    ``asr_model`` is duck-typed: ``_cfg.preprocessor`` (the preprocessor config), ``_cfg.sample_rate``, ``encoder`` (the
    B200 ``ConformerEncoder``), ``decoder`` (the B200 ``ConvASRDecoder``) and ``tokenizer`` (``ids_to_text``).
    ``batch_size`` is the number of windows per encoder forward; the results do not depend on it."""

    def __init__(self, asr_model, frame_len: float = 1.6, total_buffer: float = 4.0, batch_size: int = 4):
        if not isinstance(asr_model.encoder, ConformerEncoder):
            raise TypeError("FrameBatchASR (B200): asr_model.encoder must be conformer_nemo_b200.ConformerEncoder")
        if not isinstance(asr_model.decoder, ConvASRDecoder):
            raise TypeError("FrameBatchASR (B200): asr_model.decoder must be conformer_nemo_b200.ConvASRDecoder")
        if int(batch_size) < 1:
            raise ValueError("batch_size must be >= 1")
        self.asr_model = asr_model
        self.encoder, self.decoder = asr_model.encoder, asr_model.decoder
        self.tokenizer = getattr(asr_model, "tokenizer", None)
        self.frame_len, self.total_buffer, self.batch_size = frame_len, total_buffer, int(batch_size)
        self.sample_rate = _field(asr_model._cfg, "sample_rate")
        pcfg = _field(asr_model._cfg, "preprocessor")
        kwargs = {k: v for k, v in (pcfg.items() if isinstance(pcfg, Mapping) else vars(pcfg).items())
                  if not str(k).startswith("_")}  # drops Hydra's _target_
        kwargs.update(dither=0.0, pad_to=0, normalize="None")  # what the reference sets for its raw_preprocessor
        self.raw_preprocessor = AudioToMelSpectrogramPreprocessor(**kwargs)
        stride = _field(pcfg, "window_stride")
        self.n_frame_len = _frames(frame_len, stride, "frame_len")
        self.n_buffer_len = _frames(total_buffer, stride, "total_buffer")
        if self.n_frame_len > self.n_buffer_len:
            raise ValueError(f"frame_len ({frame_len} s) is longer than total_buffer ({total_buffer} s)")
        self.n_feat = self.raw_preprocessor.nfilt
        if self.n_feat != self.encoder._feat_in:
            raise ValueError(f"the preprocessor gives {self.n_feat} features, the encoder takes {self.encoder._feat_in}")
        self.window_tokens = self.encoder.output_frames(self.n_buffer_len)  # Lw: predictions per window
        self.blank_id = self.decoder.num_classes_with_blank - 1
        self.reset()

    def reset(self) -> None:
        self.all_preds: List[np.ndarray] = []
        self.unmerged: List[int] = []
        self._samples = None

    def read_audio_file(self, audio, delay: int, model_stride_in_secs: float) -> None:
        """``audio``: 1-D float samples at the model's rate (array or tensor).  Like the reference, appends
        ``int(delay * model_stride_in_secs * sample_rate)`` zero samples.  Audio decoding stays with the caller."""
        pad = int(delay * model_stride_in_secs * self.sample_rate)
        self._samples = (_waveform(audio), pad)

    def transcribe(self, tokens_per_chunk: int, delay: int) -> str:
        if self._samples is None:
            raise RuntimeError("FrameBatchASR.transcribe: call read_audio_file first")
        samples, pad = self._samples
        ids, preds = self.decode([samples], pad, tokens_per_chunk, delay)
        start, end = self._slice(tokens_per_chunk, delay)
        self.all_preds = preds[0]
        self.unmerged = [int(p) for pred in self.all_preds for p in pred[start:end]]
        return self.tokenizer.ids_to_text(ids[0])

    def _slice(self, tokens_per_chunk: int, delay: int) -> Tuple[int, int]:
        start = self.window_tokens - 1 - int(delay)
        if start < 0:  # Python would index from the end
            raise ValueError(f"delay={delay} reaches before the start of a window of {self.window_tokens} predictions")
        if int(tokens_per_chunk) < 1:
            raise ValueError("tokens_per_chunk must be >= 1")
        return start, min(start + int(tokens_per_chunk), self.window_tokens)

    @torch.no_grad()
    def decode(self, audios: Sequence, pad: int, tokens_per_chunk: int, delay: int, timeline: list = None):
        """The pipeline for many files: ``audios`` 1-D waveforms, each followed by ``pad`` zero samples.  Returns (merged
        ids per file, per-window arg-max predictions per file as int64 numpy rows).  ``timeline``: a list that receives
        (stage, CUDA event) pairs, one event recorded at the start and one at the end of every stage (tools/bench_buffered.py)."""
        start, end = self._slice(tokens_per_chunk, delay)
        wavs = [_waveform(a) for a in audios]
        if not wavs:
            return [], []
        dev = next(self.encoder.parameters()).device
        pre = self.raw_preprocessor
        n_samples = [int(w.numel()) + int(pad) for w in wavs]
        seq_len = pre.get_seq_len(torch.tensor(n_samples, dtype=torch.int64)).tolist()  # the device's float32 formula
        n_win = [n // self.n_frame_len + 1 for n in seq_len]  # the first chunk that does not fit is the last one
        first = np.concatenate([[0], np.cumsum(n_win[:-1])]).astype(np.int64)
        n_files, n_windows, fl, W = len(wavs), int(sum(n_win)), self.n_frame_len, self.n_buffer_len
        with torch.cuda.device(dev):
            _mark(timeline, "start")
            # Raw log-mel.  With a trailing zero pad longer than n_fft / 2 + 1 samples the reflect padding of a file alone
            # and the zero padding of a batch row read the same zeros (pre-emphasis included), so the features of a file in
            # the batch equal its features alone bit for bit.  With a shorter pad each file runs on its own.
            shared = int(pad) >= pre.n_fft // 2 + 2
            groups = [list(range(n_files))] if shared else [[i] for i in range(n_files)]
            parts = []
            for g in groups:
                x = torch.zeros(len(g), max(n_samples[i] for i in g), dtype=torch.float32, device=dev)
                for r, i in enumerate(g):
                    x[r, :wavs[i].numel()] = _to_device(wavs[i], dev)
                lens = _to_device(torch.tensor([n_samples[i] for i in g], dtype=torch.int64), dev)
                parts.append(pre.get_features(x, lens))
            if len(parts) == 1:
                feats, feat_len = parts[0]
            else:
                feats = torch.empty(n_files, self.n_feat, max(f.shape[2] for f, _ in parts), device=dev)
                feat_len = torch.empty(n_files, dtype=torch.int64, device=dev)
                for i, (f, ln) in enumerate(parts):  # frames behind seq_len are never read
                    feats[i, :, :f.shape[2]] = f[0]
                    feat_len[i] = ln[0]
            _mark(timeline, "raw_logmel")
            # every window of every file, normalised
            first_dev = _to_device(torch.from_numpy(first.astype(np.int32)), dev)
            windows = torch.empty(n_windows, self.n_feat, W, dtype=torch.float32, device=dev)
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            vp = ctypes.c_void_p
            _lib.check(_lib.load_library().cfb_op_feature_buffers(
                vp(feats.data_ptr()), n_files, self.n_feat, feats.shape[2], vp(feat_len.data_ptr()), vp(first_dev.data_ptr()),
                n_windows, fl, W, vp(windows.data_ptr()), stream), None, "cfb_op_feature_buffers")
            _mark(timeline, "windows")
            # encoder + head in chunks of batch_size windows (each chunk's output is consumed before the next forward:
            # with CUDA graphs on, the encoder returns its graph's static buffer)
            best = torch.empty(n_windows, self.window_tokens, dtype=torch.int32, device=dev)
            for i in range(0, n_windows, self.batch_size):
                enc, _ = self.encoder(audio_signal=windows[i:i + self.batch_size])
                _mark(timeline, "encoder")
                best[i:i + self.batch_size] = self.decoder.forward_with_predictions(enc, _int32_predictions=True)[1]
                _mark(timeline, "head")
            # merge: the kept slice of every window, concatenated per file, then the greedy collapse
            width, most = end - start, max(n_win)
            rows = [[int(first[f]) + min(k, n_win[f] - 1) for k in range(most)] for f in range(n_files)]
            merged = best[:, start:end][_to_device(torch.tensor(rows, dtype=torch.int64), dev)].reshape(n_files, most * width)
            merged_len = _to_device(torch.tensor([n * width for n in n_win], dtype=torch.int32), dev)
            tokens, n_tokens = ctc_collapse_device(merged, merged_len, self.blank_id)
            _mark(timeline, "merge")
            host = torch.cat([n_tokens, tokens.flatten(), best.flatten()]).cpu().numpy()  # the one read back
        counts = host[:n_files]
        toks = host[n_files:n_files + tokens.numel()].reshape(n_files, -1)
        preds = host[n_files + tokens.numel():].reshape(n_windows, self.window_tokens).astype(np.int64)
        ids = [toks[f, :counts[f]].tolist() for f in range(n_files)]
        return ids, [list(preds[first[f]:first[f] + n_win[f]]) for f in range(n_files)]


def buffered_ctc_transcribe(asr_model, audios: Sequence, frame_len: float, total_buffer: float, tokens_per_chunk: int,
                            delay: int, model_stride_in_secs: float, batch_size: int = 4) -> List[List[int]]:
    """Buffered CTC inference of many files, every window of every file batched together: one id list per file, each
    equal to what ``FrameBatchASR`` gives for that file alone (``read_audio_file`` + ``transcribe`` before the tokenizer).
    ``audios``: 1-D waveforms at the model's rate, each padded with ``int(delay * model_stride_in_secs * sample_rate)``
    zero samples as the reference does.  A ``FrameBatchASR`` kept across calls (its ``decode``) also keeps its front end's
    filter bank on the device."""
    asr = FrameBatchASR(asr_model, frame_len, total_buffer, batch_size)
    pad = int(delay * model_stride_in_secs * asr.sample_rate)
    return asr.decode(audios, pad, tokens_per_chunk, delay)[0]


def _waveform(audio) -> torch.Tensor:
    if isinstance(audio, (str, bytes, os.PathLike)):
        raise NotImplementedError("FrameBatchASR (B200) takes samples, not a path: decode the audio file first")
    t = audio if torch.is_tensor(audio) else torch.from_numpy(np.ascontiguousarray(audio, dtype=np.float32))
    if t.dim() != 1:
        raise ValueError(f"audio must be 1-D samples, got shape {tuple(t.shape)}")
    return t.to(torch.float32)


def _mark(timeline, stage: str) -> None:
    if timeline is not None:
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        timeline.append((stage, ev))


def _to_device(t: torch.Tensor, dev) -> torch.Tensor:
    """Host tensors go through pinned memory so that the copy does not wait for the device."""
    if t.is_cuda:
        return t
    return t.contiguous().pin_memory().to(dev, non_blocking=True)
