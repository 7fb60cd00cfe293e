"""Buffered long-audio inference on the B200: drop-ins for the reference's ``FrameBatchASR`` (CTC) and
``BatchedFrameASRRNNT`` (transducer) of nemo/collections/asr/parts/utils/streaming_utils.py (``AudioFeatureIterator``,
``FeatureFrameBufferer``, ``BatchedFeatureFrameBufferer``, ``FrameBatchASR``, ``BatchedFrameASRRNNT``), restated in
oracle/buffered_oracle.py and oracle/buffered_rnnt_oracle.py.

A long recording is not run through one full-context forward.  Its raw log-mel features (no normalisation) are cut into
``frame_len`` chunks; every chunk becomes the right edge of a ``total_buffer`` window, normalised on its own statistics;
every window goes through the encoder.  CTC keeps, from each window's greedy predictions, the ``tokens_per_chunk`` that
end ``delay`` frames before the window's end, concatenates them over the file and collapses them.  The transducer decodes
every window from a blank state and keeps the tokens emitted at the window's middle frames (the "middle token" merge),
concatenated over the file without a collapse.

Here all of it stays on the device, for many files at once: one raw log-mel call (``cfb_op_logmel_raw``), one window
kernel (``cfb_op_feature_buffers``), the encoder in chunks of windows, then the head's arg-max or the greedy transducer
decode (``cfb_op_rnnt_greedy``) of each chunk, and a gather of the kept tokens.  The host waits for the device once, at
the end.
"""
from __future__ import annotations

import ctypes
import os
from collections.abc import Mapping
from typing import Callable, List, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .ctc_head import ConvASRDecoder, ctc_collapse_device
from .encoder import ConformerEncoder
from .preprocessor import AudioToMelSpectrogramPreprocessor
from .rnnt import GreedyBatchedRNNTInfer, RNNTDecoder, RNNTJoint


def _field(obj, name):
    return obj[name] if isinstance(obj, Mapping) else getattr(obj, name)


def _optional(obj, name):
    if obj is None:
        return None
    return obj.get(name) if isinstance(obj, Mapping) else getattr(obj, name, None)


def _frames(seconds: float, stride: float, what: str) -> int:
    """Feature frames in ``seconds``.  The reference truncates ``seconds / stride`` with int(); a ratio that is not whole
    (within 1e-6) makes its chunk boundaries drift on long files, so it is refused here."""
    ratio = seconds / stride
    n = int(round(ratio))
    if n < 1 or abs(ratio - n) > 1e-6:
        raise ValueError(f"{what} / window_stride = {ratio!r} is not a positive whole number of feature frames")
    return n


class _BufferedASR:
    """What the buffered CTC and transducer classes share: the raw front end built from the model's preprocessor config,
    the chunk and window widths, and the device pipeline from waveforms to the encoder output of every window."""

    _name = None  # the class the error messages name

    def __init__(self, asr_model, frame_len: float, total_buffer: float):
        if not isinstance(asr_model.encoder, ConformerEncoder):
            raise TypeError(f"{self._name} (B200): asr_model.encoder must be conformer_nemo_b200.ConformerEncoder")
        self.asr_model = asr_model
        self.encoder = asr_model.encoder
        self.tokenizer = getattr(asr_model, "tokenizer", None)
        self.frame_len, self.total_buffer = frame_len, total_buffer
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
        self.window_tokens = self.encoder.output_frames(self.n_buffer_len)  # Lw: encoder frames per window

    def _windows(self, wavs: List[torch.Tensor], pad: int, dev, timeline) -> Tuple[torch.Tensor, np.ndarray, List[int]]:
        """Raw log-mel of the waveforms (each followed by ``pad`` zero samples), then every normalised window of every
        file: (windows (n_windows, F, W) fp32, first window of each file, windows per file).  Enqueue-only."""
        pre = self.raw_preprocessor
        n_samples = [int(w.numel()) + int(pad) for w in wavs]
        seq_len = pre.get_seq_len(torch.tensor(n_samples, dtype=torch.int64)).tolist()  # the device's float32 formula
        n_win = [n // self.n_frame_len + 1 for n in seq_len]  # the first chunk that does not fit is the last one
        first = np.concatenate([[0], np.cumsum(n_win[:-1])]).astype(np.int64)
        n_files, n_windows, fl, W = len(wavs), int(sum(n_win)), self.n_frame_len, self.n_buffer_len
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
        first_dev = _to_device(torch.from_numpy(first.astype(np.int32)), dev)
        windows = torch.empty(n_windows, self.n_feat, W, dtype=torch.float32, device=dev)
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        vp = ctypes.c_void_p
        _lib.check(_lib.load_library().cfb_op_feature_buffers(
            vp(feats.data_ptr()), n_files, self.n_feat, feats.shape[2], vp(feat_len.data_ptr()), vp(first_dev.data_ptr()),
            n_windows, fl, W, vp(windows.data_ptr()), stream), None, "cfb_op_feature_buffers")
        _mark(timeline, "windows")
        return windows, first, n_win

    def _encode(self, windows: torch.Tensor, per_forward: int, consume: Callable, timeline) -> None:
        """The encoder over ``windows`` in chunks of ``per_forward``; ``consume(i, encoded)`` gets the output of windows
        ``[i, i + len)`` and must enqueue all its reads of it before it returns: with CUDA graphs on, the encoder returns its
        graph's static buffer, which the next forward overwrites."""
        for i in range(0, windows.shape[0], per_forward):
            enc, _ = self.encoder(audio_signal=windows[i:i + per_forward])
            _mark(timeline, "encoder")
            consume(i, enc)


class FrameBatchASR(_BufferedASR):
    """``FrameBatchASR(asr_model, frame_len=1.6, total_buffer=4.0, batch_size=4)`` as in the reference.

    ``asr_model`` is duck-typed: ``_cfg.preprocessor`` (the preprocessor config), ``_cfg.sample_rate``, ``encoder`` (the
    B200 ``ConformerEncoder``), ``decoder`` (the B200 ``ConvASRDecoder``) and ``tokenizer`` (``ids_to_text``).
    ``batch_size`` is the number of windows per encoder forward; the results do not depend on it."""

    _name = "FrameBatchASR"

    def __init__(self, asr_model, frame_len: float = 1.6, total_buffer: float = 4.0, batch_size: int = 4):
        if not isinstance(asr_model.decoder, ConvASRDecoder):
            raise TypeError("FrameBatchASR (B200): asr_model.decoder must be conformer_nemo_b200.ConvASRDecoder")
        if int(batch_size) < 1:
            raise ValueError("batch_size must be >= 1")
        super().__init__(asr_model, frame_len, total_buffer)
        self.decoder = asr_model.decoder
        self.batch_size = int(batch_size)
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
        self._samples = (_waveform(audio, self._name), pad)

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
        wavs = [_waveform(a, self._name) for a in audios]
        if not wavs:
            return [], []
        dev = next(self.encoder.parameters()).device
        n_files = len(wavs)
        with torch.cuda.device(dev):
            windows, first, n_win = self._windows(wavs, pad, dev, timeline)
            n_windows = windows.shape[0]
            # encoder + head in chunks of batch_size windows
            best = torch.empty(n_windows, self.window_tokens, dtype=torch.int32, device=dev)

            def head(i, enc):
                best[i:i + self.batch_size] = self.decoder.forward_with_predictions(enc, _int32_predictions=True)[1]
                _mark(timeline, "head")

            self._encode(windows, self.batch_size, head, timeline)
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


class BatchedFrameASRRNNT(_BufferedASR):
    """``BatchedFrameASRRNNT(asr_model, frame_len=1.6, total_buffer=4.0, batch_size=32, max_steps_per_timestep=5,
    stateful_decoding=False)`` as in the reference, with the "middle token" merge of its ``transcribe``.

    ``asr_model`` is duck-typed: ``_cfg.preprocessor``, ``_cfg.sample_rate``, optionally ``_cfg.decoding.greedy.max_symbols``
    (absent: ``None``, no limit per frame), the B200 ``encoder`` (``ConformerEncoder``), ``decoder`` (``RNNTDecoder``)
    and ``joint`` (``RNNTJoint``), and ``tokenizer`` (``ids_to_text``).  ``batch_size`` is the number of files
    ``read_audio_file`` takes, as in the reference; ``windows_per_forward`` is the number of windows per encoder forward,
    and the results do not depend on it.  ``max_steps_per_timestep`` is kept as an attribute; the symbol limit per frame
    is the model's ``decoding.greedy.max_symbols``, as with the reference's decoding object."""

    _name = "BatchedFrameASRRNNT"

    def __init__(self, asr_model, frame_len: float = 1.6, total_buffer: float = 4.0, batch_size: int = 32,
                 max_steps_per_timestep: int = 5, stateful_decoding: bool = False, windows_per_forward: int = 256):
        if stateful_decoding:
            raise NotImplementedError("BatchedFrameASRRNNT (B200): stateful_decoding (partial hypotheses across windows); "
                                      "every window is decoded from a blank state")
        if not isinstance(getattr(asr_model, "decoder", None), RNNTDecoder):
            raise TypeError("BatchedFrameASRRNNT (B200): asr_model.decoder must be conformer_nemo_b200.RNNTDecoder")
        if not isinstance(getattr(asr_model, "joint", None), RNNTJoint):
            raise TypeError("BatchedFrameASRRNNT (B200): asr_model.joint must be conformer_nemo_b200.RNNTJoint")
        if int(batch_size) < 1 or int(windows_per_forward) < 1:
            raise ValueError("batch_size and windows_per_forward must be >= 1")
        super().__init__(asr_model, frame_len, total_buffer)
        max_symbols = _optional(_optional(_optional(asr_model._cfg, "decoding"), "greedy"), "max_symbols")
        if max_symbols is not None and int(max_symbols) < 1:
            raise ValueError(f"decoding.greedy.max_symbols must be >= 1 or None, got {max_symbols!r}")
        self.max_symbols = None if max_symbols is None else int(max_symbols)
        self.decoder, self.joint = asr_model.decoder, asr_model.joint
        self.blank_id = self.decoder.blank_idx
        self.greedy = GreedyBatchedRNNTInfer(self.decoder, self.joint, blank_index=self.blank_id,
                                             max_symbols_per_step=self.max_symbols)
        self.batch_size, self.windows_per_forward = int(batch_size), int(windows_per_forward)
        self.max_steps_per_timestep = max_steps_per_timestep
        self.stateful_decoding = False
        # token capacity of a window's first decode: it cannot overflow with a symbol limit; without one a window that
        # outgrows it is decoded again with room for all of its tokens
        Lw = self.window_tokens
        self.initial_capacity = Lw * self.max_symbols if self.max_symbols is not None else 4 * Lw + 64
        self.reset()

    def reset(self) -> None:
        self.all_preds: List[List[np.ndarray]] = [[] for _ in range(self.batch_size)]
        self.unmerged: List[List[int]] = [[] for _ in range(self.batch_size)]
        self._samples = None

    def read_audio_file(self, audios: Sequence, delay: int, model_stride_in_secs: float) -> None:
        """``audios``: exactly ``batch_size`` 1-D float waveforms at the model's rate (arrays or tensors).  Like the
        reference, each gets ``int(delay * model_stride_in_secs * sample_rate)`` zero samples appended."""
        if isinstance(audios, (str, bytes, os.PathLike)):
            _waveform(audios, self._name)
        if len(audios) != self.batch_size:
            raise ValueError(f"read_audio_file takes batch_size = {self.batch_size} files, got {len(audios)}")
        pad = int(delay * model_stride_in_secs * self.sample_rate)
        self._samples = ([_waveform(a, self._name) for a in audios], pad)

    def transcribe(self, tokens_per_chunk: int, delay: int) -> List[str]:
        if self._samples is None:
            raise RuntimeError("BatchedFrameASRRNNT.transcribe: call read_audio_file first")
        samples, pad = self._samples
        ids, decodes = self.decode(samples, pad, tokens_per_chunk, delay)
        self.all_preds = [[tokens for tokens, _ in d] for d in decodes]
        self.unmerged = ids
        return [self.tokenizer.ids_to_text(i) for i in ids]

    def _slice(self, tokens_per_chunk: int, delay: int) -> Tuple[int, int]:
        """Frames ``[lo, hi)`` of a window whose tokens are kept: the reference's
        ``alignment[Lw - offset - delay : Lw - offset - delay + tokens_per_chunk]`` with ``offset = 0 if delay == Lw else 1``."""
        Lw, delay = self.window_tokens, int(delay)
        if delay < 0:
            raise ValueError(f"delay must be >= 0, got {delay}")
        lo = Lw - (0 if delay == Lw else 1) - delay
        if lo < 0:  # Python would index from the end
            raise ValueError(f"delay={delay} reaches before the start of a window of {Lw} encoder frames")
        if int(tokens_per_chunk) < 1:
            raise ValueError("tokens_per_chunk must be >= 1")
        return lo, min(lo + int(tokens_per_chunk), Lw)

    def _decode_windows(self, windows: torch.Tensor, cap: int, timeline):
        """Encoder and greedy decode of ``windows`` with room for ``cap`` tokens each: (tokens, timesteps (n, cap) int32,
        n_tokens (n,) int32 -- the full count, also when it exceeds ``cap`` --, flags (1,) int32).  Enqueue-only."""
        n, dev = windows.shape[0], windows.device
        i32 = dict(dtype=torch.int32, device=dev)
        tokens, steps = torch.empty(n, cap, **i32), torch.empty(n, cap, **i32)
        counts, flags = torch.empty(n, **i32), torch.zeros(1, **i32)
        lens = torch.full((min(n, self.windows_per_forward),), self.window_tokens, **i32)

        def decode(i, enc):
            out = self.greedy.decode_arrays(enc, lens[:enc.shape[0]], max_tokens=cap)
            j = i + enc.shape[0]
            tokens[i:j], steps[i:j], counts[i:j] = out["tokens"], out["timesteps"], out["n_tokens"]
            torch.bitwise_or(flags, out["flags"], out=flags)
            _mark(timeline, "decode")

        self._encode(windows, self.windows_per_forward, decode, timeline)
        return tokens, steps, counts, flags

    @torch.no_grad()
    def decode(self, audios: Sequence, pad: int, tokens_per_chunk: int, delay: int, timeline: list = None):
        """The pipeline for any number of files: ``audios`` 1-D waveforms, each followed by ``pad`` zero samples.  Returns
        (merged ids per file, per file the decode of each window as (tokens, timesteps) int64 numpy arrays).
        ``timeline``: a list that receives (stage, CUDA event) pairs (tools/bench_buffered_rnnt.py)."""
        lo, hi = self._slice(tokens_per_chunk, delay)
        wavs = [_waveform(a, self._name) for a in audios]
        if not wavs:
            return [], []
        dev = next(self.encoder.parameters()).device
        n_files, Lw = len(wavs), self.window_tokens
        with torch.cuda.device(dev):
            windows, first, n_win = self._windows(wavs, pad, dev, timeline)
            n_windows = windows.shape[0]
            cap = self.initial_capacity
            tokens, steps, counts, flags = self._decode_windows(windows, cap, timeline)
            first_dev = _to_device(torch.from_numpy(first), dev)
            n_win_dev = _to_device(torch.tensor(n_win, dtype=torch.int64), dev)
            kept_cap = min(cap, (hi - lo) * self.max_symbols) if self.max_symbols is not None else cap
            merged, merged_len = merge_middle_tokens(tokens, steps, counts, first_dev, n_win_dev, max(n_win), kept_cap,
                                                     lo, hi, Lw)
            _mark(timeline, "merge")
            head = torch.cat([flags, counts, merged_len]).cpu()  # the one wait for the device
            if int(head[0]) & 2:
                raise RuntimeError("GreedyBatchedRNNTInfer (B200): runaway emission with max_symbols_per_step=None "
                                   "(4096 symbols at one frame)")
            n = head[1:1 + n_windows]
            if int(n.max()) > cap:
                # Some windows outgrew the capacity (max_symbols None only): encoder and decode again for those alone, with
                # room for all of their tokens.  Both are deterministic and independent of the other windows of a call, so
                # this gives the bits of one decode with the larger capacity.
                rows = torch.nonzero(n > cap).flatten()
                big = int(n.max())
                t2, s2, c2, f2 = self._decode_windows(windows[rows.to(dev)], big, None)
                grown = torch.empty(n_windows, big, dtype=torch.int32, device=dev)
                grown[:, :cap] = tokens
                tokens = grown.index_copy_(0, rows.to(dev), t2)
                grown = torch.empty(n_windows, big, dtype=torch.int32, device=dev)
                grown[:, :cap] = steps
                steps = grown.index_copy_(0, rows.to(dev), s2)
                cap = kept_cap = big
                merged, merged_len = merge_middle_tokens(tokens, steps, counts, first_dev, n_win_dev, max(n_win), kept_cap,
                                                         lo, hi, Lw)
                head = torch.cat([f2, c2, merged_len]).cpu()
                if int(head[0]) & 2 or not torch.equal(head[1:1 + rows.numel()], n[rows]):
                    raise RuntimeError("BatchedFrameASRRNNT (B200): a window decoded again gave another token count")
            merged_len_h = head[-n_files:]
            # read exactly what the counts say: a buffer sized for the bound holds Lw * max_symbols entries per window
            wm, wt = max(int(merged_len_h.max()), 1), max(int(n.max()), 1)
            host = torch.cat([merged[:, :wm].flatten(), tokens[:, :wt].flatten(), steps[:, :wt].flatten()]).cpu().numpy()
        ids_h = host[:n_files * wm].reshape(n_files, wm)
        toks_h = host[n_files * wm:n_files * wm + n_windows * wt].reshape(n_windows, wt).astype(np.int64)
        steps_h = host[n_files * wm + n_windows * wt:].reshape(n_windows, wt).astype(np.int64)
        ids = [ids_h[f, :int(merged_len_h[f])].tolist() for f in range(n_files)]
        n = n.numpy()
        decodes = [[(toks_h[w, :n[w]].copy(), steps_h[w, :n[w]].copy()) for w in range(first[f], first[f] + n_win[f])]
                   for f in range(n_files)]
        return ids, decodes


def merge_middle_tokens(tokens: torch.Tensor, timesteps: torch.Tensor, n_tokens: torch.Tensor, first: torch.Tensor,
                        n_win: torch.Tensor, max_windows: int, kept_cap: int, lo: int, hi: int, frames: int):
    """The middle-token merge with tensor ops and no synchronisation.  Window ``w`` keeps its tokens whose timestep lies in
    ``[lo, hi)``; a file's result is the concatenation of its windows' kept tokens in window order (no collapse).

    ``tokens`` / ``timesteps`` (n_windows, cap) int32 with ``n_tokens`` valid entries per row (clipped at ``cap``),
    timesteps non-decreasing; windows of file ``f`` are rows ``first[f] .. first[f] + n_win[f] - 1``; ``kept_cap`` bounds
    the kept tokens of one window; ``frames`` is the window's frame count (> every timestep).  Returns (merged
    (n_files, max_windows * kept_cap) int32, valid up to merged_len, merged_len (n_files,) int32)."""
    n_windows, cap = tokens.shape
    dev = tokens.device
    n_files = first.numel()
    col = torch.arange(cap, device=dev)
    n = n_tokens.clamp(max=cap).to(torch.int64)
    # past the last token the row is padded with `frames`, which sorts after every timestep and after hi
    ts = torch.where(col[None, :] < n[:, None], timesteps, torch.full_like(timesteps, frames))
    bounds = torch.tensor([lo, hi], dtype=timesteps.dtype, device=dev).expand(n_windows, 2).contiguous()
    ab = torch.searchsorted(ts, bounds)
    a, b = ab[:, 0], ab[:, 1]
    kept = b - a
    file_of = torch.repeat_interleave(torch.arange(n_files, device=dev), n_win, output_size=n_windows)
    excl = torch.cumsum(kept, 0) - kept                      # exclusive prefix sum over all windows
    off = excl - excl[first][file_of]                        # ... restarted at every file's first window
    merged_len = torch.zeros(n_files, dtype=torch.int64, device=dev).index_add_(0, file_of, kept)
    width = max_windows * kept_cap
    keep = (col[None, :] >= a[:, None]) & (col[None, :] < b[:, None])
    dst = file_of[:, None] * width + off[:, None] + (col[None, :] - a[:, None])
    dst = torch.where(keep, dst, torch.full_like(dst, n_files * width))  # everything not kept lands in one spare slot
    flat = torch.zeros(n_files * width + 1, dtype=tokens.dtype, device=dev)
    flat.scatter_(0, dst.flatten(), tokens.flatten())
    return flat[:-1].view(n_files, width), merged_len.to(torch.int32)


def buffered_rnnt_transcribe(asr_model, audios: Sequence, frame_len: float, total_buffer: float, tokens_per_chunk: int,
                             delay: int, model_stride_in_secs: float, windows_per_forward: int = 256) -> List[List[int]]:
    """Buffered transducer inference of any number of files, every window of every file batched together: one id list per
    file, each equal to what ``BatchedFrameASRRNNT`` gives for that file (``unmerged`` after ``transcribe``).  ``audios``:
    1-D waveforms at the model's rate, each padded with ``int(delay * model_stride_in_secs * sample_rate)`` zero samples
    as the reference does."""
    asr = BatchedFrameASRRNNT(asr_model, frame_len, total_buffer, batch_size=max(len(audios), 1),
                              windows_per_forward=windows_per_forward)
    pad = int(delay * model_stride_in_secs * asr.sample_rate)
    return asr.decode(audios, pad, tokens_per_chunk, delay)[0]


def _waveform(audio, name: str) -> torch.Tensor:
    if isinstance(audio, (str, bytes, os.PathLike)):
        raise NotImplementedError(f"{name} (B200) takes samples, not a path: decode the audio file first")
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
