"""CPU oracle of buffered long-audio CTC inference -- TEST INFRASTRUCTURE ONLY (imported by tests/ and tools/; the
product path is conformer-nemo_b200/buffered.py on the kernels behind cfb_op_logmel_raw / cfb_op_feature_buffers).

Restates, line by line, ``AudioFeatureIterator``, ``FeatureFrameBufferer`` and ``FrameBatchASR`` of
nemo/collections/asr/parts/utils/streaming_utils.py:455-684, with the buffers in numpy float32 as the reference keeps
them.  The raw front end is ``raw_filterbank_features``: the steps of ``frontend_oracle.filterbank_features`` without
its normalisation (what the reference's ``raw_preprocessor`` computes: dither 0, pad_to 0, normalize "None", for which
normalize_batch returns its input unchanged).  The model pieces come from the other oracles:
``conformer_oracle.encoder_forward`` followed by ``ctc_head_oracle``.  ``load_reference_streaming_utils`` executes the
unmodified reference module when its tree is mounted.

Not confirmed against the reference text (the reference tree is not reachable where this was written; like the beam
search oracle, these are restated from the published source and are checked by
tests/test_buffered.py::test_oracle_matches_live_reference_when_mounted whenever the tree is mounted):
  * the silence constant ZERO_LEVEL_SPEC_DB_VAL = -16.635 that fills a fresh buffer when ``preprocessor.log`` is set
    (0.0 otherwise);
  * the statistics of a window: np.mean and np.std with numpy's default ddof 0, and CONSTANT = 1e-5 added to the std;
  * the extra all-zero chunk: the iterator's first chunk that does not fit is zero-filled past the end and is the last
    one, so a file of n frames has n // frame_len + 1 chunks, the last all zeros when frame_len divides n;
  * the slice bounds ``decoded[len(decoded) - 1 - delay : len(decoded) - 1 - delay + tokens_per_chunk]``;
  * the pad of ``read_audio_file``: ``int(delay * model_stride_in_secs * sample_rate)`` zero samples appended.
"""
from __future__ import annotations

import importlib
import os
import sys
import types
from typing import Callable, List

import numpy as np
import torch

from oracle import conformer_oracle as oc
from oracle import ctc_head_oracle as ho
from oracle import frontend_oracle as fo

ZERO_LEVEL_SPEC_DB_VAL = -16.635  # log-mel value of a zero signal


def raw_filterbank_features(x: torch.Tensor, lengths: torch.Tensor, window: torch.Tensor, fb: torch.Tensor, *, n_fft=512,
                            hop=160, preemph=0.97, log_guard=2.0 ** -24):
    """FilterbankFeatures.forward in eval mode (features.py:358-453) with normalize "None" and pad_to 0: the steps of
    ``frontend_oracle.filterbank_features`` up to the log, then frames t >= seq_len set to 0.  x (B, L) fp32, lengths (B,)
    samples -> (features (B, n_mels, 1 + L // hop) fp32, seq_len (B,) int64)."""
    seq_len = fo.seq_len_frames(lengths, n_fft, hop)
    if preemph is not None:
        x = torch.cat((x[:, 0].unsqueeze(1), x[:, 1:] - preemph * x[:, :-1]), dim=1)
    spec = torch.view_as_real(torch.stft(x, n_fft=n_fft, hop_length=hop, win_length=window.numel(), center=True,
                                         window=window.float(), return_complex=True))
    power = torch.sqrt(spec.pow(2).sum(-1)).pow(2.0)
    feat = torch.log(torch.matmul(fb.to(power.dtype), power) + log_guard)
    mask = torch.arange(feat.shape[-1])[None, :] >= seq_len[:, None]
    return feat.masked_fill(mask.unsqueeze(1), 0.0), seq_len


def raw_featurizer(window: torch.Tensor, fb: torch.Tensor, n_fft: int = 512, hop: int = 160, preemph: float = 0.97,
                   log_guard: float = 2.0 ** -24) -> Callable:
    """The reference's raw_preprocessor as a function (input_signal (1, L), length (1,)) -> (features, seq_len)."""
    def featurize(input_signal, length):
        return raw_filterbank_features(input_signal.float(), length, window, fb, n_fft=n_fft, hop=hop, preemph=preemph,
                                       log_guard=log_guard)
    return featurize


def ctc_model(enc_sd, enc_cfg: oc.EncoderConfig, head_sd) -> Callable:
    """asr_model(processed_signal, processed_signal_length) -> (log_probs, encoded_len, predictions) for the oracles."""
    def model(processed_signal, processed_signal_length):
        enc, enc_len = oc.encoder_forward(enc_sd, enc_cfg, processed_signal.float(), processed_signal_length)
        log_probs = ho.ctc_head_forward(head_sd, enc)
        return log_probs, enc_len, ho.greedy_predictions(log_probs)
    return model


class AudioFeatureIterator:
    def __init__(self, samples, frame_len, featurize, window_stride):
        self._samples = samples
        self._frame_len = frame_len
        self._start = 0
        self.output = True
        self.count = 0
        timestep_duration = window_stride  # preprocessor._cfg['window_stride']
        self._feature_frame_len = frame_len / timestep_duration
        audio_signal = torch.from_numpy(self._samples).unsqueeze_(0)
        audio_signal_len = torch.Tensor([self._samples.shape[0]])
        self._features, self._features_len = featurize(audio_signal, audio_signal_len)
        self._features = self._features.squeeze()

    def __iter__(self):
        return self

    def __next__(self):
        if not self.output:
            raise StopIteration
        last = int(self._start + self._feature_frame_len)
        if last <= self._features_len[0]:
            frame = self._features[:, self._start:last].cpu()
            self._start = last
        else:
            frame = np.zeros([self._features.shape[0], int(self._feature_frame_len)], dtype='float32')
            samp_len = int(self._features_len[0]) - self._start
            frame[:, 0:samp_len] = self._features[:, self._start:int(self._features_len[0])].cpu()
            self.output = False
        self.count += 1
        return frame


class FeatureFrameBufferer:
    """``dtype``: the reference keeps float32 buffers; float64 gives the high-precision reference for kernel tests."""

    def __init__(self, n_feat, window_stride, frame_len=1.6, batch_size=4, total_buffer=4.0, log=True, dtype=np.float32):
        self.ZERO_LEVEL_SPEC_DB_VAL = ZERO_LEVEL_SPEC_DB_VAL if log else 0.0
        self.dtype = dtype
        self.frame_len = frame_len
        timestep_duration = window_stride
        self.n_frame_len = int(frame_len / timestep_duration)
        total_buffer_len = int(total_buffer / timestep_duration)
        self.n_feat = n_feat
        self.buffer = np.ones([self.n_feat, total_buffer_len], dtype=dtype) * self.ZERO_LEVEL_SPEC_DB_VAL
        self.batch_size = batch_size
        self.signal_end = False
        self.frame_reader = None
        self.feature_buffer_len = total_buffer_len
        self.feature_buffer = np.ones([self.n_feat, self.feature_buffer_len], dtype=dtype) * self.ZERO_LEVEL_SPEC_DB_VAL
        self.frame_buffers = []
        self.buffered_features_size = 0
        self.reset()
        self.buffered_len = 0

    def reset(self):
        self.buffer = np.ones(shape=self.buffer.shape, dtype=self.dtype) * self.ZERO_LEVEL_SPEC_DB_VAL
        self.prev_char = ''
        self.unmerged = []
        self.frame_buffers = []
        self.buffered_len = 0
        self.feature_buffer = np.ones([self.n_feat, self.feature_buffer_len], dtype=self.dtype) * self.ZERO_LEVEL_SPEC_DB_VAL

    def get_batch_frames(self):
        if self.signal_end:
            return []
        batch_frames = []
        for frame in self.frame_reader:
            batch_frames.append(np.copy(frame))
            if len(batch_frames) == self.batch_size:
                return batch_frames
        self.signal_end = True
        return batch_frames

    def get_frame_buffers(self, frames):
        self.frame_buffers = []
        for frame in frames:
            self.buffer[:, :-self.n_frame_len] = self.buffer[:, self.n_frame_len:]
            self.buffer[:, -self.n_frame_len:] = frame
            self.buffered_len += frame.shape[1]
            self.frame_buffers.append(np.copy(self.buffer))
        return self.frame_buffers

    def set_frame_reader(self, frame_reader):
        self.frame_reader = frame_reader
        self.signal_end = False

    def _update_feature_buffer(self, feat_frame):
        self.feature_buffer[:, :-feat_frame.shape[1]] = self.feature_buffer[:, feat_frame.shape[1]:]
        self.feature_buffer[:, -feat_frame.shape[1]:] = feat_frame
        self.buffered_features_size += feat_frame.shape[1]

    def get_norm_consts_per_frame(self, batch_frames):
        norm_consts = []
        for i, frame in enumerate(batch_frames):
            self._update_feature_buffer(frame)
            mean_from_buffer = np.mean(self.feature_buffer, axis=1)
            stdev_from_buffer = np.std(self.feature_buffer, axis=1)
            norm_consts.append((mean_from_buffer.reshape(self.n_feat, 1), stdev_from_buffer.reshape(self.n_feat, 1)))
        return norm_consts

    def normalize_frame_buffers(self, frame_buffers, norm_consts):
        CONSTANT = 1e-5
        for i, frame_buffer in enumerate(frame_buffers):
            frame_buffers[i] = (frame_buffer - norm_consts[i][0]) / (norm_consts[i][1] + CONSTANT)

    def get_buffers_batch(self):
        batch_frames = self.get_batch_frames()
        while len(batch_frames) > 0:
            frame_buffers = self.get_frame_buffers(batch_frames)
            norm_consts = self.get_norm_consts_per_frame(batch_frames)
            if len(frame_buffers) == 0:
                continue
            self.normalize_frame_buffers(frame_buffers, norm_consts)
            return frame_buffers
        return []


def file_windows(samples: np.ndarray, featurize, n_feat, window_stride, frame_len, total_buffer, dtype=np.float32):
    """Every normalised window FeatureFrameBufferer produces for one (already padded) file, in order: (n, F, W)."""
    bufferer = FeatureFrameBufferer(n_feat, window_stride, frame_len, 4, total_buffer, dtype=dtype)
    bufferer.set_frame_reader(AudioFeatureIterator(samples, frame_len, featurize, window_stride))
    out = []
    while True:
        batch = bufferer.get_buffers_batch()
        if not batch:
            return np.stack(out)
        out += batch


class FrameBatchASR:
    """The reference class with its model pieces passed in: ``featurize`` (raw_featurizer), ``model`` (ctc_model)."""

    def __init__(self, featurize, model, n_feat, window_stride, sample_rate, blank_id, frame_len=1.6, total_buffer=4.0,
                 batch_size=4):
        self.frame_bufferer = FeatureFrameBufferer(n_feat, window_stride, frame_len, batch_size, total_buffer)
        self.featurize, self.model = featurize, model
        self.window_stride, self.sample_rate = window_stride, sample_rate
        self.batch_size = batch_size
        self.blank_id = blank_id
        self.frame_len = frame_len
        self.reset()

    def reset(self):
        self.prev_char = ''
        self.unmerged = []
        self.all_logits = []
        self.all_preds = []
        self.toks_unmerged = []
        self.frame_buffers = []
        self.frame_bufferer.reset()

    def read_audio_file(self, samples: np.ndarray, delay, model_stride_in_secs):
        samples = np.pad(samples, (0, int(delay * model_stride_in_secs * self.sample_rate)))
        frame_reader = AudioFeatureIterator(samples, self.frame_len, self.featurize, self.window_stride)
        self.frame_bufferer.set_frame_reader(frame_reader)

    def infer_logits(self):
        frame_buffers = self.frame_bufferer.get_buffers_batch()
        while len(frame_buffers) > 0:
            self.frame_buffers += frame_buffers[:]
            self._get_batch_preds(frame_buffers[:])
            frame_buffers = self.frame_bufferer.get_buffers_batch()

    def _get_batch_preds(self, signals):
        # AudioBuffersDataLayer + DataLoader(batch_size) + speech_collate_fn: equal-length buffers, stacked
        for i in range(0, len(signals), self.batch_size):
            chunk = signals[i:i + self.batch_size]
            feat_signal = torch.stack([torch.as_tensor(s, dtype=torch.float32) for s in chunk])
            feat_signal_len = torch.full((len(chunk),), signals[0].shape[1], dtype=torch.int64)
            log_probs, encoded_len, predictions = self.model(feat_signal, feat_signal_len)
            self.all_logits += list(torch.unbind(log_probs))  # kept here for the tests' margin check only
            for pred in torch.unbind(predictions):
                self.all_preds.append(pred.cpu().numpy())

    def transcribe(self, tokens_per_chunk: int, delay: int) -> List[int]:
        """Returns the merged ids (the reference hands them to tokenizer.ids_to_text)."""
        self.infer_logits()
        self.unmerged = []
        for pred in self.all_preds:
            decoded = pred.tolist()
            self.unmerged += decoded[len(decoded) - 1 - delay:len(decoded) - 1 - delay + tokens_per_chunk]
        return self.greedy_merge(self.unmerged)

    def greedy_merge(self, preds):
        decoded_prediction = []
        previous = self.blank_id
        for p in preds:
            if (p != previous or previous == self.blank_id) and p != self.blank_id:
                decoded_prediction.append(p)
            previous = p
        return decoded_prediction


def load_reference_streaming_utils():
    """Returns the reference ``parts/utils/streaming_utils.py`` module (``AudioFeatureIterator``, ``FeatureFrameBufferer``,
    ``FrameBatchASR``), executed unmodified through oracle/reference_loader.py's stub packages.  Its imports that are
    absent here get inert stand-ins: omegaconf, the model classes (``EncDecCTCModelBPE`` only builds FrameBatchASR's raw
    preprocessor, which the tests replace), audio_utils (file decoding) and the nemo.core dataset symbols."""
    from oracle import reference_loader as rl

    rl.load_reference_collation()  # stub packages, nemo.utils.logging, features.py, nemo.core.classes datasets
    name = "nemo.collections.asr.parts.utils.streaming_utils"
    if name in sys.modules:
        return sys.modules[name]
    if "omegaconf" not in sys.modules or not hasattr(sys.modules["omegaconf"].OmegaConf, "set_struct"):
        om = sys.modules.get("omegaconf") or types.ModuleType("omegaconf")
        om.MISSING, om.ListConfig, om.DictConfig = "???", list, dict
        om.OmegaConf = type("OmegaConf", (), {"set_struct": staticmethod(lambda *a, **k: None),
                                              "to_container": staticmethod(lambda c, **k: c)})
        om.open_dict = lambda c: __import__("contextlib").nullcontext(c)
        sys.modules["omegaconf"] = om
    models = types.ModuleType("nemo.collections.asr.models")
    models.__path__ = [os.path.join(rl.REFERENCE_ROOT, "nemo/collections/asr/models")]
    sys.modules.setdefault(models.__name__, models)
    for mod_name, attrs in (("nemo.collections.asr.models.ctc_bpe_models", ("EncDecCTCModelBPE",)),
                            ("nemo.collections.asr.models.ctc_models", ("EncDecCTCModel",)),
                            ("nemo.collections.asr.models.rnnt_bpe_models", ("EncDecRNNTBPEModel",)),
                            ("nemo.collections.asr.parts.utils.audio_utils", ())):
        if mod_name not in sys.modules:
            m = types.ModuleType(mod_name)
            for a in attrs:
                setattr(m, a, type(a, (), {}))
            sys.modules[mod_name] = m
    sys.modules["nemo.collections.asr.parts.utils.audio_utils"].get_samples = lambda *a, **k: (_ for _ in ()).throw(
        NotImplementedError("audio decoding stand-in"))
    classes = sys.modules["nemo.core.classes"]
    classes.IterableDataset = torch.utils.data.IterableDataset
    sys.modules["nemo.core"].classes = classes
    return importlib.import_module(name)
