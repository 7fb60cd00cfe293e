"""CPU oracle of buffered long-audio transducer inference -- TEST INFRASTRUCTURE ONLY (imported by tests/ and tools/; the
product path is conformer-nemo_b200/buffered.py: BatchedFrameASRRNNT on the kernels behind cfb_op_logmel_raw /
cfb_op_feature_buffers / cfb_op_rnnt_greedy).

Restates, line by line, the transducer classes of nemo/collections/asr/parts/utils/streaming_utils.py:
``BatchedFeatureFrameBufferer``, ``BatchedFrameASRRNNT`` (``_get_batch_preds``, ``transcribe``, ``_alignment_decoder``)
and ``inplace_buffer_merge``, with the buffers in numpy float32 as the reference keeps them.  The pieces shared with the
CTC path (``AudioFeatureIterator``, ``FeatureFrameBufferer``, the raw front end ``raw_featurizer``) come from
oracle/buffered_oracle.py.  The model pieces come from the other oracles: ``conformer_oracle.encoder_forward`` followed by
``rnnt_oracle.rnnt_greedy_decode`` (``rnnt_model``, whose hypotheses carry alignments rebuilt from the decode's
decisions).  ``buffered_oracle.load_reference_streaming_utils`` executes the unmodified reference module, transducer
classes included, when its tree is mounted.

Not confirmed against the reference text (the reference tree is not reachable where this was written; like the CTC
buffered oracle, these are restated from the published source and are checked by
tests/test_buffered_rnnt.py::test_oracle_matches_live_reference_when_mounted whenever the tree is mounted):
  * that ``BatchedFeatureFrameBufferer`` normalises exactly as ``FeatureFrameBufferer`` does (each file keeps its own
    ``W``-wide buffer; population std, 1e-5 added to it);
  * that a file's ``signal_end_index`` is its chunk count, so ``transcribe`` keeps every window of it;
  * the slice ``alignment[Lw - offset - delay : Lw - offset - delay + tokens_per_chunk]`` with
    ``offset = 0 if delay == len(alignment) else 1``, ``len(alignment)`` being the window's encoder frames;
  * that ``inplace_buffer_merge`` only concatenates, and that ``greedy_merge`` of the transducer class hands the
    concatenation to ``tokenizer.ids_to_text`` without a collapse.
"""
from __future__ import annotations

from typing import List

import numpy as np
import torch

from oracle import conformer_oracle as oc
from oracle import rnnt_oracle as ro
from oracle.buffered_oracle import AudioFeatureIterator, FeatureFrameBufferer


class RNNTHypothesis:
    """The fields of a greedy_batch hypothesis that BatchedFrameASRRNNT reads (preserve_alignments on)."""

    def __init__(self, y_sequence, timestep, alignments):
        self.y_sequence, self.timestep, self.alignments = y_sequence, timestep, alignments


def alignments_from_decode(tokens, timesteps, length: int, max_symbols, blank: int) -> List[list]:
    """The alignment greedy_batch keeps with preserve_alignments: per encoder frame the list of its decisions as
    (logits, label), the symbols emitted there and then the blank that moved on (none after ``max_symbols`` symbols).
    Only the labels are rebuilt (from ``rnnt_oracle.decisions``); the logits slot holds None, the merge never reads it."""
    out = [[] for _ in range(length)]
    for t, _, label in ro.decisions(list(tokens), list(timesteps), length, max_symbols, blank):
        out[t].append((None, label))
    return out


def rnnt_model(enc_sd, enc_cfg: oc.EncoderConfig, dec_sd, joint_sd, max_symbols, activation: str = "relu"):
    """The transducer model pieces BatchedFrameASRRNNT calls, for the oracles: ``model(processed_signal,
    processed_signal_length) -> (encoded, encoded_len)`` and ``model.decode(encoded, encoded_len) -> hypotheses``
    (``decoding.rnnt_decoder_predictions_tensor(..., return_hypotheses=True)`` of greedy_batch with alignments).
    ``model.results`` keeps the rnnt_oracle results of every window (their decision margins judge ties)."""
    class Model:
        blank = dec_sd["prediction.embed.weight"].shape[0] - 1

        def __init__(self):
            self.results: List[ro.RNNTGreedyResult] = []

        def __call__(self, processed_signal, processed_signal_length):
            return oc.encoder_forward(enc_sd, enc_cfg, processed_signal.float(), processed_signal_length)

        def decode(self, encoded, encoded_len):
            res = ro.rnnt_greedy_decode(encoded, encoded_len, dec_sd, joint_sd, max_symbols, activation, False)
            self.results += res
            return [RNNTHypothesis(torch.tensor(r.tokens, dtype=torch.int64), list(r.timesteps),
                                   alignments_from_decode(r.tokens, r.timesteps, r.length, max_symbols, self.blank))
                    for r in res]
    return Model()


class BatchedFeatureFrameBufferer(FeatureFrameBufferer):
    """Batched variant of FeatureFrameBufferer where the batch dimension is the independent audio files."""

    def __init__(self, n_feat, window_stride, frame_len=1.6, batch_size=4, total_buffer=4.0, log=True, dtype=np.float32):
        super().__init__(n_feat, window_stride, frame_len, batch_size, total_buffer, log, dtype)
        timestep_duration = window_stride
        total_buffer_len = int(total_buffer / timestep_duration)
        self.buffer = np.ones([batch_size, self.n_feat, total_buffer_len], dtype=dtype) * self.ZERO_LEVEL_SPEC_DB_VAL
        self.all_frame_reader = [None for _ in range(self.batch_size)]
        self.signal_end = [False for _ in range(self.batch_size)]
        self.signal_end_index = [None for _ in range(self.batch_size)]
        self.buffer_number = 0
        self.reset()
        del self.buffered_len
        del self.buffered_features_size

    def reset(self):
        super().reset()
        self.feature_buffer = np.ones([self.batch_size, self.n_feat, self.feature_buffer_len],
                                      dtype=self.dtype) * self.ZERO_LEVEL_SPEC_DB_VAL
        self.all_frame_reader = [None for _ in range(self.batch_size)]
        self.signal_end = [False for _ in range(self.batch_size)]
        self.signal_end_index = [None for _ in range(self.batch_size)]
        self.buffer_number = 0

    def get_batch_frames(self):
        if all(self.signal_end):
            return []
        batch_frames = []
        for idx, frame_reader in enumerate(self.all_frame_reader):
            try:
                frame = next(frame_reader)
                batch_frames.append(np.copy(frame))
            except StopIteration:
                batch_frames.append(None)
                self.signal_end[idx] = True
                if self.signal_end_index[idx] is None:
                    self.signal_end_index[idx] = self.buffer_number
        self.buffer_number += 1
        return batch_frames

    def get_frame_buffers(self, frames):
        self.frame_buffers = []
        for idx in range(self.batch_size):
            frame = frames[idx]
            if frame is not None:
                self.buffer[idx, :, :-self.n_frame_len] = self.buffer[idx, :, self.n_frame_len:]
                self.buffer[idx, :, -self.n_frame_len:] = frame
                self.frame_buffers.append([np.copy(self.buffer[idx])])
            else:
                self.buffer[idx, :, :] *= 0.0
                self.frame_buffers.append([np.copy(self.buffer[idx])])
        return self.frame_buffers

    def set_frame_reader(self, frame_reader, idx):
        self.all_frame_reader[idx] = frame_reader
        self.signal_end[idx] = False
        self.signal_end_index[idx] = None

    def _update_feature_buffer(self, feat_frame, idx):
        if feat_frame is not None:
            self.feature_buffer[idx, :, :-feat_frame.shape[1]] = self.feature_buffer[idx, :, feat_frame.shape[1]:]
            self.feature_buffer[idx, :, -feat_frame.shape[1]:] = feat_frame
        else:
            self.feature_buffer[idx, :, :] *= 0.0

    def get_norm_consts_per_frame(self, batch_frames):
        for idx, frame in enumerate(batch_frames):
            self._update_feature_buffer(frame, idx)
        mean_from_buffer = np.mean(self.feature_buffer, axis=2, keepdims=True)
        stdev_from_buffer = np.std(self.feature_buffer, axis=2, keepdims=True)
        return (mean_from_buffer, stdev_from_buffer)

    def normalize_frame_buffers(self, frame_buffers, norm_consts):
        CONSTANT = 1e-5
        for i in range(len(frame_buffers)):
            frame_buffers[i] = (frame_buffers[i] - norm_consts[0][i]) / (norm_consts[1][i] + CONSTANT)

    def get_buffers_batch(self):
        batch_frames = self.get_batch_frames()
        while len(batch_frames) > 0:
            frame_buffers = self.get_frame_buffers(batch_frames)
            norm_consts = self.get_norm_consts_per_frame(batch_frames)
            self.normalize_frame_buffers(frame_buffers, norm_consts)
            return frame_buffers
        return []


def inplace_buffer_merge(buffer, data, timesteps, model=None):
    """streaming_utils.py's merge of the middle-token path: the kept ids of a window are appended to the file's buffer."""
    if timesteps < 1:
        buffer += data
        return buffer
    if len(buffer) == 0:
        buffer += data
        return buffer
    buffer += data
    return buffer


class BatchedFrameASRRNNT:
    """The reference class with its model pieces passed in: ``featurize`` (raw_featurizer), ``model`` (rnnt_model).
    ``transcribe`` returns the merged ids of every file (the reference hands each list to tokenizer.ids_to_text)."""

    def __init__(self, featurize, model, n_feat, window_stride, sample_rate, blank_id, frame_len=1.6, total_buffer=4.0,
                 batch_size=32, max_steps_per_timestep=5, stateful_decoding=False):
        self.featurize, self.model = featurize, model
        self.window_stride, self.sample_rate = window_stride, sample_rate
        self.blank_id, self.frame_len, self.batch_size = blank_id, frame_len, batch_size
        self.max_steps_per_timestep = max_steps_per_timestep
        self.stateful_decoding = stateful_decoding
        self.frame_bufferer = BatchedFeatureFrameBufferer(n_feat, window_stride, frame_len, batch_size, total_buffer)
        self.reset()

    def reset(self):
        self.unmerged = []
        self.frame_buffers = []
        self.all_alignments = [[] for _ in range(self.batch_size)]
        self.all_preds = [[] for _ in range(self.batch_size)]
        self.all_timestamps = [[] for _ in range(self.batch_size)]
        self.previous_hypotheses = None
        self.batch_index_map = {idx: idx for idx in range(self.batch_size)}
        self.signals = [None for _ in range(self.batch_size)]  # AudioBuffersDataLayer of every file
        self.frame_bufferer.reset()

    def read_audio_file(self, audios, delay, model_stride_in_secs):
        assert len(audios) == self.batch_size
        for idx in range(self.batch_size):
            samples = np.pad(audios[idx], (0, int(delay * model_stride_in_secs * self.sample_rate)))
            frame_reader = AudioFeatureIterator(samples, self.frame_len, self.featurize, self.window_stride)
            self.frame_bufferer.set_frame_reader(frame_reader, idx)

    def infer_logits(self):
        frame_buffers = self.frame_bufferer.get_buffers_batch()
        while len(frame_buffers) > 0:
            self.frame_buffers += frame_buffers[:]
            for idx, buffer in enumerate(frame_buffers):
                self.signals[idx] = buffer[:]
            self._get_batch_preds()
            frame_buffers = self.frame_bufferer.get_buffers_batch()

    def _get_batch_preds(self):
        feat_signals, feat_signal_lens, new_batch_keys = [], [], []
        for idx in range(self.batch_size):
            if self.frame_bufferer.signal_end[idx]:
                continue
            # DataLoader(batch_size=1, collate_fn=speech_collate_fn) over the file's one buffer
            feat_signal = torch.as_tensor(np.asarray(self.signals[idx]), dtype=torch.float32).reshape(
                1, *np.shape(self.signals[idx])[-2:])
            feat_signals.append(feat_signal)
            feat_signal_lens.append(torch.tensor([feat_signal.shape[-1]], dtype=torch.int64))
            new_batch_keys.append(idx)
        if len(feat_signals) == 0:
            return
        feat_signal = torch.cat(feat_signals, 0)
        feat_signal_len = torch.cat(feat_signal_lens, 0)
        encoded, encoded_len = self.model(processed_signal=feat_signal, processed_signal_length=feat_signal_len)
        best_hyp = self.model.decode(encoded, encoded_len)
        for idx, hyp in enumerate(best_hyp):
            global_index_key = new_batch_keys[idx]
            if not self.frame_bufferer.signal_end[global_index_key]:
                self.all_alignments[global_index_key].append(hyp.alignments)
        preds = [hyp.y_sequence for hyp in best_hyp]
        for idx, pred in enumerate(preds):
            global_index_key = new_batch_keys[idx]
            if not self.frame_bufferer.signal_end[global_index_key]:
                self.all_preds[global_index_key].append(pred.cpu().numpy())
        timestamps = [hyp.timestep for hyp in best_hyp]
        for idx, timestep in enumerate(timestamps):
            global_index_key = new_batch_keys[idx]
            if not self.frame_bufferer.signal_end[global_index_key]:
                self.all_timestamps[global_index_key].append(timestep)
        if len(new_batch_keys) != len(self.batch_index_map):
            for new_batch_idx, global_index_key in enumerate(new_batch_keys):
                self.batch_index_map[global_index_key] = new_batch_idx

    def transcribe(self, tokens_per_chunk: int, delay: int) -> List[List[int]]:
        self.infer_logits()
        self.unmerged = [[] for _ in range(self.batch_size)]
        for idx, alignments in enumerate(self.all_alignments):
            signal_end_idx = self.frame_bufferer.signal_end_index[idx]
            if signal_end_idx is None:
                raise ValueError("Signal did not end")
            for a_idx, alignment in enumerate(alignments):
                if delay == len(alignment):  # chunk size = buffer size
                    offset = 0
                else:
                    offset = 1
                alignment = alignment[len(alignment) - offset - delay:len(alignment) - offset - delay + tokens_per_chunk]
                ids, toks = self._alignment_decoder(alignment, None, self.blank_id)
                if len(ids) > 0 and a_idx < signal_end_idx:
                    self.unmerged[idx] = inplace_buffer_merge(self.unmerged[idx], ids, delay)
        return [self.greedy_merge(self.unmerged[idx]) for idx in range(self.batch_size)]

    def _alignment_decoder(self, alignments, tokenizer, blank_id):
        s, ids = [], []
        for t in range(len(alignments)):
            for u in range(len(alignments[t])):
                _, token_id = alignments[t][u]
                token_id = int(token_id)
                if token_id != blank_id:
                    if tokenizer is not None:
                        s.append(tokenizer.ids_to_tokens([token_id])[0])
                    ids.append(token_id)
        return ids, s

    def greedy_merge(self, preds):
        return [p for p in preds]
