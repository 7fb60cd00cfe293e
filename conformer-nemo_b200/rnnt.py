"""Transducer decoder, joint and greedy-batch inference on the B200 encoder output: drop-ins for
``nemo.collections.asr.modules.RNNTDecoder`` (modules/rnnt.py:51-611), ``nemo.collections.asr.modules.RNNTJoint``
(modules/rnnt.py:613-1084) and ``GreedyBatchedRNNTInfer`` (parts/submodules/rnnt_greedy_decoding.py:358-616) for
inference with ``decoding.strategy = greedy_batch`` (configs/conformer_transducer_bpe.yaml:139-177).

Same constructor arguments, same ``state_dict`` keys (``prediction.embed.weight``, ``prediction.dec_rnn.lstm.*_l0``,
``pred.*``, ``enc.*``, ``joint_net.{n}.*``), same call
``greedy(encoder_output=(B, D, T), encoded_lengths=(B,)) -> (List[Hypothesis],)`` with ``y_sequence`` / ``timestep`` /
``score`` / ``dec_state`` / ``length`` filled like the reference does.  The whole decode -- joint.enc over every frame,
then the symbol loop with the LSTM and the joint -- runs in libcfb.so (``cfb_op_rnnt_greedy``, csrc/rnnt_greedy.cu)
with ONE device-to-host read at the end; the reference synchronises once per symbol step.  ``decoding.strategy = beam``
(parts/submodules/rnnt_beam_decoding.py, ``BeamRNNTInfer``) runs in ``cfb_op_rnnt_beam`` (csrc/rnnt_beam.cu).  No CPU
fallback; training (``forward`` over label sequences, the transducer loss) stays with the reference modules.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field
from typing import Any, Dict, List, Optional, Tuple, Union

import torch
from torch import nn

from . import _lib

_ACTIVATIONS = {"relu": 0, "sigmoid": 1, "tanh": 2}
_MAX_HYPS = 2048  # entries of a hypothesis list of cfb_op_rnnt_beam (shared memory)


@dataclass
class Hypothesis:
    """The fields of parts/utils/rnnt_utils.py:33-82 that greedy decoding fills."""
    score: float
    y_sequence: Union[List[int], torch.Tensor]
    text: Optional[str] = None
    dec_out: Optional[List[torch.Tensor]] = None
    dec_state: Optional[Any] = None
    timestep: Union[List[int], torch.Tensor] = field(default_factory=list)
    alignments: Optional[Any] = None
    length: Union[int, torch.Tensor] = 0
    y: Optional[List[torch.Tensor]] = None
    lm_state: Optional[Any] = None
    lm_scores: Optional[torch.Tensor] = None
    tokens: Optional[Any] = None
    last_token: Optional[torch.Tensor] = None


class _LSTMDropout(nn.Module):
    """Parameter container with the key layout of common/parts/rnn.py:151-226 (``lstm.weight_ih_l0`` ...)."""

    def __init__(self, input_size, hidden_size, forget_gate_bias, weights_init_scale, hidden_hidden_bias_scale):
        super().__init__()
        self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=1)
        if forget_gate_bias is not None:  # rnn.py:212-219
            with torch.no_grad():
                self.lstm.bias_ih_l0[hidden_size:2 * hidden_size].fill_(forget_gate_bias)
                self.lstm.bias_hh_l0[hidden_size:2 * hidden_size] *= float(hidden_hidden_bias_scale)
        with torch.no_grad():
            for p in self.parameters():
                p *= float(weights_init_scale)


class RNNTDecoder(nn.Module):
    def __init__(self, prednet: Dict[str, Any], vocab_size: int, normalization_mode: Optional[str] = None,
                 random_state_sampling: bool = False, blank_as_pad: bool = True):
        super().__init__()
        self.pred_hidden = prednet["pred_hidden"]
        self.pred_rnn_layers = prednet["pred_rnn_layers"]
        self.blank_idx = vocab_size
        self.vocab_size = vocab_size
        self.blank_as_pad = blank_as_pad
        self.random_state_sampling = random_state_sampling
        if normalization_mode not in (None, "batch", "layer"):
            raise ValueError(f"unknown norm={normalization_mode}")  # common/parts/rnn.py:80-81
        unsupported = []
        if self.pred_rnn_layers != 1:
            unsupported.append(f"pred_rnn_layers={self.pred_rnn_layers} (the Conformer-Transducer recipes use 1)")
        if normalization_mode is not None:
            unsupported.append(f"normalization_mode={normalization_mode!r}")
        if not blank_as_pad:
            unsupported.append("blank_as_pad=False (greedy_batch needs the padding-row embedding)")
        if prednet.get("t_max") is not None:
            unsupported.append("t_max (chrono initialisation is a training-time choice)")
        if prednet.get("rnn_hidden_size", -1) not in (-1, self.pred_hidden):
            unsupported.append("rnn_hidden_size != pred_hidden (projected LSTM)")
        if self.pred_hidden % 4:
            unsupported.append("pred_hidden not a multiple of 4")
        if unsupported:
            raise NotImplementedError("RNNTDecoder (B200): " + "; ".join(unsupported))
        self.prediction = nn.ModuleDict({
            "embed": nn.Embedding(vocab_size + 1, self.pred_hidden, padding_idx=self.blank_idx),  # rnnt.py:327
            "dec_rnn": _LSTMDropout(self.pred_hidden, self.pred_hidden, prednet.get("forget_gate_bias", 1.0),
                                    prednet.get("weights_init_scale", 1.0), prednet.get("hidden_hidden_bias_scale", 0.0)),
        })
        self.eval()

    def forward(self, *args, **kwargs):
        raise NotImplementedError("RNNTDecoder (B200) serves greedy inference through GreedyBatchedRNNTInfer; the "
                                  "teacher-forced forward over label sequences is training code and stays with the reference")


class RNNTJoint(nn.Module):
    def __init__(self, jointnet: Dict[str, Any], num_classes: int, vocabulary: Optional[List] = None,
                 log_softmax: Optional[bool] = None, preserve_memory: bool = False, fuse_loss_wer: bool = False,
                 fused_batch_size: Optional[int] = None, experimental_fuse_loss_wer: Any = None):
        super().__init__()
        self.vocabulary = vocabulary
        self._vocab_size = num_classes
        self._num_classes = num_classes + 1  # + blank (rnnt.py:741)
        if experimental_fuse_loss_wer is not None:
            fuse_loss_wer = experimental_fuse_loss_wer
        if fuse_loss_wer and fused_batch_size is None:  # rnnt.py:754-755
            raise ValueError("If `fuse_loss_wer` is set, then `fused_batch_size` cannot be None!")
        self.log_softmax = log_softmax
        self.encoder_hidden = jointnet["encoder_hidden"]
        self.pred_hidden = jointnet["pred_hidden"]
        self.joint_hidden = jointnet["joint_hidden"]
        self.activation = str(jointnet["activation"]).lower()
        if self.activation not in _ACTIVATIONS:  # rnnt.py:1023-1024
            raise ValueError("Unsupported activation for joint step - please pass one of [relu, sigmoid, tanh]")
        if self.encoder_hidden % 8 or self.joint_hidden % 4:
            raise NotImplementedError("RNNTJoint (B200): encoder_hidden must be a multiple of 8 and joint_hidden of 4")
        dropout = jointnet.get("dropout", 0.0)
        self.pred = nn.Linear(self.pred_hidden, self.joint_hidden)
        self.enc = nn.Linear(self.encoder_hidden, self.joint_hidden)
        act = {"relu": nn.ReLU(inplace=True), "sigmoid": nn.Sigmoid(), "tanh": nn.Tanh()}[self.activation]
        layers = [act] + ([nn.Dropout(p=dropout)] if dropout else []) + [nn.Linear(self.joint_hidden, self._num_classes)]
        self.joint_net = nn.Sequential(*layers)  # the output Linear sits at index 2 when dropout != 0, like rnnt.py:1039-1043
        self.eval()

    @property
    def num_classes_with_blank(self):
        return self._num_classes

    def forward(self, *args, **kwargs):
        raise NotImplementedError("RNNTJoint (B200) serves greedy inference through GreedyBatchedRNNTInfer; the (B, T, U, V) "
                                  "joint tensor and the fused loss / WER are training code and stay with the reference")


class _DeviceRNNTInfer:
    """What the greedy and the beam decoder share: fp32 copies of the decoder / joint weights and their refresh, the
    checks and layout of the encoder output and lengths, and the device scratch buffer of the decode."""

    _name = None  # the class the error messages name

    def __init__(self, decoder_model: RNNTDecoder, joint_model: RNNTJoint):
        self.decoder = decoder_model
        self.joint = joint_model
        self._packed = None
        self._scratch = None

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)

    def invalidate(self):
        """Call after changing decoder / joint parameters (they are re-read on the next call)."""
        self._packed = None

    def _sources(self):
        dec, jn = self.decoder, self.joint
        lstm = dec.prediction["dec_rnn"].lstm
        out = [m for m in jn.joint_net if isinstance(m, nn.Linear)][-1]
        return (dec.prediction["embed"].weight, lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0,
                jn.pred.weight, jn.pred.bias, jn.enc.weight, jn.enc.bias, out.weight, out.bias)

    def _fingerprint(self):
        """Identity of the source parameters: storage, dtype and in-place version counter.  The kernel decodes from fp32
        COPIES of them, so ``decoder.half()``, ``.to(dtype)``, re-assigning a Parameter or an in-place update (optimizer
        step, ``load_state_dict``) must refresh the copies -- checked on every call (eleven tuple compares)."""
        return tuple((p.data_ptr(), p.dtype, p._version) for p in self._sources())

    def _prepare(self, device):
        f = lambda t: t.detach().to(device=device, dtype=torch.float32).contiguous()
        dec, jn = self.decoder, self.joint
        lstm = dec.prediction["dec_rnn"].lstm
        out = [m for m in jn.joint_net if isinstance(m, nn.Linear)][-1]
        t = dict(embed=f(dec.prediction["embed"].weight), w_ih=f(lstm.weight_ih_l0), w_hh=f(lstm.weight_hh_l0),
                 b_ih=f(lstm.bias_ih_l0), b_hh=f(lstm.bias_hh_l0), w_pred=f(jn.pred.weight), b_pred=f(jn.pred.bias),
                 w_enc=f(jn.enc.weight), b_enc=f(jn.enc.bias), w_out=f(out.weight), b_out=f(out.bias))
        if float(t["embed"][self._blank_index].abs().max()) != 0.0:
            raise NotImplementedError(f"{self._name} (B200): the blank row of prediction.embed must be the zero padding row")
        w = _lib.CfbRnntWeights()
        w.enc_hidden, w.pred_hidden, w.joint_hidden = jn.encoder_hidden, dec.pred_hidden, jn.joint_hidden
        w.num_classes_with_blank, w.activation = jn.num_classes_with_blank, _ACTIVATIONS[jn.activation]
        for k, v in t.items():
            setattr(w, k, ctypes.cast(ctypes.c_void_p(v.data_ptr()), ctypes.POINTER(ctypes.c_float)))
        self._packed = (w, t, device, self._fingerprint())

    def _inputs(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor):
        """Checks the (B, D, T) encoder output, refreshes the weight copies if needed and returns the weights, the
        contiguous (B, T, D) fp32 / bf16 encoder output and the int32 lengths on its device."""
        jn = self.joint
        if encoder_output.dim() != 3 or encoder_output.size(1) != jn.encoder_hidden:
            raise TypeError(f"encoder_output must be (B, {jn.encoder_hidden}, T), got {tuple(encoder_output.shape)}")
        if not encoder_output.is_cuda:
            raise RuntimeError(f"{self._name} (B200) has no CPU path: encoder_output must be a CUDA tensor")
        device = encoder_output.device
        if self._packed is None or self._packed[2] != device or self._packed[3] != self._fingerprint():
            self._prepare(device)
        x = encoder_output.transpose(1, 2)  # the encoder returns the transposed view of a contiguous (B, T, D) buffer
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        lens = encoded_lengths.to(device=device, dtype=torch.int32).contiguous()
        return self._packed[0], x, lens

    def _scratch_ptr(self, nbytes: int, device) -> ctypes.c_void_p:
        """A 256-byte aligned device buffer of `nbytes`, kept between calls."""
        if self._scratch is None or self._scratch.numel() < nbytes + 256 or self._scratch.device != device:
            self._scratch = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
        return ctypes.c_void_p((self._scratch.data_ptr() + 255) // 256 * 256)


class GreedyBatchedRNNTInfer(_DeviceRNNTInfer):
    """rnnt_greedy_decoding.py:358-616 (the ``blank_as_pad`` branch)."""

    _name = "GreedyBatchedRNNTInfer"

    def __init__(self, decoder_model: RNNTDecoder, joint_model: RNNTJoint, blank_index: int,
                 max_symbols_per_step: Optional[int] = None, preserve_alignments: bool = False):
        if preserve_alignments:
            raise NotImplementedError("GreedyBatchedRNNTInfer (B200): preserve_alignments is a debugging aid of the reference")
        if blank_index != decoder_model.blank_idx or blank_index != joint_model.num_classes_with_blank - 1:
            raise ValueError("blank_index must be len(vocabulary) for the decoder and the joint (blank_as_pad)")
        if decoder_model.pred_hidden != joint_model.pred_hidden:
            raise ValueError("decoder pred_hidden and joint pred_hidden differ")
        super().__init__(decoder_model, joint_model)
        self._blank_index = blank_index
        self._SOS = blank_index
        self.max_symbols = max_symbols_per_step
        self.preserve_alignments = False

    @torch.no_grad()
    def decode_arrays(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor, max_tokens: Optional[int] = None):
        """Device-side result: dict of tokens / timesteps (B, max_tokens) int32, n_tokens (B) int32, scores (B) fp32,
        h / c (B, H) fp32.  Enqueue-only (no synchronisation)."""
        w, x, lens = self._inputs(encoder_output, encoded_lengths)
        device = x.device
        b, t, d = x.shape
        max_symbols = 0 if self.max_symbols is None else int(self.max_symbols)
        if max_tokens is None:
            max_tokens = t * max_symbols if 0 < max_symbols <= 8 else 4 * t + 64
        max_tokens = max(int(max_tokens), 1)
        lib = _lib.load_library()
        need = lib.cfb_rnnt_greedy_scratch_bytes(d, w.pred_hidden, w.joint_hidden, b, t)
        sptr = self._scratch_ptr(need, device)
        out = dict(tokens=torch.empty(b, max_tokens, dtype=torch.int32, device=device),
                   timesteps=torch.empty(b, max_tokens, dtype=torch.int32, device=device),
                   n_tokens=torch.empty(b, dtype=torch.int32, device=device),
                   scores=torch.empty(b, dtype=torch.float32, device=device),
                   h=torch.empty(b, w.pred_hidden, dtype=torch.float32, device=device),
                   c=torch.empty(b, w.pred_hidden, dtype=torch.float32, device=device),
                   flags=torch.zeros(1, dtype=torch.int32, device=device))
        vp = lambda tensor: ctypes.c_void_p(tensor.data_ptr())
        with torch.cuda.device(device):
            rc = lib.cfb_op_rnnt_greedy(ctypes.byref(w), vp(x), _lib.CFB_F32 if x.dtype == torch.float32 else _lib.CFB_BF16,
                                        vp(lens), b, t, max_symbols, max_tokens, vp(out["tokens"]), vp(out["timesteps"]),
                                        vp(out["n_tokens"]), vp(out["scores"]), vp(out["h"]), vp(out["c"]), vp(out["flags"]),
                                        sptr, need, ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream))
        _lib.check(rc, None, "cfb_op_rnnt_greedy")
        out["_keepalive"] = (x, lens)
        return out

    @torch.no_grad()
    def forward(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor,
                partial_hypotheses: Optional[List[Hypothesis]] = None) -> Tuple[List[Hypothesis]]:
        if partial_hypotheses is not None:  # rnnt_greedy_decoding.py:461-462
            raise NotImplementedError("`partial_hypotheses` support is not supported")
        t = encoder_output.size(2)
        max_tokens = None
        while True:
            out = self.decode_arrays(encoder_output, encoded_lengths, max_tokens)
            n = out["n_tokens"].cpu()  # the one synchronisation of the decode
            flags = int(out["flags"].cpu())
            if flags & 2:
                raise RuntimeError("GreedyBatchedRNNTInfer (B200): runaway emission with max_symbols_per_step=None "
                                   "(4096 symbols at one frame)")
            if flags == 0:
                break
            max_tokens = int(n.max()) + t  # some utterance outgrew the token buffer: run again with room for all of it
        width = max(int(n.max()), 1)
        tokens = out["tokens"][:, :width].cpu().long()
        steps = out["timesteps"][:, :width].cpu()
        scores, h, c = out["scores"].cpu(), out["h"].cpu(), out["c"].cpu()
        lens_cpu = encoded_lengths.to("cpu")
        any_emitted = bool((n > 0).any())
        hyps = []
        for i in range(tokens.size(0)):
            k = int(n[i])
            # pack_hypotheses (rnnt_greedy_decoding.py:43-57): y_sequence as a LongTensor, the state on the CPU; the state is
            # None only when no utterance of the batch ever emitted (`hidden` stays None, :611-614)
            state = ([h[i]], [c[i]]) if any_emitted else None
            hyps.append(Hypothesis(score=float(scores[i]), y_sequence=tokens[i, :k].clone(), timestep=steps[i, :k].tolist(),
                                   dec_state=state, length=lens_cpu[i]))
        return (hyps,)


@dataclass
class NBestHypotheses:
    """parts/utils/rnnt_utils.py: the sorted n-best list of one utterance (``return_best_hypothesis=False``)."""
    n_best_hypotheses: Optional[List[Hypothesis]]


class BeamRNNTInfer(_DeviceRNNTInfer):
    """``decoding.strategy = beam`` (parts/submodules/rnnt_beam_decoding.py, ``BeamRNNTInfer``): ``search_type='default'``
    (default_beam_search) and, for ``beam_size == 1``, the class's own sample-level greedy_search.  The search for every
    utterance of the batch runs in one persistent kernel (``cfb_op_rnnt_beam``, csrc/rnnt_beam.cu) with one device-to-host
    read at the end; the reference decodes one utterance at a time and synchronises once per hypothesis expansion.

    Hypotheses are filled like the reference's pack_hypotheses: ``y_sequence`` a LongTensor with its leading blank,
    ``timestep`` with its leading -1 (greedy_search: neither), ``score`` the double sum of log-probabilities,
    ``dec_state`` the LSTM state ``(h, c)`` as (1, 1, H) CPU tensors (None for greedy_search before its first label),
    ``length`` the utterance's encoded length.  TSD / ALSD / MAES, language models, alignments and partial hypotheses raise
    NotImplementedError."""

    _name = "BeamRNNTInfer"

    def __init__(self, decoder_model: RNNTDecoder, joint_model: RNNTJoint, beam_size: int, search_type: str = "default",
                 score_norm: bool = True, return_best_hypothesis: bool = True, tsd_max_sym_exp_per_step: Optional[int] = 50,
                 alsd_max_target_len: Union[int, float] = 1.0, nsc_max_timesteps_expansion: int = 1,
                 nsc_prefix_alpha: int = 1, maes_num_steps: int = 2, maes_prefix_alpha: int = 1,
                 maes_expansion_gamma: float = 2.3, maes_expansion_beta: int = 2,
                 language_model: Optional[Dict[str, Any]] = None, softmax_temperature: float = 1.0,
                 preserve_alignments: bool = False, ngram_lm_model: Optional[str] = None, ngram_lm_alpha: float = 0.0):
        if beam_size < 1:
            raise ValueError("Beam search size cannot be less than 1!")
        if search_type not in ("default", "tsd", "alsd", "nsc", "maes"):
            raise NotImplementedError(f"The search type ({search_type}) supplied is not supported!\n"
                                      "Please use one of : (default, tsd, alsd, nsc)")
        if beam_size > 1 and search_type != "default":
            raise NotImplementedError(f"BeamRNNTInfer (B200): search_type={search_type!r} (only 'default' runs on the device)")
        if language_model is not None or ngram_lm_model is not None:
            raise NotImplementedError("BeamRNNTInfer (B200): language-model fusion")
        if preserve_alignments:
            raise NotImplementedError("BeamRNNTInfer (B200): preserve_alignments is a debugging aid of the reference")
        if not softmax_temperature > 0:
            raise ValueError("softmax_temperature must be positive")
        if decoder_model.pred_hidden != joint_model.pred_hidden:
            raise ValueError("decoder pred_hidden and joint pred_hidden differ")
        if decoder_model.blank_idx != joint_model.num_classes_with_blank - 1:
            raise ValueError("the decoder's blank index must be the joint's last class (blank_as_pad)")
        super().__init__(decoder_model, joint_model)
        self.blank = decoder_model.blank_idx
        self.vocab_size = decoder_model.vocab_size
        self.search_type = search_type
        self.return_best_hypothesis = return_best_hypothesis
        self.beam_size = beam_size
        self.score_norm = score_norm
        self.max_candidates = beam_size
        self.softmax_temperature = float(softmax_temperature)
        self.preserve_alignments = False
        self._blank_index = self.blank

    def widths(self) -> Tuple[int, int]:
        """(beam, beam_k) of default_beam_search: hypotheses that end a frame, non-blank candidates per expansion."""
        beam = min(self.beam_size, self.vocab_size + 1)
        return beam, min(beam, self.vocab_size)

    def default_caps(self, t: int) -> Dict[str, int]:
        """First-try capacities for T frames; the decode is repeated with larger ones when an utterance outgrows them."""
        beam, beam_k = self.widths()
        x = 8 * beam + 8
        return dict(max_expansions=x, max_hyps=min(x * (beam_k + 1) + 8, _MAX_HYPS), max_nodes=(t + 1) * 2 * beam * beam_k + 64,
                    max_states=(t + 1) * beam + 64, max_len=t + 64)

    @torch.no_grad()
    def decode_arrays(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor, caps: Optional[Dict[str, int]] = None):
        """Device-side result (enqueue-only): n_hyps (B), lengths (B, X), tokens / timesteps (B, X, L) int32, scores (B, X)
        fp64, h / c (B, X, H) fp32, stats (B, 4) int32, flags (1); X = max_expansions, L = max_len of ``caps``."""
        w, x, lens = self._inputs(encoder_output, encoded_lengths)
        device = x.device
        b, t, d = x.shape
        caps = dict(self.default_caps(t), **(caps or {}))
        c = _lib.CfbRnntBeamCaps()
        for k, v in caps.items():
            setattr(c, k, int(v))
        lib = _lib.load_library()
        need = lib.cfb_rnnt_beam_scratch_bytes(d, w.pred_hidden, w.joint_hidden, w.num_classes_with_blank, b, t,
                                               ctypes.byref(c))
        sptr = self._scratch_ptr(need, device)
        X, L, H = c.max_expansions, c.max_len, w.pred_hidden
        i32 = dict(dtype=torch.int32, device=device)
        out = dict(n_hyps=torch.empty(b, **i32), lengths=torch.zeros(b, X, **i32), tokens=torch.empty(b, X, L, **i32),
                   timesteps=torch.empty(b, X, L, **i32), scores=torch.empty(b, X, dtype=torch.float64, device=device),
                   h=torch.empty(b, X, H, dtype=torch.float32, device=device),
                   c=torch.empty(b, X, H, dtype=torch.float32, device=device), stats=torch.empty(b, 4, **i32),
                   flags=torch.zeros(1, **i32))
        vp = lambda tensor: ctypes.c_void_p(tensor.data_ptr())
        with torch.cuda.device(device):
            rc = lib.cfb_op_rnnt_beam(ctypes.byref(w), vp(x), _lib.CFB_F32 if x.dtype == torch.float32 else _lib.CFB_BF16,
                                      vp(lens), b, t, self.beam_size, int(bool(self.score_norm)), self.softmax_temperature,
                                      ctypes.byref(c), vp(out["n_hyps"]), vp(out["lengths"]), vp(out["tokens"]),
                                      vp(out["timesteps"]), vp(out["scores"]), vp(out["h"]), vp(out["c"]), vp(out["stats"]),
                                      vp(out["flags"]), sptr, need,
                                      ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream))
        _lib.check(rc, None, "cfb_op_rnnt_beam")
        out["_keepalive"] = (x, lens)
        out["caps"] = caps
        return out

    @torch.no_grad()
    def forward(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor,
                partial_hypotheses: Optional[List[Hypothesis]] = None):
        if partial_hypotheses is not None:
            raise NotImplementedError("BeamRNNTInfer (B200): partial_hypotheses")
        t = encoder_output.size(2)
        caps = self.default_caps(t)
        for _ in range(24):
            out = self.decode_arrays(encoder_output, encoded_lengths, caps)
            flags = int(out["flags"].cpu())  # the one synchronisation of the decode
            if flags == 0:
                break
            # some utterance outgrew a capacity: run again with the exhausted ones grown
            if flags & 4 and caps["max_hyps"] >= _MAX_HYPS:
                raise NotImplementedError(f"BeamRNNTInfer (B200): a frame needs more than {_MAX_HYPS} list entries "
                                          "(the hypothesis lists live in shared memory)")
            caps = dict(caps)
            for bit, k in ((2, "max_expansions"), (4, "max_hyps"), (8, "max_nodes"), (16, "max_states"), (32, "max_len")):
                if flags & bit:
                    caps[k] *= 4
            if flags & 2:  # more expansions per frame also need longer lists
                caps["max_hyps"] = max(caps["max_hyps"], caps["max_expansions"] * (self.widths()[1] + 1) + 8)
            caps["max_hyps"] = min(caps["max_hyps"], _MAX_HYPS)
        else:
            raise RuntimeError(f"BeamRNNTInfer (B200): capacities still exceeded after growing them to {caps}")
        self.last_caps = caps  # what this batch needed (pass to decode_arrays to skip the growth next time)
        n = out["n_hyps"].cpu()
        lengths, tokens, steps = out["lengths"].cpu(), out["tokens"].cpu(), out["timesteps"].cpu()
        scores, h, c = out["scores"].cpu(), out["h"].cpu(), out["c"].cpu()
        lens_cpu = encoded_lengths.to("cpu")
        greedy = self.beam_size == 1
        H = h.size(-1)
        hypotheses = []
        for i in range(n.size(0)):
            nbest = []
            for r in range(int(n[i])):
                k = int(lengths[i, r])
                emitted = k > 0
                state = (h[i, r].view(1, 1, H).clone(), c[i, r].view(1, 1, H).clone()) if (emitted or not greedy) else None
                nbest.append(Hypothesis(score=float(scores[i, r]), y_sequence=tokens[i, r, :k].long().clone(),
                                        timestep=steps[i, r, :k].tolist(), dec_state=state, length=lens_cpu[i]))
            hypotheses.append(nbest[0] if self.return_best_hypothesis else NBestHypotheses(nbest))
        return (hypotheses,)


class GreedyRNNTInfer(GreedyBatchedRNNTInfer):
    """``decoding.strategy = greedy`` (rnnt_greedy_decoding.py:191-355): the reference decodes one utterance at a time with
    the same per-utterance rule, so tokens, timesteps and scores are those of the batched decode (module docstring of
    oracle/rnnt_oracle.py); here the whole batch still runs in one launch.  Differences in what the Hypothesis carries, kept:
    ``dec_state`` is None for an utterance that emitted nothing (:277, :330-346) and ``last_token`` holds the last symbol."""

    @torch.no_grad()
    def forward(self, encoder_output: torch.Tensor, encoded_lengths: torch.Tensor,
                partial_hypotheses: Optional[List[Hypothesis]] = None) -> Tuple[List[Hypothesis]]:
        (hyps,) = super().forward(encoder_output, encoded_lengths, partial_hypotheses)
        for h in hyps:
            if len(h.y_sequence) == 0:
                h.dec_state = None
            else:
                h.last_token = int(h.y_sequence[-1])
        return (hyps,)
