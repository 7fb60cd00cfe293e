"""CPU oracle of the transducer beam search (``decoding.strategy = beam``, ``search_type = default``) -- TEST
INFRASTRUCTURE ONLY.

Restates, in plain Python lists and torch fp32 on the CPU, ``BeamRNNTInfer.default_beam_search``, ``greedy_search`` (what
``beam_size == 1`` switches to), ``sort_nbest`` and the per-utterance loop of ``BeamRNNTInfer.forward``
(parts/submodules/rnnt_beam_decoding.py).  The prediction network and the joint are those of oracle/rnnt_oracle.py.

Per utterance, with V non-blank classes, blank = V, ``beam = min(beam_size, V + 1)`` and ``beam_k = min(beam, V)``:

    kept = [Hyp(score=0.0, y=[blank], state=zeros, timestep=[-1])]
    for t in range(encoded_len):
        hyps, kept = kept, []
        while True:
            best = max(hyps, key=score)                    # first maximal element, in list order
            hyps.remove(best)
            g, state' = prediction(best)                   # LSTM on best.y[-1] (blank -> zero input) from best.state;
                                                           # cached per y sequence, so a pure function of y
            lp = log_softmax(joint(f_t, g) / temperature)  # fp32, V + 1 classes
            for (v, k) in topk(lp[:V], beam_k) + [(lp[blank], blank)]:
                new = best with score += float(v)          # Python float: scores accumulate in double
                if k == blank: kept.append(new)            # same y, same state
                else: new.y += [k]; new.timestep += [t]; new.state = state'; hyps.append(new)
            hyps_max = max(h.score for h in hyps)
            most = sorted([h for h in kept if h.score > hyps_max], key=score)   # stable, ascending
            if len(most) >= beam: kept = most; break       # not truncated to beam
    return sort_nbest(kept)   # by score / len(y) (y with its leading blank) if score_norm else score, descending, stable

``greedy_search`` (beam_size == 1): per frame, up to 5 joint evaluations; the arg-max over all V + 1 log-probabilities
(first index on ties) either ends the frame (blank) or is appended with its log-probability added to the score.  Its
hypothesis has no leading blank in ``y`` nor -1 in ``timestep``, and ``dec_state`` None while nothing was emitted.

Every decision records the gap that settled it (``BeamResult.margins``): the ``max`` pick (best minus second-best score),
the top-k boundary (k-th minus (k+1)-th non-blank log-probability), the break test (smallest |kept score - hyps_max|),
the final sort (smallest gap between adjacent sort keys) and, in greedy mode, top-1 minus top-2.  Another implementation
that differs from this oracle is only wrong if it differs on a case whose smallest margin is above fp32 summation noise.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from .rnnt_oracle import _ACT, lstm_cell

GREEDY_MAX_SYMBOLS = 5  # greedy_search's hard-coded symbols per frame


@dataclass
class BeamHyp:
    score: float                      # Hypothesis.score (double)
    y: List[int]                      # Hypothesis.y_sequence (leading blank in beam mode)
    timestep: List[int]               # Hypothesis.timestep (leading -1 in beam mode)
    h: Optional[torch.Tensor] = None  # Hypothesis.dec_state (H,) each; None in greedy mode before the first symbol
    c: Optional[torch.Tensor] = None


@dataclass
class BeamResult:
    nbest: List[BeamHyp] = field(default_factory=list)                  # sorted as sort_nbest returns it
    margins: List[Tuple[str, int, float]] = field(default_factory=list)  # (decision kind, frame, gap)
    expansions: int = 0                                                 # hypotheses popped (joint evaluations)
    length: int = 0

    @property
    def min_margin(self) -> float:
        return min((m for _, _, m in self.margins), default=float("inf"))


def _weights(dec_sd, joint_sd):
    f32 = lambda t: t.detach().to(torch.float32).cpu()
    if "prediction.dec_rnn.lstm.weight_ih_l1" in dec_sd:
        raise NotImplementedError("oracle restates the one-layer prediction network of the Conformer-Transducer recipes")
    out_keys = sorted(k for k in joint_sd if k.startswith("joint_net.") and k.endswith(".weight"))
    return dict(embed=f32(dec_sd["prediction.embed.weight"]),
                w_ih=f32(dec_sd["prediction.dec_rnn.lstm.weight_ih_l0"]), w_hh=f32(dec_sd["prediction.dec_rnn.lstm.weight_hh_l0"]),
                b_ih=f32(dec_sd["prediction.dec_rnn.lstm.bias_ih_l0"]), b_hh=f32(dec_sd["prediction.dec_rnn.lstm.bias_hh_l0"]),
                wp=f32(joint_sd["pred.weight"]), bp=f32(joint_sd["pred.bias"]),
                we=f32(joint_sd["enc.weight"]), be=f32(joint_sd["enc.bias"]),
                wj=f32(joint_sd[out_keys[-1]]), bj=f32(joint_sd[out_keys[-1][:-6] + "bias"]))


def beam_widths(beam_size: int, vocab_size: int) -> Tuple[int, int]:
    """(beam, beam_k) of default_beam_search for V = vocab_size non-blank classes."""
    beam = min(beam_size, vocab_size + 1)
    return beam, min(beam, vocab_size)


class _Model:
    def __init__(self, w, activation, temperature):
        self.w, self.act, self.temperature = w, _ACT[activation], temperature
        self.blank = w["embed"].shape[0] - 1
        self.hid = w["w_hh"].shape[1]
        self.cache: Dict[tuple, tuple] = {}

    def predict(self, y, h, c):
        """score_hypothesis: (g = joint.pred(LSTM output), h', c') for the last label of y from state (h, c)."""
        key = tuple(y)
        if key not in self.cache:
            w = self.w
            x = torch.zeros(self.hid) if y[-1] == self.blank else w["embed"][y[-1]]
            h2, c2 = lstm_cell(x, h, c, w["w_ih"], w["w_hh"], w["b_ih"], w["b_hh"])
            self.cache[key] = (F.linear(h2, w["wp"], w["bp"]), h2, c2)
        return self.cache[key]

    def logprobs(self, f, g):
        w = self.w
        return torch.log_softmax(F.linear(self.act(f + g), w["wj"], w["bj"]) / self.temperature, dim=-1)


def _beam_one(m: _Model, encp, length, beam_size, score_norm) -> BeamResult:
    blank, V = m.blank, m.blank
    beam, beam_k = beam_widths(beam_size, V)
    res = BeamResult(length=length)
    zeros = torch.zeros(m.hid)
    kept = [BeamHyp(0.0, [blank], [-1], zeros, zeros)]
    for t in range(length):
        hyps, kept = kept, []
        while True:
            best = max(hyps, key=lambda x: x.score)
            others = sorted((x.score for x in hyps if x is not best), reverse=True)
            res.margins.append(("pick", t, best.score - others[0] if others else float("inf")))
            hyps.remove(best)
            g, h2, c2 = m.predict(best.y, best.h, best.c)
            lp = m.logprobs(encp[t], g)
            res.expansions += 1
            top = lp[:V].topk(beam_k)
            if beam_k < V:
                nxt = lp[:V].topk(beam_k + 1).values
                res.margins.append(("topk", t, float(nxt[beam_k - 1] - nxt[beam_k])))
            for v, k in list(zip(top.values.tolist(), top.indices.tolist())) + [(float(lp[blank]), blank)]:
                if k == blank:
                    kept.append(BeamHyp(best.score + float(v), best.y[:], best.timestep[:], best.h, best.c))
                else:
                    hyps.append(BeamHyp(best.score + float(v), best.y + [k], best.timestep + [t], h2, c2))
            hyps_max = float(max(hyps, key=lambda x: x.score).score)
            res.margins.append(("break", t, min(abs(x.score - hyps_max) for x in kept)))
            most = sorted([x for x in kept if x.score > hyps_max], key=lambda x: x.score)
            if len(most) >= beam:
                kept = most
                break
    key = (lambda x: x.score / len(x.y)) if score_norm else (lambda x: x.score)
    res.nbest = sorted(kept, key=key, reverse=True)
    keys = [key(x) for x in res.nbest]
    if len(keys) > 1:
        res.margins.append(("sort", length, min(a - b for a, b in zip(keys, keys[1:]))))
    return res


def _greedy_one(m: _Model, encp, length) -> BeamResult:
    blank = m.blank
    res = BeamResult(length=length)
    hyp = BeamHyp(0.0, [], [], None, None)
    zeros = torch.zeros(m.hid)
    g, h, c = m.predict([blank], zeros, zeros)  # empty y: the SOS (blank) input from the zero state
    for t in range(length):
        for _ in range(GREEDY_MAX_SYMBOLS):
            lp = m.logprobs(encp[t], g)
            res.expansions += 1
            top2 = lp.topk(2).values
            res.margins.append(("argmax", t, float(top2[0] - top2[1])))
            v, k = lp.max(dim=-1)
            k = int(k)
            if k == blank:
                break
            hyp.y.append(k)
            hyp.score += float(v)
            hyp.h, hyp.c = h, c
            hyp.timestep.append(t)
            g, h, c = m.predict([blank] + hyp.y, h, c)
    res.nbest = [hyp]
    return res


def rnnt_beam_decode(encoded: torch.Tensor, encoded_len: torch.Tensor, dec_sd, joint_sd, beam_size: int,
                     activation: str = "relu", score_norm: bool = True, temperature: float = 1.0) -> List[BeamResult]:
    """encoded (B, D, T) as the encoder returns it; dec_sd / joint_sd = state_dicts of RNNTDecoder / RNNTJoint.
    One BeamResult per utterance, each decoded alone (BeamRNNTInfer.forward's loop)."""
    if beam_size < 1:
        raise ValueError("Beam search size cannot be less than 1!")
    w = _weights(dec_sd, joint_sd)
    x = encoded.detach().to(torch.float32).cpu().transpose(1, 2)
    encp = F.linear(x, w["we"], w["be"])  # joint.enc over every frame
    out = []
    for b in range(x.shape[0]):
        m = _Model(w, activation, temperature)  # the cache lives for one utterance
        n = int(encoded_len[b])
        out.append(_greedy_one(m, encp[b], n) if beam_size == 1 else _beam_one(m, encp[b], n, beam_size, score_norm))
    return out


def first_difference(got: List[Tuple[List[int], List[int]]], want: BeamResult):
    """None if the n-best lists agree on (y, timestep) in order; otherwise (rank, what differs)."""
    exp = [(h.y, h.timestep) for h in want.nbest]
    if len(got) != len(exp):
        return (min(len(got), len(exp)), f"{len(got)} hypotheses instead of {len(exp)}")
    for r, (a, b) in enumerate(zip(got, exp)):
        if list(a[0]) != list(b[0]) or list(a[1]) != list(b[1]):
            return (r, f"y {list(a[0])[:12]}... vs {list(b[0])[:12]}...")
    return None


def random_beam_state_dicts(enc_hidden: int, pred_hidden: int, joint_hidden: int, vocab_size: int, seed: int,
                            blank_bias: float = 0.0, sharpness: float = 1.0):
    """rnnt_oracle.random_rnnt_state_dicts with the output layer's weights scaled by ``sharpness``: random joints give
    nearly flat distributions, where a beam search keeps only the all-blank path (every label costs an extra
    log-probability); sharper ones make labels win and hypotheses branch like a trained model's."""
    from .rnnt_oracle import random_rnnt_state_dicts

    dec, joint = random_rnnt_state_dicts(enc_hidden, pred_hidden, joint_hidden, vocab_size, seed, blank_bias)
    joint["joint_net.2.weight"] = joint["joint_net.2.weight"] * sharpness
    return dec, joint


def load_reference_beam_class():
    """The reference's ``BeamRNNTInfer`` (parts/submodules/rnnt_beam_decoding.py), executed unmodified with the stub
    packages and framework stand-ins that reference_loader.load_reference_rnnt_classes registers."""
    import importlib
    import sys

    from . import reference_loader as rl

    rl.load_reference_rnnt_classes()
    name = "nemo.collections.asr.parts.submodules.rnnt_beam_decoding"
    if name not in sys.modules:
        importlib.import_module(name)
    return sys.modules[name].BeamRNNTInfer
