"""Generates tests/golden/rnnt_beam/*.npz: the n-best lists of the transducer beam search (decoding.strategy = beam,
search_type = default; beam_size 1 is greedy_search) on seeded weights and encoder outputs.

    python tests/golden/make_golden_rnnt_beam.py

With the unmodified reference reachable (oracle/reference_loader.py: $CONFORMER_REF or an install under the repository)
the lists come from its ``BeamRNNTInfer``; otherwise from oracle/rnnt_beam_oracle.py, the restatement of it that
tests/test_rnnt_beam.py checks against the reference whenever it is reachable.  ``source`` in each file says which.
The files live in a subdirectory so that the greedy tests' ``rnnt_*.npz`` pattern does not pick them up.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import reference_loader as rl  # noqa: E402
from oracle import rnnt_beam_oracle as bo  # noqa: E402

OUT = os.path.join(HERE, "rnnt_beam")
SHARPNESS = 5.0  # output-layer scale (rnnt_beam_oracle.random_beam_state_dicts): hypotheses branch
# name: (enc_hidden, pred_hidden, joint_hidden, vocab, lens, beam, score_norm, activation, temperature, blank_bias, seed)
CASES = {
    "beam2_relu": (48, 64, 56, 30, [12, 0, 7, 1, 10], 2, True, "relu", 1.0, 1.0, 0),
    "beam4_relu_raw": (48, 64, 56, 30, [14, 9, 1, 0], 4, False, "relu", 1.0, 1.0, 1),
    "beam8_tanh": (32, 40, 48, 20, [10, 6, 1], 8, True, "tanh", 1.0, 3.0, 2),
    "beam4_tanh_temp": (32, 40, 48, 20, [11, 8], 4, True, "tanh", 1.7, 1.0, 3),
    "beam8_small_vocab": (32, 40, 48, 5, [9, 4, 0, 1], 8, True, "relu", 1.0, 1.0, 4),  # beam and beam_k clipped by V
    "beam1_greedy": (48, 64, 56, 30, [15, 0, 6, 1], 1, True, "relu", 1.0, 1.5, 5),
}


def run_reference(dims, dec_sd, joint_sd, x, lens, beam, score_norm, activation, temperature):
    e, p, j, v = dims
    dec_cls, joint_cls, _ = rl.load_reference_rnnt_classes()
    beam_cls = bo.load_reference_beam_class()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        dec = dec_cls(prednet=dict(pred_hidden=p, pred_rnn_layers=1, dropout=0.1), vocab_size=v)
    joint = joint_cls(jointnet=dict(encoder_hidden=e, pred_hidden=p, joint_hidden=j, activation=activation, dropout=0.1),
                      num_classes=v)
    dec.load_state_dict(dec_sd, strict=True)
    joint.load_state_dict(joint_sd, strict=True)
    kw = dict(beam_size=beam, search_type="default", score_norm=score_norm, return_best_hypothesis=False)
    if temperature != 1.0:
        kw["softmax_temperature"] = temperature
    (nbest,) = beam_cls(dec, joint, **kw)(encoder_output=x, encoded_lengths=lens)
    out = []
    for nb in nbest:
        hyps = nb.n_best_hypotheses
        out.append([(float(h.score), [int(t) for t in h.y_sequence], [int(t) for t in h.timestep]) for h in hyps])
    return out


def main():
    torch.set_num_threads(1)
    os.makedirs(OUT, exist_ok=True)
    live = rl.reference_available()
    source = (f"unmodified reference BeamRNNTInfer loaded from {os.path.basename(rl.REFERENCE_ROOT.rstrip('/'))}" if live
              else "oracle/rnnt_beam_oracle.py restatement (reference not reachable at generation time)")
    for name, (e, p, j, v, lens, beam, score_norm, activation, temperature, blank_bias, seed) in CASES.items():
        dec_sd, joint_sd = bo.random_beam_state_dicts(e, p, j, v, seed, blank_bias, SHARPNESS)
        t = max(lens)
        x = torch.randn(len(lens), e, t, generator=torch.Generator().manual_seed(200 + seed))
        lens_t = torch.tensor(lens, dtype=torch.int64)
        res = bo.rnnt_beam_decode(x, lens_t, dec_sd, joint_sd, beam, activation, score_norm, temperature)
        if live:
            lists = run_reference((e, p, j, v), dec_sd, joint_sd, x, lens_t, beam, score_norm, activation, temperature)
        else:
            lists = [[(h.score, h.y, h.timestep) for h in r.nbest] for r in res]
        n = max(len(lst) for lst in lists)
        width = max(len(y) for lst in lists for _, y, _ in lst) or 1
        counts = np.array([len(lst) for lst in lists])
        lengths = np.zeros((len(lens), n), dtype=np.int64)
        tokens = np.full((len(lens), n, width), -2, dtype=np.int64)
        steps = np.full_like(tokens, -2)
        scores = np.zeros((len(lens), n), dtype=np.float64)
        for b, lst in enumerate(lists):
            for r, (s, y, ts) in enumerate(lst):
                lengths[b, r] = len(y)
                tokens[b, r, :len(y)] = y
                steps[b, r, :len(ts)] = ts
                scores[b, r] = s
        np.savez_compressed(
            os.path.join(OUT, name + ".npz"), source=np.array(source), encoder_output=x.numpy(), encoded_lengths=lens_t.numpy(),
            dims=np.array([e, p, j, v]), beam_size=np.array(beam), score_norm=np.array(score_norm),
            activation=np.array(activation), temperature=np.array(temperature), blank_bias=np.array(blank_bias),
            weight_seed=np.array(seed), sharpness=np.array(SHARPNESS), counts=counts, lengths=lengths, tokens=tokens, timesteps=steps, scores=scores,
            weight_checksum=np.array(float(sum(w.double().sum() for w in list(dec_sd.values()) + list(joint_sd.values())))))
        print(name, "n-best sizes", counts.tolist(), "best lengths", lengths[:, 0].tolist(),
              "smallest oracle decision margin %.1e" % min(r.min_margin for r in res))
    print(source)


if __name__ == "__main__":
    main()
