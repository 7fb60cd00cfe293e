"""Bit-identity of the transducer decoders between two builds of libcfb.so (for example this tree's and one built from an
earlier commit): both decode the same seeded inputs, each library in a process of its own, and every output array must
be bitwise equal.  The decoders combine partial results in a fixed order, so any difference is a bug, not rounding.

    python tools/rnnt_parity.py --reference-lib OTHER/libcfb.so [--lib conformer-nemo_b200/lib/libcfb.so]

Cases (Conformer-Transducer Large decoder / joint, 512/640/640/1025, max_symbols 30): greedy with CFB_RNNT_CLUSTER=0
(row-partitioned kernel) and unset (the kernel selection's default) at 32 x 500 and 7 x 120 frames, fp32 and bf16 encoder
output; beam search with beam sizes 1, 2 and 4 at 32 x 100 frames.  Needs a GPU.
"""
import argparse
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DIMS = (512, 640, 640, 1024)


def _inputs(b, t, seed, dtype):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, DIMS[0], t, generator=g)
    lens = torch.randint(t // 2, t + 1, (b,), generator=g)
    lens[0] = t
    if b > 5:
        lens[5] = 2
    return (x.bfloat16() if dtype == "bf16" else x).cuda(), lens.cuda()


def _modules():
    import conformer_nemo_b200 as cn
    from oracle import rnnt_oracle as ro

    e, p, j, v = DIMS
    dec_sd, joint_sd = ro.random_rnnt_state_dicts(*DIMS, seed=7, blank_bias=1.1)
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=p, pred_rnn_layers=1, dropout=0.1), vocab_size=v)
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=e, pred_hidden=p, joint_hidden=j, activation="relu", dropout=0.1),
                         num_classes=v)
    dec.load_state_dict(dec_sd)
    joint.load_state_dict(joint_sd)
    return dec.cuda(), joint.cuda()


def _masked(t, keep):
    t = t.cpu()
    return torch.where(keep, t, torch.zeros_like(t))


def dump(lib_path, out_path):
    """Decodes every case with the library at `lib_path`; saves the outputs (entries past a row's length zeroed)."""
    import conformer_nemo_b200 as cn
    from conformer_nemo_b200 import _lib

    _lib.LIB_PATH = os.path.abspath(lib_path)
    dec, joint = _modules()
    greedy = cn.GreedyBatchedRNNTInfer(dec, joint, blank_index=DIMS[3], max_symbols_per_step=30)
    res = {}
    for cluster in ("0", None):
        if cluster is None:
            os.environ.pop("CFB_RNNT_CLUSTER", None)
        else:
            os.environ["CFB_RNNT_CLUSTER"] = cluster
        for b, t in ((32, 500), (7, 120)):
            for dtype in ("fp32", "bf16"):
                x, lens = _inputs(b, t, 11 + b, dtype)
                out = greedy.decode_arrays(x, lens)
                n = out["n_tokens"].cpu()
                valid = torch.arange(out["tokens"].size(1))[None] < n[:, None].long()
                r = {k: out[k].cpu() for k in ("n_tokens", "scores", "h", "c", "flags")}
                r["tokens"] = _masked(out["tokens"], valid)
                r["timesteps"] = _masked(out["timesteps"], valid)
                res[f"greedy cluster={cluster or 'default'} {b}x{t} {dtype}"] = r
    os.environ.pop("CFB_RNNT_CLUSTER", None)
    x, lens = _inputs(32, 100, 5, "bf16")
    for beam_size in (1, 2, 4):
        beam = cn.BeamRNNTInfer(dec, joint, beam_size=beam_size, return_best_hypothesis=False)
        try:
            beam(encoder_output=x, encoded_lengths=lens)  # grows the capacities to what this batch needs
        except NotImplementedError as e:  # the search outgrew the list limit: both builds must say so
            res[f"beam {beam_size} 32x100 bf16"] = dict(not_run=torch.tensor(list(str(e).encode())))
            continue
        out = beam.decode_arrays(x, lens, beam.last_caps)
        n, lengths = out["n_hyps"].cpu(), out["lengths"].cpu()
        rows = torch.arange(lengths.size(1))[None] < n[:, None].long()  # (B, X) hypotheses written
        pos = (torch.arange(out["tokens"].size(2))[None, None] < lengths[..., None].long()) & rows[..., None]
        r = dict(n_hyps=n, lengths=_masked(lengths, rows), stats=out["stats"].cpu(), flags=out["flags"].cpu(),
                 scores=_masked(out["scores"], rows), h=_masked(out["h"], rows[..., None]), c=_masked(out["c"], rows[..., None]),
                 tokens=_masked(out["tokens"], pos), timesteps=_masked(out["timesteps"], pos))
        res[f"beam {beam_size} 32x100 bf16"] = r
    torch.save(res, out_path)


def _bits(t):
    return t.view(torch.int64) if t.dtype == torch.float64 else (t.view(torch.int32) if t.dtype == torch.float32 else t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-lib", required=True)
    ap.add_argument("--lib", default=os.path.join(ROOT, "conformer-nemo_b200", "lib", "libcfb.so"))
    ap.add_argument("--dump", nargs=2, metavar=("LIB", "OUT"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump:
        dump(*args.dump)
        return
    with tempfile.TemporaryDirectory() as tmp:
        outs = []
        for i, lib in enumerate((args.reference_lib, args.lib)):
            path = os.path.join(tmp, f"{i}.pt")
            subprocess.run([sys.executable, os.path.abspath(__file__), "--reference-lib", "-", "--dump", lib, path], check=True)
            outs.append(torch.load(path))
    ref, new = outs
    bad = 0
    for case, r in ref.items():
        diff = [k for k in r if not torch.equal(_bits(r[k]), _bits(new[case][k]))]
        size = f"{int(r['n_tokens'].sum())} symbols" if "n_tokens" in r else (
            f"{int(r['lengths'].sum())} labels in the n-best lists" if "lengths" in r else "not run: list limit")
        print(f"{case}: {'identical' if not diff else 'DIFFERENT: ' + ', '.join(diff)} ({size})")
        bad += bool(diff)
    print("RNNT_PARITY_OK" if bad == 0 else f"RNNT_PARITY_FAILED: {bad} case(s)")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
