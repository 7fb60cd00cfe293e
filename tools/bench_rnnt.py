"""Transducer greedy decode benchmark (SURVEY.md 8(f) rank 4): Conformer-Transducer Large decoder / joint sizes
(configs/conformer_transducer_bpe.yaml: enc 512, pred 640, joint 640, 1024 BPE classes, max_symbols 30) on a batch of
B x T' encoder frames (default 32 x 500 = 32 utterances of 20 s).  Random weights emit nothing sensible, so the blank
bias is calibrated (with the kernel itself) to a speech-like symbol rate (--rate symbols per frame, default 0.2).

    python tools/bench_rnnt.py [--batch 32] [--frames 500] [--steps 20] [--cpu-sample 2]

Prints one JSON line: audio-s/s of the decode alone (encoder output resident in HBM), the end-to-end figure through
GreedyBatchedRNNTInfer.forward (hypotheses on the host), symbols, and the CPU oracle timed on a bounded sample of the same
batch.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import conformer_nemo_b200 as cn  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--frames", type=int, default=500)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rate", type=float, default=0.2)
    ap.add_argument("--cpu-sample", type=int, default=2)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    args = ap.parse_args()
    from oracle import rnnt_oracle as ro  # weights generator + cpu_baseline leg only

    dims = (512, 640, 640, 1024)
    B, T = args.batch, args.frames
    x = torch.randn(B, 512, T, generator=torch.Generator().manual_seed(1234))
    if args.dtype == "bf16":
        x = x.bfloat16()
    lens = torch.full((B,), T, dtype=torch.int64)
    xg, lg = x.cuda(), lens.cuda()

    def modules(bias):
        dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=0, blank_bias=bias)
        dec = cn.RNNTDecoder(prednet=dict(pred_hidden=640, pred_rnn_layers=1, dropout=0.1), vocab_size=1024)
        joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=512, pred_hidden=640, joint_hidden=640, activation="relu",
                                           dropout=0.1), num_classes=1024)
        dec.load_state_dict(dec_sd)
        joint.load_state_dict(joint_sd)
        return dec_sd, joint_sd, cn.GreedyBatchedRNNTInfer(dec.cuda(), joint.cuda(), 1024, 30)

    lo, hi = 0.5, 2.0  # symbols per frame fall with the bias: bisect
    for _ in range(12):
        bias = 0.5 * (lo + hi)
        dec_sd, joint_sd, greedy = modules(bias)
        n = greedy.decode_arrays(xg, lg, max_tokens=30 * T)["n_tokens"].float().sum().item() / (B * T)
        if n > args.rate:
            lo = bias
        else:
            hi = bias
    symbols_per_frame = n
    out = greedy.decode_arrays(xg, lg)
    torch.cuda.synchronize()
    n_tok = out["n_tokens"].cpu()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.warmup):
        greedy.decode_arrays(xg, lg)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        greedy.decode_arrays(xg, lg)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    t0 = time.perf_counter()
    for _ in range(args.steps):
        greedy(encoder_output=xg, encoded_lengths=lg)
    e2e_ms = (time.perf_counter() - t0) / args.steps * 1e3
    audio_s = B * T * 0.04  # 40 ms per encoder frame (10 ms hop x 4 subsampling)
    line = dict(metric="transducer greedy decode audio-sec/sec", value=audio_s / (ms * 1e-3), unit="audio-sec/sec",
                ms_per_batch=ms, e2e=dict(value=audio_s / (e2e_ms * 1e-3), ms_per_batch=e2e_ms,
                                          mode="GreedyBatchedRNNTInfer.forward: decode + hypotheses on the host"),
                config=dict(workload=f"Conformer-Transducer Large decoder/joint (512/640/640/1025), {B} x {T} frames, max_symbols 30",
                            encoder_output_dtype=args.dtype, blank_bias=bias, symbols_per_frame=symbols_per_frame),
                symbols=int(n_tok.sum()), gpu_launches=5)
    if args.cpu_sample > 0:
        k = min(args.cpu_sample, B)
        torch.set_num_threads(os.cpu_count() or 1)
        ro.rnnt_greedy_decode(x[:1].float(), lens[:1], dec_sd, joint_sd, 30, "relu", False)
        t0 = time.perf_counter()
        ro.rnnt_greedy_decode(x[:k].float(), lens[:k], dec_sd, joint_sd, 30, "relu", False)
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = dict(value=k * T * 0.04 / dt, unit="audio-sec/sec", cores=torch.get_num_threads(), kind="port",
                                    sample=f"{k} of the batch's utterances, oracle/rnnt_oracle.py (torch fp32 CPU)")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
