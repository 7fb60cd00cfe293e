"""Transducer beam search benchmark (decoding.strategy = beam): Conformer-Transducer Large decoder / joint sizes
(enc 512, pred 640, joint 640, 1024 BPE classes) on B x T' encoder frames (default 32 x 500 = 32 utterances of 20 s), the
blank bias calibrated with the greedy kernel to a speech-like symbol rate as in tools/bench_rnnt.py.

    python tools/bench_rnnt_beam.py [--batch 32] [--frames 500] [--beams 1,2,4,8] [--steps 3] [--out FILE]

For every beam size: ms per batch and audio-s/s of cfb_op_rnnt_beam (encoder output resident in HBM, capacities already
grown to what the batch needs, so one launch sequence per decode), expansions per frame (hypotheses popped = lock-step
work items) and the end-to-end BeamRNNTInfer.forward time.  The greedy kernel on the same input
and the CPU oracle (oracle/rnnt_beam_oracle.py, the restatement of the reference's BeamRNNTInfer) on a bounded sample
of frames are timed beside it.  Prints one JSON document; --out also writes it to a file.
"""
import argparse
import json
import os
import subprocess
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
    ap.add_argument("--beams", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--rate", type=float, default=0.2)
    ap.add_argument("--cpu-frames", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from oracle import rnnt_beam_oracle as bo  # CPU leg only
    from oracle import rnnt_oracle as ro

    dims = (512, 640, 640, 1024)
    B, T = args.batch, args.frames
    x = torch.randn(B, 512, T, generator=torch.Generator().manual_seed(1234)).bfloat16()
    lens = torch.full((B,), T, dtype=torch.int64)
    xg, lg = x.cuda(), lens.cuda()

    def modules(bias):
        dec_sd, joint_sd = ro.random_rnnt_state_dicts(*dims, seed=0, blank_bias=bias)
        dec = cn.RNNTDecoder(prednet=dict(pred_hidden=640, pred_rnn_layers=1, dropout=0.1), vocab_size=1024)
        joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=512, pred_hidden=640, joint_hidden=640, activation="relu",
                                           dropout=0.1), num_classes=1024)
        dec.load_state_dict(dec_sd)
        joint.load_state_dict(joint_sd)
        return dec_sd, joint_sd, dec.cuda(), joint.cuda()

    lo, hi = 0.5, 2.0  # greedy symbols per frame fall with the blank bias: bisect (as tools/bench_rnnt.py)
    for _ in range(12):
        bias = 0.5 * (lo + hi)
        dec_sd, joint_sd, dec, joint = modules(bias)
        greedy = cn.GreedyBatchedRNNTInfer(dec, joint, 1024, 30)
        n = greedy.decode_arrays(xg, lg, max_tokens=30 * T)["n_tokens"].float().sum().item() / (B * T)
        if n > args.rate:
            lo = bias
        else:
            hi = bias
    audio_s = B * T * 0.04  # 40 ms per encoder frame (10 ms hop x 4 subsampling)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / args.steps

    greedy_ms = timed(lambda: greedy.decode_arrays(xg, lg))
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    doc = dict(metric="transducer beam search audio-sec/sec", device=props.name, nvidia_smi=smi,
               config=dict(workload=f"Conformer-Transducer Large decoder/joint (512/640/640/1025), {B} x {T} frames, bf16 "
                                    "encoder output", blank_bias=bias, greedy_symbols_per_frame=n, steps=args.steps),
               greedy=dict(ms_per_batch=greedy_ms, value=audio_s / (greedy_ms * 1e-3), unit="audio-sec/sec",
                           mode="cfb_op_rnnt_greedy, max_symbols 30"),
               beams={})
    for beam_size in [int(b) for b in args.beams.split(",")]:
        beam = cn.BeamRNNTInfer(dec, joint, beam_size=beam_size)
        try:
            (hyps,) = beam(encoder_output=xg, encoded_lengths=lg)  # grows the capacities to what this batch needs
        except NotImplementedError as e:
            doc["beams"][str(beam_size)] = dict(not_run=str(e))
            print(json.dumps({str(beam_size): doc["beams"][str(beam_size)]}), flush=True)
            continue
        caps = beam.last_caps
        out = beam.decode_arrays(xg, lg, caps)
        assert int(out["flags"].cpu()) == 0
        stats = out["stats"].cpu()
        ms = timed(lambda: beam.decode_arrays(xg, lg, caps))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            beam.decode_arrays(xg, lg, caps)["flags"].cpu()
        e2e_ms = (time.perf_counter() - t0) / args.steps * 1e3
        expansions = int(stats[:, 0].sum())
        doc["beams"][str(beam_size)] = dict(
            ms_per_batch=ms, value=audio_s / (ms * 1e-3), unit="audio-sec/sec", decode_arrays_with_sync_ms=e2e_ms,
            expansions_per_frame=expansions / (B * T), max_expansions_at_one_frame=int(stats[:, 3].max()),
            prefix_tree_nodes_max=int(stats[:, 1].max()), state_slots_max=int(stats[:, 2].max()),
            best_hypothesis_labels_per_frame=sum(len(h.y_sequence) - (beam_size > 1) for h in hyps) / (B * T),
            caps=caps)
        print(json.dumps({str(beam_size): doc["beams"][str(beam_size)]}), flush=True)
    if args.cpu_frames > 0:
        tf = min(args.cpu_frames, T)
        torch.set_num_threads(os.cpu_count() or 1)
        cpu = {}
        for beam_size in [int(b) for b in args.beams.split(",")]:
            t0 = time.perf_counter()
            bo.rnnt_beam_decode(x[:1, :, :tf].float(), lens[:1].clamp(max=tf), dec_sd, joint_sd, beam_size, "relu", True)
            dt = time.perf_counter() - t0
            cpu[str(beam_size)] = dict(value=tf * 0.04 / dt, unit="audio-sec/sec")
        doc["cpu_baseline"] = dict(per_beam=cpu, cores=torch.get_num_threads(), kind="port",
                                   sample=f"1 utterance x {tf} frames, oracle/rnnt_beam_oracle.py (torch fp32 CPU, "
                                          "the restatement of BeamRNNTInfer; the reference itself was not reachable)")
    text = json.dumps(doc)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
