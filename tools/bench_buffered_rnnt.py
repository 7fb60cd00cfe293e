"""Buffered long-audio transducer inference (BatchedFrameASRRNNT / buffered_rnnt_transcribe) against one full-context pass.

    python tools/bench_buffered_rnnt.py [--reps 3] [--out buffered_rnnt_b200.json]

Model: Conformer-Transducer-L dimensions (encoder d_model 512, 17 layers, 8 heads, 80 mel bins; prediction network and
joint 640 wide; 1025 joint classes = 1024 tokens + blank; decoding.greedy.max_symbols 30), random weights, the blank
bias calibrated to about 0.2 symbols per encoder frame as tools/bench_pipeline.py does (bisection on the one-pass
decode of 8 x 20 s).  Workloads: 16 files x 5 min and 64 files x 1 min of synthetic 16 kHz audio, already on the device.
Each path is timed from the waveforms on the device to the ids on the host (host clock, the call ends in the read of the
ids), warmed up first, median of --reps runs.

* buffered: frame_len 1.6 s, total_buffer 4.0 s, tokens_per_chunk 40 and delay 70 (model_stride_in_secs 0.04), every
  window of every file batched, 256 windows per encoder forward (CUDA graphs on), every chunk's windows decoded by the
  greedy kernel before the next forward.  Per-stage device times (raw log-mel, windows, encoder, decode, merge) come from
  CUDA events recorded between the stages in a separate run.
* one pass: the normalising front end, one encoder forward over the whole files and the greedy decode of them.
The card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STRIDE_SECS = 0.04  # window_stride 0.01 x subsampling_factor 4
MAX_SYMBOLS = 30    # configs/conformer_transducer_bpe.yaml decoding.greedy.max_symbols
PRE = dict(sample_rate=16000, window_size=0.025, window_stride=0.01, window="hann", normalize="per_feature", n_fft=512,
           features=80, dither=1e-5, pad_to=0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def build_model():
    import types

    import torch

    import conformer_nemo_b200 as cn
    from oracle import conformer_oracle as oc
    from oracle import rnnt_oracle as ro

    cfg = oc.EncoderConfig(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    enc.load_state_dict(oc.random_state_dict(cfg, 0), strict=False)
    enc = enc.cuda().eval()
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=640, pred_rnn_layers=1, dropout=0.1), vocab_size=1024).cuda()
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=512, pred_hidden=640, joint_hidden=640, activation="relu", dropout=0.1),
                         num_classes=1024).cuda()
    model = types.SimpleNamespace(_cfg={"sample_rate": 16000, "preprocessor": dict(PRE),
                                        "decoding": {"strategy": "greedy_batch", "greedy": {"max_symbols": MAX_SYMBOLS}}},
                                  encoder=enc, decoder=dec, joint=joint, tokenizer=None)

    # calibrate the blank bias to ~0.2 symbols per encoder frame (random weights would emit at every frame)
    pre = cn.AudioToMelSpectrogramPreprocessor(**PRE).cuda()
    g = torch.Generator(device="cuda").manual_seed(99)
    x = 0.1 * torch.randn(8, 20 * 16000, device="cuda", generator=g)
    with torch.no_grad():
        f, flen = pre(input_signal=x, length=torch.full((8,), x.shape[1], device="cuda"), check_lengths=False)
        encoded, elen = enc(audio_signal=f, length=flen)
        encoded = encoded.clone()
    frames = int(elen.sum())

    def rate(bias):
        dec_sd, joint_sd = ro.random_rnnt_state_dicts(512, 640, 640, 1024, seed=0, blank_bias=bias)
        dec.load_state_dict(dec_sd)
        joint.load_state_dict(joint_sd)
        greedy = cn.GreedyBatchedRNNTInfer(dec, joint, 1024, MAX_SYMBOLS)
        n = greedy.decode_arrays(encoded, elen, max_tokens=MAX_SYMBOLS * encoded.shape[2])["n_tokens"]
        return n.float().sum().item() / frames

    lo, hi = 0.5, 3.0
    for _ in range(10):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if rate(mid) > 0.2 else (lo, mid)
    symbols = rate(hi)
    return model, torch, hi, symbols


def timed(fn, reps):
    import torch

    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
    return out, sorted(times)[len(times) // 2], times


def stage_times(timeline):
    out = {}
    for (_, a), (name, b) in zip(timeline, timeline[1:]):
        out[name] = out.get(name, 0.0) + a.elapsed_time(b)
    return out


def run_workload(model, torch, n_files, seconds, reps):
    import conformer_nemo_b200 as cn

    g = torch.Generator(device="cuda").manual_seed(n_files)
    audios = [0.1 * torch.randn(seconds * 16000, device="cuda", generator=g) for _ in range(n_files)]
    audio_s = n_files * seconds
    tpc = math.ceil(1.6 / STRIDE_SECS)
    delay = math.ceil((1.6 + (4.0 - 1.6) / 2) / STRIDE_SECS)
    pad = int(delay * STRIDE_SECS * 16000)
    res = {"workload": f"{n_files} x {seconds} s", "audio_seconds": audio_s, "tokens_per_chunk": tpc, "delay": delay}

    model.encoder.enable_cuda_graphs(True)
    asr = cn.BatchedFrameASRRNNT(model, 1.6, 4.0, batch_size=n_files, windows_per_forward=256)
    asr.decode(audios, pad, tpc, delay)  # warm-up: graph capture, filter bank upload
    (ids, decodes), med, all_t = timed(lambda: asr.decode(audios, pad, tpc, delay), reps)
    n_windows = sum(len(d) for d in decodes)
    window_tokens = sum(len(t) for d in decodes for t, _ in d)
    timeline = []
    asr.decode(audios, pad, tpc, delay, timeline=timeline)
    torch.cuda.synchronize()
    res["buffered"] = {
        "windows_per_forward": 256, "windows": n_windows, "seconds_median": med, "seconds_all": all_t,
        "audio_s_per_s": audio_s / med, "stage_ms": stage_times(timeline), "tokens_out": sum(len(i) for i in ids),
        "window_symbols_per_encoder_frame": window_tokens / (n_windows * asr.window_tokens)}
    model.encoder.enable_cuda_graphs(False)

    pre = cn.AudioToMelSpectrogramPreprocessor(**PRE).cuda()
    greedy = cn.GreedyBatchedRNNTInfer(model.decoder, model.joint, 1024, MAX_SYMBOLS)
    x = torch.stack(audios)
    lens = torch.full((n_files,), x.shape[1], dtype=torch.int64, device="cuda")

    def one_pass(timeline=None):
        def mark(name):
            if timeline is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                timeline.append((name, e))
        with torch.no_grad():
            mark("start")
            f, flen = pre(input_signal=x, length=lens, check_lengths=False)
            mark("logmel")
            enc, enc_len = model.encoder(audio_signal=f, length=flen)
            mark("encoder")
            (hyps,) = greedy(encoder_output=enc, encoded_lengths=enc_len)  # ends in the read of the hypotheses
            mark("decode")
        return hyps

    try:
        one_pass()
        hyps, med1, all1 = timed(one_pass, reps)
        tl = []
        one_pass(tl)
        torch.cuda.synchronize()
    except (RuntimeError, torch.cuda.OutOfMemoryError) as e:  # recorded, not hidden: the buffered figures stand alone
        res["one_pass"] = {"error": str(e)[:500]}
        return res
    res["one_pass"] = {"seconds_median": med1, "seconds_all": all1, "audio_s_per_s": audio_s / med1,
                       "stage_ms": stage_times(tl), "encoder_frames_per_file": int(enc_frames(model, x.shape[1])),
                       "tokens_out": sum(len(h.y_sequence) for h in hyps)}
    res["buffered_over_one_pass_speed"] = res["buffered"]["audio_s_per_s"] / res["one_pass"]["audio_s_per_s"]
    return res


def enc_frames(model, n_samples):
    return model.encoder.output_frames(n_samples // 160 + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "buffered_rnnt_b200.json"))
    ap.add_argument("--workloads", default="16x300,64x60")
    args = ap.parse_args()
    model, torch, bias, symbols = build_model()
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0),
              "model": "Conformer-Transducer-L dims (encoder d_model 512, 17 layers, 8 heads; prediction network and joint "
                       "640; 1025 joint classes; max_symbols 30), random weights, bf16 encoder",
              "blank_bias": bias, "calibrated_symbols_per_encoder_frame": symbols,
              "buffered_settings": {"frame_len": 1.6, "total_buffer": 4.0, "model_stride_in_secs": STRIDE_SECS},
              "workloads": []}
    for w in args.workloads.split(","):
        n, s = (int(v) for v in w.split("x"))
        result["workloads"].append(run_workload(model, torch, n, s, args.reps))
        print(json.dumps(result["workloads"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"card": result["card"], "out": args.out}))


if __name__ == "__main__":
    main()
