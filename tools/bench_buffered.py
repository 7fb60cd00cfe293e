"""Buffered long-audio CTC inference (FrameBatchASR / buffered_ctc_transcribe) against one full-context pass.

    python tools/bench_buffered.py [--reps 3] [--out buffered_b200.json]

Model: Conformer-L dimensions (d_model 512, 17 layers, 8 heads, 80 mel bins), random weights, a 1025-class CTC head
(1024 tokens + blank).  Workloads: 16 files x 5 min and 64 files x 1 min of synthetic 16 kHz audio, already on the
device.  Each path is timed from the waveforms on the device to the ids on the host (host clock, the call ends in the
read of the ids), warmed up first, median of --reps runs.

* buffered: frame_len 1.6 s, total_buffer 4.0 s, tokens_per_chunk and delay as NeMo's buffered CTC script computes them
  (40 and 70 with model_stride_in_secs 0.04), every window of every file batched, batch_size 256 windows per encoder
  forward (CUDA graphs on); also batch_size 4, the reference's default, once.  Per-stage device times (raw log-mel,
  windows, encoder, head, merge) come from CUDA events recorded between the stages in a separate run.
* one pass: the normalising front end, one encoder forward over the whole files, the head and the greedy collapse.
The window kernel's bytes (windows written + raw features read once) over its time are compared with 7.7 TB/s, the
HBM3e bandwidth of the B200 data sheet.  The card name and power limit are read in the same run.
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

HBM_TBS = 7.7
STRIDE_SECS = 0.04  # window_stride 0.01 x subsampling_factor 4
PRE = dict(sample_rate=16000, window_size=0.025, window_stride=0.01, window="hann", normalize="per_feature", n_fft=512,
           features=80, dither=1e-5, pad_to=16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def build_model():
    import types

    import torch

    import conformer_nemo_b200 as cn
    from oracle import conformer_oracle as oc
    from oracle import ctc_head_oracle as ho

    cfg = oc.EncoderConfig(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=17, d_model=512, n_heads=8)
    enc.load_state_dict(oc.random_state_dict(cfg, 0), strict=False)
    dec = cn.ConvASRDecoder(feat_in=512, num_classes=1024)
    dec.load_state_dict(ho.random_head_state_dict(512, 1024, 1))
    return types.SimpleNamespace(_cfg={"sample_rate": 16000, "preprocessor": dict(PRE)}, encoder=enc.cuda().eval(),
                                 decoder=dec.cuda(), tokenizer=None), torch


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
    from conformer_nemo_b200.buffered import FrameBatchASR

    g = torch.Generator(device="cuda").manual_seed(n_files)
    audios = [0.1 * torch.randn(seconds * 16000, device="cuda", generator=g) for _ in range(n_files)]
    audio_s = n_files * seconds
    tpc = math.ceil(1.6 / STRIDE_SECS)
    delay = math.ceil((1.6 + (4.0 - 1.6) / 2) / STRIDE_SECS)
    pad = int(delay * STRIDE_SECS * 16000)
    res = {"workload": f"{n_files} x {seconds} s", "audio_seconds": audio_s, "tokens_per_chunk": tpc, "delay": delay}

    model.encoder.enable_cuda_graphs(True)
    asr = FrameBatchASR(model, 1.6, 4.0, batch_size=256)
    asr.decode(audios, pad, tpc, delay)  # warm-up: graph capture, filter bank upload
    (ids, _), med, all_t = timed(lambda: asr.decode(audios, pad, tpc, delay), reps)
    n_windows = sum(n // asr.n_frame_len + 1 for n in asr.raw_preprocessor.get_seq_len(
        torch.tensor([seconds * 16000 + pad] * n_files)).tolist())
    timeline = []
    asr.decode(audios, pad, tpc, delay, timeline=timeline)
    torch.cuda.synchronize()
    stages = stage_times(timeline)
    n_frames = seconds * 16000 // 160 + 1 + pad // 160
    win_bytes = n_windows * 80 * 400 * 4 + n_files * 80 * n_frames * 4
    res["buffered"] = {
        "batch_size": 256, "windows": n_windows, "seconds_median": med, "seconds_all": all_t, "audio_s_per_s": audio_s / med,
        "stage_ms": stages, "tokens_out": sum(len(i) for i in ids),
        "window_kernel": {"bytes": win_bytes, "ms": stages["windows"], "tb_per_s": win_bytes / stages["windows"] / 1e9,
                          "fraction_of_7.7_tb_per_s": win_bytes / stages["windows"] / 1e9 / HBM_TBS}}
    small = FrameBatchASR(model, 1.6, 4.0, batch_size=4)
    small.decode(audios, pad, tpc, delay)
    (ids4, _), med4, _ = timed(lambda: small.decode(audios, pad, tpc, delay), 1)
    res["buffered_batch_size_4"] = {"seconds": med4, "audio_s_per_s": audio_s / med4, "same_ids_as_batch_size_256": ids4 == ids}
    model.encoder.enable_cuda_graphs(False)

    pre = cn.AudioToMelSpectrogramPreprocessor(**PRE).cuda()
    x = torch.stack(audios)
    lens = torch.full((n_files,), x.shape[1], dtype=torch.int64, device="cuda")

    def one_pass(timeline=None):
        def mark(name):
            if timeline is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                timeline.append((name, e))
        mark("start")
        f, flen = pre(input_signal=x, length=lens, check_lengths=False)
        mark("logmel")
        enc, enc_len = model.encoder(audio_signal=f, length=flen)
        mark("encoder")
        tokens, n_tokens = model.decoder.greedy_tokens(enc, enc_len)
        mark("head_and_collapse")
        return torch.cat([n_tokens, tokens.flatten()]).cpu()

    try:
        one_pass()
        _, med1, all1 = timed(one_pass, reps)
        tl = []
        one_pass(tl)
        torch.cuda.synchronize()
    except (RuntimeError, torch.cuda.OutOfMemoryError) as e:  # recorded, not hidden: the buffered figures stand alone
        res["one_pass"] = {"error": str(e)[:500]}
        return res
    res["one_pass"] = {"seconds_median": med1, "seconds_all": all1, "audio_s_per_s": audio_s / med1,
                       "stage_ms": stage_times(tl), "encoder_frames_per_file": x.shape[1] // 160 + 1}
    res["buffered_over_one_pass_speed"] = res["buffered"]["audio_s_per_s"] / res["one_pass"]["audio_s_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "buffered_b200.json"))
    ap.add_argument("--workloads", default="16x300,64x60")
    args = ap.parse_args()
    model, torch = build_model()
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0),
              "model": "Conformer-L dims (d_model 512, 17 layers, 8 heads), random weights, 1025-class CTC head, bf16",
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
