#!/usr/bin/env python
"""Benchmark of the Conformer encoder forward (BASELINE.json metric: audio-seconds per second, RTFx).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this repository's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's algorithm on host cores
    python bench.py --steps K --dump-outputs bench_outputs/A # also write the last timed step's outputs (two builds
                                                             # given the same arguments see the same inputs)

A step = one forward pass of the encoder over one synthetic batch.  Workload at every N: BASELINE.json configs[1],
Conformer-CTC Large encoder (d_model 512, 17 layers, 8 heads, ff x4, striding x4), batch 32 x 20 s (T = 2000 mel
frames, full lengths) PER GPU (weak scaling, utterances are independent, no data-path collective).
The same line carries `strong`: BASELINE.json configs[2] (cfg3) measured with the same encoder in the same process --
ONE global batch of 64 mixed-length utterances (2-30 s) LPT-sharded over the N ranks, every rank running its share in
the packed variable-length layout (cfb_forward_packed): the strong-scaling curve of the split the north star names.

Printed JSON (one line, rank 0):
  value     whole-job audio-s/s with inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through ConformerEncoder.forward with HOST buffers: pinned H2D of the features and D2H of
            (encoded, encoded_len) inside the timed region
  roofline  dominant kernel family (tcgen05 GEMMs): algorithmic FLOPs / CUDA-event time, against the measured
            sustained bf16 peak in MEASURED_PEAKS.json; `kernels` lists every kernel family the same way
  cpu_baseline  the oracle (CPU restatement of the reference, oracle/conformer_oracle.py) timed on this box's host
            cores on a bounded sample of the same workload
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Conformer-L encoder audio-sec/sec (RTFx)"
UNIT = "audio-sec/sec"
FRAME_SEC = 0.01  # 10 ms hop (configs/conformer_ctc_bpe.yaml:83)

WORKLOADS = {
    # name: (encoder kwargs, batch, frames)
    "cfg2": (dict(feat_in=80, n_layers=17, d_model=512, n_heads=8), 32, 2000),
    "cfg2_18l": (dict(feat_in=80, n_layers=18, d_model=512, n_heads=8), 32, 2000),
    # cfg3: 64 mixed-length utterances (one global batch, sharded over the ranks); batch/frames decided by the plan
    "cfg3": (dict(feat_in=80, n_layers=17, d_model=512, n_heads=8), None, None),
    "cfg4": (dict(feat_in=80, n_layers=18, d_model=256, n_heads=4), 256, 400),
    "cfg5": (dict(feat_in=80, n_layers=17, d_model=512, n_heads=8), 1, 30000),
    # cfg1: BASELINE.json configs[0], the reference's own CPU-runnable case (Small: d_model 176, dk 44), 4 x 10 s
    "cfg1": (dict(feat_in=80, n_layers=16, d_model=176, n_heads=4), 4, 1000),
    "tiny": (dict(feat_in=80, n_layers=2, d_model=256, n_heads=4), 4, 400),
}


def workload_config(name, n_gpus):
    kw, b, t = WORKLOADS[name]
    if b is None:
        return {
            "workload": f"{name}: Conformer-Transducer Large encoder d_model={kw['d_model']} layers={kw['n_layers']} "
                        f"heads={kw['n_heads']}, ONE global batch of 64 utterances of 2-30 s (mixed lengths, padding "
                        f"masks), LPT-sharded into length-bucketed sub-batches over {n_gpus} GPU(s)",
            "global_batch": 64, "parallelism": f"dp{n_gpus} (no collective, strong scaling)",
            "l2": ("no flush between steps: a step streams the 230 MB of bf16 weights plus the rank's activations "
                   f"(first-conv output alone ~{2070 / n_gpus:.0f} MB at this GPU count) through the 126 MB L2"),
        }
    # activations one layer touches (token-major buffers of engine.cu's plan) + the first conv's output, per step
    rows = b * _out_frames(t)[1]
    d = kw["d_model"]
    ws_mb = (rows * d * (4 + 2 + 8 + 8 + 2 + 2 + 2) + b * _out_frames(t)[0] * 40 * d * 2) / 1e6
    return {
        "workload": f"{name}: Conformer encoder d_model={kw['d_model']} layers={kw['n_layers']} heads={kw['n_heads']} "
                    f"ff_x4 conv_k31 striding_x4, batch {b} x {t * FRAME_SEC:.0f} s ({t} mel frames, full lengths) per GPU",
        "per_gpu_batch": b, "frames": t, "global_batch": b * n_gpus, "parallelism": f"dp{n_gpus} (no collective)",
        "l2": (f"working set per step (~{ws_mb:.0f} MB of activations) exceeds the 126 MB L2; no flush needed" if ws_mb > 126 else
               f"working set per step (~{ws_mb:.0f} MB) FITS in the 126 MB L2 and the steps run back to back without a "
               "flush: an L2-warm number, not comparable with the HBM roofline"),
    }


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(tflops=float(p.get("bf16_tflops_sustained", 1399.7)), gbs=float(p.get("hbm_gbs", 6454.6)),
                    burst=float(p.get("bf16_tflops", 1703.6)),
                    source="MEASURED_PEAKS.json (sustained bf16, copy bandwidth)")
    return dict(tflops=1400.0, gbs=6650.0, burst=1700.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, sampled in-process through NVML (pynvml) every 20 ms.
    (A looping nvidia-smi subprocess was measured to perturb the timed steps through its start-up.)"""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._active = threading.Event()
        self.thread = None
        self.err = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if visible:
                ids = [v for v in visible.split(",") if v.strip() != ""]
                if idx < len(ids) and ids[idx].strip().isdigit():
                    idx = int(ids[idx])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def _loop(self):
        nv = self.nv
        masks = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                    r = get_reasons(self.handle)
                    for name, m in masks.items():
                        if r & m:
                            self.reasons.add(name)
                except Exception as e:  # pragma: no cover
                    self.err = repr(e)
            time.sleep(0.02)

    def mark(self):
        """Begin recording (called right before the timed region)."""
        self._active.set()

    def stop(self):
        self._active.clear()
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        sm = sorted(self.samples)
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
               "reasons": sorted(self.reasons), "source": "NVML, 20 ms period, timed region only"}
        if self.err:
            out["error"] = self.err
        return out


def build_encoder(kw, device):
    import conformer_nemo_b200 as cn

    torch.manual_seed(0)
    enc = cn.ConformerEncoder(**kw)
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():  # SURVEY 8(c): the defaults of these are degenerate (zeros / identity)
        for layer in enc.layers:
            layer.self_attn.pos_bias_u.copy_(torch.randn(layer.self_attn.pos_bias_u.shape, generator=g) * 0.1)
            layer.self_attn.pos_bias_v.copy_(torch.randn(layer.self_attn.pos_bias_v.shape, generator=g) * 0.1)
            bn = layer.conv.batch_norm
            bn.running_mean.copy_(torch.randn(bn.running_mean.shape, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(bn.running_var.shape, generator=g) * 0.5 + 0.75)
    enc.mark_weights_dirty()
    return enc.to(device).eval()


def _out_frames(t):
    t1 = (t - 1) // 2 + 1
    return t1, (t1 - 1) // 2 + 1


def algorithmic_costs(kw, batches):
    """Per-step algorithmic FLOPs (tensor-bound kernels) / bytes (memory-bound kernels), keyed by the kernel labels
    of cfb_forward, summed over the step's sub-batches.  `batches` = [[valid frames per utterance], ...].
    Formulas: SURVEY.md section 8(d): valid frames only; GEMM = 2*M*N*K on unpadded dims."""
    d, L = kw["d_model"], kw["n_layers"]
    c, ff = d, 4 * d
    f1, f2 = 40, 20
    fl, by = {}, {}

    def add(dst, key, val):
        dst[key] = dst.get(key, 0) + val

    for lens in batches:
        t1s = [_out_frames(t)[0] for t in lens]
        t2s = [_out_frames(t)[1] for t in lens]
        n = sum(t2s)                       # valid encoder frames
        n1 = sum(t1s)
        t2_max = max(t2s)
        add(fl, "subsample conv 2", 2 * 9 * c * c * n * f2)
        add(fl, "pre_encode.out", 2 * n * f2 * c * d)
        add(fl, "linear_pos", 2 * (2 * t2_max - 1) * d * d * L)
        add(fl, "qkv projection", L * 2 * n * d * 3 * d)
        add(fl, "linear_out", L * 2 * n * d * d)
        add(fl, "pointwise_conv1+glu", L * 2 * n * d * 2 * d)
        add(fl, "pointwise_conv2", L * 2 * n * d * d)
        add(fl, "linear1+swish", 2 * L * 2 * n * d * ff)
        add(fl, "linear2", 2 * L * 2 * n * d * ff)
        add(fl, "rel-pos attention", L * 6 * sum(v * v for v in t2s) * d)
        add(by, "subsample conv 0", sum(lens) * 80 * 4 + n1 * f1 * c * 2)
        add(by, "norm_feed_forward", (L + 1) * n * d * 6)  # norm_feed_forward1 of layers > 0 rides on norm_out
        add(by, "norm_self_att", L * n * d * 6)
        add(by, "norm_conv", L * n * d * 6)
        add(by, "norm_out", (L - 1) * n * d * 10 + n * d * 8)  # reads x, writes x (fp32) + the next bf16 operand
        add(by, "depthwise conv", L * (n * d * 4 + 31 * d * 4))
        # fused conv-module tail (conv_tail.cu): g (bf16) in, x (fp32) read + write; 2*n*d*d FLOPs need less time
        add(by, "depthwise+pointwise_conv2", L * (n * d * 10 + 32 * d * 4 + d * d * 2))
    return fl, by


def gemm_algorithmic_bytes(kw, batches):
    """Per-step compulsory bytes of the GEMM family (operands read once, result written once; the fp32 residual
    stream is read and written by the reduce-add epilogues), keyed like algorithmic_costs."""
    d, L = kw["d_model"], kw["n_layers"]
    ff, f2 = 4 * d, 20
    by = {}
    for lens in batches:
        t2s = [_out_frames(t)[1] for t in lens]
        n, p = sum(t2s), 2 * max(t2s) - 1
        def add(key, m, nn, k, out_b, launches, resid=False):
            by[key] = by.get(key, 0) + launches * (m * k * 2 + nn * k * 2 + m * nn * out_b * (2 if resid else 1))
        add("pre_encode.out", n, d, f2 * d, 4, 1)
        add("linear_pos", p, L * d, d, 2, 1)
        add("qkv projection", n, 3 * d, d, 2, L)
        by["qkv projection"] += L * n * d * 2  # the q + v copy
        add("linear_out", n, d, d, 4, L, resid=True)
        add("pointwise_conv1+glu", n, 2 * d, d, 1, L)  # GLU halves the output: d bf16 columns = 2d * 1 byte
        add("pointwise_conv2", n, d, d, 4, L, resid=True)
        add("linear1+swish", n, ff, d, 2, 2 * L)
        add("linear2", n, d, ff, 4, 2 * L, resid=True)
    return by


GEMM_LABELS = ["pre_encode.out", "linear_pos", "qkv projection", "linear_out", "pointwise_conv1+glu", "pointwise_conv2",
               "linear1+swish", "linear2"]  # the fused depthwise+pointwise_conv2 kernel is not gemm_tc_kernel: reported apart


def measure_pipelines(enc, device, steps=5, warmup=2, batch=32, seconds=20):
    """The widened rows composed around the SAME encoder (SURVEY.md 8(f), DESIGN.md 9-13): pinned host waveforms ->
    log-mel kernels -> encoder (graph replay) -> (a) CTC head + greedy collapse, (b) transducer greedy decode -> token ids
    on the host.  Random-init heads of the recipes' sizes (the modules' own initialisers), blank biases calibrated so that
    both decoders emit a speech-like 0.2 symbols per encoder frame.  Wall clock over whole batches, everything included."""
    import conformer_nemo_b200 as cn

    n_samp = seconds * 16000
    audio = (torch.randn(batch, n_samp, generator=torch.Generator().manual_seed(0)) * 0.1).pin_memory()
    lengths = torch.full((batch,), n_samp, dtype=torch.int64).pin_memory()
    vocab = 1024
    torch.manual_seed(0)
    pre = cn.AudioToMelSpectrogramPreprocessor(window_size=0.025, window_stride=0.01, features=80, n_fft=512, pad_to=0).to(device)
    head = cn.ConvASRDecoder(feat_in=enc._feat_out, num_classes=vocab).to(device)
    dec = cn.RNNTDecoder(prednet=dict(pred_hidden=640, pred_rnn_layers=1, dropout=0.1), vocab_size=vocab).to(device)
    joint = cn.RNNTJoint(jointnet=dict(encoder_hidden=enc._feat_out, pred_hidden=640, joint_hidden=640, activation="relu",
                                       dropout=0.1), num_classes=vocab).to(device)
    enc.enable_cuda_graphs(True)

    def front(a, n):
        feats, flen = pre(input_signal=a, length=n, check_lengths=False)
        return enc(audio_signal=feats, length=flen)

    encoded, elen = front(audio.to(device), lengths.to(device))
    encoded, elen = encoded.clone(), elen.clone()
    frames = int(elen.sum())
    head_bias = head.decoder_layers[0].bias
    out_bias = joint.joint_net[-1].bias
    base_h, base_j = float(head_bias.detach()[vocab]), float(out_bias.detach()[vocab])

    def ctc_rate(b):
        with torch.no_grad():
            head_bias[vocab] = base_h + b
        head._invalidate()  # the packed bf16 copy of the head's weights is rebuilt from the edited bias
        _, pred = head.forward_with_predictions(encoded)
        return sum(len(t) for t in cn.ctc_greedy_decode(pred, elen, vocab)) / frames

    lo, hi = 0.0, 8.0
    for _ in range(10):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if ctc_rate(mid) > 0.2 else (lo, mid)
    ctc_symbols = ctc_rate(hi)

    greedy = cn.GreedyBatchedRNNTInfer(dec, joint, vocab, 30)

    def rnnt_rate(b):
        with torch.no_grad():
            out_bias[vocab] = base_j + b
        greedy.invalidate()
        arr = greedy.decode_arrays(encoded, elen, max_tokens=30 * encoded.shape[2])
        return arr["n_tokens"].float().sum().item() / frames

    lo, hi = 0.0, 8.0
    for _ in range(10):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if rnnt_rate(mid) > 0.2 else (lo, mid)
    rnnt_symbols = rnnt_rate(hi)

    def run_ctc():
        y, yl = front(audio.to(device, non_blocking=True), lengths.to(device, non_blocking=True))
        _, pred = head.forward_with_predictions(y)
        return cn.ctc_greedy_decode(pred, yl, vocab)

    def run_rnnt():
        y, yl = front(audio.to(device, non_blocking=True), lengths.to(device, non_blocking=True))
        return greedy(encoder_output=y, encoded_lengths=yl)[0]

    res = {}
    for name, fn in (("waveform_to_ctc_ids", run_ctc), ("waveform_to_transducer_hypotheses", run_rnnt)):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) / steps * 1e3
        res[name] = {"value": round(batch * seconds / (ms * 1e-3), 1), "unit": UNIT, "ms_per_batch": round(ms, 3)}
    names = ["h2d_audio", "log_mel", "encoder", "ctc_head", "transducer_greedy_decode"]
    best = {k: float("inf") for k in names}
    for _ in range(3):  # device time of every stage (CUDA events), best of three passes
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        torch.cuda.synchronize()
        ev[0].record()
        a, n = audio.to(device, non_blocking=True), lengths.to(device, non_blocking=True)
        ev[1].record()
        feats, flen = pre(input_signal=a, length=n, check_lengths=False)
        ev[2].record()
        y, yl = enc(audio_signal=feats, length=flen)
        ev[3].record()
        head.forward_with_predictions(y)
        ev[4].record()
        greedy.decode_arrays(y, yl)
        ev[5].record()
        torch.cuda.synchronize()
        for i, k in enumerate(names):
            best[k] = min(best[k], ev[i].elapsed_time(ev[i + 1]))
    res["stage_ms"] = {k: round(v, 4) for k, v in best.items()}
    res["config"] = {"workload": f"{batch} x {seconds} s of 16 kHz audio in pinned host memory; log-mel 80; this encoder; CTC head "
                                 f"{vocab + 1} classes | transducer decoder / joint 640 / 640 / {vocab + 1}, max_symbols 30; ids on the host",
                     "ctc_symbols_per_frame": round(ctc_symbols, 4), "transducer_symbols_per_frame": round(rnnt_symbols, 4),
                     "h2d_bytes_per_batch": batch * n_samp * 4 + batch * 8, "steps": steps}
    return res


def _pin(t):
    return t.pin_memory() if torch.cuda.is_available() else t  # the reference arm also runs on GPU-less hosts


def build_batches(args, kw, rank, world, name=None):
    """The rank's sub-batches for one step: [(features (B, F, T) pinned host, lengths (B,) pinned host), ...].
    cfg3 (strong scaling): one global batch of 64 mixed-length utterances, planned over `world` ranks by
    conformer_nemo_b200.sharding.plan_shards (LPT assignment + length buckets, no communication).
    Every other workload (weak scaling): the same single full-length batch on every rank."""
    name = name or args.workload
    if WORKLOADS[name][1] is None:
        import random

        from conformer_nemo_b200.sharding import plan_shards

        rnd = random.Random(1234)  # SURVEY.md 8(d): len ~ U[200, 3000] frames, seed 1234
        lengths = [rnd.randint(200, 3000) for _ in range(64)]
        bucket = args.bucket_frames if args.bucket_frames == "auto" else int(args.bucket_frames)
        if args.packed != "off" and args.bucket_frames == "auto":
            bucket = 1 << 30  # packed layout: padding costs nothing, so a rank's share is ONE sub-batch (one launch set)
        plan = plan_shards(lengths, world, max_batch=args.max_batch, bucket_frames=bucket)
        g = torch.Generator().manual_seed(1234)
        out = []
        for sub in plan.batches[rank]:
            lens = [lengths[i] for i in sub]
            x = torch.zeros(len(sub), kw["feat_in"], max(lens))
            for row, n in enumerate(lens):
                x[row, :, :n] = torch.randn(kw["feat_in"], n, generator=g)
            out.append((_pin(x), _pin(torch.tensor(lens, dtype=torch.int64))))
        return out, sum(lengths) * FRAME_SEC, "strong", {"utterances": 64, "frames": "U[200,3000] seed 1234",
                                                         "sub_batches_rank0": len(out), "bucket_frames": args.bucket_frames,
                                                         "max_batch": args.max_batch,
                                                         "layout": "dense (padded sub-batches)" if args.packed == "off"
                                                         else "packed (cfb_forward_packed: one slot of token rows per utterance, no padding)"}
    _, b, t = WORKLOADS[name]
    g = torch.Generator().manual_seed(1234 + rank)
    x = _pin(torch.randn(b, kw["feat_in"], t, generator=g))
    ln = _pin(torch.full((b,), t, dtype=torch.int64))
    return [(x, ln)], b * t * FRAME_SEC * world, "weak", None


def measure_workload(enc, args, host_batches, audio_sec_job, device, barrier, max_over_ranks, sampler=None,
                     eager=True, keep_outputs=False):
    """Times one workload on this rank's sub-batches: device-resident steps launched eagerly, then through CUDA-graph
    replay (the headline), then end to end with host buffers.  Returns a dict; every time is the max over ranks.
    keep_outputs: the dict also holds `outputs`, the [(encoded, encoded_len), ...] of the last timed step on the host."""
    use_host_lens = args.packed != "off"
    enc.packed = True if args.packed == "on" else "auto"
    dev_batches = [(x.to(device), ln.to(device), ln.tolist() if use_host_lens else None) for x, ln in host_batches]
    main_stream = torch.cuda.current_stream(device)
    concurrent = [False]  # set once graphs with private workspaces are on: sub-batches overlap on side streams

    def step():
        """One forward of every sub-batch: [(encoded, encoded_len), ...]."""
        if concurrent[0]:
            return enc.forward_many(dev_batches, args.streams)
        return [enc(audio_signal=xd, length=ld, length_host=hl) for xd, ld, hl in dev_batches]

    enc.enable_cuda_graphs(False)
    launches_per_step = 0
    for i in range(max(args.warmup, 3)):
        for xd, ld, hl in dev_batches:
            enc(audio_signal=xd, length=ld, length_host=hl)
            if i == 0:
                launches_per_step += enc.last_launch_count()
    if args.ncu:
        return {"step": step, "launches_per_step": launches_per_step}
    # a fresh box needs a moment of sustained load before clocks / power state settle: keep warming for ~1 s
    torch.cuda.synchronize()
    t_warm = time.time()
    while time.time() - t_warm < args.settle:
        step()
        torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eager_ms = None
    if eager:
        # ---------------- the steps launched eagerly (host-side launch cost included); reported beside the headline
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
        eager_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps

    # ---------------- headline: the public forward with CUDA graphs on (ConformerEncoder.enable_cuda_graphs).
    # cfb_forward is enqueue-only (no allocation, no sync), so the wrapper captures one graph per input shape and a
    # step = copy the inputs into the graph's static buffers (device to device) + one replay of ~260 kernel nodes.
    if not args.no_graphs:
        concurrent[0] = args.streams > 1 and len(dev_batches) > 1
        enc.enable_cuda_graphs(True, max_shapes=max(4, len(dev_batches)), private_workspaces=concurrent[0])
    for _ in range(3):
        step()
    barrier()
    if sampler is not None:
        sampler.mark()
    e0.record()
    for _ in range(args.steps):
        outs = step()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler is not None else None
    outputs = None
    if keep_outputs:
        # graph replays return views of the graph's static buffers, which the end-to-end pass below overwrites.  One after
        # the other, sub-batches of one shape also replay one graph, so the last step kept only the last one's result:
        # then one more (untimed) step copies every result out before the next forward; the forward is deterministic.
        if len(dev_batches) > 1 and not concurrent[0]:
            outputs = []
            for xd, ld, hl in dev_batches:
                y, ylen = enc(audio_signal=xd, length=ld, length_host=hl)
                outputs.append((y.cpu(), ylen.cpu()))
        else:
            outputs = [(y.cpu(), ylen.cpu()) for y, ylen in outs]
    ms_step = ms_total / args.steps
    value = audio_sec_job / (ms_step / 1e3)

    # ---------------- end to end through the public API with host buffers
    # Two-deep software pipeline, as a serving loop would run it: a copy stream moves the next sub-batch's features
    # in and the previous result out while the current one computes (PCIe is full duplex).  Every sub-batch's H2D and
    # D2H are inside the timed region; the closing event waits for the last D2H.
    n_buf = 2
    shapes = [(x.shape[0], enc.output_frames(x.shape[2])) for x, _ in host_batches]
    d_out = outs[-1][0].shape[1]
    max_b = max(sh[0] for sh in shapes)
    max_bt = max(sh[0] * sh[1] for sh in shapes)
    max_in = max(x.numel() for x, _ in host_batches)
    out_host = [torch.empty(max_bt * d_out, dtype=torch.float32).pin_memory() for _ in range(n_buf)]
    olen_host = [torch.empty(max_b, dtype=torch.int32).pin_memory() for _ in range(n_buf)]
    x_stage = [torch.empty(max_in, dtype=torch.float32, device=device) for _ in range(n_buf)]
    len_stage = [torch.empty(max_b, dtype=torch.int64, device=device) for _ in range(n_buf)]
    y_stage = [torch.empty(max_bt * d_out, dtype=torch.float32, device=device) for _ in range(n_buf)]
    ylen_stage = [torch.empty(max_b, dtype=torch.int32, device=device) for _ in range(n_buf)]
    copy_stream = torch.cuda.Stream(device=device)
    ev_in = [torch.cuda.Event() for _ in range(n_buf)]        # features of the slot are on the device
    ev_used = [torch.cuda.Event() for _ in range(n_buf)]      # the forward has consumed the slot's features
    ev_out = [torch.cuda.Event() for _ in range(n_buf)]       # the slot's result is in y_stage
    ev_done = [torch.cuda.Event() for _ in range(n_buf)]      # the slot's result is in host memory
    n_sub = len(host_batches)
    host_lens = [ln.tolist() if use_host_lens else None for _, ln in host_batches]

    def e2e_run(n_steps):
        total = n_steps * n_sub
        for k in range(n_buf):
            ev_used[k].record(main_stream)
            ev_done[k].record(copy_stream)

        def h2d(i):
            k = i % n_buf
            xh, lh = host_batches[i % n_sub]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_used[k])
                x_stage[k][: xh.numel()].view_as(xh).copy_(xh, non_blocking=True)
                len_stage[k][: lh.numel()].copy_(lh, non_blocking=True)
                ev_in[k].record(copy_stream)

        h2d(0)
        for i in range(total):
            k = i % n_buf
            xh, lh = host_batches[i % n_sub]
            bb, tt = shapes[i % n_sub]
            if i + 1 < total:
                h2d(i + 1)
            main_stream.wait_event(ev_in[k])
            yy, ll = enc(audio_signal=x_stage[k][: xh.numel()].view_as(xh), length=len_stage[k][: lh.numel()],
                         length_host=host_lens[i % n_sub])
            ev_used[k].record(main_stream)
            main_stream.wait_event(ev_done[k])            # the slot's previous result has left the device
            y_stage[k][: bb * tt * d_out].view(bb, tt, d_out).copy_(yy.transpose(1, 2))
            ylen_stage[k][:bb].copy_(ll)
            ev_out[k].record(main_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_out[k])
                out_host[k][: bb * tt * d_out].copy_(y_stage[k][: bb * tt * d_out], non_blocking=True)
                olen_host[k][:bb].copy_(ylen_stage[k][:bb], non_blocking=True)
                ev_done[k].record(copy_stream)
        for k in range(n_buf):
            main_stream.wait_event(ev_done[k])

    # Several sub-batches per step (cfg3) with graphs that own their workspaces: every sub-batch is a chain
    # H2D -> forward (graph replay) -> D2H on ONE of `--streams` side streams, chains of different sub-batches overlap.
    # Sub-batches of the same shape share a graph (static buffers), so they are kept on the same stream.
    if concurrent[0]:
        side = [torch.cuda.Stream(device=device) for _ in range(args.streams)]
        x_dev = [torch.empty_like(x, device=device) for x, _ in host_batches]
        l_dev = [torch.empty_like(ln, device=device) for _, ln in host_batches]
        y_host = [torch.empty(bb, tt, d_out, dtype=torch.float32).pin_memory() for bb, tt in shapes]
        yl_host = [torch.empty(bb, dtype=torch.int32).pin_memory() for bb, _ in shapes]
        stream_of, lane_of = {}, []
        for i, (x, ln) in enumerate(host_batches):
            lane_of.append(stream_of.setdefault((tuple(x.shape), tuple(ln.tolist())), i % args.streams))

        def e2e_run(n_steps):  # noqa: F811 -- replaces the 2-deep pipeline above for this workload
            for sd_ in side:
                sd_.wait_stream(main_stream)
            for _ in range(n_steps):
                for i, (xh, lh) in enumerate(host_batches):
                    with torch.cuda.stream(side[lane_of[i]]):
                        x_dev[i].copy_(xh, non_blocking=True)
                        l_dev[i].copy_(lh, non_blocking=True)
                        yy, ll = enc(audio_signal=x_dev[i], length=l_dev[i], length_host=host_lens[i])
                        y_host[i].copy_(yy.transpose(1, 2), non_blocking=True)
                        yl_host[i].copy_(ll, non_blocking=True)
            for sd_ in side:
                main_stream.wait_stream(sd_)

    e2e_run(2)
    barrier()
    e0.record()
    e2e_run(args.steps)
    e1.record()
    barrier()
    seq_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps

    e2e = {"value": audio_sec_job / (seq_ms / 1e3), "unit": UNIT, "ms_per_step": seq_ms,
           "mode": (f"per sub-batch: pinned H2D of the features, ConformerEncoder.forward (CUDA graphs with private workspaces), D2H "
                    f"of encoded + encoded_len, as one chain on one of {args.streams} side streams; chains of different "
                    "sub-batches overlap") if concurrent[0] else
                   "per sub-batch: pinned H2D of the features, ConformerEncoder.forward (CUDA graphs on), D2H of encoded "
                   "+ encoded_len; copies of neighbouring sub-batches overlap the forward on a second stream "
                   "(2-deep pipeline)",
           "h2d_bytes_per_step": sum(x.numel() * 4 + ln.numel() * 8 for x, ln in host_batches),
           "d2h_bytes_per_step": sum(bb * tt * d_out * 4 + bb * 4 for bb, tt in shapes)}
    return {"value": value, "ms_per_step": ms_step, "eager_ms_per_step": eager_ms, "e2e": e2e, "clocks": clocks,
            "launches_per_step": launches_per_step, "step": step, "sub_batches_in_flight": args.streams if concurrent[0] else 1,
            "outputs": outputs}


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much
DUMP_WHOLE_BYTES = 1 << 20  # arrays up to this size are always written whole


def dump_outputs(out_dir, outputs):
    """Writes the [(encoded, encoded_len), ...] of one step as out_dir/encoded.npy and out_dir/encoded_len.npy (with a
    _<i> suffix per sub-batch when there are several): floating arrays as float32, integer ones as float64 (exact).
    When the arrays exceed DUMP_BYTES, each one larger than DUMP_WHOLE_BYTES is replaced by the same seeded sample of
    its flattened (C-order) elements, written as <name>.npy beside the float64 flat indices in <name>_index.npy."""
    import numpy as np

    named = {}
    for i, (y, ylen) in enumerate(outputs):
        sfx = f"_{i}" if len(outputs) > 1 else ""
        named["encoded" + sfx] = y.float().contiguous().numpy()
        named["encoded_len" + sfx] = ylen.double().numpy()
    total = sum(a.nbytes for a in named.values())
    if total > DUMP_BYTES:
        big = [k for k, a in named.items() if a.nbytes > DUMP_WHOLE_BYTES]
        headers = 1024 * (len(named) + len(big))  # a .npy header is 128 bytes
        budget = DUMP_BYTES - headers - sum(a.nbytes for k, a in named.items() if k not in big)
        frac = budget / sum(named[k].size * (named[k].itemsize + 8) for k in big)  # a sampled value + its index
        for k in big:
            a = named.pop(k).reshape(-1)
            g = torch.Generator().manual_seed(0)
            idx = torch.randperm(a.size, generator=g)[: int(a.size * frac)].sort().values.numpy()
            named[k] = a[idx]
            named[k + "_index"] = idx.astype("float64")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in named.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return sorted(named)


def packing_stats(enc, host_batches):
    """Token rows the step computes on: dense = sum B * T'max of the sub-batches, packed = the slots, valid = sum T'_b."""
    dense = sum(x.shape[0] * enc.output_frames(x.shape[2]) for x, _ in host_batches)
    packed = sum(enc.packed_rows(ln.tolist(), x.shape[2]) for x, ln in host_batches)
    valid = sum(_out_frames(int(n))[1] for _, ln in host_batches for n in ln.tolist())
    return {"token_rows_valid": valid, "token_rows_packed": packed, "token_rows_dense": dense}


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        # rank 0 prints exactly one JSON line on stdout: NCCL's own output (version banner at WARN/INFO) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=device)
    kw = WORKLOADS[args.workload][0]
    enc = build_encoder(kw, device)
    if args.share and world == 1:
        # diagnostic: this one GPU runs the share rank R of a W-rank job would run (cfg3); `value` then counts the whole
        # job's audio against this share's time, i.e. what the W-GPU job would report if R were its slowest rank
        sr, sw = (int(v) for v in args.share.split("/"))
        host_batches, audio_sec_job, scaling, extra_cfg = build_batches(args, kw, sr, sw)
        extra_cfg = dict(extra_cfg or {}, emulated_share=f"rank {sr} of {sw} on one GPU")
    else:
        host_batches, audio_sec_job, scaling, extra_cfg = build_batches(args, kw, rank, world)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        tt = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # ---------------- device-resident throughput + end to end (the headline workload)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    head = measure_workload(enc, args, host_batches, audio_sec_job, device, barrier, max_over_ranks,
                            sampler if rank == 0 else None, keep_outputs=bool(args.dump_outputs) and rank == 0)
    outputs = head.pop("outputs", None)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    step = head["step"]
    if args.ncu:
        # profiling helper: 3 warm-up steps above, ONE eager step here, nothing else (no graphs, no e2e, no JSON):
        #   ncu -s <3 * launches/step> -c <launches/step> ... python bench.py --ncu
        step()
        torch.cuda.synchronize()
        if rank == 0:
            emit({"ncu_helper": True, "launches_per_step": head["launches_per_step"]})
        return
    launches_per_step = head["launches_per_step"]

    # ---------------- per-kernel timing pass (CUDA events on the forward's stream) -> roofline
    roofline, kernels = None, None
    if rank == 0:
        pk = peaks()
        # (1) eager brackets: CUDA events recorded around every launch while the host enqueues the step
        enc.enable_cuda_graphs(False)
        enc.set_profiling(True)
        prof_steps = 3
        for _ in range(prof_steps):
            step()
        rep_eager = enc.profile_report()
        # (2) the same brackets as event-record nodes of a captured graph (one forward per sub-batch on one stream, as in
        # (1)): replayed, the intervals hold each kernel plus the node-to-node launch latency, and none of the host's
        # enqueue cost -- a 5 us kernel bracketed eagerly measures mostly how fast the host enqueues.  These are the times
        # the roofline fractions below use; the eager ones are kept beside them.
        rep, prof_how = None, None
        try:
            dev_b = [(x.to(device), ln.to(device), ln.tolist() if args.packed != "off" else None) for x, ln in host_batches]
            side = torch.cuda.Stream(device)
            side.wait_stream(torch.cuda.current_stream(device))
            with torch.cuda.stream(side):
                for xd, ld, hl in dev_b:
                    enc(audio_signal=xd, length=ld, length_host=hl)
                torch.cuda.synchronize()
                enc.set_profiling(True)  # drops the eager records; the capture below registers the brackets once
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    for xd, ld, hl in dev_b:
                        enc(audio_signal=xd, length=ld, length_host=hl)
                for _ in range(3):
                    graph.replay()
                torch.cuda.synchronize()
                rep = enc.profile_report()  # intervals of the last replay
            prof_steps_used = 1
            prof_how = ("CUDA events recorded as nodes of a captured graph of the step (single stream), intervals of the last "
                        "of 3 replays after the timed region")
            del graph
        except Exception as e:  # noqa: BLE001 -- the eager brackets remain
            sys.stderr.write(f"bench: graph-timed kernel pass failed ({e}); using the eager brackets\n")
            rep = None
        enc.set_profiling(False)
        if not rep:
            rep, prof_steps_used = rep_eager, prof_steps
            prof_how = f"CUDA events around every launch (eager), {prof_steps} extra steps after the timed region"
        prof_steps_eager, prof_steps = prof_steps, prof_steps_used
        fl, by = algorithmic_costs(kw, [ln.tolist() for _, ln in host_batches])
        kernels = {}
        # timer overhead: the engine also brackets NOTHING once per forward ("(empty bracket)": two event records back to
        # back).  A bracket around a kernel holds that fixed cost plus the kernel's own launch latency and run time; the
        # net time (and the fractions computed from it) subtracts the former only.  Raw figures are kept beside them.
        empty = rep.pop("(empty bracket)", None)
        rep_eager.pop("(empty bracket)", None)
        bracket_ms = (empty[1] / max(empty[0], 1)) if empty else 0.0

        def net_ms(n_launch, ms):
            return max(ms - n_launch * bracket_ms, 0.05 * ms)

        for label, (n_launch, ms) in rep.items():
            per_fwd_ms = ms / prof_steps
            per_fwd_net = net_ms(n_launch, ms) / prof_steps
            ent = {"launches_per_step": n_launch // prof_steps, "ms_per_step": round(per_fwd_net, 4),
                   "ms_per_step_raw_brackets": round(per_fwd_ms, 4)}
            if rep is not rep_eager and label in rep_eager:
                ent["ms_per_step_eager_brackets"] = round(rep_eager[label][1] / prof_steps_eager, 4)
            if label in fl:
                ach = fl[label] / (per_fwd_net / 1e3) / 1e12
                ent.update(bound="tensor", achieved=round(ach, 1), unit="TFLOP/s", frac=round(ach / pk["tflops"], 4),
                           frac_raw_brackets=round(fl[label] / (per_fwd_ms / 1e3) / 1e12 / pk["tflops"], 4))
            elif label in by:
                ach = by[label] / (per_fwd_net / 1e3) / 1e9
                ent.update(bound="hbm", achieved=round(ach, 1), unit="GB/s", frac=round(ach / pk["gbs"], 4),
                           frac_raw_brackets=round(by[label] / (per_fwd_ms / 1e3) / 1e9 / pk["gbs"], 4))
            kernels[label] = ent
        gemm_bytes = gemm_algorithmic_bytes(kw, [ln.tolist() for _, ln in host_batches])
        gemm_ms_raw = sum(rep[l][1] for l in GEMM_LABELS if l in rep) / prof_steps
        gemm_ms = sum(net_ms(*rep[l]) for l in GEMM_LABELS if l in rep) / prof_steps
        gemm_fl = sum(fl[l] for l in GEMM_LABELS if l in rep)
        gemm_launches = sum(rep[l][0] for l in GEMM_LABELS if l in rep) // prof_steps
        ach = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        ach_raw = gemm_fl / (gemm_ms_raw / 1e3) / 1e12 if gemm_ms_raw > 0 else 0.0
        traffic, traffic_src = None, None
        try:  # DRAM bytes per launch of the same kernels from the committed ncu --set full capture (tools/ncu_summary.py)
            with open(os.path.join(ROOT, "profiles", "ncu_traffic_gemm.json")) as f:
                tj = json.load(f)
            if args.workload == "cfg2":
                traffic, traffic_src = round(tj["traffic_bytes_per_launch"]), f"profiles/{tj['report']} ({tj['how']})"
        except (OSError, KeyError, ValueError):
            pass
        roofline = {"kernel": "gemm_tc_kernel / gemm_tc2_kernel (tcgen05 GEMM family, single CTA and CTA pair: "
                              + ", ".join(GEMM_LABELS) + ")",
                    "bound": "tensor", "achieved": round(ach, 1), "peak": pk["tflops"], "unit": "TFLOP/s",
                    "frac": round(ach / pk["tflops"], 4),
                    "achieved_raw_brackets": round(ach_raw, 1), "frac_raw_brackets": round(ach_raw / pk["tflops"], 4),
                    "bracket_overhead_ms": round(bracket_ms, 5),
                    # the timed region is short enough to run near the maximum SM clock (see `clocks`), where the
                    # burst figure is the fairer denominator: both are given
                    "peak_burst": pk["burst"], "frac_of_burst": round(ach / pk["burst"], 4), "traffic": traffic, "traffic_unit": "bytes per launch (DRAM read + write)",
                    "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": round(sum(gemm_bytes.get(l, 0) for l in GEMM_LABELS if l in rep) / max(gemm_launches, 1)),
                    "peak_source": pk["source"],
                    "launches_per_step": gemm_launches, "avg_launch_ms": round(gemm_ms / max(gemm_launches, 1), 5),
                    "share_of_step": round(gemm_ms_raw / sum(v[1] for v in rep.values()) * prof_steps, 4),
                    "how": prof_how + "; `achieved` / `frac` are net of the measured cost of an empty bracket per launch "
                           "(`bracket_overhead_ms`), the `_raw_brackets` figures are not"}

    # ---------------- strong scaling of the split the north star names (cfg3), same encoder, same process
    strong = None
    if args.strong and WORKLOADS[args.workload][0] == WORKLOADS["cfg3"][0] and WORKLOADS[args.workload][1] is not None:
        s_batches, s_audio, _, s_cfg = build_batches(args, kw, rank, world, name="cfg3")
        sm = measure_workload(enc, args, s_batches, s_audio, device, barrier, max_over_ranks, None, eager=False)
        stats = packing_stats(enc, s_batches)
        # algorithmic FLOPs of THIS rank's share (valid frames only, SURVEY.md 8(d)) against the step time: how far the
        # share is from the tensor peak once padding is gone -- the rest is the fixed cost of ~250 dependent launches
        fl_s, _ = algorithmic_costs(kw, [ln.tolist() for _, ln in s_batches])
        share_tflop = sum(v for k, v in fl_s.items()) / 1e12
        stats.update(algorithmic_tflop=round(share_tflop, 4),
                     achieved_tflops=round(share_tflop / (sm["ms_per_step"] / 1e3), 1),
                     frac_of_sustained_peak=round(share_tflop / (sm["ms_per_step"] / 1e3) / peaks()["tflops"], 4))
        strong = {"workload": workload_config("cfg3", world)["workload"], "metric": METRIC, "unit": UNIT,
                  "value": sm["value"], "ms_per_step": sm["ms_per_step"], "n_gpus": world, "steps": args.steps,
                  "scaling": "strong", "audio_sec_per_step": s_audio, "e2e": sm["e2e"],
                  "sub_batches_rank0": len(s_batches), "sub_batches_in_flight": sm["sub_batches_in_flight"],
                  "launches_per_step_rank0": sm["launches_per_step"], "rank0": stats, **(s_cfg or {})}
        if world == 1 and args.strong_sim:
            # what every rank of a 2 / 4 / 8-GPU job would run, measured one share after the other on THIS GPU (the path
            # has no communication, so a rank's time does not depend on the others); the slowest share sets the step
            sim = {}
            for w in (2, 4, 8):
                worst, per_rank = 0.0, []
                for r in range(w):
                    rb, _, _, _ = build_batches(args, kw, r, w, name="cfg3")
                    saved = args.settle
                    args.settle = 0.0
                    try:
                        m = measure_workload(enc, args, rb, s_audio, device, barrier, max_over_ranks, None, eager=False)
                    finally:
                        args.settle = saved
                    per_rank.append(round(m["ms_per_step"], 4))
                    worst = max(worst, m["ms_per_step"])
                sim[str(w)] = {"ms_per_step_slowest_rank": worst, "value": s_audio / (worst / 1e3),
                               "speedup_vs_1gpu": sm["ms_per_step"] / worst, "ms_per_rank": per_rank}
            strong["emulated_on_one_gpu"] = sim

    # ---------------- CPU baseline: the reference's own forward (or the oracle port) on the WHOLE workload batch, rank 0, N=1
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = time_cpu_arm(kw, {k: v.detach().float().cpu() for k, v in enc.state_dict().items()},
                                    [(x, ln) for x, ln in host_batches], warmup=1, steps=2, budget_s=60.0)

    pipelines = None
    if rank == 0 and world == 1 and args.pipelines and args.workload == "cfg2":
        try:
            pipelines = measure_pipelines(enc, device, steps=args.steps)
        except Exception as e:  # noqa: BLE001 -- an extra record must never cost the headline
            pipelines = {"unavailable": f"{type(e).__name__}: {e}"}

    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cfg = workload_config(args.workload, world)
    if extra_cfg:
        cfg.update(extra_cfg)
        cfg["sub_batches_in_flight"] = head["sub_batches_in_flight"]
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic (randn log-mel features, random-init weights)",
        "config": cfg, "clocks": head["clocks"], "e2e": head["e2e"],
        "gpu_launches": launches_per_step * args.steps,
        "launch_mode": "eager" if args.no_graphs else "cuda graph replay", "eager_ms_per_step": head["eager_ms_per_step"],
        "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu_baseline, "strong": strong,
        "pipelines": pipelines,
    }
    emit(line)


def cpu_forward_fn(kw, sd):
    """The CPU arm's forward: the reference's own unmodified ConformerEncoder when a reference tree is reachable
    ($CONFORMER_REF, /root/reference, or the per-pod install baseline/_ref written by oracle/install_reference.py),
    else the oracle port of its algorithm.  The only place the benchmark touches oracle/ (cpu_baseline / reference arm)."""
    from oracle import conformer_oracle as oc
    from oracle import reference_loader as rl

    cfg = oc.EncoderConfig(feat_in=kw["feat_in"], n_layers=kw["n_layers"], d_model=kw["d_model"], n_heads=kw["n_heads"])
    if sd is None:
        sd = oc.random_state_dict(cfg, 0)
    sd = {k: v for k, v in sd.items() if not k.endswith("num_batches_tracked")}
    if rl.reference_available():
        try:
            ref = rl.build_reference_encoder(cfg, sd)

            def fwd(x, length):
                with torch.no_grad():
                    return ref(audio_signal=x, length=length)

            return fwd, "reference", f"unmodified ConformerEncoder.forward loaded from {rl.REFERENCE_ROOT}"
        except Exception as e:  # pragma: no cover - fall back to the port, say why
            why = f"reference at {rl.REFERENCE_ROOT} failed to load ({type(e).__name__}: {e}); oracle port timed instead"
    else:
        why = "no reference tree reachable (looked at $CONFORMER_REF, /root/reference, baseline/_ref, oracle/_ref); oracle port"
    return (lambda x, length: oc.encoder_forward(sd, cfg, x, length)), "port", why


def time_cpu_arm(kw, sd, batches, warmup, steps, budget_s):
    """Times the CPU arm on the given sub-batches [(features (B, F, T), lengths (B,))] = one step of the workload.
    `steps` timed steps after `warmup`, cut short (never below one step) once `budget_s` seconds have been spent."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fwd, kind, how = cpu_forward_fn(kw, sd)
    batches = [(x.float(), ln.to(torch.int64)) for x, ln in batches]
    audio = sum(float(ln.sum()) for _, ln in batches) * FRAME_SEC
    t_begin = time.perf_counter()

    def one_step():
        t0 = time.perf_counter()
        for x, ln in batches:
            fwd(x, ln)
        return time.perf_counter() - t0

    done_w = 0
    for _ in range(warmup):
        one_step()
        done_w += 1
        if time.perf_counter() - t_begin > budget_s / 2:
            break
    times = []
    for _ in range(steps):
        times.append(one_step())
        if time.perf_counter() - t_begin > budget_s:
            break
    sec = sum(times) / len(times)
    cpu_model = ""
    try:
        with open("/proc/cpuinfo") as f:
            cpu_model = next((l.split(":", 1)[1].strip() for l in f if l.startswith("model name")), "")
    except OSError:
        pass
    shape = ", ".join(f"{x.shape[0]} x {x.shape[2]} frames" for x, _ in batches[:4]) + (" ..." if len(batches) > 4 else "")
    return {"value": audio / sec, "unit": UNIT, "cores": cores, "kind": kind, "sec_per_step": sec,
            "steps": len(times), "warmup": done_w, "cpu_model": cpu_model, "how": how,
            "sample": f"the whole workload step ({shape}; {audio:.0f} s of audio), fp32, torch {torch.__version__} CPU "
                      f"kernels, {cores} threads, mean of {len(times)} after {done_w} warm-up"}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores, on the b200 arm's config
    (whole workload batch per step).  --steps / --warmup are honoured unless the run would exceed ~4 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    kw = WORKLOADS[args.workload][0]
    host_batches, _, _, _ = build_batches(args, kw, 0, 1)
    res = time_cpu_arm(kw, None, host_batches, warmup=max(1, args.warmup), steps=max(1, args.steps), budget_s=240.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world,
        "steps": res["steps"], "warmup": res["warmup"], "ms_per_step": res["sec_per_step"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, world), "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.workload == "cfg2":
        # BASELINE.md section 3: cfg 1 (Small, d_model 176, 16 layers, 4 heads, 4 x 10 s) in full, the reference's own CPU case
        kw1 = dict(feat_in=80, n_layers=16, d_model=176, n_heads=4)
        g = torch.Generator().manual_seed(1234)
        b1 = [(torch.randn(4, 80, 1000, generator=g), torch.full((4,), 1000, dtype=torch.int64))]
        r1 = time_cpu_arm(kw1, None, b1, warmup=2, steps=5, budget_s=30.0)
        line["cfg1"] = {"workload": "cfg1: Conformer-CTC Small encoder d_model=176 layers=16 heads=4, batch 4 x 10 s, fp32 on the host cores",
                        **r1}
    emit(line)


_JSON_OUT = None


def emit(line: dict) -> None:
    """The contract line goes to the process's ORIGINAL stdout; everything else (NCCL's version banner, library
    chatter, stray prints) was re-pointed at stderr by main()."""
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    # stdout carries exactly one JSON line: keep a private handle to it and send file descriptor 1 to stderr, so that
    # C-level writers (NCCL prints its banner with printf at NCCL_DEBUG=VERSION / WARN) cannot get in front of it
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the throughput measurements (headline, eager, e2e, strong, pipelines); the per-kernel and "
                         "per-stage breakdowns and cpu_baseline keep their own counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--bucket-frames", default="auto",
                    help="cfg3: length-bucket width in input frames, or auto (sharding.plan_cost picks it)")
    ap.add_argument("--max-batch", type=int, default=64, help="cfg3: utterances per sub-batch at most")
    ap.add_argument("--streams", type=int, default=3,
                    help="cfg3: sub-batches of a rank in flight at once (ConformerEncoder.forward_many); 1 = one after the other")
    ap.add_argument("--packed", default="auto", choices=["auto", "on", "off"],
                    help="variable-length layout (cfb_forward_packed) for mixed-length batches: auto = when it saves >= 15 %% "
                         "of the token rows, off = dense padded sub-batches")
    ap.add_argument("--no-pipelines", dest="pipelines", action="store_false",
                    help="skip the waveform -> token ids records (log-mel + encoder + CTC head / transducer decode) of the cfg2 line")
    ap.add_argument("--no-strong", dest="strong", action="store_false",
                    help="skip the cfg3 strong-scaling sub-record of the default (cfg2) line")
    ap.add_argument("--no-strong-sim", dest="strong_sim", action="store_false",
                    help="N=1: skip the one-GPU emulation of the 2/4/8-rank shares of cfg3")
    ap.add_argument("--share", default="", help="cfg3 diagnostic on one GPU: R/W = run the share of rank R of a W-rank job")
    ap.add_argument("--settle", type=float, default=1.0, help="seconds of extra warm-up load before timing")
    ap.add_argument("--ncu", action="store_true", help="3 warm-up steps + 1 eager step only (for ncu -s/-c)")
    ap.add_argument("--no-graphs", action="store_true", help="launch every step eagerly (no CUDA graph replay)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the encoder outputs of the last timed step of the headline as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.ncu):
        ap.error("--dump-outputs needs the timed steps of the b200 arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
