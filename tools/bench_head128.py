"""Heads 128 wide against heads 64 wide: attention alone, the whole encoder, and the cfg 2 no-regression check.

    python tools/bench_head128.py [--iters 20] [--parent-lib PATH] [--out profiles/head128_b200.json]

* Attention alone (cfb_op_rel_attention, all rows full): at equal d_model, (H 8, dk 64) against (H 4, dk 128) at
  d 512 and (H 16, dk 64) against (H 8, dk 128) at d 1024, B 32 x T' 500; plus B 1 x T' 7500 at d 1024.  Each
  configuration is warmed up, then the configurations are timed in alternation, ITERS launches between CUDA events
  per round.  The op converts its bf16 positional projections to fp16 per call (the encoder does it once per forward),
  so a separate torch.profiler pass reports the attention kernel alone as well.  Algorithmic rate: 6 B T^2 H dk
  (Q K^T, Q P^T and P V) over the kernel time, and its share of the 1399.7 TFLOP/s sustained dense bf16 peak the
  project uses (BASELINE.md).
* Whole encoder, XLarge shape: d 1024, 24 layers, 32 x 20 s, bf16, CUDA-graph replay; H 8 (dk 128) beside H 16
  (dk 64), alternating.
* No regression: cfg 2 (d 512, H 8, 17 layers, 32 x 20 s, graph replay) with this build and with --parent-lib
  (libcfb.so of the parent commit), alternating, each in a fresh process.
The card name and power limit are read in the same run and written into the JSON.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_TFLOPS = 1399.7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


# ---------------------------------------------------------------------------------------------------- attention alone
def attention_cases():
    # name, B, T, H, dk
    return [("d512_h8_dk64", 32, 500, 8, 64), ("d512_h4_dk128", 32, 500, 4, 128),
            ("d1024_h16_dk64", 32, 500, 16, 64), ("d1024_h8_dk128", 32, 500, 8, 128),
            ("long_d1024_h16_dk64", 1, 7500, 16, 64), ("long_d1024_h8_dk128", 1, 7500, 8, 128)]


def bench_attention(iters, rounds):
    import ctypes

    import torch

    from conformer_nemo_b200 import _lib

    lib = _lib.load_library()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    cases = {}
    for name, B, T, H, dk in attention_cases():
        Dp = H * dk
        qkv = (torch.randn(B * T, 4 * Dp, device="cuda", generator=g) * 0.5).bfloat16()
        pos = (torch.randn(2 * T - 1, Dp, device="cuda", generator=g) * 0.5).bfloat16()
        ctx = torch.empty(B * T, Dp, device="cuda", dtype=torch.bfloat16)
        lens = torch.full((B,), T, dtype=torch.int32, device="cuda")

        def run(qkv=qkv, pos=pos, ctx=ctx, lens=lens, B=B, T=T, H=H, dk=dk):
            rc = lib.cfb_op_rel_attention(1, ctypes.c_void_p(qkv.data_ptr()), ctypes.c_void_p(pos.data_ptr()), pos.stride(0),
                                          ctypes.c_void_p(ctx.data_ptr()), ctypes.c_void_p(lens.data_ptr()), B, T, H, dk, dk,
                                          st)
            assert rc == 0, _lib.last_error(None)

        for _ in range(5):
            run()
        cases[name] = dict(run=run, B=B, T=T, H=H, dk=dk, ms=[])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for c in cases.values():
            e0.record()
            for _ in range(iters):
                c["run"]()
            e1.record()
            torch.cuda.synchronize()
            c["ms"].append(e0.elapsed_time(e1) / iters)
    # kernel time alone: torch.profiler over one more pass
    from torch.profiler import ProfilerActivity, profile

    kern = {}
    for name, c in cases.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(iters):
                c["run"]()
            torch.cuda.synchronize()
        us = [e.device_time_total / e.count for e in prof.key_averages() if "rel_attn" in e.key and e.count > 0]
        kern[name] = max(us) / 1e3 if us else None  # ms per launch
    out = {}
    for name, c in cases.items():
        fl = 6.0 * c["B"] * c["T"] ** 2 * c["H"] * c["dk"]
        best = min(c["ms"])
        k = kern[name]
        out[name] = dict(B=c["B"], T=c["T"], H=c["H"], dk=c["dk"], op_ms_rounds=[round(v, 4) for v in c["ms"]],
                         op_ms_best=round(best, 4), kernel_ms=round(k, 4) if k else None,
                         kernel_tflops=round(fl / k / 1e9, 1) if k else None,
                         kernel_share_of_peak=round(fl / k / 1e9 / PEAK_TFLOPS, 4) if k else None)
    for d, a, b in (("d512", "d512_h8_dk64", "d512_h4_dk128"), ("d1024", "d1024_h16_dk64", "d1024_h8_dk128"),
                    ("long_d1024", "long_d1024_h16_dk64", "long_d1024_h8_dk128")):
        if out[a]["kernel_ms"] and out[b]["kernel_ms"]:
            out[f"ratio_{d}_dk128_over_dk64_kernel"] = round(out[b]["kernel_ms"] / out[a]["kernel_ms"], 3)
        out[f"ratio_{d}_dk128_over_dk64_op"] = round(out[b]["op_ms_best"] / out[a]["op_ms_best"], 3)
    return out


# ---------------------------------------------------------------------------------------------------- whole encoder
def encoder_worker(d, heads, layers, steps, warmup, lib_path):
    """One configuration in this process: graph replay of a 32 x 2000-frame bf16 batch, ms per step."""
    import torch

    from conformer_nemo_b200 import _lib

    if lib_path:
        _lib.LIB_PATH = lib_path
    import conformer_nemo_b200 as cn
    from oracle import conformer_oracle as oc

    cfg = oc.EncoderConfig(feat_in=80, n_layers=layers, d_model=d, n_heads=heads)
    sd = oc.random_state_dict(cfg, 1)
    B, T = 32, 2000
    x, length = oc.synthetic_batch(B, 80, T, None, seed=2)
    enc = cn.ConformerEncoder(feat_in=80, n_layers=layers, d_model=d, n_heads=heads)
    enc.load_state_dict(sd, strict=False)
    enc = enc.cuda().eval()
    enc.enable_cuda_graphs(True)
    xs, ls = x.cuda(), length.cuda()
    for _ in range(warmup):
        enc(audio_signal=xs, length=ls)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        y, _ = enc(audio_signal=xs, length=ls)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return dict(d_model=d, n_heads=heads, dk=d // heads, layers=layers, B=B, frames=T, ms_per_step=round(ms, 3),
                audio_s_per_s=round(B * T / 100.0 / (ms / 1e3), 1), checksum=float(y.float().abs().sum()))


def spawn(d, heads, layers, steps, warmup, lib_path=None):
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", f"{d},{heads},{layers},{steps},{warmup}"]
    if lib_path:
        cmd += ["--lib", lib_path]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError(r.stdout[-3000:] + r.stderr[-3000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20, help="timed launches / steps per round (>= 20)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parent-lib", default=None, help="libcfb.so of the parent commit for the cfg 2 comparison")
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-encoder", action="store_true")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--lib", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        d, h, n_layers, steps, warmup = (int(v) for v in args.worker.split(","))
        print(json.dumps(encoder_worker(d, h, n_layers, steps, warmup, args.lib)))
        return
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing here is measured without the GPU")
    res = dict(card=card(), torch=torch.__version__, iters=args.iters, rounds=args.rounds, time=time.strftime("%Y-%m-%d %H:%M:%S"))
    res["attention"] = bench_attention(args.iters, args.rounds)
    print(json.dumps(res["attention"], indent=1), flush=True)
    if not args.skip_encoder:
        runs = {"xlarge_h8_dk128": [], "xlarge_h16_dk64": []}
        for _ in range(2):  # alternating, each in a fresh process
            runs["xlarge_h8_dk128"].append(spawn(1024, 8, 24, args.iters, args.warmup))
            runs["xlarge_h16_dk64"].append(spawn(1024, 16, 24, args.iters, args.warmup))
        res["encoder_xlarge"] = runs
        print(json.dumps(runs, indent=1), flush=True)
        if args.parent_lib:
            reg = {"cfg2_this_build": [], "cfg2_parent": []}
            for _ in range(3):
                reg["cfg2_this_build"].append(spawn(512, 8, 17, args.iters, args.warmup))
                reg["cfg2_parent"].append(spawn(512, 8, 17, args.iters, args.warmup, args.parent_lib))
            res["cfg2_regression"] = reg
            print(json.dumps(reg, indent=1), flush=True)
        else:
            res["cfg2_regression"] = "not measured (no --parent-lib)"
    res["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k in ("card", "card_after")}))


if __name__ == "__main__":
    main()
