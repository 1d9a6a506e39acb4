"""Backward cost of the input gradient at the benchmark batch (960 slices x 160 frames, eval mode, 3 layers).

  (a) frozen encoder, mel.requires_grad:        forward + input-only backward (no parameter gradient)
  (b) trainable encoder, mel without gradient:  forward + full backward (what a training step's encoder runs)
  (c) trainable encoder, mel.requires_grad:     forward + full backward + d_mel

Device events over ITERS iterations per arm after warm-up, the arms alternated in rounds so that clock drift
spreads over all three.  A separate pass with the library's profiler gives the split of (a)'s backward.
Usage: python tools/input_grad_bench.py [--iters 120] [--rounds 6]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from speaker_embedding_torch_b200 import GE2E, _native  # noqa: E402
from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=120, help="timed iterations per arm (>= 100)")
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--batch", type=int, default=960)
    ap.add_argument("--frames", type=int, default=160)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("input_grad_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = GE2E(default_hyper_parameters()).to(dev).eval()
    params = list(model.parameters())
    gen = torch.Generator(device=dev).manual_seed(1234)
    mel = bench.synth_mel(gen, args.batch, args.frames, dev)
    cot = torch.randn(args.batch, 256, device=dev, generator=gen)

    def step(arm):
        for p in params:
            p.requires_grad_(arm != "a")
            p.grad = None
        x = mel.detach().requires_grad_(arm != "b")
        model(x).backward(cot)

    for arm in "abc":
        for _ in range(5):
            step(arm)
    torch.cuda.synchronize()
    per_round = max(1, (args.iters + args.rounds - 1) // args.rounds)
    total = {arm: 0.0 for arm in "abc"}
    count = {arm: 0 for arm in "abc"}
    orders = ("abc", "cba", "bca", "acb", "cab", "bac")
    for r in range(args.rounds):
        for arm in orders[r % len(orders)]:
            step(arm)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per_round):
                step(arm)
            e1.record()
            torch.cuda.synchronize()
            total[arm] += e0.elapsed_time(e1)
            count[arm] += per_round
    ms = {arm: total[arm] / count[arm] for arm in "abc"}

    # profiler pass (separate: the events per launch slow the host)
    _native.prof_enable(True)
    prof = {}
    for arm in "abc":
        step(arm)
        torch.cuda.synchronize()
        _native.prof_report()
        for _ in range(10):
            step(arm)
        rep = _native.prof_report()
        bwd = {k: v["ms"] / 10 for k, v in rep.items()
               if "bwd" in k or "wgrad" in k or k in ("mel_grad_unpack", "attn_delta", "rows_add", "pe_alpha_grad")}
        prof[arm] = dict(backward_kernels_ms=sum(bwd.values()),
                         wgrad_ms=sum(v for k, v in bwd.items() if "wgrad" in k),
                         mel_dgrad_ms=rep.get("gemm.bwd.mel_dgrad", {}).get("ms", 0.0) / 10,
                         mel_grad_unpack_ms=rep.get("mel_grad_unpack", {}).get("ms", 0.0) / 10)
    _native.prof_enable(False)
    name, limit = card()
    print(json.dumps({"card": name, "power_limit": limit, "batch": args.batch, "frames": args.frames,
                      "iters_per_arm": count["a"], "ms_per_iter": ms, "profile": prof}))


if __name__ == "__main__":
    main()
