"""Cost of the mel front-end's backward, at a vocoder training batch and at a speaker-critic batch.

  (a) library forward:                  meldataset.mel_spectrogram, no gradient
  (b) library forward + backward:       y.requires_grad, mel.backward(g) -> spk_mel_spectrogram_backward
  (c) torch fp32 forward + backward:    the reference's ops (F.pad, torch.stft, sqrt, matmul, log-clamp) on the GPU

Sizes: 16 x 8192 samples (vocoder segments) and 64 x 44100 samples (2 s utterances at 22050 Hz), both at
1024 / 256 / 1024 with 80 mels.  Device events over ITERS iterations per arm after warm-up, the arms alternated in
rounds so that clock drift spreads over all three.  A separate pass with the library's profiler splits (b) into its
kernels.  The working sets (at most 45 MB of frame gradients) fit in the 126 MB L2; no cache flush between iterations.
Usage: python tools/mel_grad_bench.py [--iters 200] [--rounds 6]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from mel_grad_oracle import mel_spectrogram_torch  # noqa: E402
from speaker_embedding_torch_b200 import _native  # noqa: E402
from speaker_embedding_torch_b200.meldataset import mel_spectrogram  # noqa: E402

SOUND = (1024, 80, 22050, 256, 1024, 0.0, None)     # n_fft, mels, rate, hop, win, fmin, fmax
SIZES = ((16, 8192), (64, 44100))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def measure(batch, samples, iters, rounds, dev):
    gen = torch.Generator(device=dev).manual_seed(batch * samples)
    audio = (0.3 * torch.randn(batch, samples, device=dev, generator=gen)).clamp(-1, 1)
    with torch.no_grad():
        g = torch.randn(mel_spectrogram(audio, *SOUND).shape, device=dev, generator=gen)

    def step(arm):
        if arm == "a":
            with torch.no_grad():
                mel_spectrogram(audio, *SOUND)
            return
        y = audio.detach().requires_grad_(True)
        mel = mel_spectrogram(y, *SOUND) if arm == "b" else mel_spectrogram_torch(y, *SOUND)
        mel.backward(g)

    for arm in "abc":
        for _ in range(10):
            step(arm)
    torch.cuda.synchronize()
    per_round = max(1, (iters + rounds - 1) // rounds)
    total = {arm: 0.0 for arm in "abc"}
    count = {arm: 0 for arm in "abc"}
    orders = ("abc", "cba", "bca", "acb", "cab", "bac")
    for r in range(rounds):
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
    step("b")
    torch.cuda.synchronize()
    _native.prof_report()
    for _ in range(20):
        step("b")
    rep = _native.prof_report()
    _native.prof_enable(False)
    kernels = {k: dict(ms=v["ms"] / v["launches"], gflops=v["flops"] / v["launches"] / 1e9,
                       mbytes=v["bytes"] / v["launches"] / 1e6) for k, v in rep.items()}
    return dict(batch=batch, samples=samples, iters_per_arm=count["a"], ms_per_iter=ms, kernels=kernels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200, help="timed iterations per arm (>= 100)")
    ap.add_argument("--rounds", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("mel_grad_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    results = [measure(b, s, args.iters, args.rounds, dev) for b, s in SIZES]
    name, limit = card()
    print(json.dumps({"card": name, "power_limit": limit, "results": results}))


if __name__ == "__main__":
    main()
