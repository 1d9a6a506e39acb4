"""Encoder cost against Mel_Dim, one process, the Mel_Dim arms alternated in rounds so that clock drift spreads over all.

  infer   inference d-vectors per second, 960 slices x 160 frames, eval (one fp16 plane)
  train   the 64 x 15 x 160 training step: train() with dropout, GE2E loss, backward, clip 1.0 + fused RAdam
  critic  a frozen encoder as critic: forward + backward of a cotangent into d_mel, 960 x 160, eval

Device events over ITERS iterations per arm and workload after warm-up.  The card's name and power limit are read in
the same run and printed with the numbers.
Usage: python tools/mel_dim_bench.py [--mel-dims 40,64,80,128] [--iters 60] [--rounds 4]
"""
import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from speaker_embedding_torch_b200 import GE2E, GE2E_Loss  # noqa: E402
from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters  # noqa: E402
from speaker_embedding_torch_b200.Radam import RAdam  # noqa: E402
from tools.input_grad_bench import card  # noqa: E402

SPEAKERS, UTTS, FRAMES, INFER_BATCH = 64, 15, 160, 960


def synth_mel(gen, batch, mel_dim, frames, device):
    x = torch.randn(batch, mel_dim, frames, generator=gen, device=device)
    return (-5.0 + 2.0 * x).clamp_(math.log(1e-5), 2.0)


def arm(mel_dim, device):
    hp = default_hyper_parameters()
    hp.Sound.Mel_Dim = mel_dim
    torch.manual_seed(0)
    model = GE2E(hp).to(device)
    critic = GE2E(hp).to(device).eval()
    critic.load_state_dict(model.state_dict())
    for p in critic.parameters():
        p.requires_grad_(False)
    crit = GE2E_Loss().to(device)
    opt = RAdam(model.parameters(), lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, max_grad_norm=1.0)
    gen = torch.Generator(device=device).manual_seed(1234 + mel_dim)
    train_mel = synth_mel(gen, SPEAKERS * UTTS, mel_dim, FRAMES, device)
    infer_mel = synth_mel(gen, INFER_BATCH, mel_dim, FRAMES, device)
    cot = torch.randn(INFER_BATCH, 256, generator=gen, device=device)

    def train():
        model.train()
        opt.zero_grad(set_to_none=True)
        crit(model(train_mel), UTTS).backward()
        opt.step()

    def infer():
        model.eval()
        with torch.no_grad():
            model(infer_mel)

    def frozen_critic():
        x = infer_mel.detach().requires_grad_(True)
        critic(x).backward(cot)

    return {"train": train, "infer": infer, "critic": frozen_critic}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mel-dims", default="40,64,80,128")
    ap.add_argument("--iters", type=int, default=60, help="timed iterations per arm and workload")
    ap.add_argument("--rounds", type=int, default=4)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("mel_dim_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    dims = [int(v) for v in args.mel_dims.split(",")]
    arms = {c: arm(c, dev) for c in dims}
    for c in dims:
        for fn in arms[c].values():
            for _ in range(3):
                fn()
    torch.cuda.synchronize()
    per_round = max(1, (args.iters + args.rounds - 1) // args.rounds)
    total = {(c, w): 0.0 for c in dims for w in ("train", "infer", "critic")}
    count = dict.fromkeys(total, 0)
    for r in range(args.rounds):
        order = dims if r % 2 == 0 else dims[::-1]
        for w in ("train", "infer", "critic"):
            for c in order:
                fn = arms[c][w]
                fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(per_round):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                total[(c, w)] += e0.elapsed_time(e1)
                count[(c, w)] += per_round
    name, limit = card()
    rows = {}
    for c in dims:
        ms = {w: total[(c, w)] / count[(c, w)] for w in ("train", "infer", "critic")}
        rows[c] = {"train_step_ms": ms["train"], "infer_dvectors_per_s": INFER_BATCH / ms["infer"] * 1e3,
                   "infer_ms": ms["infer"], "critic_fwd_bwd_ms": ms["critic"]}
    print(json.dumps({"card": name, "power_limit": limit, "iters_per_arm": count[(dims[0], "train")],
                      "train": "%d x %d x %d" % (SPEAKERS, UTTS, FRAMES), "infer": "%d x %d" % (INFER_BATCH, FRAMES),
                      "mel_dim": rows}))


if __name__ == "__main__":
    main()
