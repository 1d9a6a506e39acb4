"""Variable-length utterances on one GPU: GE2E.embed_utterances against the length-bucket workaround, a frozen critic's
forward + backward against a per-utterance loop, and the kernel times of the segmented head and the ragged fold.

    python tools/utterance_bench.py [--out DIR] [--utterances 4096] [--reps 5]

Prints the card's name and power limit (read in the same run), then one JSON line per measurement; the arms of (a)
and (b) alternate inside one process.  Kernel times come from a separate pass with the library's launch profiler.

The workaround arms do slightly less work than embed_utterances: they crop every utterance to the largest window on
the hop grid that fits (the tail frames are dropped), and the per-utterance loop of (b) back-propagates each
utterance's own critic loss instead of the batch mean (the same gradient up to the 1 / 64 factor).  Neither changes
what is timed: one encoder forward + backward per utterance against one for the whole batch.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # noqa: BLE001
        q = "unknown (%s)" % e
    return q


def timed(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--utterances", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("utterance_bench needs a CUDA device")
    from oracle import synth
    from speaker_embedding_torch_b200 import GE2E, _native as N
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices, utterance_slices

    info = {"card": card()}
    print(json.dumps(info))
    lines = [info]
    m = GE2E(default_hyper_parameters())
    m.load_state_dict({k: torch.as_tensor(v) for k, v in synth.make_state(1).items()}, strict=True)
    m = m.cuda().eval()
    T, O_ = 160, 80
    hop = T - O_
    rng = np.random.RandomState(0)

    # ---- (a) verification-sized set: embed_utterances against length buckets through embed_windows
    U = args.utterances
    lengths = rng.randint(50, 2001, size=U)
    data = torch.randn(80, int(lengths.sum()), device="cuda") - 4.0
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    mels = [data[:, s:s + L] for s, L in zip(starts.tolist(), lengths.tolist())]
    slices = int(utterance_slices(lengths, T, O_)[1][-1])
    # bucket workaround: crop every utterance to the largest hop-grid window that fits (short ones reflect-padded
    # to T), group by window length, one embed_windows call per bucket
    buckets = {}
    for i, L in enumerate(lengths.tolist()):
        S = max(1, (L - O_) // hop) if L >= T else 1
        buckets.setdefault(S, []).append(i)
    pads = {}
    for S, idx in buckets.items():
        W = S * hop + O_
        ws = []
        for i in idx:
            x = mels[i]
            if x.size(1) < W:
                left = (W - x.size(1)) // 2
                x = torch.nn.functional.pad(x[None], (left, W - x.size(1) - left), mode="reflect")[0] \
                    if x.size(1) > (W - x.size(1)) // 2 + 1 else x.repeat(1, W // x.size(1) + 1)[:, :W]
            ws.append(x[:, :W])
        pads[S] = torch.stack(ws)
    bucket_slices = sum(S * len(idx) for S, idx in buckets.items())

    def run_utt():
        with torch.no_grad():
            m.embed_utterances(mels, T, O_)

    def run_buckets():
        with torch.no_grad():
            for S, w in pads.items():
                m.embed_windows(w, T, O_)

    run_utt(); run_buckets()
    ta, tb = [], []
    for _ in range(args.reps):
        ta += timed(run_utt, 1)
        tb += timed(run_buckets, 1)
    for name, t, sl in (("embed_utterances", ta, slices), ("buckets_embed_windows", tb, bucket_slices)):
        rec = dict(arm=name, utterances=U, slices=sl, T=T, O=O_, buckets=len(buckets) if "bucket" in name else 1,
                   median_s=float(np.median(t)), min_s=float(np.min(t)),
                   utt_per_s=U / float(np.median(t)), slices_per_s=sl / float(np.median(t)))
        print(json.dumps(rec)); lines.append(rec)

    # ---- (b) frozen critic, forward + backward, 64 generated mels of 200-1500 frames
    for p in m.parameters():
        p.requires_grad_(False)
    lens_b = rng.randint(200, 1501, size=64)
    gen = [torch.randn(80, int(L), device="cuda") - 4.0 for L in lens_b]
    target = torch.nn.functional.normalize(torch.randn(64, 256, device="cuda"), dim=1)

    def crit(d, t):
        return (1.0 - torch.nn.functional.cosine_similarity(d, t, dim=1)).mean()

    def run_seg():
        xs = [g.clone().requires_grad_(True) for g in gen]
        crit(m.embed_utterances(xs, T, O_), target).backward()

    def run_loop():
        # per utterance: the hop-grid window that fits, Overlapped_Slices, forward (short ones reflect-padded)
        loss = 0.0
        for u, g in enumerate(gen):
            x = g.clone().requires_grad_(True)
            S = max(1, (x.size(1) - O_) // hop)
            W = S * hop + O_
            sl = Overlapped_Slices(x[None, :, :W], T, O_)
            loss = crit(m(sl, S), target[u:u + 1])
            loss.backward()

    run_seg(); run_loop()
    sa, sb = [], []
    for _ in range(args.reps):
        sa += timed(run_seg, 1)
        sb += timed(run_loop, 1)
    for name, t in (("critic_embed_utterances", sa), ("critic_per_utterance_loop", sb)):
        rec = dict(arm=name, mels=64, frames=int(lens_b.sum()), median_s=float(np.median(t)), min_s=float(np.min(t)))
        print(json.dumps(rec)); lines.append(rec)

    # ---- (c) kernel times of the new kernels (separate profiler pass)
    torch.cuda.synchronize()
    N.prof_enable(True)
    N.prof_report()
    with torch.no_grad():
        m.embed_utterances(mels, T, O_)
    run_seg()
    rep = N.prof_report()
    N.prof_enable(False)
    for tag in ("head_fwd_seg", "head_bwd_seg", "mel_grad_fold", "head_fwd", "mel_pack_ragged"):
        if tag in rep:
            rec = dict(kernel=tag, launches=rep[tag]["launches"], ms=rep[tag]["ms"],
                       us_per_launch=1e3 * rep[tag]["ms"] / max(rep[tag]["launches"], 1))
            print(json.dumps(rec)); lines.append(rec)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "utterance_bench.jsonl"), "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
