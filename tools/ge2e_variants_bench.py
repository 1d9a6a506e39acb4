"""Cost of the GE2E loss variants: one spk_ge2e_loss_ex call (forward + backward) per mode at N = 64, 256 and 4096
speakers x 15 utterances x 256.

Each arm captures REPS calls in a CUDA graph, as `bench.py --workload ge2e` does, and the replay is timed with CUDA
events.  The four modes of one N are alternated in ROUNDS rounds in one process, so that clock drift spreads over all of
them; the best replay of each arm is reported.  The card's name and power limit are read in the same run and printed
with the numbers.
Usage: python tools/ge2e_variants_bench.py [--speakers 64,256,4096] [--rounds 5]
"""
import argparse
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from speaker_embedding_torch_b200 import _native as NV  # noqa: E402
from tools.input_grad_bench import card  # noqa: E402

UTTS, DIM, REPS = 15, 256, 20
MODES = {"softmax/inclusive": 0, "softmax/exclusive": NV.GE2E_EXCLUSIVE, "contrast/inclusive": NV.GE2E_CONTRAST,
         "contrast/exclusive": NV.GE2E_CONTRAST | NV.GE2E_EXCLUSIVE}


def graph_arm(emb, n, mode, stream):
    """A CUDA graph of REPS loss calls with gradients in `mode`, warmed up."""
    lib = NV.lib()
    wsb = lib.spk_ge2e_workspace_bytes_ex(n, UTTS, mode)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    scal = torch.zeros(3, dtype=torch.float32, device="cuda")
    d_emb = torch.empty_like(emb)
    wt, bs = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")

    def call():
        NV.check(lib.spk_ge2e_loss_ex(NV.ptr(emb), n, UTTS, DIM, mode, NV.ptr(wt), NV.ptr(bs),
                                      ctypes.c_void_p(scal.data_ptr()), NV.ptr(d_emb),
                                      ctypes.c_void_p(scal.data_ptr() + 4), ctypes.c_void_p(scal.data_ptr() + 8),
                                      NV.ptr(ws), wsb, NV.stream_ptr()), "spk_ge2e_loss_ex")
    with torch.cuda.stream(stream):
        for _ in range(3):
            call()
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for _ in range(REPS):
                call()
        graph.replay()
        stream.synchronize()
    return graph, (ws, scal, d_emb, wt, bs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--speakers", default="64,256,4096")
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("this benchmark needs a CUDA device")
    stream = torch.cuda.Stream()
    rows = {}
    for n in (int(s) for s in args.speakers.split(",")):
        gen = torch.Generator(device="cuda").manual_seed(n)
        emb = torch.nn.functional.normalize(torch.randn(n * UTTS, DIM, generator=gen, device="cuda"), dim=1)
        arms = {name: graph_arm(emb, n, mode, stream) for name, mode in MODES.items()}
        best = {name: None for name in MODES}
        with torch.cuda.stream(stream):              # the replay runs on the current stream: the events' stream
            for _ in range(args.rounds):
                for name, (graph, _) in arms.items():
                    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0.record(stream)
                    graph.replay()
                    t1.record(stream)
                    stream.synchronize()
                    us = t0.elapsed_time(t1) * 1e3 / REPS
                    best[name] = us if best[name] is None else min(best[name], us)
        rows[n] = {name: round(us, 2) for name, us in best.items()}
        del arms
    name, limit = card()
    print(json.dumps({"card": name, "power_limit": limit, "per_speaker": UTTS, "dim": DIM, "calls_per_graph": REPS,
                      "rounds": args.rounds, "us_per_call_fwd_bwd": rows}))


if __name__ == "__main__":
    main()
