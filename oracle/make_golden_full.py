"""Generate tests/golden/train_full_case{0,1,2}.npz: the UNMODIFIED reference (fp64, eval mode) on the BASELINE batch.

TEST INFRASTRUCTURE.  Needs a checkout of the reference (SPK_REFERENCE), ~16 GB of RAM and a few minutes per case:

    SPK_REFERENCE=<reference checkout> python oracle/make_golden_full.py

Cases: 64 speakers x 15 utterances x T frames for T in {160, 140, 180} (BASELINE.json configs[1]; the benchmark draws
one T from [140, 180] per step).  Stored per case, one file each so that every file stays under 1 MB: loss, a third of
the 960 d-vectors (fp32; seeded rows, ``make_golden.sample_rows(960, 320)``, under ``case<i>_dvec_rows``), and for
every parameter the gradient norm plus a 4096-element fingerprint (seeded indices,
``make_golden.fingerprint_indices(numel, 4096)``) -- ~100 k sampled gradient elements per case, enough to estimate the
global relative L2 error to a few percent of itself.  Inputs and weights are regenerated from ``oracle/synth.py`` seeds
at test time.
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import synth  # noqa: E402
from oracle.make_golden import fingerprint_indices, load_reference, ref_model, sample_rows  # noqa: E402

FP_K = 4096
DVEC_ROWS = 320
CASES = [  # (state_seed, mel_seed, N, M, T)
    (61, 601, 64, 15, 160),
    (62, 602, 64, 15, 140),
    (63, 603, 64, 15, 180),
]


def main():
    GE2E, GE2E_Loss, hp = load_reference()
    torch.set_num_threads(os.cpu_count() or 1)
    for i, (ss, ms, N, M, T) in enumerate(CASES):
        out = {}
        t0 = time.time()
        state = synth.make_state(ss)
        mel = synth.make_mel(ms, N * M, T)
        m = ref_model(GE2E, hp, state, torch.float64)
        crit = GE2E_Loss().double()
        for p in m.parameters():
            p.requires_grad_(True)
        d = m(torch.as_tensor(mel).double())
        loss = crit(d, M)
        loss.backward()
        out["case%d_loss" % i] = loss.detach().numpy()
        rows = out["case%d_dvec_rows" % i] = sample_rows(N * M, DVEC_ROWS)
        out["case%d_dvec" % i] = d.detach().numpy()[rows].astype(np.float32)
        for name, p in m.named_parameters():
            g = p.grad.numpy().reshape(-1)
            out["case%d_gnorm_%s" % (i, name)] = np.array(np.linalg.norm(g))
            out["case%d_gsamp_%s" % (i, name)] = g[fingerprint_indices(g.size, FP_K)]
        out["case%d_dw" % i] = crit.weight.grad.numpy()
        out["case%d_meta" % i] = np.array([ss, ms, N, M, T], dtype=np.int64)
        out["fp_k"] = np.array(FP_K)
        path = os.path.join(ROOT, "tests", "golden", "train_full_case%d.npz" % i)
        np.savez_compressed(path, **out)
        print("case", i, (ss, ms, N, M, T), "loss", float(loss), "%.0f s" % (time.time() - t0), path,
              os.path.getsize(path), flush=True)
        del m, d, loss


if __name__ == "__main__":
    main()
