"""Generate tests/golden/*.npz by running the UNMODIFIED reference modules on seeded inputs.

TEST INFRASTRUCTURE.  Run in the authoring container only (needs /root/reference):

    python oracle/make_golden.py

The fixtures hold only seeds/shapes and the reference's outputs (d-vectors, loss,
gradient fingerprints); inputs and weights are regenerated from ``oracle/synth.py``.
/root/reference is never read at test time.
"""
import os
import sys
import warnings

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = os.environ.get("SPK_REFERENCE", "/root/reference")

from oracle import synth  # noqa: E402

FP_IDX_SEED = 20240611


def fingerprint_indices(numel, k=64):
    rng = np.random.default_rng(FP_IDX_SEED + numel)
    return rng.integers(0, numel, size=min(k, numel))


def sample_rows(rows, k):
    """Sorted seeded sample of ``k`` distinct row indices out of ``rows``: the rows of an output too large to store
    whole (a golden file stays under 1 MB) that the file keeps, next to the values under ``<name>_rows``."""
    rng = np.random.default_rng(FP_IDX_SEED + rows)
    return np.sort(rng.choice(rows, size=min(k, rows), replace=False))


def stored_rows(golden, key):
    """Index of the rows a golden file holds of an output: ``golden[key]`` when it keeps a sample, else every row."""
    return golden[key] if key in golden.files else slice(None)


def load_reference():
    sys.path.insert(0, REF)
    warnings.filterwarnings("ignore")
    from Modules import GE2E, GE2E_Loss      # the reference's own modules
    from Arg_Parser import Recursive_Parse
    hp = Recursive_Parse(yaml.load(open(os.path.join(REF, "Hyper_Parameters.yaml")), Loader=yaml.Loader))
    return GE2E, GE2E_Loss, hp


def ref_model(GE2E, hp, state, dtype):
    m = GE2E(hp)
    sd = {k: torch.as_tensor(v) for k, v in state.items()}
    m.load_state_dict(sd, strict=True)
    return m.to(dtype).eval()


def main():
    GE2E, GE2E_Loss, hp = load_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.manual_seed(0)

    # ---- encoder forward cases ---------------------------------------------------------
    enc = {}
    cases = [  # (state_seed, mel_seed, B, T, samples)
        (11, 101, 6, 24, 1),
        (12, 102, 10, 64, 5),
        (13, 103, 4, 177, 1),
        (14, 104, 3, 1, 1),
        (15, 105, 2, 400, 1),
        (16, 106, 5, 160, 1),
    ]
    for i, (ss, ms, B, T, S) in enumerate(cases):
        state = synth.make_state(ss)
        mel = synth.make_mel(ms, B, T)
        for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
            m = ref_model(GE2E, hp, state, dt)
            with torch.no_grad():
                d = m(torch.as_tensor(mel).to(dt), S)
            enc["case%d_%s" % (i, tag)] = d.numpy()
        enc["case%d_meta" % i] = np.array([ss, ms, B, T, S], dtype=np.int64)
    enc["num_cases"] = np.array(len(cases))
    np.savez_compressed(os.path.join(out_dir, "encoder_forward.npz"), **enc)

    # ---- GE2E loss cases ---------------------------------------------------------------
    los = {}
    lcases = [  # (seed, N, M, unit_norm, w, b)
        (201, 2, 2, 1, 10.0, -5.0),
        (202, 7, 5, 1, 10.0, -5.0),
        (203, 9, 4, 0, 7.0, -3.0),
        (204, 64, 15, 1, 10.0, -5.0),
        (205, 33, 3, 0, 12.5, 1.5),
    ]
    for i, (sd, N, M, un, w, b) in enumerate(lcases):
        E = synth.make_embeddings(sd, N, M, unit_norm=bool(un))
        rows = slice(None)
        if N * M > 240:                       # the 960 x 256 dE of case 3 is kept as a quarter of its rows
            rows = los["case%d_rows" % i] = sample_rows(N * M, 240)
        for tag, dt in (("f32", torch.float32), ("f64", torch.float64)):
            crit = GE2E_Loss(init_weight=w, init_bias=b).to(dt)
            e = torch.as_tensor(E).to(dt).requires_grad_(True)
            loss = crit(e, M)
            loss.backward()
            los["case%d_%s_loss" % (i, tag)] = loss.detach().numpy()
            if tag == "f64":                  # the fp32 run is checked through its loss only
                los["case%d_%s_dE" % (i, tag)] = e.grad.numpy()[rows]
            los["case%d_%s_dw" % (i, tag)] = crit.weight.grad.numpy()
            los["case%d_%s_db" % (i, tag)] = (crit.bias.grad if crit.bias.grad is not None
                                               else torch.zeros(())).numpy()
        los["case%d_meta" % i] = np.array([sd, N, M, un, w, b], dtype=np.float64)
    los["num_cases"] = np.array(len(lcases))
    np.savez_compressed(os.path.join(out_dir, "ge2e_loss.npz"), **los)

    # ---- full training-step gradients (eval mode: dropout off, SURVEY.md D9) ------------
    trn = {}
    tcases = [  # (state_seed, mel_seed, N, M, T)
        (21, 301, 3, 2, 24),
        (22, 302, 4, 3, 50),
    ]
    for i, (ss, ms, N, M, T) in enumerate(tcases):
        state = synth.make_state(ss)
        mel = synth.make_mel(ms, N * M, T)
        m = ref_model(GE2E, hp, state, torch.float64)
        crit = GE2E_Loss().double()
        for p in m.parameters():
            p.requires_grad_(True)
        d = m(torch.as_tensor(mel).double())
        loss = crit(d, M)
        loss.backward()
        trn["case%d_loss" % i] = loss.detach().numpy()
        trn["case%d_dvec" % i] = d.detach().numpy()
        for name, p in m.named_parameters():
            g = p.grad.numpy().reshape(-1)
            trn["case%d_gnorm_%s" % (i, name)] = np.array(np.linalg.norm(g))
            trn["case%d_gsamp_%s" % (i, name)] = g[fingerprint_indices(g.size)]
        trn["case%d_dw" % i] = crit.weight.grad.numpy()
        trn["case%d_meta" % i] = np.array([ss, ms, N, M, T], dtype=np.int64)
    trn["num_cases"] = np.array(len(tcases))
    np.savez_compressed(os.path.join(out_dir, "train_grads.npz"), **trn)

    # ---- optimiser: reference RAdam + Modified_Noam_Scheduler trajectories ---------------
    from Radam import RAdam
    from Noam_Scheduler import Modified_Noam_Scheduler
    rng = np.random.default_rng(77)
    p0 = rng.standard_normal(257).astype(np.float64)
    grads = rng.standard_normal((12, 257)).astype(np.float64)
    p = torch.nn.Parameter(torch.as_tensor(p0.copy()))
    opt = RAdam([p], lr=2e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0)
    sch = Modified_Noam_Scheduler(opt, base=4000)
    traj, lrs = [], []
    for g in grads:
        p.grad = torch.as_tensor(g.copy())
        lrs.append(opt.param_groups[0]["lr"])
        opt.step()
        sch.step()
        traj.append(p.detach().numpy().copy())
    np.savez_compressed(os.path.join(out_dir, "radam.npz"), p0=p0, grads=grads,
                        traj=np.stack(traj), lrs=np.array(lrs))
    for f in sorted(os.listdir(out_dir)):
        print(f, os.path.getsize(os.path.join(out_dir, f)))


if __name__ == "__main__":
    main()
