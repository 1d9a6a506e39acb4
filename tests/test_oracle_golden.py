"""Pin the CPU oracle (oracle/ge2e_oracle.py) against the reference's own outputs.

The fixtures under tests/golden/ were produced by oracle/make_golden.py, which runs the
unmodified reference modules (/root/reference/Modules.py, Radam.py, Noam_Scheduler.py).
"""
import os

import numpy as np
import torch

from oracle import ge2e_oracle as O
from oracle import synth
from oracle.make_golden import fingerprint_indices, sample_rows, stored_rows


def test_encoder_forward_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "encoder_forward.npz"))
    for i in range(int(g["num_cases"])):
        ss, ms, B, T, S = [int(v) for v in g["case%d_meta" % i]]
        state = synth.make_state(ss)
        mel = synth.make_mel(ms, B, T)
        d64 = O.encoder_forward(O.to_torch_state(state, torch.float64), torch.as_tensor(mel).double(), S).numpy()
        assert d64.shape == (B // S, 256)
        np.testing.assert_allclose(d64, g["case%d_f64" % i], rtol=0, atol=1e-12)
        d32 = O.encoder_forward(O.to_torch_state(state, torch.float32), torch.as_tensor(mel), S).numpy()
        # fp32 vs the reference's fp32 run: same math, different summation order
        np.testing.assert_allclose(d32, g["case%d_f32" % i], rtol=0, atol=5e-6)
        np.testing.assert_allclose(np.linalg.norm(d64, axis=1), 1.0, atol=1e-12)


def test_ge2e_loss_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "ge2e_loss.npz"))
    for i in range(int(g["num_cases"])):
        sd, N, M, un, w, b = g["case%d_meta" % i]
        N, M = int(N), int(M)
        E = synth.make_embeddings(int(sd), N, M, unit_norm=bool(un))
        rows = stored_rows(g, "case%d_rows" % i)
        # autograd through the restated loss
        e = torch.as_tensor(E).double().requires_grad_(True)
        wt = torch.tensor(float(w), dtype=torch.float64, requires_grad=True)
        bt = torch.tensor(float(b), dtype=torch.float64, requires_grad=True)
        loss = O.ge2e_loss(e, M, wt, bt)
        loss.backward()
        np.testing.assert_allclose(loss.item(), g["case%d_f64_loss" % i], rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(e.grad.numpy()[rows], g["case%d_f64_dE" % i], rtol=0, atol=1e-13)
        np.testing.assert_allclose(wt.grad.item(), g["case%d_f64_dw" % i], rtol=1e-10, atol=1e-14)
        # closed form (what the fused kernel implements)
        l2, dE, dw, db = O.ge2e_loss_and_grads_closed_form(E, M, float(w), float(b))
        np.testing.assert_allclose(l2, g["case%d_f64_loss" % i], rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(dE, e.grad.numpy(), rtol=0, atol=2e-13)
        np.testing.assert_allclose(dE[rows], g["case%d_f64_dE" % i], rtol=0, atol=1e-13)
        np.testing.assert_allclose(dw, g["case%d_f64_dw" % i], rtol=1e-10, atol=1e-14)
        assert abs(db) < 1e-12 and abs(float(g["case%d_f64_db" % i])) < 1e-12
        # the reference's own fp32 run agrees with fp64 to fp32 round-off
        np.testing.assert_allclose(g["case%d_f32_loss" % i], g["case%d_f64_loss" % i], rtol=2e-5, atol=1e-6)


def test_chunked_closed_form_equals_closed_form():
    E = synth.make_embeddings(77, 37, 5, unit_norm=False)
    a = O.ge2e_loss_and_grads_closed_form(E, 5, 7.0, -3.0)
    b = O.ge2e_closed_form_chunked(E, 5, 7.0, -3.0, rows_per_chunk=16)
    np.testing.assert_allclose(a[0], b[0], rtol=1e-13)
    np.testing.assert_allclose(a[1], b[1], rtol=0, atol=1e-15)
    np.testing.assert_allclose(a[2], b[2], rtol=1e-11, atol=1e-16)
    assert abs(b[3]) < 1e-12


def test_explicit_dropout_scales_reach_every_site():
    """The oracle's 13 dropout sites take explicit keep-scales (what the GPU mask test feeds it): all-ones scales
    reproduce eval mode, and zeroing any single site changes the output."""
    state = O.to_torch_state(synth.make_state(3), torch.float64)
    mel = torch.as_tensor(synth.make_mel(5, 4, 12)).double()
    B, T, D, F, H = 4, 12, 256, 1024, 4
    shapes = {0: (B, T, D)}
    for l in range(3):
        shapes.update({1 + 4 * l: (B, H, T, T), 2 + 4 * l: (B, T, D), 3 + 4 * l: (B, T, F), 4 + 4 * l: (B, T, D)})
    ones = {k: torch.ones(v, dtype=torch.float64) for k, v in shapes.items()}
    base = O.encoder_forward(state, mel, 1)
    np.testing.assert_allclose(O.encoder_forward(state, mel, 1, drop_scales=ones).numpy(), base.numpy(), atol=1e-14)
    assert len(shapes) == 13
    for site in shapes:
        ds = dict(ones)
        ds[site] = torch.zeros(shapes[site], dtype=torch.float64)
        out = O.encoder_forward(state, mel, 1, drop_scales=ds)
        assert (out - base).abs().max() > 1e-6, site


def test_full_batch_golden_is_complete(golden_dir):
    for i in range(3):
        g = np.load(os.path.join(golden_dir, "train_full_case%d.npz" % i))
        assert int(g["fp_k"]) == 4096
        ss, ms, N, M, T = [int(v) for v in g["case%d_meta" % i]]
        assert (N, M) == (64, 15) and T in (140, 160, 180)
        rows = g["case%d_dvec_rows" % i]
        np.testing.assert_array_equal(rows, sample_rows(N * M, 320))
        assert g["case%d_dvec" % i].shape == (320, 256)
        np.testing.assert_allclose(np.linalg.norm(g["case%d_dvec" % i].astype(np.float64), axis=1), 1.0, atol=1e-6)
        names = [n for n, _ in synth.state_shapes() if not n.endswith(".pe")]
        assert all("case%d_gsamp_%s" % (i, n) in g for n in names)


def test_train_step_grads_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "train_grads.npz"))
    for i in range(int(g["num_cases"])):
        ss, ms, N, M, T = [int(v) for v in g["case%d_meta" % i]]
        loss, d, grads = O.train_step_grads(synth.make_state(ss), synth.make_mel(ms, N * M, T), M)
        np.testing.assert_allclose(loss, g["case%d_loss" % i], rtol=1e-11)
        np.testing.assert_allclose(d, g["case%d_dvec" % i], atol=1e-12)
        np.testing.assert_allclose(grads["loss.weight"], g["case%d_dw" % i], rtol=1e-9, atol=1e-14)
        n = 0
        for name, _ in synth.state_shapes():
            if name.endswith(".pe"):
                continue
            gr = grads[name].reshape(-1)
            ref_norm = float(g["case%d_gnorm_%s" % (i, name)])
            np.testing.assert_allclose(np.linalg.norm(gr), ref_norm, rtol=1e-9, atol=1e-14)
            np.testing.assert_allclose(gr[fingerprint_indices(gr.size)], g["case%d_gsamp_%s" % (i, name)],
                                       rtol=0, atol=1e-11 * max(1.0, ref_norm))
            n += 1
        assert n == 43


def test_radam_noam_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "radam.npz"))
    p = g["p0"].copy()
    m = np.zeros_like(p)
    v = np.zeros_like(p)
    for t, grad in enumerate(g["grads"]):
        lr = O.modified_noam_lr(2e-3, t, 4000)
        np.testing.assert_allclose(lr, g["lrs"][t], rtol=1e-12)
        O.radam_step(p, grad, m, v, t + 1, lr, eps=1e-6)
        # the reference steps in fp32 (Radam.py:36,41: grad.float(), p.data.float())
        np.testing.assert_allclose(p, g["traj"][t], rtol=0, atol=2e-6)


def test_state_layout_is_the_reference_layout():
    shapes = synth.state_shapes()
    assert len(shapes) == 44
    assert sum(int(np.prod(s)) for n, s in shapes if not n.endswith(".pe")) == 2456321
