"""Parity where the benchmark runs (BASELINE.json configs[1]: 64 speakers x 15 utterances x 140..180 frames) and in
the regimes the small-batch tests do not reach: very short and very long slices, train-mode dropout masks.

Reference values: tests/golden/train_full_case*.npz = the UNMODIFIED reference in fp64 on the full batch
(oracle/make_golden_full.py; a seeded third of the d-vectors is stored); the fp64 oracle elsewhere.  Tolerances are
BASELINE.json's: cosine >= 0.9999 per d-vector, relative loss / gradient error <= 1e-3.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth
from oracle.make_golden import fingerprint_indices

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _model(seed):
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    state = synth.make_state(seed)
    m = GE2E(default_hyper_parameters())
    m.load_state_dict({k: torch.as_tensor(v) for k, v in state.items()}, strict=True)
    return m.cuda(), state


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


def _full_case(golden_dir, i, precision):
    from speaker_embedding_torch_b200 import GE2E_Loss
    g = np.load(os.path.join(golden_dir, "train_full_case%d.npz" % i))
    ss, ms, N, M, T = [int(v) for v in g["case%d_meta" % i]]
    k = int(g["fp_k"])
    m, _ = _model(ss)
    m.eval()                                            # parity is defined with dropout off (SURVEY.md D9)
    m.train_precision = precision
    crit = GE2E_Loss().cuda()
    d = m(torch.as_tensor(synth.make_mel(ms, N * M, T)).cuda())
    loss = crit(d, M)
    loss.backward()
    torch.cuda.synchronize()
    ref_loss = float(g["case%d_loss" % i])
    rows = g["case%d_dvec_rows" % i]
    cos = _cos(d.detach().cpu().numpy().astype(np.float64)[rows], g["case%d_dvec" % i].astype(np.float64))
    num = den = 0.0
    worst = ("", 0.0)
    norm_dev = 0.0
    for name, p in m.named_parameters():
        gr = p.grad.detach().cpu().numpy().astype(np.float64).reshape(-1)
        ref_norm = float(g["case%d_gnorm_%s" % (i, name)])
        norm_dev = max(norm_dev, abs(np.linalg.norm(gr) - ref_norm) / max(ref_norm, 1e-30))
        samp = g["case%d_gsamp_%s" % (i, name)]
        got = gr[fingerprint_indices(gr.size, k)]
        # weight every tensor's sample by numel / samples so the estimate is of the GLOBAL relative L2 error
        wgt = gr.size / float(len(samp))
        num += wgt * ((got - samp) ** 2).sum()
        den += wgt * (samp ** 2).sum()
        rel = np.linalg.norm(got - samp) / max(np.linalg.norm(samp), 1e-30)
        if rel > worst[1]:
            worst = (name, rel)
    dw_ref = float(g["case%d_dw" % i])
    return dict(frames=T, precision=precision, loss=loss.item(), ref_loss=ref_loss,
                loss_rel=abs(loss.item() - ref_loss) / abs(ref_loss), min_cos=float(cos.min()),
                grad_rel=float((num / den) ** 0.5), worst_tensor=worst[0], worst_rel=float(worst[1]),
                max_norm_dev=float(norm_dev), dw_rel=abs(crit.weight.grad.item() - dw_ref) / abs(dw_ref))


@pytest.mark.parametrize("case", [0, 1, 2])
def test_full_batch_train_step_matches_the_reference(golden_dir, case):
    """64 x 15 x {160, 140, 180}: loss, the stored d-vectors and the gradient of every parameter against the
    reference's own fp64 run, at the default training precision."""
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    default_precision = GE2E(default_hyper_parameters()).train_precision
    r = _full_case(golden_dir, case, default_precision)
    print("full-size parity:", json.dumps(r))
    assert r["loss_rel"] <= 1e-3, r
    assert r["min_cos"] >= 0.9999, r
    assert r["grad_rel"] <= 1e-3, r
    assert r["max_norm_dev"] <= 2e-3, r
    assert r["dw_rel"] <= 1e-3, r
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parity_full.jsonl"), "a") as f:
            f.write(json.dumps(r) + "\n")


def test_full_batch_other_precisions_are_recorded(golden_dir):
    """Two fp16 planes (the default: 22-bit mantissa, 3 MMAs per product) and three (6 MMAs) on the full batch: both
    inside the tolerance, recorded side by side (with bf16 planes, round 1, two planes were marginal: 8e-4)."""
    rows = [_full_case(golden_dir, 0, p) for p in (2, 3)]
    for r in rows:
        print("full-size parity:", json.dumps(r))
        assert r["loss_rel"] <= 1e-3 and r["min_cos"] >= 0.9999, r
        assert r["grad_rel"] <= 1e-3, r
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parity_full.jsonl"), "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


def _grad_rel(m, g_ref):
    num = den = 0.0
    worst = ("", 0.0)
    for name, p in m.named_parameters():
        gr = p.grad.detach().cpu().numpy().astype(np.float64)
        r = g_ref[name]
        num += ((gr - r) ** 2).sum()
        den += (r ** 2).sum()
        rel = np.linalg.norm(gr - r) / max(np.linalg.norm(r), 1e-30)
        if rel > worst[1]:
            worst = (name, rel)
    return (num / den) ** 0.5, worst


@pytest.mark.parametrize("nspk,utt,frames", [(4, 3, 1), (4, 3, 7), (3, 2, 8), (2, 2, 300), (2, 2, 1024)])
def test_gradients_at_the_ends_of_the_frame_range(nspk, utt, frames):
    """T < 8 (compact last-layer buffers smaller than a row), T > 256 (multi-chunk softmax, unfused attention) and the
    T = 1024 limit, forward and backward against the fp64 oracle."""
    from speaker_embedding_torch_b200 import GE2E_Loss
    m, state = _model(37)
    m.eval()
    crit = GE2E_Loss().cuda()
    mel = synth.make_mel(700 + frames, nspk * utt, frames)
    d = m(torch.as_tensor(mel).cuda())
    loss = crit(d, utt)
    loss.backward()
    torch.cuda.synchronize()
    loss_ref, d_ref, g_ref = O.train_step_grads(state, mel, utt)
    assert abs(loss.item() - loss_ref) <= 1e-3 * abs(loss_ref)
    assert _cos(d.detach().cpu().numpy().astype(np.float64), d_ref).min() >= 0.9999
    rel, worst = _grad_rel(m, g_ref)
    assert rel <= 1e-3, (rel, worst)
    # inference path (one plane) on the same input
    with torch.no_grad():
        d1 = m(torch.as_tensor(mel).cuda())
    assert _cos(d1.cpu().numpy().astype(np.float64), d_ref).min() >= 0.9999


def _site_scales(seed, p_pe, p, B, T, heads, layers, pruned, device):
    """Keep-scales of all 13 sites in the oracle's layouts, read back from the library (spk_dropout_keep)."""
    from speaker_embedding_torch_b200 import _native
    Tp = (T + 7) // 8 * 8
    D, F = 256, 1024
    ds, rates = {}, {}

    def keep(site, numel, prob):
        k = _native.dropout_keep(seed, prob, site, numel, device).double().cpu()
        rates[site] = (float((k > 0).double().mean()), numel, prob)
        nz = k[k > 0]
        q = round(prob * 65536) / 65536.0
        assert nz.numel() == 0 or torch.allclose(nz, torch.full_like(nz, 1.0 / (1.0 - q)), rtol=1e-6)
        return k

    ds[0] = keep(0, B * T * D, p_pe).view(B, T, D)
    for l in range(layers):
        last = pruned and l == layers - 1
        if not last:
            ds[1 + 4 * l] = keep(1 + 4 * l, B * heads * T * Tp, p).view(B, heads, T, Tp)[..., :T]
            ds[2 + 4 * l] = keep(2 + 4 * l, B * T * D, p).view(B, T, D)
            ds[3 + 4 * l] = keep(3 + 4 * l, B * T * F, p).view(B, T, F)
            ds[4 + 4 * l] = keep(4 + 4 * l, B * T * D, p).view(B, T, D)
        else:
            # the pruned last layer only evaluates the t = 0 query row of every slice: its masks are indexed on the
            # compact [B, .] buffers; rows t > 0 of that layer never reach the d-vector, any mask will do there
            a = torch.ones(B, heads, T, T, dtype=torch.float64)
            a[:, :, 0, :] = keep(1 + 4 * l, B * heads * Tp, p).view(B, heads, Tp)[..., :T]
            ds[1 + 4 * l] = a
            for site, width in ((2 + 4 * l, D), (3 + 4 * l, F), (4 + 4 * l, D)):
                t = torch.ones(B, T, width, dtype=torch.float64)
                t[:, 0, :] = keep(site, B * width, p).view(B, width)
                ds[site] = t
    return ds, rates


@pytest.mark.parametrize("prune", [1, 0])
def test_train_mode_masks_are_the_same_in_forward_and_backward(prune):
    """All 13 dropout sites (Modules.py:103 + 4 per encoder layer): the masks are a pure function of (seed, site,
    element); fed to the fp64 oracle they must reproduce the train-mode d-vectors (sites applied in the forward, with
    scale 1/(1-p)) AND the train-mode gradients (the backward regenerates the same masks).  Keep rates within 4 sigma
    of 1 - p per site."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    nspk, utt, T = 4, 3, 44
    B = nspk * utt
    try:
        _native.set_option("prune_last_layer", prune)
        m, state = _model(51)
        m.train()
        crit = GE2E_Loss().cuda()
        mel = synth.make_mel(801, B, T)
        torch.manual_seed(4242)
        seed = int(torch.empty((), dtype=torch.int64).random_().item())      # what GE2E.forward will draw
        torch.manual_seed(4242)
        d = m(torch.as_tensor(mel).cuda())
        loss = crit(d, utt)
        loss.backward()
        torch.cuda.synchronize()
    finally:
        _native.set_option("prune_last_layer", 1)
    ds, rates = _site_scales(seed, 0.1, 0.1, B, T, 4, 3, bool(prune), "cuda")
    assert len(ds) == 13
    for site, (rate, n, prob) in rates.items():
        sigma = (prob * (1 - prob) / n) ** 0.5
        assert abs(rate - (1 - prob)) <= 4 * sigma + 1e-4, (site, rate, n)
    loss_ref, d_ref, g_ref = O.train_step_grads(state, mel, utt, drop_scales=ds)
    assert _cos(d.detach().cpu().numpy().astype(np.float64), d_ref).min() >= 0.9999
    assert abs(loss.item() - loss_ref) <= 1e-3 * abs(loss_ref)
    rel, worst = _grad_rel(m, g_ref)
    assert rel <= 1e-3, (rel, worst)
    # and it is not the eval-mode answer
    _, d_eval, _ = O.train_step_grads(state, mel, utt)
    assert _cos(d.detach().cpu().numpy().astype(np.float64), d_eval).min() < 0.9999
