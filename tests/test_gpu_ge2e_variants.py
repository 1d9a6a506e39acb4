"""The GE2E paper's loss variants (contrast loss, exclusive own-speaker centroids) on the GPU: small-N and tensor-core
paths against the fp64 closed form, which tests/test_ge2e_variant_oracle.py pins to a literal restatement of the paper's
equations; the tie rule, the refusals, and a training step through the encoder against autograd in fp64."""
import ctypes

import numpy as np
import pytest
import torch

from ge2e_variant_oracle import (MODES, ge2e_variant_closed_form_chunked, mode_bits, planted_embeddings,
                                 train_step_grads_variant)
from oracle import synth

pytestmark = pytest.mark.gpu

W, B = 5.0, 2.0            # logits w cos - b in the sigmoid's sensitive range, so the contrast gradients are not tiny
SMALL = [(3, 7), (5, 13), (64, 15), (65, 3), (100, 9), (128, 15), (129, 2), (192, 5), (255, 3)]
TENSOR_CORE = [(256, 3), (261, 5), (1024, 15), (4096, 15)]


def _fixture(n, m, method, seed):
    unit = n % 2 == 1
    if method == "contrast":           # a clear strongest impostor in every row (checked against the oracle below)
        return planted_embeddings(seed, n, m, unit_norm=unit)
    return synth.make_embeddings(seed, n, m, unit_norm=unit)


def _run(E, m, method, centroids, grad=True):
    from speaker_embedding_torch_b200 import GE2E_Loss
    crit = GE2E_Loss(init_weight=W, init_bias=B, loss_method=method, centroids=centroids).cuda()
    e = torch.as_tensor(E).cuda().requires_grad_(grad)
    if not grad:
        with torch.no_grad():
            return crit(e, m).item(), None, None, None
    loss = crit(e, m)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), e.grad.cpu().numpy().astype(np.float64), crit.weight.grad.item(), crit.bias.grad.item()


def _check(out, ref, method):
    loss, dE, dw, db = out
    l_ref, dE_ref, dw_ref, db_ref = ref[:4]
    assert abs(loss - l_ref) <= 2e-5 * max(1.0, abs(l_ref)), (loss, l_ref)
    assert np.linalg.norm(dE - dE_ref) / np.linalg.norm(dE_ref) <= 3e-4
    assert abs(dw - dw_ref) <= 2e-4 * abs(dw_ref) + 1e-6, (dw, dw_ref)
    if method == "contrast":
        assert abs(db - db_ref) <= 2e-4 * abs(db_ref) + 1e-6, (db, db_ref)
    else:
        assert abs(db) <= 1e-5


@pytest.mark.parametrize("method,centroids", MODES)
@pytest.mark.parametrize("n,m", SMALL + TENSOR_CORE)
def test_variants_match_the_closed_form(method, centroids, n, m):
    """Every tile shape of the small-N row stage with N, M >= 2, and the tensor-core path; the forward-only call gives
    the loss of the gradient call."""
    E = _fixture(n, m, method, 2100 + n)
    ref = ge2e_variant_closed_form_chunked(E, m, W, B, method, centroids)
    if method == "contrast":
        assert ref[4].min() > 1e-5, ref[4].min()      # k* cannot flip under fp32 rounding
    out = _run(E, m, method, centroids)
    _check(out, ref, method)
    l_ng = _run(E, m, method, centroids, grad=False)[0]
    assert abs(l_ng - out[0]) <= 1e-6 * max(1.0, abs(out[0]))


@pytest.mark.parametrize("n", [4, 256])
@pytest.mark.parametrize("centroids", ["inclusive", "exclusive"])
def test_contrast_ties_go_to_the_lowest_speaker(n, centroids):
    """Speakers 1 and 2 have identical rows, so their centroids, and their logits in every other row, tie exactly;
    the strongest impostor is speaker 1, so its centroid gets the gradient and speaker 2's does not."""
    m = 3
    E = planted_embeddings(3100 + n, n, m)
    E[:m] = (E[:m] + 2.0 * E[m:2 * m]) / 3.0       # speaker 0 leans towards speaker 1 (and so to its twin)
    E[2 * m:3 * m] = E[m:2 * m]
    ref = ge2e_variant_closed_form_chunked(E, m, W, B, "contrast", centroids)
    dE_ref = ref[1]
    assert np.abs(dE_ref[m:2 * m] - dE_ref[2 * m:3 * m]).max() > 0.01 * np.abs(dE_ref).max()
    out = _run(E, m, "contrast", centroids)
    _check(out, ref, "contrast")
    dE = out[1]
    twin = np.linalg.norm(dE[m:2 * m] - dE_ref[m:2 * m]) + np.linalg.norm(dE[2 * m:3 * m] - dE_ref[2 * m:3 * m])
    assert twin <= 3e-4 * np.linalg.norm(dE_ref[m:3 * m])


def _abi_call(fn, E, n, m, mode, grad=True):
    from speaker_embedding_torch_b200 import _native as N
    L = N.lib()
    emb = torch.as_tensor(E).cuda()
    wt = torch.tensor(W, device="cuda")
    bt = torch.tensor(B, device="cuda")
    scal = torch.zeros(3, device="cuda")
    d_emb = torch.empty_like(emb) if grad else None
    wsb = L.spk_ge2e_workspace_bytes(n, m) if fn == "spk_ge2e_loss" else L.spk_ge2e_workspace_bytes_ex(n, m, mode)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    d_w = ctypes.c_void_p(scal.data_ptr() + 4) if grad else None
    d_b = ctypes.c_void_p(scal.data_ptr() + 8) if grad else None
    args = [N.ptr(emb), n, m, 256] + ([] if fn == "spk_ge2e_loss" else [mode])
    args += [N.ptr(wt), N.ptr(bt), ctypes.c_void_p(scal.data_ptr()), N.ptr(d_emb), d_w, d_b, N.ptr(ws), wsb,
             N.stream_ptr()]
    rc = getattr(L, fn)(*args)
    torch.cuda.synchronize()
    return rc, scal.cpu().numpy().astype(np.float64), None if d_emb is None else d_emb.cpu().numpy().astype(np.float64)


@pytest.mark.parametrize("n,m", [(3, 7), (64, 15), (255, 3), (261, 5), (1024, 15)])
def test_mode_zero_of_the_variant_entry_point_is_the_reference_loss(n, m):
    """Mode 0 runs the kernels of spk_ge2e_loss (not bit-exact: fp32 atomics)."""
    E = synth.make_embeddings(4100 + n, n, m, unit_norm=False)
    rc0, s0, d0 = _abi_call("spk_ge2e_loss", E, n, m, 0)
    rc1, s1, d1 = _abi_call("spk_ge2e_loss_ex", E, n, m, 0)
    assert rc0 == 0 and rc1 == 0
    assert abs(s1[0] - s0[0]) <= 2e-6 * max(1.0, abs(s0[0]))
    assert abs(s1[1] - s0[1]) <= 2e-6 * max(1e-3, abs(s0[1]))
    assert np.linalg.norm(d1 - d0) / np.linalg.norm(d0) <= 2e-6


def test_refusals():
    from speaker_embedding_torch_b200 import GE2E_Loss
    E = synth.make_embeddings(7, 4, 3)
    e = torch.as_tensor(E).cuda().requires_grad_(True)
    with pytest.raises(RuntimeError, match="at least 2 utterances"):
        GE2E_Loss(centroids="exclusive").cuda()(e, 1)
    with pytest.raises(RuntimeError, match="at least 2 speakers"):
        GE2E_Loss(loss_method="contrast").cuda()(e, 12)
    with pytest.raises(RuntimeError, match="at least 2 speakers"):
        with torch.no_grad():
            GE2E_Loss(loss_method="contrast", centroids="exclusive").cuda()(e, 12)
    for mode in (2, 1 << 9, 0x101 | 0x10000):
        rc, _, _ = _abi_call("spk_ge2e_loss_ex", E, 4, 3, mode)
        assert rc == -22
    with pytest.raises(ValueError):
        GE2E_Loss(loss_method="triplet")
    with pytest.raises(ValueError):
        GE2E_Loss(centroids="Exclusive")
    # a refused call leaves the scalars alone: nothing ran
    rc, s, _ = _abi_call("spk_ge2e_loss_ex", E, 4, 1, mode_bits("softmax", "exclusive"))
    assert rc == -22 and not s.any()


def test_training_step_through_the_encoder():
    """8 speakers x 5 utterances x 160 frames, eval mode, contrast loss with exclusive centroids: every parameter
    gradient against autograd through the fp64 encoder restatement and the literal variant loss."""
    from speaker_embedding_torch_b200 import GE2E, GE2E_Loss
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    spk, utt, frames, seed = 8, 5, 160, 43
    state = synth.make_state(seed)
    mel = synth.make_mel(700 + seed, spk * utt, frames)
    model = GE2E(default_hyper_parameters())
    model.load_state_dict({k: torch.as_tensor(v) for k, v in state.items()}, strict=True)
    model = model.cuda().eval()
    crit = GE2E_Loss(init_weight=W, init_bias=B, loss_method="contrast", centroids="exclusive").cuda()
    d = model(torch.as_tensor(mel).cuda())
    loss = crit(d, utt)
    loss.backward()
    torch.cuda.synchronize()
    loss_ref, d_ref, g_ref = train_step_grads_variant(state, mel, utt, "contrast", "exclusive", W, B)
    # the untrained encoder's d-vectors are close together; this seed keeps every row's strongest impostor 1.5e-4
    # (in cosine) ahead of the next one, far outside the two-plane encoder's error
    assert ge2e_variant_closed_form_chunked(d_ref, utt, W, B, "contrast", "exclusive")[4].min() > 1e-4
    assert abs(loss.item() - loss_ref) <= 1e-3 * abs(loss_ref)
    num = den = 0.0
    for name, p in model.named_parameters():
        r = g_ref[name]
        num += float(((p.grad.double().cpu().numpy() - r) ** 2).sum())
        den += float((r ** 2).sum())
    assert (num / den) ** 0.5 <= 1e-3, (num / den) ** 0.5
    for p, name in ((crit.weight, "loss.weight"), (crit.bias, "loss.bias")):
        r = float(g_ref[name])
        assert abs(p.grad.item() - r) <= 1e-3 * abs(r), (name, p.grad.item(), r)
