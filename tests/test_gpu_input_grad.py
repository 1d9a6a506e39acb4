"""Input gradients of the encoder: dL/d(mel) from spk_encoder_backward_input, and the backward of a frozen encoder that
computes no parameter gradient.

* The input gradient is compared with the fp64 oracle forced onto the library's own ReLU gates and dropout masks
  (test_gpu_stage_parity.py, B2), at the same GRAD_REL bound as the parameter gradients.
* A frozen encoder (every parameter ``requires_grad=False``) gives the same ``mel.grad`` bit for bit as a trainable
  one: the data path has no atomics, and skipping the parameter-gradient work changes nothing on it.
* Asking for ``mel.grad`` changes neither the d-vectors nor the parameter gradients, and spk_encoder_backward itself
  matches a fingerprint recorded with the library before spk_encoder_backward_input existed.

Bounds follow test_gpu_stage_parity.py: about 5x the worst value measured on a B200 (1000 W power limit), written
beside each bound.  Each test prints its figures as one JSON line.
"""
import ctypes
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth

D, F, H = 256, 1024, 4
DEV = "cuda"
GOLDEN_BWD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "encoder_backward_fingerprint.npz")

GRAD_REL = 1e-4           # 1.1e-5   mel.grad, relative L2 against the gate-forced fp64 oracle (fp16 features, against
                          #          the fp64 gradient rounded to fp16: 6.7e-5)
PARAM_REORDER = 2.5e-6    # 4.4e-7   parameter gradients with / without mel.requires_grad: fp32 atomics reordered
                          #          (the same call twice: 4.1e-7); fingerprint of spk_encoder_backward: 3.1e-7
E2E_REL = 1e-3            # 2.4e-4   the project's relative gradient tolerance against fp64 without gate forcing


def _record(kind, **kw):
    print("input grad:", json.dumps(dict(kind=kind, **kw)))


# ---- host: argument errors come back before any CUDA call
def test_backward_input_rejects_missing_outputs_without_a_device():
    from speaker_embedding_torch_b200 import _native as N
    if not os.path.exists(N.LIB_PATH):
        N.build()
    L = N.lib()
    cfg = N.EncoderConfig(80, 256, 4, 1024, 3, 1024, 0.1, 0.1)
    w, g = N.EncoderParams(), N.EncoderParams()
    fake = ctypes.c_void_p(4096)          # never dereferenced: the checks come first
    args = (12, 44, 1, 2, 0, ctypes.c_uint64(0))
    rc = L.spk_encoder_backward_input(ctypes.byref(cfg), ctypes.byref(w), None, None, fake, *args, fake, 1 << 20, None)
    assert rc == -22
    assert b"both NULL" in L.spk_last_error()
    rc = L.spk_encoder_backward_input(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(g), fake, fake, *args, None,
                                      1 << 20, None)
    assert rc == -22
    assert b"null argument" in L.spk_last_error()


# ---- GEMM shape of the input dgrad: N = 80 (a tail on a 64- or 128-wide tile), B MN-major, fp32 out
@pytest.mark.gpu
@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("m", [1000, 7680])
@pytest.mark.parametrize("block_n", [0, 64])
def test_mel_dgrad_gemm_shape_matches_fp64(planes, m, block_n):
    from speaker_embedding_torch_b200 import _native as N
    n, k = 80, 256
    torch.manual_seed(m + planes)
    A = torch.randn(m, k, device=DEV)
    Bt = torch.randn(k, n, device=DEV)          # the packed prenet weight [256, 80], read MN-major
    a_s, b_s = N.split_pack(A, planes), N.split_pack(Bt, planes)
    ref = N.split_unpack(a_s).double() @ N.split_unpack(b_s).double()
    out = N.gemm(a_s, b_s, planes, m, n, k, b_mn=True, out_f32=True, block_n=block_n)
    torch.cuda.synchronize()
    err = float((out.double() - ref).abs().max() / ref.abs().max())
    _record("gemm", planes=planes, m=m, block_n=block_n, err=err)
    assert err <= (2e-6 if planes == 1 else 2e-5), err     # the bound of test_gpu_gemm.py at K = 256 (7e-7 / 1.3e-6)


# ---- helpers
def _oracle_with_mel(state, mel, utt, samples=1, drop_scales=None, relu_masks=None, cotangent=None):
    """fp64 oracle: (d-vectors, dL/d(mel), {param: grad}) under the GE2E loss (utt) or a cotangent."""
    from test_gpu_stage_parity import _dstate
    st = {k: v.clone().requires_grad_(not k.endswith(".pe")) for k, v in _dstate(state).items()}
    x = mel.detach().double().clone().requires_grad_(True)
    layers = sum(1 for k in st if k.endswith("norm1.weight"))
    d = O.encoder_forward(st, x, samples=samples, layers=layers, drop_scales=drop_scales, relu_masks=relu_masks)
    if cotangent is None:
        O.ge2e_loss(d, utt, torch.tensor(10.0, dtype=torch.float64, device=DEV),
                    torch.tensor(-5.0, dtype=torch.float64, device=DEV)).backward()
    else:
        d.backward(cotangent.double())
    return d.detach(), x.grad, {k: v.grad for k, v in st.items() if v.requires_grad}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _step_with_mel(m, mel, utt, training, samples=1, cotangent=None):
    """_train_step of the stage-parity tests with mel.requires_grad: -> (seed, d, mel.grad)."""
    from test_gpu_stage_parity import _train_step
    x = mel.clone().requires_grad_(True)
    seed, d, _, _ = _train_step(m, x, utt, training, samples=samples, cotangent=cotangent)
    return seed, d, x.grad


def _gate_forced(m, state, mel, utt, training, prune, samples=1, cotangent=None):
    from test_gpu_parity_full import _site_scales
    from test_gpu_stage_parity import _relu_masks
    B, T = mel.shape[0], mel.shape[2]
    seed, d, g = _step_with_mel(m, mel, utt, training, samples, cotangent)
    masks = _relu_masks(m, B, T, prune)
    ds = None
    if training:
        ds, _ = _site_scales(seed, m._cfg.pe_dropout, m._cfg.dropout, B, T, H, 3, bool(prune), DEV)
        ds = {k: v.to(DEV) for k, v in ds.items()}
    d_ref, g_ref, _ = _oracle_with_mel(state, mel, utt, samples, ds, masks, cotangent)
    return d, g, d_ref, g_ref


MEL_CASES = [
    # (speakers, utterances, frames, training, prune)
    (4, 3, 24, False, 1),
    (3, 2, 177, False, 1),
    (2, 2, 300, False, 1),       # materialised attention (T > 192)
    (4, 3, 44, True, 1),
    (4, 3, 44, True, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("nspk,utt,T,training,prune", MEL_CASES)
def test_mel_grad_matches_gate_forced_fp64(nspk, utt, T, training, prune):
    from test_gpu_stage_parity import _Options, _model
    B = nspk * utt
    with _Options(prune_last_layer=prune):
        m, state = _model(71)
        mel = torch.as_tensor(synth.make_mel(2300 + T, B, T)).to(DEV)
        d, g, d_ref, g_ref = _gate_forced(m, state, mel, utt, training, prune)
    err = _rel(g, g_ref)
    _record("mel_grad", case=[nspk, utt, T, training, prune], err=err)
    assert g.dtype == torch.float32 and g.shape == mel.shape
    assert err <= GRAD_REL, err


@pytest.mark.gpu
def test_mel_grad_with_samples_and_a_random_cotangent():
    B, T, S = 20, 48, 5
    from test_gpu_stage_parity import _model
    m, state = _model(72)
    mel = torch.as_tensor(synth.make_mel(2400, B, T)).to(DEV)
    cot = torch.randn(B // S, D, generator=torch.Generator().manual_seed(5), dtype=torch.float64).float().to(DEV)
    _, g, _, g_ref = _gate_forced(m, state, mel, None, True, 1, samples=S, cotangent=cot)
    err = _rel(g, g_ref)
    _record("mel_grad_samples5", err=err)
    assert err <= GRAD_REL, err


@pytest.mark.gpu
def test_fp16_features_get_an_fp16_gradient():
    from test_gpu_stage_parity import _model
    B, T, utt = 12, 64, 3
    m, state = _model(73)
    mel = torch.as_tensor(synth.make_mel(2500, B, T)).to(DEV).half()
    d, g, d_ref, g_ref = _gate_forced(m, state, mel, utt, False, 1)
    assert g.dtype == torch.float16
    err = _rel(g, g_ref.half())        # against the fp64 gradient rounded to fp16
    _record("mel_grad_fp16", err=err)
    assert err <= GRAD_REL, err


@pytest.mark.gpu
def test_benchmark_size_mel_grad_matches_gate_forced_fp64():
    from test_gpu_stage_parity import _model
    B, T, utt = 960, 160, 15
    m, state = _model(74)
    mel = torch.as_tensor(synth.make_mel(2600, B, T)).to(DEV)
    _, g, _, g_ref = _gate_forced(m, state, mel, utt, False, 1)
    err = _rel(g, g_ref)
    _record("mel_grad_960x160", err=err)
    assert err <= GRAD_REL, err


# ---- frozen critic
def _critic_loss(d, target):
    return (1.0 - torch.nn.functional.cosine_similarity(d, target, dim=1)).mean()


def _critic_run(m, mel, target, trainable, training, profile=False):
    from speaker_embedding_torch_b200 import _native as N
    for p in m.parameters():
        p.requires_grad_(trainable)
        p.grad = None
    m.train(training)
    x = mel.clone().requires_grad_(True)
    torch.manual_seed(77)                  # the dropout seed GE2E.forward draws
    d = m(x)
    loss = _critic_loss(d, target)
    rep = None
    if profile:
        torch.cuda.synchronize()
        N.prof_enable(True)
        N.prof_report()
    loss.backward()
    torch.cuda.synchronize()
    if profile:
        rep = N.prof_report()
        N.prof_enable(False)
    return d.detach(), x.grad, rep


@pytest.mark.gpu
@pytest.mark.parametrize("T,training", [(44, False), (44, True), (300, False)])
def test_frozen_critic_input_grad_is_the_trainable_one(T, training):
    from test_gpu_stage_parity import _model
    B = 12
    m, _ = _model(75)
    mel = torch.as_tensor(synth.make_mel(2700 + T, B, T)).to(DEV)
    target = torch.randn(B, D, generator=torch.Generator().manual_seed(3)).to(DEV)
    d_t, g_t, rep_t = _critic_run(m, mel, target, True, training, profile=True)
    assert all(p.grad is not None for p in m.parameters())
    fresh, _ = _model(75)
    d_f, g_f, rep_f = _critic_run(fresh, mel, target, False, training, profile=True)
    _record("frozen_critic", T=T, training=training, max_abs=float((g_f - g_t).abs().max()),
            tags=sorted(rep_f))
    assert torch.equal(d_f, d_t)
    assert torch.equal(g_f, g_t)
    assert all(p.grad is None for p in fresh.parameters())
    assert fresh._arena is None                       # no gradient arena was allocated
    assert not [t for t in rep_f if "wgrad" in t], sorted(rep_f)
    assert "gemm.bwd.mel_dgrad" in rep_f and "mel_grad_unpack" in rep_f
    assert "gemm.bwd.qkv_wgrad" in rep_t or "gemm.last.bwd.kv_wgrad" in rep_t


# ---- nothing else moves
@pytest.mark.gpu
def test_mel_requires_grad_changes_neither_dvectors_nor_parameter_gradients():
    from test_gpu_stage_parity import _model, _rel_errors
    B, T, utt = 12, 44, 3
    m, _ = _model(76)
    m.eval()
    mel = torch.as_tensor(synth.make_mel(2800, B, T)).to(DEV)
    from speaker_embedding_torch_b200 import GE2E_Loss
    crit = GE2E_Loss().to(DEV)

    def run(want_mel):
        m.zero_grad(set_to_none=True)
        x = mel.clone().requires_grad_(want_mel)
        d = m(x)
        crit(d, utt).backward()
        torch.cuda.synchronize()
        return d.detach(), {n: p.grad.clone() for n, p in m.named_parameters()}

    d0, g0 = run(False)
    d1, g1 = run(True)
    d2, g2 = run(False)
    errs = _rel_errors(g1, g0)
    spread = _rel_errors(g2, g0)                      # the same call twice: the atomics' own reordering
    worst = max(errs.items(), key=lambda kv: kv[1])
    _record("param_grads_with_mel", worst=worst, spread=max(spread.values()))
    assert torch.equal(d0, d1) and torch.equal(d0, d2)
    assert worst[1] <= PARAM_REORDER, worst


def _fingerprint(m, seed=78):
    """Seeded trainable backward through spk_encoder_backward, reduced to a few thousand values: the d-vectors, and
    per parameter gradient its fp64 norm plus 256 elements at a fixed stride."""
    from speaker_embedding_torch_b200 import GE2E_Loss
    B, T, utt = 12, 44, 3
    mel = torch.as_tensor(synth.make_mel(seed, B, T)).to(DEV)
    crit = GE2E_Loss().to(DEV)
    m.eval()
    m.zero_grad(set_to_none=True)
    d = m(mel)
    crit(d, utt).backward()
    torch.cuda.synchronize()
    out = {"dvec": d.detach().cpu().numpy()}
    for n, p in m.named_parameters():
        g = p.grad.detach().reshape(-1)
        idx = torch.arange(0, g.numel(), max(1, g.numel() // 256), device=g.device)[:256]
        out["norm/" + n] = np.array([float(g.double().norm())])
        out["elem/" + n] = g[idx].cpu().numpy()
    return out


@pytest.mark.gpu
def test_encoder_backward_matches_the_recorded_fingerprint():
    """spk_encoder_backward (no input gradient) against values recorded with the library as it was before
    spk_encoder_backward_input was added: d-vectors bit for bit, gradients within fp32-atomic reordering."""
    from test_gpu_stage_parity import _model
    m, _ = _model(79)
    ref = np.load(GOLDEN_BWD)
    got = _fingerprint(m)
    assert np.array_equal(got["dvec"], ref["dvec"])
    worst = 0.0
    for k in ref.files:
        if k == "dvec":
            continue
        a, b = got[k].astype(np.float64), ref[k].astype(np.float64)
        scale = float(ref["norm/" + k.split("/", 1)[1]][0]) if k.startswith("elem/") else abs(b).max()
        worst = max(worst, float(np.abs(a - b).max() / max(scale, 1e-30)))
    _record("fingerprint", worst=worst)
    assert worst <= PARAM_REORDER, worst


# ---- gradient-scale contract for d_mel
@pytest.mark.gpu
def test_mel_grad_gradient_scale_contract():
    from test_gpu_stage_parity import _Options, _model, _relu_masks
    B, T = 12, 44
    m, state = _model(91)
    for p in m.parameters():
        p.requires_grad_(False)
    mel = torch.as_tensor(synth.make_mel(1600, B, T)).to(DEV)
    cot = torch.randn(B, D, generator=torch.Generator().manual_seed(9)).to(DEV)
    _, g1 = _step_with_mel(m, mel, None, False, cotangent=cot)[1:]
    masks = _relu_masks(m, B, T, 1)
    _, g_ref, _ = _oracle_with_mel(state, mel, None, relu_masks=masks, cotangent=cot)
    for c in (2.0 ** -20, 2.0 ** 16, 2.0 ** 24):      # the same planes at another scale: exact
        gc = _step_with_mel(m, mel, None, False, cotangent=cot * c)[2]
        assert torch.equal(gc, g1 * c), c
    errs = {}
    for k in (8, 12, 15):
        with _Options(grad_scale_log2=k):
            gk = _step_with_mel(m, mel, None, False, cotangent=cot)[2]
        errs[k] = _rel(gk, g_ref)
    _record("mel_grad_scale", errs=errs)
    for k, v in errs.items():
        assert v <= GRAD_REL, (k, v)
    bad = cot.clone()
    bad[3, 17] = float("nan")
    gn = _step_with_mel(m, mel, None, False, cotangent=bad)[2]
    assert not torch.isfinite(gn).all()


# ---- end to end: a generator trained through a frozen critic
@pytest.mark.gpu
def test_generator_gradient_through_a_frozen_critic_matches_fp64():
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices
    from test_gpu_stage_parity import _dstate, _model
    U, S, L, hop, zdim = 4, 5, 64, 32, 16
    W = S * hop + (L - hop)
    m, state = _model(80)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    torch.manual_seed(81)
    gen = torch.nn.Linear(zdim, 80 * W).to(DEV)
    with torch.no_grad():
        gen.weight.mul_(4.0)
        gen.bias.fill_(-5.0)                         # log-mel-like values
    z = torch.randn(U, zdim, device=DEV)
    target = torch.nn.functional.normalize(torch.randn(U, D, device=DEV), dim=1)

    def graph(g, encoder, zz, tt):
        mel = g(zz).view(U, 80, W)
        return _critic_loss(encoder(Overlapped_Slices(mel, L, L - hop)), tt)

    loss = graph(gen, lambda x: m(x, S), z, target)
    loss.backward()
    gen64 = torch.nn.Linear(zdim, 80 * W).to(DEV, torch.float64)
    with torch.no_grad():
        gen64.weight.copy_(gen.weight.double())
        gen64.bias.copy_(gen.bias.double())
    st = _dstate(state)
    loss64 = graph(gen64, lambda x: O.encoder_forward(st, x, samples=S, layers=3), z.double(), target.double())
    loss64.backward()
    err_w = _rel(gen.weight.grad, gen64.weight.grad)
    err_b = _rel(gen.bias.grad, gen64.bias.grad)
    _record("generator", loss=float(loss), loss64=float(loss64), err_w=err_w, err_b=err_b)
    assert err_w <= E2E_REL and err_b <= E2E_REL, (err_w, err_b)
    assert all(p.grad is None for p in m.parameters())


if __name__ == "__main__":
    # python tests/test_gpu_input_grad.py --write-fingerprint PATH: record _fingerprint with the library on sys.path
    if len(sys.argv) == 3 and sys.argv[1] == "--write-fingerprint":
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from test_gpu_stage_parity import _model
        np.savez_compressed(sys.argv[2], **_fingerprint(_model(79)[0]))
