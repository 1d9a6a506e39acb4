"""Mel_Dim other than 80: every multiple of 8 in [16, 256], in the forward, the backward and both input gradients.

* Host: the workspace query accepts exactly that rule and names it when it refuses; GE2E builds the prenet from
  Sound.Mel_Dim.
* The GEMM shapes that only other mel counts reach (prenet K, input dgrad N, prenet wgrad N) against fp64 through
  spk_gemm.
* The encoder at C in {16, 40, 64, 128, 256} against the fp64 oracle (oracle.ge2e_oracle, which reads the prenet's
  shape): inference, training gradients, input gradients of the dense, ragged and one-plane paths, the collation paths,
  the mel front-end to d-vector chain and the formats.

The model is synth.make_state with the prenet replaced by a [256, C, 1] weight at the reference's init scale
(xavier-uniform, ReLU gain) plus a 0.1 relative perturbation (SURVEY.md D11).  Bounds are those of the 80-channel
tests they mirror (test_gpu_encoder.py, test_gpu_input_grad.py, test_gpu_utterances.py); each GPU test prints its
figures as one JSON line.
"""
import ctypes
import json
import math
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth

D, F, H = 256, 1024, 4
DEV = "cuda"
MEL_DIMS = [16, 40, 64, 128, 256]
COS_MIN = 0.9999          # d-vectors in eval precision (one fp16 plane) against fp64
E2E_REL = 1e-3            # the project's relative tolerance for loss and gradients against fp64 (test_gpu_parity_full.py)
GRAD_REL = 1e-4           # input and per-tensor gradients against the gate-forced fp64 oracle (test_gpu_input_grad.py)
ONE_PLANE_REL = 5e-2      # input gradient of a one-plane training plan (fp16 operands) against fp64: that plan's own
                          # accuracy, 3.4e-2 at 80 mels and 2.8e-2 at 256 on a B200 (two planes: 6.6e-5 / 9.6e-5)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


def _record(kind, **kw):
    print("mel dim:", json.dumps(dict(kind=kind, **kw)))


def _hp(mel_dim, layers=3):
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    hp = default_hyper_parameters()
    hp.Sound.Mel_Dim = mel_dim
    hp.GE2E.Transformer.Num_Layers = layers
    return hp


def _state(seed, mel_dim):
    state = synth.make_state(seed)
    rng = np.random.default_rng(seed + 7919 * mel_dim)
    bound = math.sqrt(2.0) * math.sqrt(6.0 / (mel_dim + D))
    w = rng.uniform(-bound, bound, (D, mel_dim, 1))
    state["prenet.weight"] = (w + 0.1 * bound * rng.standard_normal(w.shape)).astype(np.float32)
    return state


def _model(seed, mel_dim):
    from speaker_embedding_torch_b200 import GE2E
    state = _state(seed, mel_dim)
    m = GE2E(_hp(mel_dim))
    m.load_state_dict({k: torch.as_tensor(v) for k, v in state.items()}, strict=True)
    return m.to(DEV), state


def _mel(seed, batch, frames, mel_dim):
    return torch.as_tensor(synth.make_mel(seed, batch, frames, mel_dim=mel_dim)).to(DEV)


def _cos_min(a, b):
    return float(torch.nn.functional.cosine_similarity(a.double(), b.double(), dim=1).min())


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _cfg(mel_dim):
    from speaker_embedding_torch_b200 import _native as N
    return N.EncoderConfig(mel_dim, 256, 4, 1024, 3, 1024, 0.1, 0.1)


def _lib():
    from speaker_embedding_torch_b200 import _native as N
    if not os.path.exists(N.LIB_PATH):
        N.build()
    return N.lib()


# ------------------------------------------------------------------------------------------------
# host
@pytest.mark.parametrize("mel_dim", list(range(16, 257, 8)))
def test_every_legal_mel_dim_has_a_workspace(mel_dim):
    L = _lib()
    cfg = _cfg(mel_dim)
    for args in ((10, 64, 5, 1, 0), (12, 160, 1, 2, 1), (12, 160, 1, 1, 1), (4, 300, 1, 2, 1)):
        assert L.spk_encoder_workspace_bytes(ctypes.byref(cfg), *args) > 0, (mel_dim, args, L.spk_last_error())


def test_workspace_does_not_grow_up_to_80_mels():
    """dX lives in a region every training plan has anyway: the workspace depends on Mel_Dim only through x0 and the
    packed prenet weight."""
    L = _lib()
    for args in ((10, 64, 5, 1, 0), (12, 160, 1, 2, 1), (12, 160, 1, 1, 1), (960, 160, 1, 2, 1)):
        sizes = [L.spk_encoder_workspace_bytes(ctypes.byref(_cfg(c)), *args) for c in (16, 40, 64, 80)]
        assert sizes == sorted(sizes) and sizes[-1] > 0, (args, sizes)


@pytest.mark.parametrize("mel_dim", [0, 8, 12, 60, 100, 264])
def test_illegal_mel_dim_is_rejected_with_the_rule(mel_dim):
    L = _lib()
    cfg = _cfg(mel_dim)
    assert L.spk_encoder_workspace_bytes(ctypes.byref(cfg), 10, 64, 5, 1, 0) == 0
    assert b"must be a multiple of 8 in [16, 256]" in L.spk_last_error(), L.spk_last_error()


def test_ge2e_builds_its_prenet_from_mel_dim():
    from speaker_embedding_torch_b200 import GE2E
    m = GE2E(_hp(40))
    sd = m.state_dict()
    assert len(sd) == 44
    assert tuple(sd["prenet.weight"].shape) == (256, 40, 1)
    assert [k for k, _ in synth.state_shapes(mel_dim=40)] == list(sd)
    assert m._cfg.mel_dim == 40


# ------------------------------------------------------------------------------------------------
# GEMM shapes reached only by other mel counts
def _gemm_err(out, ref):
    return float((out.double() - ref).abs().max() / ref.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("c", [16, 24, 40, 136, 256])
@pytest.mark.parametrize("planes", [1, 2])
def test_prenet_gemm_shapes_match_fp64(c, planes):
    """prenet (and prenet_gate): K = C, N = 256, single-CTA and CTA-pair kernels (bit-identical to each other)."""
    from speaker_embedding_torch_b200 import _native as N
    m = 1000
    torch.manual_seed(c + planes)
    a = N.split_pack(torch.randn(m, c, device=DEV), planes)
    b = N.split_pack(torch.randn(D, c, device=DEV), planes)
    ref = N.split_unpack(a).double() @ N.split_unpack(b).double().t()
    outs = []
    try:
        for mode in (0, 1):
            N.set_option("gemm_cta_pairs", mode)
            outs.append(N.gemm(a, b, planes, m, D, c, out_f32=True).clone())
    finally:
        N.set_option("gemm_cta_pairs", 1)
    torch.cuda.synchronize()
    err = _gemm_err(outs[1], ref)
    _record("gemm_prenet", c=c, planes=planes, err=err)
    assert torch.equal(outs[0], outs[1])
    assert err <= (2e-6 if planes == 1 else 2e-5), err          # the bound of test_gpu_gemm.py


@pytest.mark.gpu
@pytest.mark.parametrize("c", [16, 24, 40, 136, 256])
@pytest.mark.parametrize("block_n", [0, 64])
def test_mel_dgrad_gemm_shapes_match_fp64(c, block_n):
    """mel_dgrad: K = 256, N = C, MN-major B, fp32 out."""
    from speaker_embedding_torch_b200 import _native as N
    m, planes = 7680, 2
    torch.manual_seed(c + block_n)
    a = N.split_pack(torch.randn(m, D, device=DEV), planes)
    b = N.split_pack(torch.randn(D, c, device=DEV), planes)
    ref = N.split_unpack(a).double() @ N.split_unpack(b).double()
    out = N.gemm(a, b, planes, m, c, D, b_mn=True, out_f32=True, block_n=block_n)
    torch.cuda.synchronize()
    err = _gemm_err(out, ref)
    _record("gemm_mel_dgrad", c=c, block_n=block_n, err=err)
    assert err <= 2e-5, err


@pytest.mark.gpu
@pytest.mark.parametrize("c", [16, 24, 40, 136, 256])
def test_prenet_wgrad_gemm_shapes_match_fp64(c):
    """prenet_wgrad: M = 256, N = C, K = tokens, both operands MN-major, split-K into fp32 atomics."""
    from speaker_embedding_torch_b200 import _native as N
    k, planes, ksplit = 4000, 2, 4
    torch.manual_seed(c)
    a = N.split_pack(torch.randn(k, D, device=DEV), planes)      # dU [tokens, 256]
    b = N.split_pack(torch.randn(k, c, device=DEV), planes)      # x0 [tokens, C]
    ref = N.split_unpack(a).double().t() @ N.split_unpack(b).double()
    out = torch.zeros(D, c, device=DEV)
    N.gemm(a, b, planes, D, c, k, a_mn=True, b_mn=True, atomic_out=out, ksplit=ksplit)
    torch.cuda.synchronize()
    err = _gemm_err(out, ref)
    _record("gemm_prenet_wgrad", c=c, err=err)
    assert err <= 2e-5 * (k / 256) ** 0.5, err


# ------------------------------------------------------------------------------------------------
# 1: inference
@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 64, 160, 240, 300])
@pytest.mark.parametrize("c", MEL_DIMS)
def test_inference_matches_fp64(c, T):
    m, state = _model(201, c)
    m.eval()
    st = {k: torch.as_tensor(v).to(DEV, torch.float64) for k, v in state.items()}
    for samples in (1, 5):
        mel = _mel(4000 + T + samples, 4 * samples, T, c)
        with torch.no_grad():
            d = m(mel, samples)
        ref = O.encoder_forward(st, mel.double(), samples=samples)
        cos = _cos_min(d, ref)
        _record("inference", c=c, T=T, samples=samples, cos_min=cos)
        assert d.shape == (4, D)
        assert cos >= COS_MIN, (samples, cos)


# ------------------------------------------------------------------------------------------------
# 2: training (two planes, eval masks)
def _pooled_rel(m, g_ref):
    num = sum(float(((p.grad.double() - g_ref[n]) ** 2).sum()) for n, p in m.named_parameters())
    den = sum(float((g_ref[n] ** 2).sum()) for n, _ in m.named_parameters())
    return (num / den) ** 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("nspk,utt,T", [(2, 3, 64), (3, 5, 160), (4, 4, 300)])
@pytest.mark.parametrize("c", MEL_DIMS)
def test_training_step_matches_fp64(c, nspk, utt, T):
    """Loss and d-vectors against the plain fp64 oracle; the pooled gradient against the fp64 oracle forced onto the
    kernels' own ReLU gates, as in test_gpu_stage_parity.py.  Unforced, one prenet pre-activation within rounding of
    zero takes the other branch: at C = 256, 2 x 3 x 64 that moves the prenet gradients by 7 % with two planes and
    with three alike (B200), while they agree with the gate-forced oracle to 1.2e-5.  The unforced pooled error is
    recorded beside it."""
    from test_gpu_stage_parity import _oracle, _relu_masks, _train_step
    B = nspk * utt
    m, state = _model(202, c)
    mel = _mel(4100 + T, B, T, c)
    _, d, loss, _ = _train_step(m, mel, utt, False)
    loss_ref, d_ref, g_ref = _oracle(state, mel, utt)
    masks = _relu_masks(m, B, T, 1)
    _, _, g_gate = _oracle(state, mel, utt, relu_masks=masks)
    loss_rel = abs(loss.item() - loss_ref) / abs(loss_ref)
    rec = dict(c=c, case=[nspk, utt, T], loss_rel=loss_rel, grad_rel=_pooled_rel(m, g_gate),
               grad_rel_unforced=_pooled_rel(m, g_ref), cos_min=_cos_min(d, d_ref))
    if c in (40, 128) and T == 160:
        rec["prenet_w"] = _rel(m.prenet.weight.grad, g_gate["prenet.weight"])
        rec["prenet_b"] = _rel(m.prenet.bias.grad, g_gate["prenet.bias"])
    _record("training", **rec)
    assert loss_rel <= E2E_REL and rec["grad_rel"] <= E2E_REL, rec
    assert rec["cos_min"] >= COS_MIN, rec
    if "prenet_w" in rec:
        assert rec["prenet_w"] <= GRAD_REL and rec["prenet_b"] <= GRAD_REL, rec


# ------------------------------------------------------------------------------------------------
# 3: input gradients
@pytest.mark.gpu
@pytest.mark.parametrize("c", MEL_DIMS)
def test_features_grad_through_forward(c):
    """features.grad with trainable and frozen parameters, fp32 and fp16 features, against fp64 autograd through the
    oracle forced onto the kernels' ReLU gates; repeated calls are bit-identical, and so are trainable and frozen."""
    from test_gpu_input_grad import _oracle_with_mel
    from test_gpu_stage_parity import _relu_masks
    B, T = 12, 96
    m, state = _model(203, c)
    m.eval()
    m._debug_keep_ws = True
    cot = torch.randn(B, D, generator=torch.Generator().manual_seed(c)).to(DEV)
    mel = _mel(4200 + c, B, T, c)

    def grad_of(x0, trainable):
        for p in m.parameters():
            p.requires_grad_(trainable)
            p.grad = None
        x = x0.clone().requires_grad_(True)
        m(x).backward(cot)
        torch.cuda.synchronize()
        return x.grad

    for dtype in (torch.float32, torch.float16):
        x0 = mel.to(dtype)
        g = grad_of(x0, True)
        masks = _relu_masks(m, B, T, 1)
        again = grad_of(x0, True)
        frozen = grad_of(x0, False)
        _, g_ref, _ = _oracle_with_mel(state, x0.float(), None, relu_masks=masks, cotangent=cot)
        err = _rel(g, g_ref.to(dtype))
        _record("features_grad", c=c, dtype=str(dtype), err=err)
        assert g.dtype == dtype and g.shape == (B, c, T)
        assert torch.equal(g, again)
        assert torch.equal(g, frozen)
        assert err <= GRAD_REL, (dtype, err)


@pytest.mark.gpu
@pytest.mark.parametrize("c", MEL_DIMS)
def test_ragged_data_grad_through_embed_utterances(c):
    """Lengths that are reflect-padded (1, 3, T - 1), exact (T) and cropped across several slices."""
    from speaker_embedding_torch_b200.Modules import utterance_slices
    from test_gpu_stage_parity import _relu_masks
    from test_gpu_utterances import _oracle
    T, O_ = 64, 32
    lengths = [1, 3, T - 1, T, T + 1, 2 * T + 5, 3 * T]
    m, state = _model(204, c)
    m.eval()
    m._debug_keep_ws = True
    for p in m.parameters():
        p.requires_grad_(False)
    mels = [_mel(4300 + c + i, 1, L, c)[0] for i, L in enumerate(lengths)]
    cot = torch.randn(len(lengths), D, generator=torch.Generator().manual_seed(c + 1)).to(DEV)

    def run():
        xs = [x.clone().requires_grad_(True) for x in mels]
        m.embed_utterances(xs, T, O_).backward(cot)
        torch.cuda.synchronize()
        return torch.cat([x.grad for x in xs], dim=1)

    g = run()
    table, seg = utterance_slices(lengths, T, O_)
    masks = _relu_masks(m, table.size(0), T, 1)
    again = run()
    _, g_ref, _ = _oracle(state, torch.cat(mels, dim=1), table, seg, T, cot, None, masks)
    err = _rel(g, g_ref)
    _record("ragged_grad", c=c, slices=int(seg[-1]), err=err)
    assert torch.equal(g, again)
    assert err <= GRAD_REL, err


@pytest.mark.gpu
def test_one_plane_training_plan_input_grad_at_256_mels():
    """A one-plane backward plan keeps the fewest gradient bytes per token; dX (4 * 256 bytes per token) must still
    fit where it is written.  Against fp64 and against the two-plane plan."""
    from test_gpu_input_grad import _oracle_with_mel
    c, B, T = 256, 16, 160
    m, state = _model(205, c)
    m.eval()
    mel = _mel(4400, B, T, c)
    cot = torch.randn(B, D, generator=torch.Generator().manual_seed(12)).to(DEV)

    def grad_of(precision):
        m.train_precision = precision
        m.zero_grad(set_to_none=True)
        x = mel.clone().requires_grad_(True)
        m(x).backward(cot)
        torch.cuda.synchronize()
        return x.grad

    g1 = grad_of(1)
    g1b = grad_of(1)
    g2 = grad_of(2)
    _, g_ref, _ = _oracle_with_mel(state, mel, None, cotangent=cot)
    rec = dict(one_vs_fp64=_rel(g1, g_ref), one_vs_two=_rel(g1, g2), two_vs_fp64=_rel(g2, g_ref))
    _record("one_plane_256", **rec)
    assert torch.equal(g1, g1b)
    assert bool(torch.isfinite(g1).all())
    assert rec["one_vs_fp64"] <= ONE_PLANE_REL and rec["one_vs_two"] <= ONE_PLANE_REL, rec
    assert rec["two_vs_fp64"] <= E2E_REL, rec


# ------------------------------------------------------------------------------------------------
# 4: collation paths
@pytest.mark.gpu
@pytest.mark.parametrize("c", MEL_DIMS)
def test_embed_windows_equals_the_sliced_forward(c):
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices
    m, _ = _model(206, c)
    m.eval()
    frame, overlap, samples = 64, 32, 5
    windows = _mel(4500 + c, 7, samples * (frame - overlap) + overlap, c)
    with torch.no_grad():
        for w in (windows, windows.half()):
            ref = m(Overlapped_Slices(w.float(), frame, overlap), samples)
            assert torch.equal(m.embed_windows(w, frame, overlap), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("c", MEL_DIMS)
def test_device_collater_equals_the_host_restatement(c):
    from speaker_embedding_torch_b200.Datasets import Collater
    np.random.seed(c)
    lengths = [[30, 64, 65], [100, 12, 250], [1, 2, 80]]
    feats = [[(synth.make_mel(4600 + 10 * s + u, 1, L, mel_dim=c)[0].astype(np.float16), s)
              for u, L in enumerate(row)] for s, row in enumerate(lengths)]
    batch = Collater(60, 90)(feats)
    assert batch.data.shape[0] == c
    dense = batch.dense().to(DEV)
    m, _ = _model(207, c)
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(batch.to(DEV)), m(dense))


# ------------------------------------------------------------------------------------------------
# 5: mel front-end -> embed_utterances -> cosine critic -> audio
@pytest.mark.gpu
@pytest.mark.parametrize("c", [40, 128])
def test_audio_grad_through_mel_spectrogram_and_embed_utterances(c):
    from mel_grad_oracle import mel_spectrogram_torch
    from speaker_embedding_torch_b200.Modules import utterance_slices
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    from test_gpu_stage_parity import _dstate
    from test_gpu_utterances import _dense, _seg_head
    sound = dict(n_fft=1024, num_mels=c, sampling_rate=22050, hop_size=256, win_size=1024, fmin=0, fmax=None)
    frames = [40, 64, 150]
    T, O_ = 64, 32
    m, state = _model(208, c)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    torch.manual_seed(c)
    y0 = [0.3 * torch.randn(1, f * 256, device=DEV) for f in frames]
    target = torch.nn.functional.normalize(torch.randn(len(frames), D, device=DEV), dim=1)

    def critic(d, t):
        return (1.0 - torch.nn.functional.cosine_similarity(d, t, dim=1)).mean()

    ys = [y.clone().requires_grad_(True) for y in y0]
    mels = [mel_spectrogram(y, **sound)[0] for y in ys]
    assert [x.shape for x in mels] == [(c, f) for f in frames]
    loss = critic(m.embed_utterances(mels, T, O_), target)
    loss.backward()

    ys64 = [y.double().requires_grad_(True) for y in y0]
    data64 = torch.cat([mel_spectrogram_torch(y, **sound)[0] for y in ys64], dim=1)
    table, seg = utterance_slices(frames, T, O_)
    st = _dstate(state)
    _, inter = O.encoder_forward(st, _dense(data64, table, T), layers=3, return_intermediates=True)
    loss64 = critic(_seg_head(st, inter["layer2"], seg), target.double())
    loss64.backward()
    err = _rel(torch.cat([y.grad[0] for y in ys]), torch.cat([y.grad[0] for y in ys64]))
    _record("audio_grad", c=c, loss=float(loss.detach()), loss64=float(loss64), err=err)
    assert err <= E2E_REL, err


# ------------------------------------------------------------------------------------------------
# 6: formats
@pytest.mark.gpu
def test_arena_round_trip_at_64_mels(tmp_path):
    from speaker_embedding_torch_b200 import Export
    c = 64
    m, _ = _model(209, c)
    m.eval()
    path = str(tmp_path / "encoder.spkw")
    header = Export.export_arena(m, path)
    assert header["config"]["Mel_Dim"] == c
    m2 = Export.model_from_arena(path, DEV)
    mel = _mel(4700, 6, 100, c)
    with torch.no_grad():
        assert torch.equal(m2(mel), m(mel))


@pytest.mark.gpu
def test_trace_at_64_mels(tmp_path):
    import yaml
    from speaker_embedding_torch_b200.Trace import Tracer
    c = 64
    m, _ = _model(210, c)
    hp = {"Sound": {"Mel_Dim": c},
          "GE2E": {"Embedding_Size": 256, "Positional_Encoding": {"Max_Position": 1024, "Dropout_Rate": 0.1},
                   "Transformer": {"Num_Layers": 3, "Head": 4, "Dropout_Rate": 0.1}}}
    hp_path, ckpt = str(tmp_path / "hp.yaml"), str(tmp_path / "S_1.pt")
    yaml.safe_dump(hp, open(hp_path, "w"))
    torch.save({"Model": m.state_dict(), "Steps": 1}, ckpt)
    tracer = Tracer(hp_path, ckpt)
    x = torch.rand(1, c, 400, device=DEV)
    lengths = torch.LongTensor([400]).to(DEV)
    traced = torch.jit.trace(tracer, (x, lengths), check_trace=False)
    assert str(traced.inlined_graph).count("spkemb::encoder_infer") == 1
    xb = _mel(4800, 4, 200, c)
    m.eval()
    with torch.no_grad():
        torch.testing.assert_close(traced(xb, lengths), m(xb), atol=0, rtol=0)


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "Modules.py")),
                    reason="needs a reference checkout, staged to baseline/_ref by build() from SPK_REFERENCE")
def test_state_dict_loads_into_the_reference_ge2e():
    import importlib.util
    import warnings
    c = 40
    m, _ = _model(211, c)
    sys.path.insert(0, REF)
    try:
        spec = importlib.util.spec_from_file_location("reference_Modules_mel_dim", os.path.join(REF, "Modules.py"))
        ref_mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref_mod)
    finally:
        sys.path.remove(REF)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref_model = ref_mod.GE2E(_hp(c)).eval()
    ref_model.load_state_dict({k: v.cpu() for k, v in m.state_dict().items()}, strict=True)
    mel = synth.make_mel(4900, 10, 80, mel_dim=c)
    with torch.no_grad():
        want = ref_model(torch.as_tensor(mel), 5)
        m.eval()
        got = m(torch.as_tensor(mel).to(DEV), 5).cpu()
    assert _cos_min(got, want) >= COS_MIN


# ------------------------------------------------------------------------------------------------
# 7: errors
@pytest.mark.gpu
def test_wrong_channel_count_is_rejected():
    m, _ = _model(212, 40)
    m.eval()
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="Mel_Dim"):
            m(_mel(5000, 2, 64, 80))
    with pytest.raises(RuntimeError, match="Mel_Dim"):
        m.embed_utterances([_mel(5001, 1, 64, 80)[0]], 64, 32)
