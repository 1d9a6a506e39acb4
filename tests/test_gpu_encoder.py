"""Encoder forward / backward parity on the GPU, through the drop-in modules (C ABI underneath).

Forward: against the reference's own d-vectors (tests/golden/encoder_forward.npz, fp64 run of
/root/reference/Modules.py) -- tolerance from BASELINE.json: cosine >= 0.9999 per d-vector.
Backward: against the fp64 oracle (itself pinned to the reference by tests/test_oracle_golden.py)
and the reference's gradient fingerprints (tests/golden/train_grads.npz) -- relative loss / global
gradient error <= 1e-3.  Parity is defined in eval mode (dropout masks cannot match, SURVEY.md D9).
"""
import os

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth
from oracle.make_golden import fingerprint_indices

pytestmark = pytest.mark.gpu


def _model(seed, layers=3):
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    hp = default_hyper_parameters()
    hp.GE2E.Transformer.Num_Layers = layers
    state = synth.make_state(seed)
    m = GE2E(hp)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in state.items() if k in m.state_dict()}, strict=True)
    return m.cuda(), state


def _cos(a, b):
    return (a * b).sum(1) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))


@pytest.mark.parametrize("precision,min_cos,max_abs", [(1, 0.9999, 4e-3), (2, 0.99999999, 2e-5)])
def test_forward_matches_reference_golden(golden_dir, precision, min_cos, max_abs):
    g = np.load(os.path.join(golden_dir, "encoder_forward.npz"))
    for i in range(int(g["num_cases"])):
        ss, ms, B, T, S = [int(v) for v in g["case%d_meta" % i]]
        m, _ = _model(ss)
        m.eval()
        m.eval_precision = precision
        with torch.no_grad():
            d = m(torch.as_tensor(synth.make_mel(ms, B, T)).cuda(), S)
        torch.cuda.synchronize()
        assert d.shape == (B // S, 256) and d.dtype == torch.float32
        d = d.cpu().numpy().astype(np.float64)
        ref = g["case%d_f64" % i]
        assert _cos(d, ref).min() >= min_cos, (i, B, T, S, _cos(d, ref).min())
        assert np.abs(d - ref).max() <= max_abs, (i, np.abs(d - ref).max())
        np.testing.assert_allclose(np.linalg.norm(d, axis=1), 1.0, atol=1e-5)


def test_forward_full_size_batch_properties():
    """BASELINE size (960 slices x 160 frames): unit norm, determinism, batch-composition independence."""
    m, state = _model(7)
    m.eval()
    mel = torch.as_tensor(synth.make_mel(70, 960, 160)).cuda()
    with torch.no_grad():
        d1 = m(mel)
        d2 = m(mel)
        d_part = m(mel[100:132])
    torch.cuda.synchronize()
    assert torch.equal(d1, d2)
    torch.testing.assert_close(d1.norm(dim=1), torch.ones(960, device="cuda"), atol=1e-5, rtol=0)
    torch.testing.assert_close(d1[100:132], d_part, atol=1e-6, rtol=0)      # slices are independent
    ref = O.encoder_forward(O.to_torch_state(state, torch.float32), mel[:8].cpu(), 1).numpy()
    assert _cos(d1[:8].cpu().numpy(), ref).min() >= 0.9999


def test_multislice_inference_chunks_whole_utterances():
    """5 x 64-frame slices with samples=5 (Inference.py:95-115): chunked == unchunked; mean is taken
    over the slices of one utterance before projection (Modules.py:55-56)."""
    m, state = _model(8)
    m.eval()
    mel = torch.as_tensor(synth.make_mel(80, 35, 64)).cuda()
    with torch.no_grad():
        full = m(mel, 5)
        m.max_slices_per_call = 12                 # -> chunks of 10 slices = 2 utterances
        chunked = m(mel, 5)
    torch.cuda.synchronize()
    assert full.shape == (7, 256)
    torch.testing.assert_close(full, chunked, atol=1e-6, rtol=0)
    ref = O.encoder_forward(O.to_torch_state(state, torch.float64), mel.cpu().double(), 5).numpy()
    assert _cos(full.cpu().numpy().astype(np.float64), ref).min() >= 0.9999
    with pytest.raises(RuntimeError, match="invalid"):
        with torch.no_grad():
            m(mel, 4)                              # 35 slices are not a multiple of 4


def _grad_errors(m, g_ref):
    num = den = 0.0
    worst = ("", 0.0)
    for name, p in m.named_parameters():
        g = p.grad.detach().cpu().numpy().astype(np.float64)
        r = g_ref[name]
        num += ((g - r) ** 2).sum()
        den += (r ** 2).sum()
        rel = np.linalg.norm(g - r) / max(np.linalg.norm(r), 1e-30)
        if rel > worst[1]:
            worst = (name, rel)
    return (num / den) ** 0.5, worst


@pytest.mark.parametrize("nspk,utt,frames", [(3, 2, 24), (4, 3, 50), (10, 4, 24), (2, 2, 128), (4, 3, 160), (3, 2, 177)])
def test_train_step_grads_match_oracle(nspk, utt, frames):
    from speaker_embedding_torch_b200 import GE2E_Loss
    m, state = _model(33)
    m.eval()
    crit = GE2E_Loss().cuda()
    mel = synth.make_mel(500 + frames, nspk * utt, frames)
    d = m(torch.as_tensor(mel).cuda())
    loss = crit(d, utt)
    loss.backward()
    torch.cuda.synchronize()
    loss_ref, d_ref, g_ref = O.train_step_grads(state, mel, utt)
    assert abs(loss.item() - loss_ref) <= 1e-3 * abs(loss_ref)
    assert _cos(d.detach().cpu().numpy().astype(np.float64), d_ref).min() >= 0.9999
    rel_all, worst = _grad_errors(m, g_ref)
    assert rel_all <= 1e-3, (rel_all, worst)
    assert abs(crit.weight.grad.item() - float(g_ref["loss.weight"])) <= 1e-3 * abs(float(g_ref["loss.weight"]))
    assert abs(crit.bias.grad.item()) <= 1e-6


def test_train_step_grads_match_reference_fingerprints(golden_dir):
    from speaker_embedding_torch_b200 import GE2E_Loss
    g = np.load(os.path.join(golden_dir, "train_grads.npz"))
    for i in range(int(g["num_cases"])):
        ss, ms, N, M, T = [int(v) for v in g["case%d_meta" % i]]
        m, _ = _model(ss)
        m.eval()
        crit = GE2E_Loss().cuda()
        loss = crit(m(torch.as_tensor(synth.make_mel(ms, N * M, T)).cuda()), M)
        loss.backward()
        torch.cuda.synchronize()
        assert abs(loss.item() - float(g["case%d_loss" % i])) <= 1e-3 * abs(float(g["case%d_loss" % i]))
        num = den = 0.0
        for name, p in m.named_parameters():
            gr = p.grad.detach().cpu().numpy().astype(np.float64).reshape(-1)
            ref_norm = float(g["case%d_gnorm_%s" % (i, name)])
            assert abs(np.linalg.norm(gr) - ref_norm) <= 2e-3 * ref_norm + 1e-12, name
            samp = g["case%d_gsamp_%s" % (i, name)]
            num += ((gr[fingerprint_indices(gr.size)] - samp) ** 2).sum()
            den += (samp ** 2).sum()
        assert (num / den) ** 0.5 <= 1e-3


def test_dropout_train_mode_is_seeded_and_unbiased():
    from speaker_embedding_torch_b200 import GE2E_Loss
    m, _ = _model(9)
    crit = GE2E_Loss().cuda()
    mel = torch.as_tensor(synth.make_mel(90, 12, 40)).cuda()
    m.train()
    torch.manual_seed(1)
    d1 = m(mel)
    torch.manual_seed(1)
    d2 = m(mel)
    torch.manual_seed(2)
    d3 = m(mel)
    assert torch.equal(d1, d2) and not torch.equal(d1, d3)          # mask = f(seed)
    loss = crit(d1, 3)
    loss.backward()
    torch.cuda.synchronize()
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())
    m.eval()
    d_eval = m(mel).detach()
    # averaged over masks the train-mode d-vectors stay close to the eval ones
    m.train()
    acc = torch.zeros_like(d_eval)
    for s in range(24):
        torch.manual_seed(100 + s)
        acc += m(mel).detach()
    cos = torch.nn.functional.cosine_similarity(acc, d_eval, dim=1)
    assert cos.min().item() > 0.9


def test_dropout_zero_equals_eval():
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    hp = default_hyper_parameters()
    hp.GE2E.Positional_Encoding.Dropout_Rate = 0.0
    hp.GE2E.Transformer.Dropout_Rate = 0.0
    m = GE2E(hp)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in synth.make_state(4).items()})
    m = m.cuda()
    mel = torch.as_tensor(synth.make_mel(41, 6, 30)).cuda()
    m.train()
    a = m(mel).detach()
    m.eval()
    b = m(mel).detach()
    torch.testing.assert_close(a, b, atol=1e-7, rtol=0)


def test_shape_and_device_errors():
    m, _ = _model(5)
    m.eval()
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="Mel_Dim"):
            m(torch.zeros(2, 64, 16, device="cuda"))
        with pytest.raises(RuntimeError, match="frames"):
            m(torch.zeros(2, 80, 1025, device="cuda"))
        out = m(torch.zeros(3, 80, 1, device="cuda"))                 # T = 1 edge case
    assert out.shape == (3, 256) and torch.isfinite(out).all()


def test_last_layer_pruning_is_exact():
    """Only the t = 0 query of the last layer is consumed (Modules.py:54): the pruned path (default) and the
    dense path must give the same d-vectors and gradients, in eval and with the same dropout seed."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    mel = torch.as_tensor(synth.make_mel(77, 8, 150)).cuda()
    results = {}
    try:
        for prune in (1, 0):
            _native.set_option("prune_last_layer", prune)
            m, _ = _model(21)
            m.eval()
            crit = GE2E_Loss().cuda()
            with torch.no_grad():
                d_inf = m(mel).clone()
            d = m(mel)
            crit(d, 4).backward()
            torch.cuda.synchronize()
            results[prune] = (d_inf, d.detach().clone(), {n: p.grad.clone() for n, p in m.named_parameters()})
    finally:
        _native.set_option("prune_last_layer", 1)
    torch.testing.assert_close(results[1][0], results[0][0], atol=2e-3, rtol=0)        # bf16 inference path
    torch.testing.assert_close(results[1][1], results[0][1], atol=2e-6, rtol=0)        # fp32-equivalent training path
    num = sum(float(((results[1][2][n] - results[0][2][n]).double() ** 2).sum()) for n in results[0][2])
    den = sum(float((results[0][2][n].double() ** 2).sum()) for n in results[0][2])
    assert (num / den) ** 0.5 <= 2e-4


@pytest.mark.parametrize("frames", [1, 24, 64, 128, 129, 160, 177, 200, 256])
def test_fused_inference_attention_matches_unfused_and_oracle(frames):
    """The one-kernel tcgen05 attention of the inference path (scores stay in TMEM / shared memory) against the
    GEMM + softmax + GEMM composition and the fp64 oracle."""
    from speaker_embedding_torch_b200 import _native
    m, state = _model(44)
    m.eval()
    mel = torch.as_tensor(synth.make_mel(300 + frames, 6, frames)).cuda()
    out = {}
    try:
        for fused in (1, 0):
            _native.set_option("fused_inference_attention", fused)
            with torch.no_grad():
                out[fused] = m(mel).clone()
            torch.cuda.synchronize()
    finally:
        _native.set_option("fused_inference_attention", 1)
    ref = O.encoder_forward(O.to_torch_state(state, torch.float64), mel.cpu().double(), 1).numpy()
    for fused in (1, 0):
        assert _cos(out[fused].cpu().numpy().astype(np.float64), ref).min() >= 0.9999, fused
    torch.testing.assert_close(out[1], out[0], atol=4e-3, rtol=0)


def test_embed_windows_equals_host_sliced_forward():
    """Overlapping slices cut inside the prenet load (spk_mel_view) == the reference collater's slices
    (Inference.py:103-110) fed through forward(features, samples): bit-identical d-vectors, fp32 and fp16 windows,
    several utterance counts (including one that is chunked by max_slices_per_call)."""
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices
    m, _ = _model(11)
    m.eval()
    frame, overlap, samples = 64, 32, 5
    required = samples * (frame - overlap) + overlap
    for utts in (1, 7, 33):
        windows = torch.as_tensor(synth.make_mel(300 + utts, utts, required)).cuda()
        with torch.no_grad():
            ref = m(Overlapped_Slices(windows, frame, overlap), samples)
            got = m.embed_windows(windows, frame, overlap)
            assert got.shape == (utts, 256)
            assert torch.equal(got, ref)
            half = windows.half()
            ref16 = m(Overlapped_Slices(half.float(), frame, overlap), samples)
            assert torch.equal(m.embed_windows(half, frame, overlap), ref16)
    m.max_slices_per_call = 10                      # two utterances per call
    with torch.no_grad():
        assert torch.equal(m.embed_windows(windows, frame, overlap), ref)
    with pytest.raises(RuntimeError):
        m.embed_windows(windows[:, :, :40], frame, overlap)
    m.train()
    with pytest.raises(RuntimeError):
        m.embed_windows(windows, frame, overlap)


def test_fp16_patterns_are_upcast_in_the_prenet_load():
    """The reference stores patterns as fp16 (Pattern_Generator.py:123) and upcasts on the host (Datasets.py:84);
    here fp16 features go to the device as they are: same d-vectors and gradients as the host-upcast input."""
    from speaker_embedding_torch_b200 import GE2E_Loss
    m, _ = _model(12)
    mel16 = torch.as_tensor(synth.make_mel(120, 4 * 3, 50)).cuda().half()
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(mel16), m(mel16.float()))
    crit = GE2E_Loss().cuda()
    grads = []
    for x in (mel16, mel16.float()):
        m.zero_grad(set_to_none=True)
        crit(m(x), 3).backward()
        grads.append(torch.cat([p.grad.flatten() for p in m.parameters()]).clone())
    # same inputs after the upcast; the split-K weight gradients use fp32 atomics, so not bit-for-bit
    rel = float((grads[0] - grads[1]).norm() / grads[1].norm())
    assert rel < 1e-5, rel


@pytest.mark.parametrize("frames", [1, 7, 16, 40, 100, 128, 129, 144, 160, 177, 192])
@pytest.mark.parametrize("train", [False, True])
def test_fused_training_attention_matches_materialised_path(frames, train):
    """The fused tcgen05 attention of the training path (forward: probabilities stay in TMEM; backward: recomputed
    from the saved row statistics and the keep-bit mask) against the GEMM + softmax + GEMM composition it replaces:
    same d-vectors and same gradients, in eval mode and -- same seed, hence same dropout masks -- in train mode."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    nspk, utt = 3, 2
    mel = torch.as_tensor(synth.make_mel(400 + frames, nspk * utt, frames)).cuda()
    res = {}
    try:
        for fused in (1, 0):
            _native.set_option("fused_training_attention", fused)
            m, _ = _model(45)
            m.train(train)
            crit = GE2E_Loss().cuda()
            torch.manual_seed(77)
            d = m(mel)
            crit(d, utt).backward()
            torch.cuda.synchronize()
            res[fused] = (d.detach().clone(), torch.cat([p.grad.flatten() for p in m.parameters()]).clone())
    finally:
        _native.set_option("fused_training_attention", 1)
    torch.testing.assert_close(res[1][0], res[0][0], atol=3e-6, rtol=0)
    rel = float((res[1][1] - res[0][1]).double().norm() / res[0][1].double().norm())
    # Two approximations of the same gradient, each held to 1e-3 against the oracle.  Typical agreement is ~3e-5; the
    # bound leaves room for ONE ReLU gate whose pre-activation lies within the forward rounding error of zero and that
    # opens in one path only -- at 6 x T x 1024 gates such an element alone moves the gradient by ~1e-3 (the
    # unmodified reference in fp32 shows the same against its fp64 run: tools/full_parity_probe.py flips).
    assert rel <= 2e-3, rel


def test_fused_training_attention_falls_back_beyond_its_frame_limit():
    """T > 192 uses the materialised path (checked against the oracle in test_gpu_parity_full); the option is a no-op."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    mel = torch.as_tensor(synth.make_mel(499, 4, 200)).cuda()
    out = {}
    try:
        for fused in (1, 0):
            _native.set_option("fused_training_attention", fused)
            m, _ = _model(46)
            m.eval()
            d = m(mel)
            GE2E_Loss().cuda()(d, 2).backward()
            out[fused] = torch.cat([p.grad.flatten() for p in m.parameters()]).clone()
    finally:
        _native.set_option("fused_training_attention", 1)
    # identical kernels either way; only the split-K weight gradients' fp32 atomics reorder
    assert float((out[1] - out[0]).norm() / out[0].norm()) < 1e-5


@pytest.mark.parametrize("case", [0, 1, 2])
def test_device_collation_equals_the_host_collated_forward(golden_dir, case):
    """Training collation inside the prenet load (spk_encoder_forward_ragged): crop / numpy-style reflect-pad / fp16
    upcast of a ragged batch give exactly the d-vectors and gradients of the reference collater's dense tensor
    (tests/golden/collate.npz holds the reference collater's output for the same seeds)."""
    from oracle.make_golden_collate import make_batch
    from speaker_embedding_torch_b200 import GE2E_Loss
    from speaker_embedding_torch_b200.Datasets import Collater
    g = np.load(os.path.join(golden_dir, "collate.npz"))
    seed, spk, utt, tmin, tmax, lo, hi = [int(v) for v in g["case%d_meta" % case]]
    np.random.seed(seed)
    ragged = Collater(tmin, tmax)(make_batch(seed, spk, utt, lo, hi))
    dense = torch.as_tensor(g["case%d_out" % case]).cuda()             # the reference collater's tensor
    m, _ = _model(13)
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(ragged.to("cuda", non_blocking=True)), m(dense))
    crit = GE2E_Loss().cuda()
    grads = []
    for x in (ragged.cuda(), dense):
        m.zero_grad(set_to_none=True)
        d = m(x)
        crit(d, utt).backward()
        grads.append((d.detach().clone(), torch.cat([p.grad.flatten() for p in m.parameters()]).clone()))
    assert torch.equal(grads[0][0], grads[1][0])
    assert float((grads[0][1] - grads[1][1]).norm() / grads[1][1].norm()) < 1e-5     # fp32 atomics reorder only
    with pytest.raises(RuntimeError):
        m(ragged)                                                        # host tensors: no CPU path


@pytest.mark.parametrize("precision,min_cos", [(1, 0.9999), (2, 1 - 1e-9), (3, 1 - 1e-9)])
def test_inference_at_every_precision_against_the_oracle(precision, min_cos):
    """eval_precision 1 / 2 run the fused-LayerNorm GEMM instantiations (one / two planes), 3 the separate LayerNorm pass;
    all against the fp64 oracle, and the fused path against the unfused one."""
    from speaker_embedding_torch_b200 import _native
    m, state = _model(5)
    m.eval()
    m.eval_precision = precision
    mel = synth.make_mel(77, 24, 150)
    st = {k: torch.as_tensor(v).double() for k, v in state.items()}
    ref = O.encoder_forward(st, torch.as_tensor(mel).double()).numpy()
    out = {}
    try:
        for fused in (1, 0):
            _native.set_option("fused_layernorm", 2 * fused)
            with torch.no_grad():
                out[fused] = m(torch.as_tensor(mel).cuda()).double().cpu().numpy()
    finally:
        _native.set_option("fused_layernorm", 2)
    for d in out.values():
        cos = (d * ref).sum(1) / (np.linalg.norm(d, axis=1) * np.linalg.norm(ref, axis=1))
        assert cos.min() >= min_cos, cos.min()
    assert np.abs(out[1] - out[0]).max() <= (5e-4 if precision == 1 else 2e-6)


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("frames", [24, 160])
def test_fused_layernorm_training_forward_matches_the_separate_pass(frames, train):
    """EPI_LN in the training forward (z planes and row statistics written by the GEMM epilogue) against GEMM + ln_fwd:
    same d-vectors, same gradients (the backward reads the stashed z / statistics of either path)."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    nspk, utt = 3, 2
    mel = torch.as_tensor(synth.make_mel(900 + frames, nspk * utt, frames)).cuda()
    res = {}
    try:
        for level in (2, 1):
            _native.set_option("fused_layernorm", level)
            m, _ = _model(46)
            m.train(train)
            crit = GE2E_Loss().cuda()
            torch.manual_seed(78)
            d = m(mel)
            crit(d, utt).backward()
            torch.cuda.synchronize()
            res[level] = (d.detach().clone(), torch.cat([p.grad.flatten() for p in m.parameters()]).clone())
    finally:
        _native.set_option("fused_layernorm", 2)
    torch.testing.assert_close(res[2][0], res[1][0], atol=3e-6, rtol=0)
    rel = float((res[2][1] - res[1][1]).double().norm() / res[1][1].double().norm())
    assert rel <= 2e-3, rel       # typically ~1e-5; the bound leaves room for one ReLU gate (see the fused-attention test)


@pytest.mark.parametrize("frames", [1, 15, 16, 17, 100, 128, 129, 160, 191, 192])
def test_two_cta_inference_attention_matches_the_one_cta_kernel(frames):
    """attn_fwd_kernel<1, 8, false> (two CTAs per SM, T <= 192) against attn_fused_fwd_kernel on the same input, and both
    against the fp64 oracle (one fp16 plane: cosine >= 0.9999)."""
    from speaker_embedding_torch_b200 import _native
    m, state = _model(9)
    m.eval()
    mel = synth.make_mel(300 + frames, 7, frames)
    st = {k: torch.as_tensor(v).double() for k, v in state.items()}
    ref = O.encoder_forward(st, torch.as_tensor(mel).double()).numpy()
    out = {}
    try:
        for two in (1, 0):
            _native.set_option("inference_attention_two_ctas", two)
            with torch.no_grad():
                out[two] = m(torch.as_tensor(mel).cuda()).double().cpu().numpy()
    finally:
        _native.set_option("inference_attention_two_ctas", 1)
    for d in out.values():
        cos = (d * ref).sum(1) / (np.linalg.norm(d, axis=1) * np.linalg.norm(ref, axis=1))
        assert cos.min() >= 0.9999, cos.min()
    assert np.abs(out[1] - out[0]).max() <= 5e-4


@pytest.mark.parametrize("frames", [1, 16, 100, 129, 160, 192])
@pytest.mark.parametrize("train", [False, True])
def test_two_cta_training_attention_forward_matches_the_one_cta_kernel(frames, train):
    """attn_fwd_kernel<2, 8, true> (two CTAs per SM, one operand buffer for K then V) against
    attn_fwd_kernel<2, 16, false>: same d-vectors, same saved statistics / keep bits (checked through the gradients of
    the shared backward)."""
    from speaker_embedding_torch_b200 import GE2E_Loss, _native
    nspk, utt = 3, 2
    mel = torch.as_tensor(synth.make_mel(500 + frames, nspk * utt, frames)).cuda()
    res = {}
    try:
        for two in (1, 0):
            _native.set_option("training_attention_two_ctas", two)
            m, _ = _model(47)
            m.train(train)
            crit = GE2E_Loss().cuda()
            torch.manual_seed(79)
            d = m(mel)
            crit(d, utt).backward()
            torch.cuda.synchronize()
            res[two] = (d.detach().clone(), torch.cat([p.grad.flatten() for p in m.parameters()]).clone())
    finally:
        _native.set_option("training_attention_two_ctas", 1)
    torch.testing.assert_close(res[1][0], res[0][0], atol=3e-6, rtol=0)
    rel = float((res[1][1] - res[0][1]).double().norm() / res[0][1].double().norm())
    assert rel <= 2e-3, rel
