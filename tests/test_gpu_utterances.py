"""Variable-length utterances: the slicing rule (Modules.utterance_slices), the segmented head, the ragged input-gradient
fold (spk_encoder_forward_segments / spk_encoder_backward_segments) and GE2E.embed_utterances.

* Equal lengths on the hop grid give exactly the slices of embed_windows, and the d-vectors bit for bit.
* Uniform segments are spk_encoder_forward_ragged at samples = S: the same d-vectors and input gradient bit for bit.
* Mixed lengths (1, 2, 3 frames, T, T + 1, long ones) meet the fp64 oracle, which runs ge2e_oracle.encoder_forward on
  the np.pad / cropped slices and restates the segmented head here.
* Gradients are checked against the fp64 oracle forced onto the library's own ReLU gates and dropout masks, as in
  test_gpu_input_grad.py, at the same GRAD_REL bound.
Each GPU test prints its figures as one JSON line.
"""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from oracle import ge2e_oracle as O
from oracle import synth

D, F, H = 256, 1024, 4
DEV = "cuda"
GRAD_REL = 1e-4           # bound of test_gpu_input_grad.py (input and parameter gradients against gate-forced fp64)
COS_MIN = 0.9999          # d-vectors in eval precision (one fp16 plane) against fp64
FOLD_REL = 1e-6           # the fold against torch autograd through an index gather (summation order only)
PARAM_REORDER = 2.5e-6    # parameter gradients: fp32 atomics in another order (test_gpu_input_grad.py); the weight
                          # gradients are split-K GEMMs that meet in fp32 atomics, so not even the same call twice is
                          # bit-identical there, and two calls are compared to this bound instead of bit for bit
E2E_REL = 1e-3            # the project's relative gradient tolerance against fp64 without gate forcing


def _record(kind, **kw):
    print("utterances:", json.dumps(dict(kind=kind, **kw)))


# ------------------------------------------------------------------------------------------------
# host: the slicing rule
def _rule(L, T, O_):
    h = T - O_
    if L <= T:
        return [0]
    S = -(-(L - T) // h) + 1
    return [min(s * h, L - T) for s in range(S)]


@pytest.mark.parametrize("T,O_", [(160, 80), (64, 32), (64, 0), (300, 100), (7, 6)])
def test_utterance_slices_follow_the_rule(T, O_):
    from speaker_embedding_torch_b200.Modules import utterance_slices
    h = T - O_
    lengths = [1, 2, 3, T - 1, T, T + 1, T + h, 4 * h + T, 5000]
    lengths = [L for L in lengths if L >= 1]
    table, seg = utterance_slices(lengths, T, O_)
    assert table.dtype == torch.int32 and seg.dtype == torch.int32
    start, rows = 0, 0
    for u, L in enumerate(lengths):
        offs = _rule(L, T, O_)
        assert int(seg[u]) == rows and int(seg[u + 1]) == rows + len(offs)
        for k, off in enumerate(offs):
            assert table[rows + k].tolist() == [start, L, off]
        rows += len(offs)
        start += L
    assert int(seg[-1]) == table.size(0)
    starts = [7 * u for u in range(len(lengths))]
    table2, seg2 = utterance_slices(lengths, T, O_, starts)
    assert torch.equal(seg2, seg) and table2[:, 0].tolist() == [starts[int(torch.searchsorted(seg[1:], r, right=True))]
                                                              for r in range(table.size(0))]


@pytest.mark.parametrize("T,O_,S", [(160, 80, 5), (64, 32, 3), (50, 0, 4)])
def test_aligned_lengths_give_the_slices_of_overlapped_slices(T, O_, S):
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices, utterance_slices
    W = S * (T - O_) + O_
    table, seg = utterance_slices([W, W], T, O_)
    windows = torch.arange(W, dtype=torch.float32).view(1, 1, W).repeat(2, 1, 1)
    offs = Overlapped_Slices(windows, T, O_)[:, 0, 0].long().tolist()
    assert table[:, 2].tolist() == offs and seg.tolist() == [0, S, 2 * S]


# ---- host: argument errors come back before any CUDA call
def test_segment_entry_points_reject_bad_arguments_without_a_device():
    from speaker_embedding_torch_b200 import _native as N
    if not os.path.exists(N.LIB_PATH):
        N.build()
    L = N.lib()
    cfg = N.EncoderConfig(80, 256, 4, 1024, 3, 1024, 0.1, 0.1)
    w, g = N.EncoderParams(), N.EncoderParams()
    fake = ctypes.c_void_p(4096)          # never dereferenced: the checks come first
    good = N.MelRagged(4096, 0, 100, 4096)
    tail = (ctypes.c_uint64(0),)

    def fwd(mel, seg, U, B):
        return L.spk_encoder_forward_segments(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(mel), seg, U, B, 64, 1,
                                              0, *tail, fake, fake, 1 << 20, 0, None)

    def bwd(mel, seg, U, B, grads=True, d_data=fake):
        return L.spk_encoder_backward_segments(ctypes.byref(cfg), ctypes.byref(w), ctypes.byref(g) if grads else None,
                                               ctypes.byref(mel), seg, U, d_data, fake, B, 64, 2, 0, *tail, fake,
                                               1 << 20, None)

    cases = [
        ((good, fake, 0, 4), b"utterances"),                  # utterances < 1
        ((good, fake, 5, 4), b"utterances"),                  # batch < utterances
        ((good, None, 3, 4), b"not a multiple"),              # segments NULL, batch % utterances != 0
        ((N.MelRagged(0, 0, 100, 4096), fake, 2, 4), b"ragged mel"),     # no data
        ((N.MelRagged(4096, 0, 100, 0), fake, 2, 4), b"ragged mel"),     # no table
        ((N.MelRagged(4096, 2, 100, 4096), fake, 2, 4), b"ragged mel"),  # bad dtype
    ]
    for args, msg in cases:
        assert fwd(*args) == -22, args
        assert msg in L.spk_last_error(), (args, L.spk_last_error())
        assert bwd(*args) == -22, args
        assert msg in L.spk_last_error(), (args, L.spk_last_error())
    assert bwd(good, fake, 2, 4, grads=False, d_data=None) == -22
    assert b"both NULL" in L.spk_last_error()


# ---- host: RaggedMel checks its segments, and refuses a gradient it could not fold
def test_ragged_mel_rejects_bad_segments_and_overlapping_spans():
    from speaker_embedding_torch_b200 import GE2E
    from speaker_embedding_torch_b200.Arg_Parser import default_hyper_parameters
    from speaker_embedding_torch_b200.Datasets import RaggedMel
    data = torch.zeros(80, 100)
    table = torch.tensor([[0, 40, 0], [0, 40, 0], [40, 60, 0]], dtype=torch.int32)
    for bad in ([0, 2], [1, 2, 3], [0, 2, 2, 3], [0, 3, 2, 3], [0, 1, 2, 4]):
        with pytest.raises(RuntimeError, match="segments"):
            RaggedMel(data, table, 64, torch.tensor(bad, dtype=torch.int32))
    ok = RaggedMel(data, table, 64, torch.tensor([0, 2, 3], dtype=torch.int32))
    assert ok.utterances == 2 and ok.spans_disjoint()
    # slices 0 and 1 share columns: fine inside one utterance, not across two
    assert not RaggedMel(data, table, 64, torch.tensor([0, 1, 3], dtype=torch.int32)).spans_disjoint()
    assert not RaggedMel(data, table, 64).spans_disjoint(1)
    m = GE2E(default_hyper_parameters())
    for p in m.parameters():
        p.requires_grad_(False)
    over = RaggedMel(data.clone().requires_grad_(True), table, 64, torch.tensor([0, 1, 3], dtype=torch.int32))
    with pytest.raises(RuntimeError, match="overlap"):
        m(over)


# ------------------------------------------------------------------------------------------------
# GPU helpers
def _model(seed):
    from test_gpu_stage_parity import _model as model
    return model(seed)


def _gather_index(table, frames):
    """Column index [B, T] of every slice frame in the ragged array: the crop / reflect-pad of mel_pack_ragged."""
    idx = []
    for start, length, offset in table.tolist():
        t = np.arange(frames)
        if length > frames:
            col = offset + t
        else:
            col = np.pad(np.arange(length), [int(np.floor((frames - length) / 2)),
                                             int(np.ceil((frames - length) / 2))], mode="reflect")
        idx.append(start + col)
    return torch.as_tensor(np.stack(idx), dtype=torch.int64)


def _dense(data, table, frames):
    """[B, Mel, T] slices of data by index gather (differentiable: autograd folds the gradient back)."""
    idx = _gather_index(table, frames).to(data.device)
    return data[:, idx].permute(1, 0, 2)


def _seg_head(state, h_last, seg):
    """The segmented head in fp64: LayerNorm of each slice's t = 0 row, mean per segment, projection, L2 norm."""
    h0 = O._layer_norm(h_last[:, 0, :], state["transformer.norm.weight"], state["transformer.norm.bias"])
    e = torch.stack([h0[int(seg[u]):int(seg[u + 1])].mean(dim=0) for u in range(len(seg) - 1)])
    e = e @ state["projection.weight"][:, :, 0].t() + state["projection.bias"]
    return e / e.norm(p=2, dim=1, keepdim=True).clamp_min(O.NORMALIZE_EPS)


def _oracle(state, data, table, seg, frames, cotangent=None, drop_scales=None, relu_masks=None):
    from test_gpu_stage_parity import _dstate
    st = {k: v.clone().requires_grad_(not k.endswith(".pe")) for k, v in _dstate(state).items()}
    x = data.detach().double().clone().requires_grad_(True)
    _, inter = O.encoder_forward(st, _dense(x, table, frames), layers=3, return_intermediates=True,
                                 drop_scales=drop_scales, relu_masks=relu_masks)
    d = _seg_head(st, inter["layer2"], seg)
    if cotangent is not None:
        d.backward(cotangent.double())
    return d.detach(), x.grad, {k: v.grad for k, v in st.items() if v.requires_grad}


def _cos_min(a, b):
    return float(torch.nn.functional.cosine_similarity(a.double(), b.double(), dim=1).min())


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _mels(seed, lengths):
    return [torch.as_tensor(synth.make_mel(seed + i, 1, L)[0]).to(DEV) for i, L in enumerate(lengths)]


# ---- 4: equal lengths on the hop grid: embed_windows bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("T,O_,S", [(160, 80, 5), (64, 32, 3)])
def test_equal_aligned_lengths_match_embed_windows_bit_for_bit(dtype, T, O_, S):
    m, _ = _model(101)
    m.eval()
    W = S * (T - O_) + O_
    windows = torch.as_tensor(synth.make_mel(3100 + T, 24, W)).to(DEV, dtype)
    with torch.no_grad():
        ref = m.embed_windows(windows, T, O_)
        got = m.embed_utterances(list(windows), T, O_)
        padded = m.embed_utterances(windows, T, O_, lengths=[W] * 24)
    _record("vs_embed_windows", T=T, S=S, dtype=str(dtype), max_abs=float((got - ref).abs().max()))
    assert torch.equal(got, ref)
    assert torch.equal(padded, ref)


# ---- 5: uniform segments are spk_encoder_forward_ragged at samples = S
@pytest.mark.gpu
@pytest.mark.parametrize("training", [False, True])
def test_uniform_segments_are_the_ragged_forward_with_samples(training):
    from speaker_embedding_torch_b200.Datasets import RaggedMel
    m, _ = _model(102)
    U, S, T = 6, 4, 48
    lengths = [300, 190, 260, 230, 48 * 4, 210]
    table = []
    start = 0
    rng = np.random.RandomState(3)
    for L in lengths:
        for _ in range(S):
            table.append([start, L, rng.randint(0, L - T)])
        start += L
    table = torch.tensor(table, dtype=torch.int32)
    seg = torch.arange(0, U * S + 1, S, dtype=torch.int32)
    data0 = torch.as_tensor(synth.make_mel(3200, 1, start)[0]).to(DEV)
    cot = torch.randn(U, D, generator=torch.Generator().manual_seed(4)).to(DEV)

    def run(with_segments):
        m.zero_grad(set_to_none=True)
        m.train(training)
        x = data0.clone().requires_grad_(True)
        r = RaggedMel(x, table, T, seg if with_segments else None).to(DEV)
        torch.manual_seed(55)
        d = m(r) if with_segments else m(r, S)
        d.backward(cot)
        torch.cuda.synchronize()
        return d.detach(), x.grad, {n: p.grad.clone() for n, p in m.named_parameters()}

    d0, g0, p0 = run(False)
    d1, g1, p1 = run(True)
    worst = max(float((p1[n] - p0[n]).abs().max() / p0[n].abs().max().clamp_min(1e-30)) for n in p0)
    _record("uniform_segments", training=training, max_abs_grad=float((g1 - g0).abs().max()), param_worst=worst)
    assert torch.equal(d1, d0)
    assert torch.equal(g1, g0)
    assert worst <= PARAM_REORDER, worst       # fp32 atomics of the weight gradients: order only


# ---- 6: mixed lengths against fp64; an utterance alone equals the same utterance in a batch
MIXED = [1, 2, 3, 63, 64, 65, 159, 160, 161, 299, 300, 301, 777, 2000]


@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 160, 300])
def test_mixed_lengths_match_fp64_and_do_not_depend_on_the_batch(T):
    from speaker_embedding_torch_b200.Modules import utterance_slices
    m, state = _model(103)
    m.eval()
    O_ = T // 2
    mels = _mels(3300 + T, MIXED)
    with torch.no_grad():
        got = m.embed_utterances(mels, T, O_)
        alone = torch.cat([m.embed_utterances([x], T, O_) for x in mels])
    table, seg = utterance_slices(MIXED, T, O_)
    data = torch.cat(mels, dim=1)
    ref, _, _ = _oracle(state, data, table, seg, T)
    cos = _cos_min(got, ref)
    diff = float((alone - got).abs().max())
    _record("mixed_fp64", T=T, slices=int(seg[-1]), cos_min=cos, alone_vs_batch=diff)
    assert cos >= COS_MIN, cos
    assert torch.equal(alone, got), diff      # no kernel choice that depends on the batch changes a d-vector


# ---- 7: input and parameter gradients against the gate-forced fp64 oracle
@pytest.mark.gpu
@pytest.mark.parametrize("T,training,prune", [(64, False, 1), (64, True, 1), (64, True, 0), (160, False, 0),
                                              (300, False, 1)])
def test_gradients_match_gate_forced_fp64(T, training, prune):
    from speaker_embedding_torch_b200.Datasets import RaggedMel
    from speaker_embedding_torch_b200.Modules import utterance_slices
    from test_gpu_parity_full import _site_scales
    from test_gpu_stage_parity import _Options, _relu_masks
    lengths = [1, 3, T - 1, T, T + 1, 2 * T + 5, 3 * T]
    O_ = T // 2
    with _Options(prune_last_layer=prune):
        m, state = _model(104)
        m.train(training)
        m._debug_keep_ws = True
        data0 = torch.cat(_mels(3400 + T, lengths), dim=1)
        table, seg = utterance_slices(lengths, T, O_)
        B, U = table.size(0), len(lengths)
        cot = torch.randn(U, D, generator=torch.Generator().manual_seed(6)).to(DEV)
        x = data0.clone().requires_grad_(True)
        torch.manual_seed(4242)
        seed = int(torch.empty((), dtype=torch.int64).random_().item())      # what GE2E.forward draws
        torch.manual_seed(4242)
        d = m(RaggedMel(x, table, T, seg).to(DEV))
        d.backward(cot)
        torch.cuda.synchronize()
        masks = _relu_masks(m, B, T, prune)
        ds = None
        if training:
            ds, _ = _site_scales(seed, m._cfg.pe_dropout, m._cfg.dropout, B, T, H, 3, bool(prune), DEV)
            ds = {k: v.to(DEV) for k, v in ds.items()}
    _, g_ref, p_ref = _oracle(state, data0, table, seg, T, cot, ds, masks)
    err = _rel(x.grad, g_ref)
    perr = {}
    for n, p in m.named_parameters():
        r = p_ref[n]
        if n.endswith("in_proj_bias"):       # the K slice is zero (softmax is shift-invariant)
            perr[n] = float((torch.cat([p.grad[:D], p.grad[2 * D:]]).double() - torch.cat([r[:D], r[2 * D:]])).norm()
                            / torch.cat([r[:D], r[2 * D:]]).norm())
        else:
            perr[n] = _rel(p.grad, r)
    worst = max(perr.items(), key=lambda kv: kv[1])
    _record("grads_fp64", T=T, training=training, prune=prune, mel=err, param_worst=worst)
    assert err <= GRAD_REL, err
    assert worst[1] <= GRAD_REL, worst


# ---- 8: data.grad of a training-collater batch
@pytest.mark.gpu
@pytest.mark.parametrize("training", [False, True])
def test_collater_batch_data_grad_matches_autograd_through_a_gather(training):
    from speaker_embedding_torch_b200.Datasets import Collater
    from speaker_embedding_torch_b200 import _native as N
    np.random.seed(7)
    lengths = [30, 64, 65, 100, 12, 250, 1, 2, 80, 40, 64, 300]
    feats = [[(synth.make_mel(3500 + i, 1, L)[0].astype(np.float32), 0)] for i, L in enumerate(lengths)]
    batch = Collater(60, 90)(feats)
    T = batch.frames
    dense_host = batch.dense()
    target = torch.randn(len(lengths), D, generator=torch.Generator().manual_seed(8)).to(DEV)

    def loss_of(d):
        return (1.0 - torch.nn.functional.cosine_similarity(d, target, dim=1)).mean()

    def run(m, trainable, ragged, profile=False):
        for p in m.parameters():
            p.requires_grad_(trainable)
            p.grad = None
        m.train(training)
        x = batch.data.to(DEV).clone().requires_grad_(True)
        torch.manual_seed(77)
        if ragged:
            r = batch.to(DEV)
            r.data = x
            d = m(r)
        else:
            dense = _dense(x, batch.table, T)
            assert torch.equal(dense.detach().cpu(), dense_host)
            d = m(dense)
        rep = None
        if profile:
            torch.cuda.synchronize()
            N.prof_enable(True)
            N.prof_report()
        loss_of(d).backward()
        torch.cuda.synchronize()
        if profile:
            rep = N.prof_report()
            N.prof_enable(False)
        return d.detach(), x.grad, rep

    m, _ = _model(105)
    d_ref, g_ref, _ = run(m, True, False)
    d_a, g_a, rep_t = run(m, True, True, profile=True)
    _, g_b, _ = run(m, True, True)
    fresh, _ = _model(105)
    d_f, g_f, rep_f = run(fresh, False, True, profile=True)
    err = _rel(g_a, g_ref)
    _record("collater_fold", training=training, T=T, err=err, tags=sorted(t for t in rep_f if "fold" in t))
    assert torch.equal(d_a, d_ref)
    assert err <= FOLD_REL, err
    assert torch.equal(g_a, g_b)                 # no atomics in the fold
    assert torch.equal(g_f, g_a)                 # frozen critic: the same data path
    assert torch.equal(d_f, d_a)
    assert all(p.grad is None for p in fresh.parameters()) and fresh._arena is None
    assert not [t for t in rep_f if "wgrad" in t], sorted(rep_f)
    assert "mel_grad_fold" in rep_f and "mel_grad_fold" in rep_t


# ---- padded form: the same d-vectors and gradients as the list form; padding columns get zero
@pytest.mark.gpu
def test_padded_form_matches_the_list_form():
    m, _ = _model(106)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    lengths = [5, 64, 200, 97]
    mels = _mels(3600, lengths)
    Lmax = max(lengths)
    padded = torch.zeros(len(lengths), 80, Lmax, device=DEV)
    for u, x in enumerate(mels):
        padded[u, :, :x.size(1)] = x
    xs = [x.clone().requires_grad_(True) for x in mels]
    xp = padded.clone().requires_grad_(True)
    cot = torch.randn(len(lengths), D, generator=torch.Generator().manual_seed(9)).to(DEV)
    d_l = m.embed_utterances(xs, 64, 32)
    d_l.backward(cot)
    d_p = m.embed_utterances(xp, 64, 32, lengths=lengths)
    d_p.backward(cot)
    assert torch.equal(d_l, d_p)
    for u, L in enumerate(lengths):
        assert torch.equal(xp.grad[u, :, :L], xs[u].grad)
        assert not xp.grad[u, :, L:].any()


# ---- chunking: max_slices_per_call cuts the batch between utterances; the pieces are the calls on their own
def _chunks(seg, max_slices):
    """Utterance ranges of embed_utterances' chunking: whole utterances, at most max_slices slices (at least one)."""
    out, u0, U = [], 0, len(seg) - 1
    while u0 < U:
        u1 = u0 + 1
        while u1 < U and int(seg[u1 + 1]) - int(seg[u0]) <= max_slices:
            u1 += 1
        out.append((u0, u1))
        u0 = u1
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("max_slices", [1, 3, 7])
def test_chunked_calls_are_the_calls_of_each_chunk(max_slices):
    from speaker_embedding_torch_b200.Modules import utterance_slices
    m, _ = _model(107)
    m.eval()
    lengths = [5, 64, 200, 97, 1, 130, 64, 300]
    T, O_ = 64, 32
    mels = _mels(3700, lengths)
    _, seg = utterance_slices(lengths, T, O_)
    parts = _chunks(seg, max_slices)
    assert len(parts) > 1
    with torch.no_grad():
        whole = m.embed_utterances(mels, T, O_)
        m.max_slices_per_call = max_slices
        chunked = m.embed_utterances(mels, T, O_)
    assert torch.equal(chunked, whole)
    # differentiable (frozen critic): every chunk is one call, its own gradient scale included
    for p in m.parameters():
        p.requires_grad_(False)
    cot = torch.randn(len(lengths), D, generator=torch.Generator().manual_seed(11)).to(DEV)
    xs = [x.clone().requires_grad_(True) for x in mels]
    d = m.embed_utterances(xs, T, O_)
    d.backward(cot)
    for u0, u1 in parts:
        ys = [x.clone().requires_grad_(True) for x in mels[u0:u1]]
        dp = m.embed_utterances(ys, T, O_)
        dp.backward(cot[u0:u1])
        assert torch.equal(dp.detach(), d.detach()[u0:u1])
        for u in range(u0, u1):
            assert torch.equal(ys[u - u0].grad, xs[u].grad), (u0, u1, u)
    xp = torch.zeros(len(lengths), 80, max(lengths), device=DEV)
    for u, x in enumerate(mels):
        xp[u, :, :x.size(1)] = x
    xp.requires_grad_(True)
    m.embed_utterances(xp, T, O_, lengths=lengths).backward(cot)
    for u, L in enumerate(lengths):
        assert torch.equal(xp.grad[u, :, :L], xs[u].grad)
    _record("chunks", max_slices=max_slices, chunks=len(parts))


# ---- 9: a waveform generator trained through the mel front-end, embed_utterances and a cosine critic
@pytest.mark.gpu
def test_generator_through_mel_spectrogram_and_embed_utterances_matches_fp64():
    from mel_grad_oracle import mel_spectrogram_torch
    from speaker_embedding_torch_b200.Modules import utterance_slices
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    from test_gpu_stage_parity import _dstate
    SOUND = dict(n_fft=1024, num_mels=80, sampling_rate=22050, hop_size=256, win_size=1024, fmin=0, fmax=None)
    frames = [40, 64, 150, 230]                      # mel frames per waveform: short (padded) to long (4 slices)
    samples = [f * 256 for f in frames]
    T, O_, zdim = 64, 32, 16
    m, state = _model(108)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    torch.manual_seed(109)
    gen = torch.nn.Linear(zdim, max(samples)).to(DEV)
    with torch.no_grad():
        gen.weight.mul_(0.05)
    z = torch.randn(len(frames), zdim, device=DEV)
    target = torch.nn.functional.normalize(torch.randn(len(frames), D, device=DEV), dim=1)

    def waves(g, zz):
        y = torch.tanh(g(zz))
        return [y[u:u + 1, :n] for u, n in enumerate(samples)]

    def critic(d, t):
        return (1.0 - torch.nn.functional.cosine_similarity(d, t, dim=1)).mean()

    ys = waves(gen, z)
    for y in ys:
        y.retain_grad()
    mels = [mel_spectrogram(y, **SOUND)[0] for y in ys]
    assert [x.size(1) for x in mels] == frames
    loss = critic(m.embed_utterances(mels, T, O_), target)
    loss.backward()

    gen64 = torch.nn.Linear(zdim, max(samples)).to(DEV, torch.float64)
    with torch.no_grad():
        gen64.weight.copy_(gen.weight.double())
        gen64.bias.copy_(gen.bias.double())
    ys64 = waves(gen64, z.double())
    for y in ys64:
        y.retain_grad()
    data64 = torch.cat([mel_spectrogram_torch(y, **SOUND)[0] for y in ys64], dim=1)
    table, seg = utterance_slices(frames, T, O_)
    st = _dstate(state)
    _, inter = O.encoder_forward(st, _dense(data64, table, T), layers=3, return_intermediates=True)
    loss64 = critic(_seg_head(st, inter["layer2"], seg), target.double())
    loss64.backward()
    err_y = _rel(torch.cat([y.grad[0] for y in ys]), torch.cat([y.grad[0] for y in ys64]))
    err_w = _rel(gen.weight.grad, gen64.weight.grad)
    _record("generator", loss=float(loss), loss64=float(loss64), err_y=err_y, err_w=err_w)
    assert err_y <= E2E_REL and err_w <= E2E_REL, (err_y, err_w)
    assert all(p.grad is None for p in m.parameters())
