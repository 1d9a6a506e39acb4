"""Backward of the mel front-end: dL/d(audio) from spk_mel_spectrogram_backward, through ``meldataset.mel_spectrogram``.

* CPU: the fp64 torch restatement of the reference's ops (mel_grad_oracle.mel_spectrogram_torch) equals the numpy
  oracle and the golden mel, and the numpy statement of the kernels' algorithm (mel_backward_np) equals fp64 autograd.
* Host: argument errors of the C entry point come back as SPK_EINVAL before any CUDA call.
* GPU: ``y.grad`` against fp64 autograd (relative L2) at every shape of the CPU check, next to the error of the same
  ops in torch fp32 on the same GPU; determinism, exact zeros under the clamp, dtypes and shapes; and a waveform
  generator trained through a mel L1 loss and a frozen GE2E critic, against the same graph in fp64.

Bounds follow test_gpu_stage_parity.py: about 5x the worst value measured on a B200 (1000 W power limit), written
beside each bound.  Each test prints its figures as one JSON line.
"""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from mel_grad_oracle import mel_backward_np, mel_spectrogram_torch
from oracle import mel_oracle
from oracle.make_golden_mel import make_audio

DEV = "cuda"
SOUND = dict(n_fft=1024, num_mels=80, sampling_rate=22050, hop_size=256, win_size=1024, fmin=0, fmax=None)

NP_REL = 1e-12            # numpy algorithm against fp64 autograd (worst measured on the CPU: 2.1e-14)
GRAD_REL = 2.5e-5         # 4.4e-6   y.grad against fp64 autograd, relative L2, random cotangent (torch fp32 on the
                          #          same GPU, the reference's own arithmetic: 1.0e-5)
E2E_REL = 1e-3            # 4.4e-5   the project's relative gradient tolerance against fp64 (generator, no gate forcing)

# (id, audio (seed, batch, samples), n_fft, hop, win, n_mels, sampling rate, fmin, fmax)
SHAPES = [
    ("golden0", (1, 3, 256 * 40), 1024, 256, 1024, 80, 22050, 0.0, None),
    ("nfft512", (9, 2, 5000), 512, 128, 512, 80, 22050, 0.0, None),
    ("nfft2048", (9, 2, 5000), 2048, 512, 2048, 80, 22050, 0.0, None),
    ("win1200", (9, 2, 5000), 2048, 512, 1200, 80, 22050, 0.0, None),
    ("fmin50_fmax7000", (9, 2, 5000), 1024, 256, 1024, 40, 16000, 50.0, 7000.0),
    ("hop300", (9, 2, 5000), 1024, 300, 800, 80, 22050, 0.0, None),
    ("shortest", (9, 2, 385), 1024, 256, 1024, 80, 22050, 0.0, None),     # samples = pad + 1: both reflections
]
IDS = [s[0] for s in SHAPES]


def _record(kind, **kw):
    print("mel grad:", json.dumps(dict(kind=kind, **kw)))


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm())


def _args(shape):
    _, _, n_fft, hop, win, mels, sr, fmin, fmax = shape
    return (n_fft, mels, sr, hop, win, fmin, fmax)


def _audio(shape):
    return make_audio(*shape[1])


def _fp64_grad(y, g, args):
    """(log-mel, dL/dy) of the reference's ops in fp64 under the cotangent g."""
    yt = torch.as_tensor(y).double().requires_grad_(True)
    mel = mel_spectrogram_torch(yt, *args)
    mel.backward(torch.as_tensor(g).to(mel.device, torch.float64))
    return mel.detach(), yt.grad


def _cotangent(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64).float()


# ---- CPU: the references
def test_torch_restatement_matches_the_numpy_oracle_and_the_golden_mel(golden_dir):
    g = np.load(os.path.join(golden_dir, "mel.npz"))
    worst_np = worst_golden = 0.0
    for i in range(int(g["num_cases"])):
        seed, batch, samples = [int(v) for v in g["case%d_meta" % i]]
        y = make_audio(seed, batch, samples)
        got = mel_spectrogram_torch(torch.as_tensor(y).double(), **SOUND).numpy()
        worst_np = max(worst_np, float(np.abs(got - mel_oracle.mel_spectrogram_np(y, **SOUND)).max()))
        worst_golden = max(worst_golden, float(np.abs(got - g["case%d_mel" % i]).max()))
    for shape in SHAPES[1:]:
        y = _audio(shape)
        got = mel_spectrogram_torch(torch.as_tensor(y).double(), *_args(shape)).numpy()
        worst_np = max(worst_np, float(np.abs(got - mel_oracle.mel_spectrogram_np(y, *_args(shape))).max()))
    _record("torch_restatement", max_abs_np=worst_np, max_abs_golden=worst_golden)
    assert worst_np <= 1e-10, worst_np
    assert worst_golden <= 1e-4, worst_golden          # the bound test_mel_frontend.py gives the numpy oracle


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_numpy_backward_matches_fp64_autograd(shape):
    y = _audio(shape)
    args = _args(shape)
    g = _cotangent(mel_spectrogram_torch(torch.as_tensor(y).double(), *args).shape, 11)
    _, want = _fp64_grad(y, g, args)
    got = mel_backward_np(y, g.numpy(), *args)
    err = _rel(got, want)
    _record("numpy_backward", shape=shape[0], err=err)
    assert got.shape == y.shape
    assert err <= NP_REL, err


def test_numpy_backward_of_silence_is_exactly_zero():
    y = np.zeros((2, 4000), dtype=np.float32)
    args = _args(SHAPES[0])
    mel = mel_spectrogram_torch(torch.as_tensor(y).double(), *args)
    assert float((mel - np.log(1e-5)).abs().max()) <= 1e-12       # every band is clamped
    g = _cotangent(mel.shape, 12)
    _, want = _fp64_grad(y, g, args)
    got = mel_backward_np(y, g.numpy(), *args)
    assert not want.any() and not got.any()


# ---- host: argument errors come back before any CUDA call
def test_backward_rejects_bad_arguments_without_a_device():
    from speaker_embedding_torch_b200 import _native as N
    if not os.path.exists(N.LIB_PATH):
        N.build()
    L = N.lib()
    fake = ctypes.c_void_p(4096)          # never dereferenced: the checks come first
    need = L.spk_mel_backward_workspace_bytes(3, 10240, 1024, 256)
    assert need == 3 * 40 * 1024 * 4
    assert L.spk_mel_backward_workspace_bytes(3, 10240, 1024, 2048) == 0      # hop > n_fft
    assert L.spk_mel_backward_workspace_bytes(3, 10240, 1000, 256) == 0

    def call(d_mel=fake, batch=3, samples=10240, n_fft=1024, hop=256, win=1024, n_mels=80, ws_bytes=need):
        return L.spk_mel_spectrogram_backward(fake, d_mel, batch, samples, n_fft, hop, win, fake, fake, fake, n_mels,
                                              fake, fake, ws_bytes, None)

    for kw, text in ((dict(d_mel=None), b"null argument"), (dict(n_fft=1000), b"n_fft 1000"),
                     (dict(hop=2048, n_fft=1024), b"hop 2048"), (dict(ws_bytes=need - 1), b"workspace"),
                     (dict(samples=384), b"cannot be reflect-padded"), (dict(n_mels=300), b"n_mels"),
                     (dict(win=2048), b"win")):
        assert call(**kw) == -22, kw
        assert text in L.spk_last_error(), (kw, L.spk_last_error())


# ---- GPU: parity
def _library_grad(y, g, args, **kw):
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    yt = torch.as_tensor(y).to(DEV).requires_grad_(True)
    mel = mel_spectrogram(yt, *args, **kw)
    mel.backward(g.to(DEV, mel.dtype))
    torch.cuda.synchronize()
    return mel.detach(), yt.grad


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_audio_grad_matches_fp64_autograd(shape):
    y = _audio(shape)
    args = _args(shape)
    mel64 = mel_spectrogram_torch(torch.as_tensor(y).double(), *args)
    g = _cotangent(mel64.shape, 13)
    _, want = _fp64_grad(y, g, args)
    mel, got = _library_grad(y, g, args)
    err = _rel(got, want)
    # the reference's own arithmetic: the same ops in torch fp32 on the same GPU
    y32 = torch.as_tensor(y).to(DEV).requires_grad_(True)
    mel_spectrogram_torch(y32, *args).backward(g.to(DEV))
    err_torch = _rel(y32.grad, want)
    _record("parity", shape=shape[0], err=err, err_torch_fp32_cuda=err_torch,
            mel_max_abs=float((mel.double().cpu() - mel64).abs().max()))
    assert got.shape == y.shape and got.dtype == torch.float32
    assert err <= GRAD_REL, err


# ---- GPU: contracts
@pytest.mark.gpu
def test_audio_grad_is_deterministic_and_the_log_mel_does_not_change():
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    y = _audio(SHAPES[0])
    args = _args(SHAPES[0])
    with torch.no_grad():
        plain = mel_spectrogram(torch.as_tensor(y).to(DEV), *args)
    g = _cotangent(plain.shape, 14)
    mel1, g1 = _library_grad(y, g, args)
    mel2, g2 = _library_grad(y, g, args)
    assert torch.equal(mel1, plain) and torch.equal(mel2, plain)
    assert torch.equal(g1, g2)
    assert plain.grad_fn is None
    assert mel_spectrogram(torch.as_tensor(y).to(DEV), *args).grad_fn is None      # no requires_grad
    yt = torch.as_tensor(y).to(DEV).requires_grad_(True)
    with torch.no_grad():
        assert mel_spectrogram(yt, *args).grad_fn is None


@pytest.mark.gpu
def test_clamped_frames_give_an_exactly_zero_gradient():
    args = _args(SHAPES[0])
    n_fft, hop = SHAPES[0][2], SHAPES[0][3]
    pad = (n_fft - hop) // 2
    y = make_audio(21, 3, 256 * 40)
    y[1] = 0.0                                                  # silent
    y[2, 5000:] = 0.0                                           # half silent
    mel64 = mel_spectrogram_torch(torch.as_tensor(y).double(), *args)
    g = _cotangent(mel64.shape, 15)
    _, got = _library_grad(y, g, args)
    _, want = _fp64_grad(y, g, args)
    got = got.cpu()
    assert not got[1].any()
    # samples of row 2 whose every covering frame (of the sample and of its mirror images) is all-zero audio
    yp = np.pad(y[2].astype(np.float64), (pad, pad), mode="reflect")
    frames = mel64.shape[2]
    silent = np.array([not yp[f * hop:f * hop + n_fft].any() for f in range(frames)])
    covered = np.zeros(yp.size, dtype=bool)                     # padded positions covered by a non-silent frame
    for f in np.nonzero(~silent)[0]:
        covered[f * hop:f * hop + n_fft] = True
    S = y.shape[1]

    def hit(p):
        return 0 <= p < covered.size and covered[p]

    zero = np.array([not hit(pad + s) and not (1 <= s <= pad and hit(pad - s))
                     and not (s <= S - 2 and hit(pad + 2 * (S - 1) - s)) for s in range(S)])
    _record("clamped", zero_samples=int(zero.sum()), nonzero_in_zero_set=int(got[2][torch.as_tensor(zero)].ne(0).sum()),
            err_row2=_rel(got[2], want[2]))
    assert zero.sum() == 4224                                   # samples 6016 .. 10239
    assert not got[2][torch.as_tensor(zero)].any()
    assert not want[2][torch.as_tensor(zero)].any()
    assert _rel(got[2], want[2]) <= GRAD_REL


@pytest.mark.gpu
def test_gradient_shape_and_dtype_follow_the_input():
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    y = torch.as_tensor(_audio(SHAPES[0]))
    args = _args(SHAPES[0])
    ref_mel, ref = _library_grad(y.numpy(), _cotangent((3, 80, 40), 16), args)
    one = y[0].to(DEV).requires_grad_(True)                     # 1-D
    mel = mel_spectrogram(one, *args)
    assert mel.shape == (1, 80, 40)
    mel.backward(_cotangent((3, 80, 40), 16)[:1].to(DEV))
    assert one.grad.shape == one.shape and one.grad.dtype == torch.float32
    assert torch.equal(one.grad, ref[0])
    for dt in (torch.float16, torch.bfloat16):
        yl = y.to(DEV, dt).requires_grad_(True)
        mel = mel_spectrogram(yl, *args)
        assert mel.dtype == torch.float32
        mel.sum().backward()
        assert yl.grad.shape == yl.shape and yl.grad.dtype == dt
        assert torch.isfinite(yl.grad.float()).all() and yl.grad.float().abs().sum() > 0
    yh = y.to(DEV).requires_grad_(True)
    g = _cotangent((3, 80, 40), 16)
    mel = mel_spectrogram(yh, *args, out_dtype=torch.float16)
    assert mel.dtype == torch.float16 and torch.equal(mel, ref_mel.half())
    mel.backward(g.to(DEV).half())
    assert yh.grad.dtype == torch.float32
    _, ref_h = _library_grad(y.numpy(), g.half().float(), args)  # the fp16 cotangent, upcast
    assert torch.equal(yh.grad, ref_h)


@pytest.mark.gpu
def test_hop_longer_than_n_fft_has_no_backward():
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    y = torch.as_tensor(make_audio(3, 1, 8000)).to(DEV).requires_grad_(True)
    mel = mel_spectrogram(y, 512, 40, 16000, 600, 512, 0.0, None)
    with pytest.raises(RuntimeError, match="hop 600"):
        mel.sum().backward()


# ---- GPU: end to end, a waveform generator trained through a mel L1 loss and a frozen critic
@pytest.mark.gpu
def test_generator_gradient_through_the_front_end_matches_fp64():
    from oracle import ge2e_oracle as O
    from speaker_embedding_torch_b200.Modules import Overlapped_Slices
    from speaker_embedding_torch_b200.meldataset import mel_spectrogram
    from test_gpu_stage_parity import _dstate, _model
    U, S, L, hop, zdim = 4, 5, 64, 32, 16
    W = S * hop + (L - hop)                                     # 192 mel frames
    samples = W * 256
    m, state = _model(90)
    m.eval()
    for p in m.parameters():
        p.requires_grad_(False)
    torch.manual_seed(91)
    gen = torch.nn.Linear(zdim, samples).to(DEV)
    z = torch.randn(U, zdim, device=DEV)
    target_d = torch.nn.functional.normalize(torch.randn(U, 256, device=DEV), dim=1)
    target_mel = mel_spectrogram_torch(torch.as_tensor(make_audio(92, U, samples)).to(DEV, torch.float64), **SOUND)

    def graph(g, front, encoder, zz, td, tm):
        mel = front(g(zz))
        l1 = (mel - tm).abs().mean()
        d = encoder(Overlapped_Slices(mel, L, L - hop))
        return l1 + (1.0 - torch.nn.functional.cosine_similarity(d, td, dim=1)).mean()

    loss = graph(gen, lambda y: mel_spectrogram(y, **SOUND), lambda x: m(x, S), z, target_d, target_mel.float())
    loss.backward()
    gen64 = torch.nn.Linear(zdim, samples).to(DEV, torch.float64)
    with torch.no_grad():
        gen64.weight.copy_(gen.weight.double())
        gen64.bias.copy_(gen.bias.double())
    st = _dstate(state)
    loss64 = graph(gen64, lambda y: mel_spectrogram_torch(y, **SOUND),
                   lambda x: O.encoder_forward(st, x, samples=S, layers=3), z.double(), target_d.double(), target_mel)
    loss64.backward()
    err_w = _rel(gen.weight.grad, gen64.weight.grad)
    err_b = _rel(gen.bias.grad, gen64.bias.grad)
    _record("generator", loss=loss.item(), loss64=loss64.item(), err_w=err_w, err_b=err_b)
    assert err_w <= E2E_REL and err_b <= E2E_REL, (err_w, err_b)
    assert all(p.grad is None for p in m.parameters())
