"""Mel front-end on the device: drop-in for ``meldataset.mel_spectrogram`` (meldataset.py:73-96).

Same call signature as the reference; ``y`` must be a CUDA tensor ``[B, samples]`` in [-1, 1] (there is no CPU path).
One kernel (``spk_mel_spectrogram``) does reflect padding, the STFT, the magnitude, the mel projection and the log;
the triangular mel filters are built once per configuration on the host (``mel_filters``, the algorithm of
``librosa.filters.mel`` with its defaults -- librosa itself is not a dependency) and cached on the device.

Like the reference's torch ops, the function is differentiable with respect to ``y``: with grad mode on and
``y.requires_grad``, autograd's backward calls ``spk_mel_spectrogram_backward``, which recomputes the forward from the
saved audio and returns dL/dy (the mel basis and the window are constants, as in the reference).  This is what a mel L1
loss on generated audio, or a speaker-consistency loss through a frozen encoder, needs.  Without grad the call is the
same single launch and returns a tensor without ``grad_fn``.

    mel = mel_spectrogram(audio.cuda(), 1024, 80, 22050, 256, 1024, 0, None)        # [B, 80, frames] fp32
    dvec = model(mel_spectrogram(...)[:, :, :T], samples)                           # wav -> d-vector without the host
    loss = (mel_spectrogram(generated, ...) - target_mel).abs().mean(); loss.backward()   # generated.grad
"""
import math

import numpy as np
import torch

from . import _native as N

_FILTERS = {}


def _hz_to_mel(f):
    f = np.asarray(f, dtype=np.float64)
    f_sp = 200.0 / 3
    min_log_hz, logstep = 1000.0, math.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_hz / f_sp + np.log(np.maximum(f, 1e-10) / min_log_hz) / logstep, f / f_sp)


def _mel_to_hz(m):
    m = np.asarray(m, dtype=np.float64)
    f_sp = 200.0 / 3
    min_log_hz, logstep = 1000.0, math.log(6.4) / 27.0
    min_log_mel = min_log_hz / f_sp
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_filters(sampling_rate, n_fft, num_mels, fmin=0.0, fmax=None):
    """Slaney-scale, area-normalised triangular filters [num_mels, n_fft // 2 + 1] fp32 (``librosa.filters.mel``
    with ``htk=False, norm='slaney'``, what meldataset.py:81 asks for)."""
    fmax = sampling_rate / 2.0 if fmax is None else fmax
    fftfreqs = np.linspace(0.0, sampling_rate / 2.0, 1 + n_fft // 2)
    mel_f = _mel_to_hz(np.linspace(_hz_to_mel(fmin), _hz_to_mel(fmax), num_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fftfreqs[None, :]
    weights = np.zeros((num_mels, 1 + n_fft // 2))
    for i in range(num_mels):
        weights[i] = np.maximum(0.0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    weights *= (2.0 / (mel_f[2:num_mels + 2] - mel_f[:num_mels]))[:, None]
    return weights.astype(np.float32)


def _device_filters(key, device):
    """-> (basis [n_mels, bins] fp32, ranges [n_mels][2], bin_ranges [bins][2]) on ``device``: the [first, last + 1)
    non-zero bin of every filter, and the [first, last + 1) filter with a non-zero weight at every bin."""
    hit = _FILTERS.get((key, device))
    if hit is None:
        basis = mel_filters(*key)
        ranges = np.zeros((basis.shape[0], 2), dtype=np.int32)
        for m, row in enumerate(basis):
            nz = np.nonzero(row)[0]
            ranges[m] = (nz[0], nz[-1] + 1) if nz.size else (0, 0)
        bin_ranges = np.zeros((basis.shape[1], 2), dtype=np.int32)
        for k, col in enumerate(basis.T):
            nz = np.nonzero(col)[0]
            bin_ranges[k] = (nz[0], nz[-1] + 1) if nz.size else (0, 0)
        hit = tuple(torch.from_numpy(a).to(device) for a in (basis, ranges, bin_ranges))
        _FILTERS[(key, device)] = hit
    return hit


def _forward(y, n_fft, num_mels, hop_size, win_size, filters, half):
    batch, samples = y.shape
    frames = N.lib().spk_mel_frames(samples, n_fft, hop_size)
    out = torch.empty((batch, num_mels, frames), dtype=torch.float16 if half else torch.float32, device=y.device)
    with torch.cuda.device(y.device):
        N.check(N.lib().spk_mel_spectrogram(N.ptr(y), batch, samples, n_fft, hop_size, win_size, N.ptr(filters[0]),
                                            N.ptr(filters[1]), num_mels, N.ptr(out), int(half),
                                            N.stream_ptr(y.device)), "spk_mel_spectrogram")
    return out


class _MelSpectrogram(torch.autograd.Function):
    """The forward kernel, with ``spk_mel_spectrogram_backward`` as its backward.  Saves only the fp32 audio."""

    @staticmethod
    def forward(ctx, y, n_fft, num_mels, hop_size, win_size, filters, half):
        ctx.save_for_backward(y)
        ctx.cfg = (n_fft, num_mels, hop_size, win_size, filters)
        return _forward(y, n_fft, num_mels, hop_size, win_size, filters, half)

    @staticmethod
    def backward(ctx, d_mel):
        (y,) = ctx.saved_tensors
        n_fft, num_mels, hop_size, win_size, (basis, ranges, bin_ranges) = ctx.cfg
        batch, samples = y.shape
        d_mel = d_mel.contiguous().float()
        d_audio = torch.empty_like(y)
        L = N.lib()
        nbytes = L.spk_mel_backward_workspace_bytes(batch, samples, n_fft, hop_size)
        # a shape the backward rejects sizes to 0 bytes; the call below then says why
        ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=y.device)
        with torch.cuda.device(y.device):
            N.check(L.spk_mel_spectrogram_backward(N.ptr(y), N.ptr(d_mel), batch, samples, n_fft, hop_size, win_size,
                                                   N.ptr(basis), N.ptr(ranges), N.ptr(bin_ranges), num_mels,
                                                   N.ptr(d_audio), N.ptr(ws), ws.numel(), N.stream_ptr(y.device)),
                    "spk_mel_spectrogram_backward")
        return d_audio, None, None, None, None, None, None


def mel_spectrogram(y, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax, center=False, out_dtype=None):
    """log-mel spectrogram [B, num_mels, frames]; ``out_dtype=torch.float16`` stores it the way the reference stores its
    patterns (Pattern_Generator.py:123).  Differentiable with respect to ``y`` (any float dtype, 1-D or 2-D: the
    gradient comes back in ``y``'s shape and dtype)."""
    if center:
        raise RuntimeError("mel_spectrogram: center=True is not what the reference uses and is not implemented")
    N.require_cuda(y, "y")
    if y.dim() == 1:
        y = y.unsqueeze(0)
    if y.dim() != 2:
        raise RuntimeError("y must be [B, samples], got %s" % (tuple(y.shape),))
    y = y.contiguous().float()
    batch, samples = y.shape
    n_fft, num_mels, hop_size, win_size = int(n_fft), int(num_mels), int(hop_size), int(win_size)
    frames = N.lib().spk_mel_frames(samples, n_fft, hop_size)
    if frames < 1 or samples <= (n_fft - hop_size) // 2:
        raise RuntimeError("mel_spectrogram: %d samples are too few for n_fft %d / hop %d" % (samples, n_fft, hop_size))
    filters = _device_filters((int(sampling_rate), n_fft, num_mels, float(fmin),
                               None if fmax is None else float(fmax)), y.device)
    half = out_dtype == torch.float16
    if torch.is_grad_enabled() and y.requires_grad:
        return _MelSpectrogram.apply(y, n_fft, num_mels, hop_size, win_size, filters, half)
    return _forward(y, n_fft, num_mels, hop_size, win_size, filters, half)
