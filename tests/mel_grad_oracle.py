"""References for the backward of the mel front-end (test infrastructure; never imported by the product).

  * ``mel_spectrogram_torch`` restates the reference's ``mel_spectrogram`` (meldataset.py:73-96) with the same torch
    ops -- ``F.pad`` reflect, ``torch.stft`` (center=False), ``sqrt(re^2 + im^2 + 1e-9)``, a matmul with the mel basis,
    ``log(clamp(., 1e-5))`` -- in whatever dtype and on whatever device ``y`` has.  In fp64, autograd through it is the
    reference gradient; in fp32 on the GPU it is the reference's own arithmetic.
  * ``mel_backward_np`` is the algorithm of the CUDA backward (csrc/melspec.cu, ``melspec_bwd_kernel`` and
    ``melspec_gather_kernel``) in numpy fp64: recompute the frame, gate the clamp, project back through the filters,
    take the adjoint of the real-FFT unpack and run the inverse N/2-point complex FFT, overlap-add, fold the reflect
    padding.  It lets the algorithm be checked against autograd without a GPU.
The existing ``oracle/mel_oracle.py`` (``mel_spectrogram_np``, ``mel_filterbank``) is the forward reference both use.
"""
import numpy as np
import torch

from oracle import mel_oracle


def _window_np(n_fft, win_size):
    n = np.arange(win_size)
    window = 0.5 - 0.5 * np.cos(2.0 * np.pi * n / win_size)          # periodic Hann (torch.hann_window)
    left = (n_fft - win_size) // 2                                   # torch.stft centres a short window in n_fft
    return np.pad(window, [left, n_fft - win_size - left])


_CONSTANTS = {}            # mel basis and window per configuration, dtype and device, as the reference caches them


def mel_spectrogram_torch(y, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax):
    """y [B, samples] (any float dtype / device) -> log-mel [B, num_mels, frames], differentiable in ``y``."""
    key = (n_fft, num_mels, sampling_rate, win_size, fmin, fmax, y.dtype, y.device)
    if key not in _CONSTANTS:
        basis = mel_oracle.mel_filterbank(sampling_rate, n_fft, num_mels, fmin, fmax)
        _CONSTANTS[key] = (torch.as_tensor(basis, dtype=y.dtype, device=y.device),
                           torch.hann_window(win_size, dtype=y.dtype, device=y.device))
    basis, window = _CONSTANTS[key]
    pad = int((n_fft - hop_size) / 2)
    yp = torch.nn.functional.pad(y.unsqueeze(1), (pad, pad), mode="reflect").squeeze(1)
    spec = torch.stft(yp, n_fft, hop_length=hop_size, win_length=win_size, window=window, center=False,
                      normalized=False, onesided=True, return_complex=True)
    spec = torch.view_as_real(spec)
    mag = torch.sqrt(spec.pow(2).sum(-1) + 1e-9)
    return torch.log(torch.clamp(torch.matmul(basis, mag), min=1e-5))


def mel_backward_np(y, g, n_fft, num_mels, sampling_rate, hop_size, win_size, fmin, fmax):
    """dL/dy [B, samples] fp64 for the cotangent g = dL/d(log-mel) [B, num_mels, frames]."""
    y = np.asarray(y, dtype=np.float64)
    g = np.asarray(g, dtype=np.float64)
    basis = mel_oracle.mel_filterbank(sampling_rate, n_fft, num_mels, fmin, fmax).astype(np.float64)
    B, S = y.shape
    N, H = n_fft, n_fft // 2
    pad = (n_fft - hop_size) // 2
    yp = np.pad(y, [[0, 0], [pad, pad]], mode="reflect")
    frames = 1 + (yp.shape[1] - N) // hop_size
    window = _window_np(N, win_size)
    idx = np.arange(N)[None, :] + hop_size * np.arange(frames)[:, None]
    seg = yp[:, idx] * window                                        # [B, frames, N]
    # 1. forward: N/2-point complex FFT of the packed frame, then the real-FFT unpack (k = 0 .. H)
    Z = np.fft.fft(seg[..., 0::2] + 1j * seg[..., 1::2], axis=-1)   # [B, frames, H]
    k = np.arange(H + 1)
    Zk, Zc = Z[..., k % H], np.conj(Z[..., (H - k) % H])
    W = np.exp(-2j * np.pi * k / N)
    X = 0.5 * (Zk + Zc) - 0.5j * W * (Zk - Zc)
    mag = np.sqrt(X.real ** 2 + X.imag ** 2 + 1e-9)
    acc = np.einsum("mk,bfk->bfm", basis, mag)
    # 2. clamp gate (torch's clamp(min=) passes the gradient at equality); 3. back through the filters
    dacc = np.where(acc >= 1e-5, np.transpose(g, (0, 2, 1)) / acc, 0.0)
    dmag = np.einsum("mk,bfm->bfk", basis, dacc)
    # 4. d|X| -> d(re, im) as one complex number G = dmag * X / |X|
    G = dmag * X / mag
    # 5. adjoint of the unpack: dZ[j] = (G[j] + conj G[H-j] + i conj(W^j) (G[j] - conj G[H-j])) / 2, j = 1 .. H-1;
    #    dZ[0] = (1 + i) Re G[0] + (1 - i) Re G[H]; then the unnormalised inverse FFT and the unpacking of the frame
    j = np.arange(1, H)
    Gj, Gm = G[..., j], np.conj(G[..., H - j])
    dZ = np.empty(G.shape[:-1] + (H,), dtype=np.complex128)
    dZ[..., 1:] = 0.5 * ((Gj + Gm) + 1j * np.conj(W[j]) * (Gj - Gm))
    dZ[..., 0] = (1 + 1j) * G[..., 0].real + (1 - 1j) * G[..., H].real
    dz = np.fft.ifft(dZ, axis=-1) * H
    dseg = np.empty_like(seg)
    dseg[..., 0::2], dseg[..., 1::2] = dz.real, dz.imag
    dseg *= window
    # 6. overlap-add into the padded signal, then fold the reflect padding back
    dpad = np.zeros_like(yp)
    for f in range(frames):
        dpad[:, f * hop_size:f * hop_size + N] += dseg[:, f]
    dy = dpad[:, pad:pad + S].copy()
    if pad:
        dy[:, 1:pad + 1] += dpad[:, pad - 1::-1]                      # padded p < pad -> sample pad - p
        right = dpad[:, pad + S:]                                    # p >= pad + S -> sample 2 (S - 1) - (p - pad)
        dy[:, S - 2 - np.arange(right.shape[1])] += right
    return dy
