"""Float64 references for training on the waveform SI-SDR: the adjoint of the iSTFT and sisdr_eval's gradient.

TEST INFRASTRUCTURE -- see ``oracle/__init__.py``.  ``istft_adjoint`` is the explicit transpose of ``stft_f64.istft``
(NumPy, direct DFT, no FFT library): <istft(Y), g> = Re <Y, istft_adjoint(g)> for every Y and real g.  ``wave_sisdr`` is
``signal_path.sisdr_eval`` over a batch with its closed-form gradient.
"""
import math

import numpy as np
import torch

from .stft_f64 import hann_periodic


def istft_adjoint(g, n_fft, hop, n_frames, window=None):
    """g: real (R, width) gradient waveform -> complex128 (R, n_frames, K) G = dL/dRe Y + i dL/dIm Y of ``stft_f64.istft``.

    Samples from hop*(n_frames-1) on (a pad_to zero fill) carry no gradient.  Written as the explicit transpose of each
    step of that istft: the trim, the envelope division, the overlap-add, the window, and the synthesis matrix of irfft
    (whose imaginary parts of DC and Nyquist are dropped, so their gradient is 0)."""
    g = np.asarray(g, dtype=np.float64)
    R = g.shape[0]
    F = int(n_frames)
    w = hann_periodic(n_fft) if window is None else np.asarray(window, dtype=np.float64)
    K = n_fft // 2 + 1
    n_out = hop * (F - 1)
    total = n_out + n_fft
    env = np.zeros(total)
    for f in range(F):
        env[f * hop:f * hop + n_fft] += w * w
    start = n_fft // 2
    m = min(n_out, g.shape[1])
    gp = np.zeros((R, total))
    gp[:, start:start + m] = g[:, :m] / env[None, start:start + m]
    frames = np.stack([gp[:, f * hop:f * hop + n_fft] * w[None, :] for f in range(F)], axis=1)    # (R, F, N)
    scale = np.full(K, 2.0)
    scale[0] = 1.0
    if n_fft % 2 == 0:
        scale[-1] = 1.0
    n = np.arange(n_fft)
    analysis = np.exp(-2j * np.pi * np.outer(n, np.arange(K)) / n_fft) * scale[None, :] / n_fft   # (N, K): basis^H / N
    G = frames @ analysis
    G[..., 0] = G[..., 0].real
    if n_fft % 2 == 0:
        G[..., -1] = G[..., -1].real
    return G


def wave_sisdr(src, tar, lengths=None, eps=1e-10):
    """sisdr_eval over a batch, float64: src, tar (B, T) -> (sisdr (B,), grad (B, T)) where grad is the closed-form gradient of
    the training loss mean_u(-sisdr_u) in src (0 from lengths[u] on).  lengths None = T."""
    src = torch.as_tensor(src, dtype=torch.float64)
    tar = torch.as_tensor(tar, dtype=torch.float64)
    B, T = src.shape
    lens = [T] * B if lengths is None else [min(T, max(0, int(n))) for n in lengths]
    sisdr = torch.zeros(B, dtype=torch.float64)
    grad = torch.zeros(B, T, dtype=torch.float64)
    ln10 = math.log(10.0)
    for b, n in enumerate(lens):
        s, t = src[b, :n], tar[b, :n]
        st, tt, ss = (s * t).sum(), (t * t).sum(), (s * s).sum()
        a = st / (tt + eps)
        e = a * t - s
        num = a * a * tt
        den = (e * e).sum() + eps
        sisdr[b] = 10.0 * torch.log10(num / den + eps)
        # d num = 2 a tt da, d den = 2 (a tt - st) da - 2 e, da = t / (tt + eps)
        da = t / (tt + eps)
        dnum = 2.0 * a * tt * da
        dden = 2.0 * (a * tt - st) * da - 2.0 * e
        dsisdr = 10.0 / (ln10 * (num / den + eps)) * (dnum * den - num * dden) / (den * den)
        grad[b, :n] = -dsisdr / B
    return sisdr, grad
