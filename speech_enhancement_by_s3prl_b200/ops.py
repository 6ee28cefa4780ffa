"""Torch-facing operator layer over the C ABI of ``libse_b200.so``.

Every function takes CUDA fp32 tensors, allocates its outputs with torch (the
library itself never allocates user-visible memory) and launches on torch's
current stream.  The differentiable operators are registered with
``torch.library.custom_op`` (+ fake + autograd) so that they compose with
autograd, ``torch.no_grad`` and graph capture.  There is NO CPU implementation:
CPU tensors raise, as does a missing library.
"""
import math

import torch

from . import _lib, dp

ACT = {"Identity": 0, "ReLU": 1, "Sigmoid": 2}
NSUMS = 6
SUPPORTED_NFFT = (256, 400, 512, 1024, 2048)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _chk(t, name, dtype=torch.float32):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"se_b200: {name} must be a CUDA tensor (there is no CPU fallback)")
    if t.dtype != dtype:
        raise RuntimeError(f"se_b200: {name} must be {dtype}, got {t.dtype}")
    return t


def _c(t, name, dtype=torch.float32):
    t = _chk(t, name, dtype)
    return None if t is None else t.contiguous()


def prepare(n_fft):
    """Create the device tables for n_fft (call before CUDA-graph capture)."""
    _lib.check(_lib.load().se_prepare(int(n_fft)), "se_prepare")


def centered_window(window, n_fft):
    """torch.stft centres a window shorter than n_fft in the frame."""
    win = window.shape[0]
    if win == n_fft:
        return window.contiguous()
    left = (n_fft - win) // 2
    return torch.nn.functional.pad(window, (left, n_fft - win - left)).contiguous()


# --------------------------------------------------------------------------- STFT / iSTFT
def stft(wavs, channel, n_fft, hop, window, power=True, phase=False, logpower=False, log_eps=1e-10):
    """wavs (B, C, T) contiguous -> dict of (B, F, K) tensors for channel ``channel``."""
    wavs = _chk(wavs, "wavs")
    assert wavs.dim() == 3 and wavs.is_contiguous()
    B, C, T = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    window = _c(window, "window")
    assert window.numel() == n_fft
    out = {}
    with torch.cuda.device(wavs.device):
        mk = lambda want: torch.empty(B, F, K, device=wavs.device, dtype=torch.float32) if want else None
        pw, ph, lg = mk(power), mk(phase), mk(logpower)
        rc = _lib.load().se_stft(wavs.data_ptr() + 4 * int(channel) * T, B, C * T, T, n_fft, hop, window.data_ptr(),
                                 float(log_eps), _p(pw), _p(ph), _p(lg), _stream())
        _lib.check(rc, "se_stft")
    if power:
        out["power"] = pw
    if phase:
        out["phase"] = ph
    if logpower:
        out["logpower"] = lg
    return out


def round4(n):
    return (int(n) + 3) // 4 * 4


def stft_padded(wavs, channel, n_fft, hop, window, logpower=True, log_eps=1e-10):
    """Fused-path variant of stft: ONE output (log-power or power) with rows padded to a multiple of
    4 floats (16-byte aligned rows for the tensor-core head).  Returns a (B, F, LD) tensor whose
    columns [K, LD) are unspecified."""
    wavs = _chk(wavs, "wavs")
    B, C, T = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = round4(K)
    window = _c(window, "window")
    with torch.cuda.device(wavs.device):
        out = torch.empty(B, F, LD, device=wavs.device, dtype=torch.float32)
        rc = _lib.load().se_stft_strided(wavs.data_ptr() + 4 * int(channel) * T, B, C * T, T, n_fft, hop, window.data_ptr(),
                                         float(log_eps), None if logpower else out.data_ptr(), None,
                                         out.data_ptr() if logpower else None, LD, _stream())
        _lib.check(rc, "se_stft_strided")
    return out


FLAG_WANT_SPEC, FLAG_SUMS_ZEROED, FLAG_MASK_IS_POWER, FLAG_WS_SELF_CLEAN = 1, 2, 4, 8


def stft_features(wavs, channel, n_fft, hop, window, logpower=True, log_eps=1e-10, stat_sums=None, self_clean=False):
    """Fused-step K1: ONE feature tensor (B, F, round4(K)) -- log-power or power -- plus the CMVN sums
    (B, round4(K), 2) float64 = [sum_f x, sum_f x^2].  If ``stat_sums`` is given it must already be zero
    (the caller zeroed its workspace once for the whole step); otherwise it is allocated and zeroed here.
    self_clean: ``stat_sums`` is the head of a persistent step workspace ``[stat_sums | K3 sums]`` (SE_FLAG_WS_SELF_CLEAN):
    this kernel zeroes the K3 sums that follow it, ``mask_istft(self_clean=True)`` zeroes ``stat_sums`` after the head."""
    wavs = _chk(wavs, "wavs")
    B, C, T = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = round4(K)
    window = _c(window, "window")
    with torch.cuda.device(wavs.device):
        out = torch.empty(B, F, LD, device=wavs.device, dtype=torch.float32)
        flags = FLAG_SUMS_ZEROED | (FLAG_WS_SELF_CLEAN if self_clean else 0)
        if stat_sums is None:
            assert not self_clean
            stat_sums = torch.empty(B, LD, 2, device=wavs.device, dtype=torch.float64)
            flags = 0
        assert stat_sums.shape == (B, LD, 2) and stat_sums.dtype == torch.float64 and stat_sums.is_contiguous()
        rc = _lib.load().se_stft_features(wavs.data_ptr() + 4 * int(channel) * T, B, C * T, T, n_fft, hop, window.data_ptr(),
                                          float(log_eps), int(bool(logpower)), out.data_ptr(), LD, stat_sums.data_ptr(), LD,
                                          flags, _stream())
        _lib.check(rc, "se_stft_features")
    return out, stat_sums


def stft_features2(wavs, channel, n_fft, hop, window, want_power=True, want_logpower=True, log_eps=1e-10, stat_sums=None):
    """Training-step K1: power and / or log-power of one channel, rows padded to round4(K), from ONE transform, plus the
    CMVN sums (B, round4(K), 2) float64 of log-power (of power if log-power is not requested).  ``stat_sums`` given =
    already zeroed by the caller.  Returns (power | None, logpower | None, stat_sums)."""
    wavs = _chk(wavs, "wavs")
    B, C, T = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = round4(K)
    window = _c(window, "window")
    assert want_power or want_logpower
    with torch.cuda.device(wavs.device):
        power = torch.empty(B, F, LD, device=wavs.device, dtype=torch.float32) if want_power else None
        logp = torch.empty(B, F, LD, device=wavs.device, dtype=torch.float32) if want_logpower else None
        flags = FLAG_SUMS_ZEROED
        if stat_sums is None:
            stat_sums = torch.empty(B, LD, 2, device=wavs.device, dtype=torch.float64)
            flags = 0
        assert stat_sums.shape == (B, LD, 2) and stat_sums.dtype == torch.float64 and stat_sums.is_contiguous()
        rc = _lib.load().se_stft_features2(wavs.data_ptr() + 4 * int(channel) * T, B, C * T, T, n_fft, hop, window.data_ptr(),
                                           float(log_eps), _p(power), _p(logp), LD, stat_sums.data_ptr(), LD, flags, _stream())
        _lib.check(rc, "se_stft_features2")
    return power, logp, stat_sums


def stft_features_pair(wavs, ch_inp, ch_tar, n_fft, hop, window, log_eps=1e-10, stat_sums=None):
    """Both K1 launches of a training / scoring step in one (register-resident geometries): power + log-power + CMVN sums of the
    input channel and the power of the target channel.  Returns (linear_inp, logpower, linear_tar, stat_sums), each (B, F, LD);
    falls back to two ``stft_features2`` / ``stft_padded`` launches where the one-launch kernel does not exist."""
    wavs = _chk(wavs, "wavs")
    B, C, T = wavs.shape
    lib = _lib.load()
    if not lib.se_stft_features_pair_supported(int(n_fft), int(hop)):
        linear_inp, logp, stat_sums = stft_features2(wavs, ch_inp, n_fft, hop, window, True, True, log_eps, stat_sums)
        return linear_inp, logp, stft_padded(wavs, ch_tar, n_fft, hop, window, logpower=False), stat_sums
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = round4(K)
    window = _c(window, "window")
    with torch.cuda.device(wavs.device):
        power2 = torch.empty(2, B, F, LD, device=wavs.device, dtype=torch.float32)
        logp = torch.empty(B, F, LD, device=wavs.device, dtype=torch.float32)
        flags = FLAG_SUMS_ZEROED
        if stat_sums is None:
            stat_sums = torch.empty(B, LD, 2, device=wavs.device, dtype=torch.float64)
            flags = 0
        assert stat_sums.shape == (B, LD, 2) and stat_sums.dtype == torch.float64 and stat_sums.is_contiguous()
        rc = lib.se_stft_features_pair(wavs.data_ptr() + 4 * int(ch_inp) * T, B, C * T, (int(ch_tar) - int(ch_inp)) * T, T, n_fft, hop,
                                       window.data_ptr(), float(log_eps), power2.data_ptr(), logp.data_ptr(), LD, stat_sums.data_ptr(),
                                       LD, flags, _stream())
        _lib.check(rc, "se_stft_features_pair")
    return power2[0], logp, power2[1], stat_sums


def linear_head_bwd_fused_supported(B, F, D_in, D_out):
    return _lib.load().se_linear_head_bwd_tc_workspace(B, F, D_in, D_out) > 0


def linear_head_bwd_fused(x, D_in, stat_sums, cmvn_eps, offset, grad_offset, D_out, activation):
    """Weight / bias gradients of the TMA head from its padded operands: x (B, F, LDx), offset and grad_offset (B, F, LDo),
    stat_sums (B, LDs, 2) float64 or None (no CMVN).  Returns (grad_W (D_out, D_in), grad_b (D_out,))."""
    B, F, LDx = x.shape
    LDo = offset.shape[2]
    assert grad_offset.shape == offset.shape and offset.is_contiguous() and grad_offset.is_contiguous() and x.is_contiguous()
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_floats = lib.se_linear_head_bwd_tc_workspace(B, F, int(D_in), int(D_out))
        if ws_floats <= 0:
            raise RuntimeError(f"se_linear_head_bwd_fused: shape (B={B}, F={F}, D_in={D_in}, D_out={D_out}) is not supported")
        ws = torch.empty(ws_floats, device=x.device)
        gw = torch.empty(D_out, D_in, device=x.device)
        gb = torch.empty(D_out, device=x.device)
        rc = lib.se_linear_head_bwd_fused(x.data_ptr(), LDx, _p(stat_sums), 0 if stat_sums is None else stat_sums.shape[1],
                                          float(cmvn_eps), offset.data_ptr(), grad_offset.data_ptr(), LDo, B, F, int(D_in),
                                          int(D_out), ACT[activation], ws.data_ptr(), ws_floats, gw.data_ptr(), gb.data_ptr(),
                                          _stream())
        _lib.check(rc, "se_linear_head_bwd_fused")
    return gw, gb


def linear_head_bwd_sisdr_supported(B, F, D_in, D_out, ldx, ld_off, ld_inp, ld_tar):
    return bool(_lib.load().se_linear_head_bwd_sisdr_supported(B, F, int(D_in), int(D_out), ldx, ld_off, ld_inp, ld_tar))


def linear_head_bwd_sisdr(x, D_in, stat_sums, cmvn_eps, offset, linear_inp, linear_tar, lengths, hop, sums3, D_out, activation, loss_eps=1e-10):
    """Weight / bias gradients of the batch-mean objective.SISDR loss on predicted = offset * linear_inp through the TMA head's
    backward with the objective's own backward folded in (no grad_offset tensor): x (B, F, LDx), offset / linear_inp / linear_tar
    (B, F, LD*) row-padded, sums3 (B, 3) from ``sisdr_mask_step``, lengths = SAMPLE lengths with ``hop`` (frame counts if hop = 0).
    Returns (grad_W (D_out, D_in), grad_b (D_out,))."""
    B, F, LDx = x.shape
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_floats = lib.se_linear_head_bwd_tc_workspace(B, F, int(D_in), int(D_out))
        if ws_floats <= 0:
            raise RuntimeError(f"se_linear_head_bwd_sisdr: shape (B={B}, F={F}, D_in={D_in}, D_out={D_out}) is not supported")
        ws = torch.empty(ws_floats, device=x.device)
        gw = torch.empty(D_out, D_in, device=x.device)
        gb = torch.empty(D_out, device=x.device)
        rc = lib.se_linear_head_bwd_sisdr(x.data_ptr(), LDx, _p(stat_sums), 0 if stat_sums is None else stat_sums.shape[1], float(cmvn_eps),
                                          offset.data_ptr(), offset.shape[2], linear_inp.data_ptr(), linear_inp.shape[2],
                                          linear_tar.data_ptr(), linear_tar.shape[2], lengths.data_ptr(), int(hop), sums3.data_ptr(),
                                          float(loss_eps), B, F, int(D_in), int(D_out), ACT[activation], ws.data_ptr(), ws_floats,
                                          gw.data_ptr(), gb.data_ptr(), _stream())
        _lib.check(rc, "se_linear_head_bwd_sisdr")
    return gw, gb


def linear_head_bwd_wsd_supported(B, F, D_in, D_out, ldx, ld_off, ld_inp, ld_tar):
    return bool(_lib.load().se_linear_head_bwd_wsd_supported(B, F, int(D_in), int(D_out), ldx, ld_off, ld_inp, ld_tar))


def linear_head_bwd_wsd(x, D_in, stat_sums, cmvn_eps, offset, linear_inp, linear_tar, lengths, hop, energy, emax, D_out, activation,
                        alpha=0.5, db_interval=30.0, loss_eps=1e-10):
    """``linear_head_bwd_sisdr`` for the batch-mean objective.WSD loss: d loss / d offset is rebuilt inside the weight-gradient
    kernel from offset / linear_inp / linear_tar (B, F, LD*) row-padded, the frame energies (B, F) and the batch maximum (1,) of
    ``wsd_energy`` (all-reduced first under data parallelism).  Returns (grad_W (D_out, D_in), grad_b (D_out,))."""
    B, F, LDx = x.shape
    lib = _lib.load()
    with torch.cuda.device(x.device):
        ws_floats = lib.se_linear_head_bwd_tc_workspace(B, F, int(D_in), int(D_out))
        if ws_floats <= 0:
            raise RuntimeError(f"se_linear_head_bwd_wsd: shape (B={B}, F={F}, D_in={D_in}, D_out={D_out}) is not supported")
        ws = torch.empty(ws_floats, device=x.device)
        gw = torch.empty(D_out, D_in, device=x.device)
        gb = torch.empty(D_out, device=x.device)
        rc = lib.se_linear_head_bwd_wsd(x.data_ptr(), LDx, _p(stat_sums), 0 if stat_sums is None else stat_sums.shape[1], float(cmvn_eps),
                                        offset.data_ptr(), offset.shape[2], linear_inp.data_ptr(), linear_inp.shape[2],
                                        linear_tar.data_ptr(), linear_tar.shape[2], lengths.data_ptr(), int(hop), energy.data_ptr(),
                                        emax.data_ptr(), float(alpha), float(db_interval), float(loss_eps), B, F, int(D_in), int(D_out),
                                        ACT[activation], ws.data_ptr(), ws_floats, gw.data_ptr(), gb.data_ptr(), _stream())
        _lib.check(rc, "se_linear_head_bwd_wsd")
    return gw, gb


def wsd_energy(linear_tar, K):
    """objective.WSD's frame energies and their maximum: linear_tar (B, F, LD) row-padded (columns >= K are not read) ->
    (energy (B, F), emax (1,) float32 -- the rank-local batch maximum, ready for ``dp.global_max``)."""
    linear_tar = _chk(linear_tar, "linear_tar")
    assert linear_tar.dim() == 3 and linear_tar.stride(2) == 1 and linear_tar.stride(1) == linear_tar.shape[2]
    B, F, LD = linear_tar.shape
    dev = linear_tar.device
    with torch.cuda.device(dev):
        energy = torch.empty(B, F, device=dev)
        emax = torch.empty(1, device=dev)
        rc = _lib.load().se_wsd_energy(linear_tar.data_ptr(), LD, B, F, int(K), energy.data_ptr(), emax.data_ptr(), _stream())
        _lib.check(rc, "se_wsd_energy")
    return energy, emax


def wsd_mask_step(offset, linear_inp, linear_tar, lengths, hop, K, energy, emax, alpha=0.5, db_interval=30.0, eps=1e-10, sums2=None,
                  sums_zeroed=False, want_grad=True):
    """The WSD objective's part of a training step on (B, F, LD) row-padded tensors (the counterpart of ``sisdr_mask_step``),
    thresholding against the maximum in ``emax`` (after ``dp.global_max`` under data parallelism).  ``lengths``: SAMPLE lengths
    with ``hop`` (frames = lengths // hop + 1) or frame counts with hop = 0.
    Returns (loss (0-dim), loss_per_utt (B,), grad_offset (B, F, LDo) or None (want_grad=False), sums2 (B, 2) float64)."""
    B, F, LDi = linear_inp.shape
    dev = linear_inp.device
    lengths = _c(lengths, "lengths", torch.int64)
    with torch.cuda.device(dev):
        if sums2 is None:
            sums2, sums_zeroed = torch.zeros(B, 2, device=dev, dtype=torch.float64), True
        out = torch.empty(B + 1, device=dev)
        grad = torch.empty_like(offset) if want_grad else None
        rc = _lib.load().se_wsd_mask_step(offset.data_ptr(), offset.shape[2], linear_inp.data_ptr(), LDi, linear_tar.data_ptr(),
                                          linear_tar.shape[2], lengths.data_ptr(), int(hop), B, F, int(K), float(alpha), float(db_interval),
                                          float(eps), energy.data_ptr(), emax.data_ptr(), sums2.data_ptr(), 1 if sums_zeroed else 0,
                                          out.data_ptr(), out[B:].data_ptr(), _p(grad), 0 if grad is None else grad.shape[2], _stream())
        _lib.check(rc, "se_wsd_mask_step")
    return out[B], out[:B], grad, sums2


def sisdr_mask_step(offset, linear_inp, linear_tar, lengths, hop, K, eps=1e-10, sums3=None, sums_zeroed=False, want_grad=True):
    """The objective's part of a training step on (B, F, LD) row-padded tensors in three launches: objective.SISDR of
    predicted = offset * linear_inp (mean over the batch, objective.py:100) and d loss / d offset.  ``lengths``: SAMPLE lengths
    (int64, device), frames = lengths // hop + 1 is taken inside the kernels (runner.py:455).
    Returns (loss (0-dim), loss_per_utt (B,), grad_offset (B, F, LDo) or None (want_grad=False: sums and losses only), sums3)."""
    B, F, LDi = linear_inp.shape
    dev = linear_inp.device
    with torch.cuda.device(dev):
        if sums3 is None:
            sums3, sums_zeroed = torch.zeros(B, 3, device=dev, dtype=torch.float64), True
        out = torch.empty(B + 1, device=dev)
        grad = torch.empty_like(offset) if want_grad else None
        rc = _lib.load().se_sisdr_mask_step(offset.data_ptr(), offset.shape[2], linear_inp.data_ptr(), LDi, linear_tar.data_ptr(),
                                            linear_tar.shape[2], lengths.data_ptr(), int(hop), B, F, int(K), float(eps), sums3.data_ptr(),
                                            1 if sums_zeroed else 0, out.data_ptr(), out[B:].data_ptr(), _p(grad),
                                            0 if grad is None else grad.shape[2], _stream())
        _lib.check(rc, "se_sisdr_mask_step")
    return out[B], out[:B], grad, sums3


def sisdr_mask_fwd(offset, linear_inp, linear_tar, stft_lengths, K, eps=1e-10, sums3=None):
    """objective.SISDR of predicted = offset * linear_inp on (B, F, LD) row-padded tensors (offset None: predicted =
    linear_inp).  Returns (loss_per_utt (B,), sums3 (B, 3) float64 for the backward)."""
    B, F, LDi = linear_inp.shape
    stft_lengths = _c(stft_lengths, "stft_lengths", torch.int64)
    with torch.cuda.device(linear_inp.device):
        if sums3 is None:
            sums3 = torch.empty(B, 3, device=linear_inp.device, dtype=torch.float64)
        loss = torch.empty(B, device=linear_inp.device)
        rc = _lib.load().se_sisdr_mask_fwd(_p(offset), 0 if offset is None else offset.shape[2], linear_inp.data_ptr(), LDi,
                                           linear_tar.data_ptr(), linear_tar.shape[2], _p(stft_lengths), B, F, int(K), float(eps),
                                           sums3.data_ptr(), loss.data_ptr(), _stream())
        _lib.check(rc, "se_sisdr_mask_fwd")
    return loss, sums3


def sisdr_mask_bwd(offset, linear_inp, linear_tar, stft_lengths, K, sums3, grad_out, eps=1e-10, ld_out=None):
    """d (sum_u grad_out[u] * loss_u) / d offset, (B, F, ld_out or LD of linear_inp); pad columns are zero."""
    B, F, LDi = linear_inp.shape
    LDg = int(ld_out or (offset.shape[2] if offset is not None else LDi))
    stft_lengths = _c(stft_lengths, "stft_lengths", torch.int64)
    grad_out = _c(grad_out, "grad_out")
    with torch.cuda.device(linear_inp.device):
        g = torch.empty(B, F, LDg, device=linear_inp.device)
        rc = _lib.load().se_sisdr_mask_bwd(_p(offset), 0 if offset is None else offset.shape[2], linear_inp.data_ptr(), LDi,
                                           linear_tar.data_ptr(), linear_tar.shape[2], _p(stft_lengths), B, F, int(K), float(eps),
                                           sums3.data_ptr(), grad_out.data_ptr(), g.data_ptr(), LDg, _stream())
        _lib.check(rc, "se_sisdr_mask_bwd")
    return g


def feature_sums(x, D):
    """x (B, F, LD) -> (B, LD, 2) float64 sums [sum_f x, sum_f x^2] of columns [0, D)."""
    x = _chk(x, "x")
    B, F, LD = x.shape
    with torch.cuda.device(x.device):
        sums = torch.zeros(B, LD, 2, device=x.device, dtype=torch.float64)
        rc = _lib.load().se_feature_sums(x.data_ptr(), LD, B, F, int(D), sums.data_ptr(), LD, _stream())
        _lib.check(rc, "se_feature_sums")
    return sums


def round_tf32(w):
    """Round fp32 values to the nearest TF32 (10-bit mantissa, ties away from zero, as cvt.rna.tf32.f32)."""
    bits = w.contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1FFF).view(torch.float32)


def linear_head_tma_supported(B, F, D_in, D_out, ldx, ldw, ld_out):
    return bool(_lib.load().se_linear_head_fused_supported(B, F, D_in, D_out, ldx, ldw, ld_out))


def linear_head_tma(x, D_in, weight_padded, bias, activation, stat_sums, cmvn_eps):
    """x (B, F, LDx), weight_padded (Dout, LDw) pre-rounded to TF32, stat_sums (B, LDs, 2) float64 or None
    -> mask (B, F, round4(Dout)) through the TMA / tcgen05 head (columns >= Dout unspecified)."""
    B, F, LDx = x.shape
    Dout, LDw = weight_padded.shape
    LDo = round4(Dout)
    with torch.cuda.device(x.device):
        out = torch.empty(B, F, LDo, device=x.device)
        rc = _lib.load().se_linear_head_fused(x.data_ptr(), LDx, _p(stat_sums), 0 if stat_sums is None else stat_sums.shape[1],
                                              float(cmvn_eps), weight_padded.data_ptr(), LDw, _p(bias), B, F, int(D_in), Dout,
                                              ACT[activation], out.data_ptr(), LDo, _stream())
        _lib.check(rc, "se_linear_head_fused")
    return out


def cmvn_stats_padded(x, D):
    """x (B, F, LD) with D valid columns -> mean, std (B, LD) (valid columns [0, D))."""
    B, F, LD = x.shape
    with torch.cuda.device(x.device):
        mean = torch.empty(B, LD, device=x.device)
        std = torch.empty(B, LD, device=x.device)
        rc = _lib.load().se_cmvn_stats_strided(x.data_ptr(), LD, B, F, D, mean.data_ptr(), std.data_ptr(), LD, _stream())
        _lib.check(rc, "se_cmvn_stats_strided")
    return mean, std


def pad_weight(weight):
    """(Dout, Din) -> contiguous (Dout, round4(Din)) zero-padded copy (16-byte aligned rows)."""
    Dout, Din = weight.shape
    LD = round4(Din)
    if LD == Din:
        return weight.contiguous()
    return torch.nn.functional.pad(weight, (0, LD - Din)).contiguous()


def linear_head_padded(x, D_in, weight_padded, bias, activation, mean, std, cmvn_eps, precision=1):
    """x (B, F, LDx), weight_padded (Dout, LDw) -> mask (B, F, round4(Dout)) (valid columns [0, Dout))."""
    B, F, LDx = x.shape
    Dout, LDw = weight_padded.shape
    LDo = round4(Dout)
    with torch.cuda.device(x.device):
        out = torch.empty(B, F, LDo, device=x.device)
        rc = _lib.load().se_linear_head_fwd_strided(x.data_ptr(), LDx, _p(mean), _p(std), 0 if mean is None else mean.shape[1],
                                                    float(cmvn_eps), weight_padded.data_ptr(), LDw, _p(bias), B, F, int(D_in), Dout,
                                                    ACT[activation], None, out.data_ptr(), None, LDo, int(precision), _stream())
        _lib.check(rc, "se_linear_head_fwd_strided")
    return out


def istft(power, phase, n_fft, hop, window, pad_to=0):
    """(B, F, K) power + phase -> (B, max(hop*(F-1), pad_to)); reference OnlinePreprocessor.istft."""
    power, phase, window = _c(power, "linears"), _c(phase, "phases"), _c(window, "window")
    B, F, K = power.shape
    assert K == n_fft // 2 + 1 and phase.shape == power.shape
    out_len = hop * (F - 1)
    width = max(out_len, int(pad_to))
    with torch.cuda.device(power.device):
        wav = torch.empty(B, width, device=power.device, dtype=torch.float32)
        rc = _lib.load().se_istft(power.data_ptr(), phase.data_ptr(), B, F, n_fft, hop, window.data_ptr(),
                                  wav.data_ptr(), width, int(pad_to), _stream())
        _lib.check(rc, "se_istft")
    return wav


def mask_istft(wavs, ch_inp, ch_tar, mask, lengths, n_fft, hop, window, pad_to, want_sums=True, want_spec=True,
               out=None, sums=None, mask_padded=False, sums_zeroed=False, mask_is_power=False, self_clean=False):
    """Fused ``istft(linear_inp * mask, phase_inp)`` straight from the noisy waveform.

    wavs (B, C, T); mask (B, F, K); lengths (B,) int64 or None.  Returns (wav (B, width), sums (B, 6) float64|None)."""
    wavs, mask, window = _chk(wavs, "wavs"), _c(mask, "mask"), _c(window, "window")
    assert wavs.dim() == 3 and wavs.is_contiguous()
    B, C, T = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    mask_stride = mask.shape[2] if mask_padded else K
    assert mask.shape == (B, F, mask_stride) and mask_stride >= K, f"mask {tuple(mask.shape)} != {(B, F, mask_stride)}"
    lengths = _c(lengths, "lengths", torch.int64)
    out_len = hop * (F - 1)
    width = max(out_len, int(pad_to))
    with torch.cuda.device(wavs.device):
        if out is None:
            out = torch.empty(B, width, device=wavs.device, dtype=torch.float32)
        if want_sums and sums is None:
            sums = torch.empty(B, NSUMS, device=wavs.device, dtype=torch.float64)
        clean = None if ch_tar is None else wavs.data_ptr() + 4 * int(ch_tar) * T
        flags = (FLAG_WANT_SPEC if want_spec else 0) | (FLAG_SUMS_ZEROED if sums_zeroed else 0)
        flags |= FLAG_MASK_IS_POWER if mask_is_power else 0     # `mask` = target power; output keeps the noisy phase
        flags |= FLAG_WS_SELF_CLEAN if self_clean else 0        # `sums` is the tail of a persistent step workspace (see stft_features)
        rc = _lib.load().se_mask_istft_ex(wavs.data_ptr() + 4 * int(ch_inp) * T, clean, C * T, mask.data_ptr(), mask_stride,
                                          _p(lengths), B, T, n_fft, hop, window.data_ptr(), out.data_ptr(), out.stride(0),
                                          int(pad_to), _p(sums) if want_sums else None, flags, _stream())
        _lib.check(rc, "se_mask_istft_ex")
    return out, (sums if want_sums else None)


def finalize_metrics(sums, lengths, T, wav=None, target_db=None, want_gain=True, want_sisdr=True, want_loss=True,
                     metric_acc=None):
    """Gain / waveform SI-SDR / spectral-SISDR terms from the sums of mask_istft; scales wav in place.
    metric_acc: float64 (3,) running [sum loss, sum SI-SDR, utterances] of an evaluation pass, updated on the device
    (the loss sum only with want_loss, the SI-SDR sum only with want_sisdr).  lengths are clamped to [0, T]."""
    B = sums.shape[0]
    dev = sums.device
    with torch.cuda.device(dev):
        gain = torch.empty(B, device=dev) if want_gain else None
        sisdr = torch.empty(B, device=dev) if want_sisdr else None
        loss = torch.empty(B, device=dev) if want_loss else None
        tdb = float("nan") if target_db is None else float(target_db)
        if metric_acc is not None:
            assert metric_acc.dtype == torch.float64 and metric_acc.numel() >= 3 and metric_acc.is_contiguous()
        rc = _lib.load().se_finalize_metrics_acc(sums.data_ptr(), _p(lengths), B, int(T), tdb, _p(wav),
                                                 0 if wav is None else wav.stride(0), 0 if wav is None else wav.shape[1],
                                                 _p(gain), _p(sisdr), _p(loss), _p(metric_acc), _stream())
        _lib.check(rc, "se_finalize_metrics_acc")
    return gain, sisdr, loss


# --------------------------------------------------------------------------- on-device batch synthesis
def mix_batch(speech, speech_len, noise, noise_len, snr_db, target_level=-25.0, eps=1e-8, T_out=None):
    """The reference's ``OnlineDataset.__getitem__`` + ``collate_fn`` for a whole batch on the GPU.

    speech (B, Ts) / noise (B, Tn) fp32 zero-padded rows with their true lengths (B,) int64, snr_db (B,) fp32.
    Returns (lengths (B,) int64, wavs (B, 3, T_out) = [noisy, speech, scaled_noise]); eps = the dataset's eps
    (dataset.py:80, 158)."""
    speech, noise = _c(speech, "speech"), _c(noise, "noise")
    speech_len, noise_len = _c(speech_len, "speech_len", torch.int64), _c(noise_len, "noise_len", torch.int64)
    snr_db = _c(snr_db.to(torch.float32), "snr_db")
    B, Ts = speech.shape
    T_out = int(T_out) if T_out is not None else Ts
    assert T_out >= Ts and noise.shape[0] == B
    with torch.cuda.device(speech.device):
        ws = torch.empty(B, 4, device=speech.device, dtype=torch.float64)
        out = torch.empty(B, 3, T_out, device=speech.device)
        rc = _lib.load().se_mix_batch(speech.data_ptr(), Ts, speech_len.data_ptr(), noise.data_ptr(), noise.shape[1],
                                      noise_len.data_ptr(), snr_db.data_ptr(), B, T_out, float(target_level), float(eps),
                                      ws.data_ptr(), out.data_ptr(), _stream())
        _lib.check(rc, "se_mix_batch")
    return speech_len, out


# --------------------------------------------------------------------------- waveform-level helpers
def sisdr_wave(src, tar, lengths=None, eps=1e-10):
    """Batched evaluation.sisdr_eval: src, tar (B, T) -> (B,) dB."""
    src, tar = _chk(src, "src"), _chk(tar, "tar")
    assert src.dim() == 2 and src.shape == tar.shape and src.stride(1) == 1 and tar.stride(1) == 1
    B, T = src.shape
    lengths = _c(lengths, "lengths", torch.int64)
    with torch.cuda.device(src.device):
        ws = torch.empty(B, 3, device=src.device, dtype=torch.float64)
        out = torch.empty(B, device=src.device)
        rc = _lib.load().se_sisdr_wave(src.data_ptr(), src.stride(0), tar.data_ptr(), tar.stride(0), _p(lengths), B, T,
                                       float(eps), ws.data_ptr(), out.data_ptr(), _stream())
        _lib.check(rc, "se_sisdr_wave")
    return out


def stoi(est, ref, lengths=None, fs=16000, want_stoi=True, want_estoi=True, acc=None, n_kept=None):
    """Batched STOI / ESTOI (pystoi 0.3.x): est = processed, ref = clean reference, both (B, T) views with unit sample stride
    (row strides may differ, e.g. a channel of a (B, C, T) batch).  Returns (stoi, estoi), each (B,) fp32 or None.
    acc: float64 (3,) device tensor += [sum stoi, sum estoi, B] (each sum only when that metric is requested).
    n_kept: optional (B,) int32 output, the frames kept by the silent-frame removal."""
    est, ref = _chk(est, "est"), _chk(ref, "ref")
    assert est.dim() == 2 and est.shape == ref.shape and est.stride(1) == 1 and ref.stride(1) == 1
    if not (want_stoi or want_estoi):
        raise ValueError("ops.stoi: request stoi, estoi or both")
    B, T = est.shape
    lengths = _c(lengths, "lengths", torch.int64)
    acc = _chk(acc, "acc", torch.float64)
    n_kept = _chk(n_kept, "n_kept", torch.int32)
    lib = _lib.load()
    ws_bytes = lib.se_stoi_workspace(B, T, int(fs))
    if ws_bytes <= 0:
        raise RuntimeError(f"se_b200.stoi: unsupported sample rate {fs} or shape {tuple(est.shape)} "
                           "(10000 / fs reduced to p / q needs p, q <= 48)")
    with torch.cuda.device(est.device):
        ws = torch.empty(ws_bytes, device=est.device, dtype=torch.uint8)
        s = torch.empty(B, device=est.device) if want_stoi else None
        e = torch.empty(B, device=est.device) if want_estoi else None
        rc = lib.se_stoi(est.data_ptr(), est.stride(0), ref.data_ptr(), ref.stride(0), _p(lengths), B, T, int(fs), ws.data_ptr(),
                         ws_bytes, _p(s), _p(e), _p(n_kept), _p(acc), _stream())
        _lib.check(rc, "se_stoi")
    return s, e


def masked_normalize_db(audio, lengths, target_db=None, ref=None, eps=1e-8):
    """utils.masked_normalize_decibel on lengths instead of (B, T) int64 masks."""
    audio = _chk(audio, "audio")
    assert audio.dim() == 2 and audio.stride(1) == 1
    B, W = audio.shape
    lengths = _c(lengths, "lengths", torch.int64)
    target_db = _c(target_db, "target_db")
    if ref is not None:
        ref = _chk(ref, "ref")
        assert ref.shape[0] == B and ref.shape[1] >= W and ref.stride(1) == 1
    with torch.cuda.device(audio.device):
        ws = torch.empty(B, 3, device=audio.device, dtype=torch.float64)
        out = torch.empty(B, W, device=audio.device)
        rc = _lib.load().se_masked_normalize_db(audio.data_ptr(), audio.stride(0), _p(lengths), B, W, _p(target_db),
                                                _p(ref), 0 if ref is None else ref.stride(0), float(eps), ws.data_ptr(),
                                                out.data_ptr(), W, _stream())
        _lib.check(rc, "se_masked_normalize_db")
    return out


def length_masks(lengths, width=None):
    """runner._get_length_masks: (B,) int64 -> (B, width or max(lengths)) int64 0/1."""
    lengths = _c(lengths, "lengths", torch.int64)
    if width is None:
        width = int(lengths.max().item())          # the reference syncs here too (runner.py:218)
    B = lengths.shape[0]
    with torch.cuda.device(lengths.device):
        out = torch.empty(B, width, device=lengths.device, dtype=torch.int64)
        _lib.check(_lib.load().se_length_masks(lengths.data_ptr(), B, width, out.data_ptr(), _stream()), "se_length_masks")
    return out


# --------------------------------------------------------------------------- features
def cmvn_stats(x):
    """x (B, F, D) -> mean, unbiased std over time, each (B, D)."""
    x = _c(x, "x")
    B, F, D = x.shape
    with torch.cuda.device(x.device):
        mean = torch.empty(B, D, device=x.device)
        std = torch.empty(B, D, device=x.device)
        _lib.check(_lib.load().se_cmvn_stats(x.data_ptr(), B, F, D, mean.data_ptr(), std.data_ptr(), _stream()), "se_cmvn_stats")
    return mean, std


def cmvn_apply_(x, mean, std, eps):
    B, F, D = x.shape
    assert x.is_contiguous()
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().se_cmvn_apply(x.data_ptr(), B, F, D, mean.data_ptr(), std.data_ptr(), float(eps), _stream()),
                   "se_cmvn_apply")
    return x


def mel(power, fb, take_log, eps, out=None, out_cols=None):
    """power (B, F, K) x fb (K, n_mels) -> (B, F, out_cols or n_mels) with the mel part in the first columns."""
    power, fb = _c(power, "power"), _c(fb, "fb")
    B, F, K = power.shape
    n_mels = fb.shape[1]
    cols = n_mels if out_cols is None else int(out_cols)
    with torch.cuda.device(power.device):
        if out is None:
            out = torch.empty(B, F, cols, device=power.device)
        rc = _lib.load().se_mel(power.data_ptr(), B * F, K, fb.data_ptr(), n_mels, int(bool(take_log)), float(eps),
                                out.data_ptr(), cols, _stream())
        _lib.check(rc, "se_mel")
    return out


_FB_RANGES = {}


def _fb_ranges(fb):
    """(n_mels, 2) int32 [first, last + 1) non-zero bin of every filter (cached per filterbank tensor)."""
    key = (fb.data_ptr(), tuple(fb.shape), str(fb.device))
    if key not in _FB_RANGES:
        nz = fb != 0
        idx = torch.arange(fb.shape[0], device=fb.device).unsqueeze(1)
        lo = torch.where(nz, idx, fb.shape[0]).amin(dim=0)
        hi = torch.where(nz, idx + 1, 0).amax(dim=0)
        lo = torch.minimum(lo, hi)                                   # an all-zero filter: empty range
        if len(_FB_RANGES) >= 8:                                     # (a module kept on the CPU makes a new device copy per call)
            _FB_RANGES.pop(next(iter(_FB_RANGES)))
        _FB_RANGES[key] = (torch.stack([lo, hi], dim=1).to(torch.int32).contiguous(), fb)   # (keeps fb alive: the key is its address)
    return _FB_RANGES[key][0]


def mel_features(power, fb, take_log, eps, order=0, cmvn=False, cmvn_eps=None, K=None):
    """K1b in one launch (two with CMVN): power (B, F, K) x fb (K, n_mels) -> (B, F, (order + 1) * n_mels) =
    [mel | delta | delta-delta] of log?(mel + eps), optionally CMVN-normalised over time.
    K: number of valid bins when ``power`` has padded rows (B, F, LD >= K), as the fused step keeps its spectra."""
    power, fb = _c(power, "power"), _c(fb, "fb")
    B, F, LDp = power.shape
    K = LDp if K is None else int(K)
    assert fb.shape[0] == K and LDp >= K
    n_mels = fb.shape[1]
    D = (int(order) + 1) * n_mels
    lib = _lib.load()
    with torch.cuda.device(power.device):
        ranges = _fb_ranges(fb)
        out = torch.empty(B, F, D, device=power.device)
        sums = torch.empty(B, D, 2, device=power.device, dtype=torch.float64) if cmvn else None
        rc = lib.se_mel_features(power.data_ptr(), LDp, B, F, K, fb.data_ptr(), ranges.data_ptr(), n_mels, int(bool(take_log)), float(eps), int(order),
                                 out.data_ptr(), D, _p(sums), _stream())
        _lib.check(rc, "se_mel_features")
        if cmvn:
            rc = lib.se_cmvn_apply_sums(out.data_ptr(), B, F, D, sums.data_ptr(), float(eps if cmvn_eps is None else cmvn_eps), _stream())
            _lib.check(rc, "se_cmvn_apply_sums")
    return out


def delta_(x, D, order):
    """x (B, F, (order+1)*D): fill column blocks 1..order with recursive regression deltas of block 0."""
    B, F, W = x.shape
    assert W == (order + 1) * D and x.is_contiguous()
    with torch.cuda.device(x.device):
        _lib.check(_lib.load().se_delta(x.data_ptr(), B, F, D, int(order), _stream()), "se_delta")
    return x


# --------------------------------------------------------------------------- objectives (custom ops + autograd)
def _stft_len_or_none(t):
    return None if t is None else t.contiguous()


@torch.library.custom_op("se_b200::sisdr_spec", mutates_args=())
def _sisdr_spec(predicted: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, eps: float) -> tuple[torch.Tensor, torch.Tensor]:
    predicted, linear_tar = _c(predicted, "predicted"), _c(linear_tar, "linear_tar")
    B, F, K = predicted.shape
    with torch.cuda.device(predicted.device):
        sums = torch.empty(B, 3, device=predicted.device, dtype=torch.float64)
        loss = torch.empty(B, device=predicted.device)
        rc = _lib.load().se_sisdr_spec_fwd(predicted.data_ptr(), linear_tar.data_ptr(), stft_len.data_ptr(), B, F, K, eps,
                                           sums.data_ptr(), loss.data_ptr(), _stream())
        _lib.check(rc, "se_sisdr_spec_fwd")
    return loss, sums


@_sisdr_spec.register_fake
def _(predicted, linear_tar, stft_len, eps):
    B = predicted.shape[0]
    return predicted.new_empty(B), predicted.new_empty(B, 3, dtype=torch.float64)


@torch.library.custom_op("se_b200::sisdr_spec_bwd", mutates_args=())
def _sisdr_spec_bwd(predicted: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, eps: float,
                    sums: torch.Tensor, grad_mean: torch.Tensor) -> torch.Tensor:
    predicted, linear_tar = _c(predicted, "predicted"), _c(linear_tar, "linear_tar")
    B, F, K = predicted.shape
    with torch.cuda.device(predicted.device):
        grad = torch.empty_like(predicted)
        g = grad_mean.reshape(B).to(torch.float32).contiguous()
        rc = _lib.load().se_sisdr_spec_bwd(predicted.data_ptr(), linear_tar.data_ptr(), stft_len.data_ptr(), B, F, K, eps,
                                           sums.data_ptr(), g.data_ptr(), grad.data_ptr(), _stream())
        _lib.check(rc, "se_sisdr_spec_bwd")
    return grad


@_sisdr_spec_bwd.register_fake
def _(predicted, linear_tar, stft_len, eps, sums, grad_mean):
    return torch.empty_like(predicted)


def _sisdr_setup(ctx, inputs, output):
    predicted, linear_tar, stft_len, eps = inputs
    ctx.save_for_backward(predicted, linear_tar, stft_len, output[1])
    ctx.eps = eps


def _sisdr_backward(ctx, grad_loss, grad_sums):
    predicted, linear_tar, stft_len, sums = ctx.saved_tensors
    grad = torch.ops.se_b200.sisdr_spec_bwd(predicted, linear_tar, stft_len, ctx.eps, sums, grad_loss)
    return grad, None, None, None


_sisdr_spec.register_autograd(_sisdr_backward, setup_context=_sisdr_setup)


def sisdr_spec(predicted, linear_tar, stft_len, eps=1e-10):
    """Per-utterance terms of objective.SISDR (their mean is the loss); differentiable in ``predicted``."""
    loss, _ = torch.ops.se_b200.sisdr_spec(predicted, linear_tar, stft_len.contiguous(), float(eps))
    return loss


@torch.library.custom_op("se_b200::l1_logspec", mutates_args=())
def _l1_logspec(log_predicted: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, eps: float) -> torch.Tensor:
    log_predicted, linear_tar = _c(log_predicted, "log_predicted"), _c(linear_tar, "linear_tar")
    B, F, K = log_predicted.shape
    with torch.cuda.device(log_predicted.device):
        acc = torch.empty(2, device=log_predicted.device, dtype=torch.float64)
        rc = _lib.load().se_l1_logspec_fwd(log_predicted.data_ptr(), linear_tar.data_ptr(), stft_len.data_ptr(), B, F, K, eps,
                                           acc.data_ptr(), _stream())
        _lib.check(rc, "se_l1_logspec_fwd")
    return acc


@_l1_logspec.register_fake
def _(log_predicted, linear_tar, stft_len, eps):
    return log_predicted.new_empty(2, dtype=torch.float64)


@torch.library.custom_op("se_b200::l1_logspec_bwd", mutates_args=())
def _l1_logspec_bwd(log_predicted: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, eps: float,
                    count: float, grad_sum: torch.Tensor) -> torch.Tensor:
    log_predicted, linear_tar = _c(log_predicted, "log_predicted"), _c(linear_tar, "linear_tar")
    B, F, K = log_predicted.shape
    with torch.cuda.device(log_predicted.device):
        grad = torch.empty_like(log_predicted)
        g = grad_sum.reshape(1).to(torch.float32).contiguous()
        rc = _lib.load().se_l1_logspec_bwd(log_predicted.data_ptr(), linear_tar.data_ptr(), stft_len.data_ptr(), B, F, K, eps,
                                           float(count), g.data_ptr(), grad.data_ptr(), _stream())
        _lib.check(rc, "se_l1_logspec_bwd")
    return grad


@_l1_logspec_bwd.register_fake
def _(log_predicted, linear_tar, stft_len, eps, count, grad_sum):
    return torch.empty_like(log_predicted)


def _l1_setup(ctx, inputs, output):
    log_predicted, linear_tar, stft_len, eps = inputs
    ctx.save_for_backward(log_predicted, linear_tar, stft_len)
    ctx.eps = eps


def _l1_backward(ctx, grad_acc):
    log_predicted, linear_tar, stft_len = ctx.saved_tensors
    # acc[0] = sum |d|: gradient of the SUM with count = 1; the caller divides by the count
    grad = torch.ops.se_b200.l1_logspec_bwd(log_predicted, linear_tar, stft_len, ctx.eps, 1.0, grad_acc[0])
    return grad, None, None, None


_l1_logspec.register_autograd(_l1_backward, setup_context=_l1_setup)


def l1_logspec_sums(log_predicted, linear_tar, stft_len, eps=1e-10):
    """(sum |log_pred - log(tar+eps)|, number of valid elements) as a float64 (2,) tensor; differentiable."""
    return torch.ops.se_b200.l1_logspec(log_predicted, linear_tar, stft_len.contiguous(), float(eps))


# --------------------------------------------------------------------------- mask head
@torch.library.custom_op("se_b200::wsd_sums", mutates_args=())
def _wsd_sums(linear_inp: torch.Tensor, offset: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, energy: torch.Tensor,
              emax: torch.Tensor, alpha: float, db_interval: float, eps: float) -> torch.Tensor:
    """objective.WSD forward from the frame energies and the batch maximum of ``wsd_energy`` -> loss (1,)."""
    linear_inp, offset, linear_tar = _c(linear_inp, "linear_inp"), _c(offset, "offset"), _c(linear_tar, "linear_tar")
    B, F, K = linear_tar.shape
    dev = linear_tar.device
    with torch.cuda.device(dev):
        sums2 = torch.empty(B, 2, device=dev, dtype=torch.float64)
        loss = torch.empty(1, device=dev)
        rc = _lib.load().se_wsd_mask_step(offset.data_ptr(), K, linear_inp.data_ptr(), K, linear_tar.data_ptr(), K, stft_len.data_ptr(), 0,
                                          B, F, K, alpha, db_interval, eps, energy.data_ptr(), emax.data_ptr(), sums2.data_ptr(), 0, None,
                                          loss.data_ptr(), None, 0, _stream())
        _lib.check(rc, "se_wsd_mask_step")
    return loss


@_wsd_sums.register_fake
def _(linear_inp, offset, linear_tar, stft_len, energy, emax, alpha, db_interval, eps):
    return linear_tar.new_empty(1)


@torch.library.custom_op("se_b200::wsd_bwd", mutates_args=())
def _wsd_bwd(linear_inp: torch.Tensor, offset: torch.Tensor, linear_tar: torch.Tensor, stft_len: torch.Tensor, alpha: float,
             db_interval: float, eps: float, energy: torch.Tensor, emax: torch.Tensor, grad_loss: torch.Tensor) -> torch.Tensor:
    linear_inp, offset, linear_tar = _c(linear_inp, "linear_inp"), _c(offset, "offset"), _c(linear_tar, "linear_tar")
    B, F, K = linear_tar.shape
    with torch.cuda.device(linear_tar.device):
        grad = torch.empty_like(offset)
        g = grad_loss.reshape(1).to(torch.float32).contiguous()
        rc = _lib.load().se_wsd_bwd(linear_inp.data_ptr(), offset.data_ptr(), linear_tar.data_ptr(), stft_len.data_ptr(), B, F, K,
                                    alpha, db_interval, eps, energy.data_ptr(), emax.data_ptr(), g.data_ptr(), grad.data_ptr(),
                                    _stream())
        _lib.check(rc, "se_wsd_bwd")
    return grad


@_wsd_bwd.register_fake
def _(linear_inp, offset, linear_tar, stft_len, alpha, db_interval, eps, energy, emax, grad_loss):
    return torch.empty_like(offset)


def _wsd_setup(ctx, inputs, output):
    linear_inp, offset, linear_tar, stft_len, energy, emax, alpha, db_interval, eps = inputs
    ctx.save_for_backward(linear_inp, offset, linear_tar, stft_len, energy, emax)
    ctx.cfg = (alpha, db_interval, eps)


def _wsd_backward(ctx, grad_loss):
    linear_inp, offset, linear_tar, stft_len, energy, emax = ctx.saved_tensors
    alpha, db_interval, eps = ctx.cfg
    grad = torch.ops.se_b200.wsd_bwd(linear_inp, offset, linear_tar, stft_len, alpha, db_interval, eps, energy, emax, grad_loss)
    return None, grad, None, None, None, None, None, None, None   # the spectra are data: only the head's offset gets a gradient


_wsd_sums.register_autograd(_wsd_backward, setup_context=_wsd_setup)


def wsd(linear_inp, offset, linear_tar, stft_len, alpha=0.5, db_interval=30.0, eps=1e-10):
    """objective.py:120-153 (+ backward w.r.t. offset).  Returns the scalar loss.  The frame energies and their maximum come first
    and the maximum is all-reduced across data-parallel ranks (``dp.global_max``) before the sums: every rank then thresholds
    voicing against the loudest frame of the GLOBAL batch, as the single-process reference does.
    That all-reduce is a collective: while a process group of world size > 1 is initialized, EVERY rank must call this for
    every batch (a call made on some ranks only -- e.g. evaluation on rank 0 alone -- waits for the others forever)."""
    stft_len = _c(stft_len, "stft_len", torch.int64)
    linear_tar = _c(linear_tar, "linear_tar")
    energy, emax = wsd_energy(linear_tar, linear_tar.shape[2])
    dp.global_max(emax)
    return torch.ops.se_b200.wsd_sums(linear_inp, offset, linear_tar, stft_len, energy, emax, float(alpha), float(db_interval),
                                      float(eps))[0]


@torch.library.custom_op("se_b200::linear_head", mutates_args=())
def _linear_head(x: torch.Tensor, mean: torch.Tensor | None, std: torch.Tensor | None, cmvn_eps: float,
                 weight: torch.Tensor, bias: torch.Tensor | None, act: int, precision: int) -> torch.Tensor:
    x, weight, bias = _c(x, "features"), _c(weight, "weight"), _c(bias, "bias")
    B, F, Din = x.shape
    Dout = weight.shape[0]
    assert weight.shape[1] == Din
    with torch.cuda.device(x.device):
        out = torch.empty(B, F, Dout, device=x.device)
        rc = _lib.load().se_linear_head_fwd(x.data_ptr(), _p(mean), _p(std), cmvn_eps, weight.data_ptr(), _p(bias), B, F, Din,
                                            Dout, act, None, out.data_ptr(), None, precision, _stream())
        _lib.check(rc, "se_linear_head_fwd")
    return out


@_linear_head.register_fake
def _(x, mean, std, cmvn_eps, weight, bias, act, precision):
    return x.new_empty(x.shape[0], x.shape[1], weight.shape[0])


@torch.library.custom_op("se_b200::linear_head_bwd", mutates_args=())
def _linear_head_bwd(x: torch.Tensor, mean: torch.Tensor | None, std: torch.Tensor | None, cmvn_eps: float,
                     weight: torch.Tensor, offset: torch.Tensor, grad_offset: torch.Tensor, act: int,
                     precision: int) -> tuple[torch.Tensor, torch.Tensor]:
    x, offset, grad_offset = _c(x, "features"), _c(offset, "offset"), _c(grad_offset, "grad_offset")
    B, F, Din = x.shape
    Dout = weight.shape[0]
    with torch.cuda.device(x.device):
        gw = torch.empty(Dout, Din, device=x.device)
        gb = torch.empty(Dout, device=x.device)
        lib = _lib.load()
        ws_floats = lib.se_linear_head_bwd_tc_workspace(B, F, Din, Dout) if precision == 1 else 0
        if ws_floats > 0:                                   # tensor-core split-K GEMM (TF32 operands, fp32 accumulate)
            ws = torch.empty(ws_floats, device=x.device)
            rc = lib.se_linear_head_bwd_tc(x.data_ptr(), Din, _p(mean), _p(std), Din, cmvn_eps, offset.data_ptr(),
                                           grad_offset.data_ptr(), Dout, B, F, Din, Dout, act, ws.data_ptr(), ws_floats,
                                           gw.data_ptr(), gb.data_ptr(), _stream())
            _lib.check(rc, "se_linear_head_bwd_tc")
            return gw, gb
        rc = lib.se_linear_head_bwd(x.data_ptr(), _p(mean), _p(std), cmvn_eps, weight.data_ptr(), offset.data_ptr(),
                                            grad_offset.data_ptr(), B, F, Din, Dout, act, gw.data_ptr(), gb.data_ptr(), _stream())
        _lib.check(rc, "se_linear_head_bwd")
    return gw, gb


@_linear_head_bwd.register_fake
def _(x, mean, std, cmvn_eps, weight, offset, grad_offset, act, precision):
    return torch.empty_like(weight), weight.new_empty(weight.shape[0])


def _head_setup(ctx, inputs, output):
    x, mean, std, cmvn_eps, weight, bias, act, precision = inputs
    ctx.save_for_backward(x, mean, std, weight, output)
    ctx.cmvn_eps, ctx.act, ctx.has_bias, ctx.precision = cmvn_eps, act, bias is not None, precision


def _head_backward(ctx, grad_out):
    x, mean, std, weight, offset = ctx.saved_tensors
    gw = gb = None
    if ctx.needs_input_grad[4] or ctx.needs_input_grad[5]:
        gw, gb = torch.ops.se_b200.linear_head_bwd(x, mean, std, ctx.cmvn_eps, weight, offset, grad_out, ctx.act, ctx.precision)
    gx = None
    if ctx.needs_input_grad[0]:
        # the recurrent heads train the LSTM below the projection (model.py:57-60, 85-91): d loss / d x = (grad_out * act'(z)) W,
        # the same projection kernel run on the transposed weight.  (With the CMVN inside the op, x would also reach the
        # output through mean / std: the named path never differentiates that, so it is refused rather than approximated.)
        if mean is not None:
            raise RuntimeError("se_b200: linear_head with fused CMVN has no gradient w.r.t. its input (normalise in autograd instead)")
        if ctx.act == ACT["Sigmoid"]:
            gz = grad_out * offset * (1.0 - offset)
        elif ctx.act == ACT["ReLU"]:
            gz = grad_out * (offset > 0).to(grad_out.dtype)
        else:
            gz = grad_out
        gx = torch.ops.se_b200.linear_head(gz.contiguous(), None, None, 0.0, weight.t().contiguous(), None, ACT["Identity"], ctx.precision)
    return gx, None, None, None, gw, (gb if ctx.has_bias else None), None, None


_linear_head.register_autograd(_head_backward, setup_context=_head_setup)


def linear_head(x, weight, bias, activation="Sigmoid", mean=None, std=None, cmvn_eps=1e-6, precision=0):
    """act(cmvn(x) W^T + b): x (B, F, Din) -> (B, F, Dout); gradients flow to weight and bias, and -- without the fused
    CMVN -- to x (the projection after a trainable recurrent body)."""
    return torch.ops.se_b200.linear_head(x, mean, std, float(cmvn_eps), weight, bias, ACT[activation], int(precision))


def linear_head_fused(x, weight, bias, activation, mean, std, cmvn_eps, linears=None, want_offset=True, precision=0):
    """Inference-only variant that can also emit predicted = linears * offset from the GEMM epilogue."""
    x, weight, bias = _c(x, "features"), _c(weight, "weight"), _c(bias, "bias")
    B, F, Din = x.shape
    Dout = weight.shape[0]
    linears = _c(linears, "linears")
    with torch.cuda.device(x.device):
        off = torch.empty(B, F, Dout, device=x.device) if want_offset else None
        pred = torch.empty(B, F, Dout, device=x.device) if linears is not None else None
        rc = _lib.load().se_linear_head_fwd(x.data_ptr(), _p(mean), _p(std), float(cmvn_eps), weight.data_ptr(), _p(bias), B, F,
                                            Din, Dout, ACT[activation], _p(linears), _p(off), _p(pred), int(precision), _stream())
        _lib.check(rc, "se_linear_head_fwd")
    return off, pred
