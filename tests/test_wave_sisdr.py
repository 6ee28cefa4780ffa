"""Training on the waveform SI-SDR: the adjoint of the iSTFT (se_istft_bwd, se_mask_istft_bwd), the differentiable ops.istft,
se_wave_sisdr_finish / objective.WaveSISDR and the training and evaluation routes that use them.

CPU: the float64 oracle's adjoint against its own iSTFT (dot-product test), its closed-form SI-SDR gradient against torch
autograd, and the new tile bodies run serially under g++ (tests/host_harness_wave.cpp) against the oracle.
GPU: the library against the same oracle, the fused training routes against the autograd route and a float64 oracle of the
whole step, the captured step, the evaluation step and two data-parallel ranks."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import signal_path, stft_f64, wave_f64

HERE = os.path.dirname(os.path.abspath(__file__))
GEOS = [(256, 128), (400, 160), (512, 256), (1024, 256), (2048, 512), (256, 64)]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = tmp_path_factory.mktemp("harness_wave") / "host_harness.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out), os.path.join(HERE, "host_harness_wave.cpp")])
    return ctypes.CDLL(str(out))


def fptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def window(n_fft, win=None):
    return stft_f64.hann_periodic(win or n_fft, n_fft)


# ----------------------------------------------------------------------------------------------------------- CPU: oracle
@pytest.mark.parametrize("n_fft,hop,T,pad", [(256, 128, 1000, 0), (400, 160, 3333, 3400), (512, 256, 4000, 0),
                                             (1024, 256, 5000, 5100), (2048, 512, 9000, 0), (256, 64, 777, 800)])
def test_istft_adjoint_dot_product(n_fft, hop, T, pad):
    rng = np.random.default_rng(T)
    F, K = T // hop + 1, n_fft // 2 + 1
    w = window(n_fft, 400 if n_fft == 400 else None)
    Y = rng.standard_normal((2, F, K)) + 1j * rng.standard_normal((2, F, K))
    width = max(hop * (F - 1), pad)
    g = rng.standard_normal((2, width))
    y = stft_f64.istft(Y, n_fft, hop, w)
    y = np.concatenate([y, np.zeros((2, width - y.shape[1]))], 1)
    lhs = (y * g).sum()
    rhs = (Y * np.conj(wave_f64.istft_adjoint(g, n_fft, hop, F, w))).real.sum()
    assert abs(lhs - rhs) <= 1e-12 * max(1.0, abs(lhs)) * 100


def _sisdr_eval_torch(s, t, eps=1e-10):
    alpha = (s * t).sum() / ((t * t).sum() + eps)
    proj = alpha * t
    resid = ((proj - s) ** 2).sum() + eps
    return 10.0 * ((proj * proj).sum() / resid + eps).log10()


@pytest.mark.parametrize("case", ["plain", "silent_reference", "zero_estimate"])
def test_oracle_wave_sisdr_gradient_matches_autograd(case):
    g = torch.Generator().manual_seed(3)
    B, T = 4, 900
    src = torch.randn(B, T, generator=g, dtype=torch.float64)
    tar = 0.7 * src + 0.3 * torch.randn(B, T, generator=g, dtype=torch.float64)
    lengths = [900, 700, 333, 1]
    if case == "silent_reference":
        tar[1] = 0.0
    if case == "zero_estimate":
        src[2] = 0.0
    sisdr, grad = wave_f64.wave_sisdr(src, tar, lengths)
    s = src.clone().requires_grad_(True)
    vals = torch.stack([_sisdr_eval_torch(s[b, :n], tar[b, :n]) for b, n in enumerate(lengths)])
    (-vals.mean()).backward()
    assert torch.isfinite(sisdr).all() and torch.isfinite(grad).all()
    torch.testing.assert_close(sisdr, vals.detach(), rtol=1e-12, atol=1e-9)
    torch.testing.assert_close(grad, s.grad, rtol=1e-7, atol=1e-12 * float(s.grad.abs().max()))   # length 1: ill-conditioned
    for b, n in enumerate(lengths):
        ref = signal_path.sisdr_eval(src[b, :n], tar[b, :n])
        assert abs(float(sisdr[b]) - ref) < 1e-9


# ------------------------------------------------------------------------------------------------- CPU: the tile bodies
def _budget(n_fft):
    # fp32 FFT: rounding grows with log2(N); relative to the largest gradient element
    return 4e-6 * np.log2(n_fft)


@pytest.mark.parametrize("n_fft,hop", GEOS)
def test_istft_bwd_tile_matches_adjoint(harness, n_fft, hop):
    rng = np.random.default_rng(n_fft + hop)
    T = 13 * hop + hop // 3
    F, K = T // hop + 1, n_fft // 2 + 1
    w = window(n_fft).astype(np.float32)
    power = (rng.random((2, F, K)) + 0.05).astype(np.float32)
    power[0, 3, 5] = 0.0                                              # grad_power 0 there, grad_phase 0 too (sqrt(P) = 0)
    phase = rng.uniform(-np.pi, np.pi, (2, F, K)).astype(np.float32)
    width = hop * (F - 1) + 37                                        # a pad_to fill that carries no gradient
    g = rng.standard_normal((2, width)).astype(np.float32)
    gp, gph = np.zeros_like(power), np.zeros_like(power)
    rc = harness.h_istft_bwd(n_fft, fptr(g), ctypes.c_longlong(width), fptr(power), fptr(phase), 2, F, hop, fptr(w), fptr(gp), fptr(gph))
    assert rc == 0
    G = wave_f64.istft_adjoint(g.astype(np.float64), n_fft, hop, F, w.astype(np.float64))
    P, ph = power.astype(np.float64), phase.astype(np.float64)
    rot = G * np.exp(-1j * ph)
    mag = np.sqrt(P)
    ref_p = np.where(P > 0, rot.real / (2 * np.where(P > 0, mag, 1.0)), 0.0)
    ref_ph = mag * rot.imag
    assert gp[0, 3, 5] == 0.0 and gph[0, 3, 5] == 0.0
    assert np.abs(gp - ref_p).max() < _budget(n_fft) * np.abs(ref_p).max()
    assert np.abs(gph - ref_ph).max() < _budget(n_fft) * np.abs(ref_ph).max()


def mask_bwd_oracle(noisy, clean, y, coef, lengths, mask, n_fft, hop, w, log_power):
    """float64 gradient of se_mask_istft_bwd: g = alpha y + beta c on t < min(len, hop (F-1)), G = istft_adjoint(g), chain rule."""
    B, T = noisy.shape
    F = T // hop + 1
    out_len = hop * (F - 1)
    g = np.zeros((B, out_len))
    for b in range(B):
        n = min(int(lengths[b]), out_len)
        g[b, :n] = coef[b, 0] * y[b, :n] + coef[b, 1] * clean[b, :n]
    G = wave_f64.istft_adjoint(g, n_fft, hop, F, w)
    X = stft_f64.stft(noisy, n_fft, hop, w)
    m = mask.astype(np.float64)
    if log_power:
        ax = np.abs(X)
        Y = np.where(ax > 0, np.exp(m / 2) * X / np.where(ax > 0, ax, 1.0), np.exp(m / 2))
        return 0.5 * (G * np.conj(Y)).real
    return np.where(m > 0, (G * np.conj(X)).real / (2 * np.sqrt(np.where(m > 0, m, 1.0))), 0.0)


def mask_bwd_inputs(n_fft, hop, T, lengths, log_power, seed=0):
    rng = np.random.default_rng(seed + n_fft + T)
    B = len(lengths)
    F, K = T // hop + 1, n_fft // 2 + 1
    wavs = (0.05 * rng.standard_normal((B, 3, T))).astype(np.float32)
    wavs[:, 1] = 0.8 * wavs[:, 0] + 0.01 * rng.standard_normal((B, T)).astype(np.float32)
    y = (0.05 * rng.standard_normal((B, T))).astype(np.float32)
    coef = rng.standard_normal((B, 2)).astype(np.float32)
    if log_power:
        mask = rng.uniform(-4.0, 1.0, (B, F, K)).astype(np.float32)
    else:
        mask = rng.uniform(0.05, 1.0, (B, F, K)).astype(np.float32)
        mask[:, ::3, ::7] = 0.0                                       # exact zeros: gradient 0
    return wavs, y, coef, mask


@pytest.mark.parametrize("n_fft,hop", GEOS)
@pytest.mark.parametrize("log_power", [False, True])
def test_mask_istft_bwd_tile_matches_adjoint(harness, n_fft, hop, log_power):
    T = 11 * hop + hop // 2 + 3                                      # T % hop != 0
    lengths = np.array([T, n_fft - 5, T - hop - 7], np.int64)         # len = T, len < N, ragged
    wavs, y, coef, mask = mask_bwd_inputs(n_fft, hop, T, lengths, log_power)
    B, _, _ = wavs.shape
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = (K + 3) // 4 * 4
    mpad = np.zeros((B, F, LD), np.float32)
    mpad[..., :K] = mask
    out = np.full((B, F, LD), 7.0, np.float32)
    w = window(n_fft).astype(np.float32)
    rc = harness.h_mask_istft_bwd(n_fft, fptr(wavs), ctypes.c_void_p(wavs.ctypes.data + 4 * T), ctypes.c_longlong(3 * T), fptr(y),
                                  ctypes.c_longlong(T), fptr(coef), fptr(lengths), fptr(mpad), ctypes.c_longlong(LD), B, T, hop, fptr(w),
                                  fptr(out), int(log_power))
    assert rc == 0
    ref = mask_bwd_oracle(wavs[:, 0].astype(np.float64), wavs[:, 1].astype(np.float64), y.astype(np.float64), coef.astype(np.float64),
                          lengths, mask, n_fft, hop, w.astype(np.float64), log_power)
    assert (out[..., K:] == 0.0).all()
    got = out[..., :K]
    assert np.isfinite(got).all()
    if not log_power:
        assert (got[mask == 0.0] == 0.0).all()
    assert np.abs(got - ref).max() < _budget(n_fft) * np.abs(ref).max()


# ------------------------------------------------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import sys
    sys.path.insert(0, HERE)
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def _tr():
    import test_train_recurrent as tr
    return tr


@pytest.fixture(autouse=True)
def _no_cudnn_tf32():
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        yield


@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (400, 160), (256, 64)])
def test_istft_autograd_matches_adjoint(se, n_fft, hop):
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(n_fft)
    B, F, K = 2, 9, n_fft // 2 + 1
    power = (torch.rand(B, F, K, generator=g) + 0.05).cuda().requires_grad_(True)
    phase = ((torch.rand(B, F, K, generator=g) * 2 - 1) * np.pi).cuda().requires_grad_(True)
    win = ops.centered_window(torch.hann_window(n_fft).cuda(), n_fft)
    pad = hop * (F - 1) + 11
    gw = torch.randn(B, pad, generator=g).cuda()
    wav = ops.istft(power, phase, n_fft, hop, win, pad_to=pad)
    (wav * gw).sum().backward()
    G = wave_f64.istft_adjoint(gw.double().cpu().numpy(), n_fft, hop, F, win.double().cpu().numpy())
    P, ph = power.detach().double().cpu().numpy(), phase.detach().double().cpu().numpy()
    rot = G * np.exp(-1j * ph)
    ref_p, ref_ph = rot.real / (2 * np.sqrt(P)), np.sqrt(P) * rot.imag
    gp, gph = power.grad.double().cpu().numpy(), phase.grad.double().cpu().numpy()
    assert np.abs(gp - ref_p).max() < 1e-4 * np.abs(ref_p).max()
    assert np.abs(gph - ref_ph).max() < 1e-4 * np.abs(ref_ph).max()
    # directional derivative: istft is smooth in (P, phase); central difference of <g, istft> along a random direction
    dP, dph = torch.randn(B, F, K, generator=g).cuda() * 0.01, torch.randn(B, F, K, generator=g).cuda() * 0.01
    with torch.no_grad():
        f = lambda e: float((ops.istft(power + e * dP, phase + e * dph, n_fft, hop, win, pad_to=pad).double() * gw.double()).sum())
        fd = (f(1.0) - f(-1.0)) / 2.0
    an = float((power.grad * dP).sum() + (phase.grad * dph).sum())
    assert fd == pytest.approx(an, rel=2e-2)


@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (1024, 256), (400, 160), (256, 64)])
@pytest.mark.parametrize("log_power", [False, True])
def test_mask_istft_bwd_matches_adjoint(se, n_fft, hop, log_power):
    from speech_enhancement_by_s3prl_b200 import ops
    T = 23 * hop + hop // 2 + 3
    lengths = np.array([T, n_fft - 5, T - hop - 7, T // 2], np.int64)
    wavs, _, coef, mask = mask_bwd_inputs(n_fft, hop, T, lengths, log_power, seed=5)
    B = len(lengths)
    F, K = T // hop + 1, n_fft // 2 + 1
    LD = ops.round4(K)
    mpad = torch.zeros(B, F, LD)
    mpad[..., :K] = torch.from_numpy(mask)
    w_c, m_c, l_c = torch.from_numpy(wavs).cuda(), mpad.cuda(), torch.from_numpy(lengths).cuda()
    win = ops.centered_window(torch.hann_window(n_fft).cuda(), n_fft)
    y, _ = ops.mask_istft(w_c, 0, 1, m_c, l_c, n_fft, hop, win, pad_to=T, want_spec=False, mask_padded=True,
                          mask_is_log_power=log_power)
    got = ops.mask_istft_bwd(w_c, 0, 1, y, torch.from_numpy(coef).cuda(), l_c, m_c, n_fft, hop, win, mask_is_log_power=log_power)
    got = got.cpu().numpy()
    ref = mask_bwd_oracle(wavs[:, 0].astype(np.float64), wavs[:, 1].astype(np.float64), y.double().cpu().numpy(),
                          coef.astype(np.float64), lengths, mask, n_fft, hop, win.double().cpu().numpy(), log_power)
    assert (got[..., K:] == 0).all() and np.isfinite(got).all()
    if not log_power:
        assert (got[..., :K][mask == 0.0] == 0.0).all()
    assert np.abs(got[..., :K] - ref).max() < 1e-4 * np.abs(ref).max()


@gpu
def test_wave_sisdr_finish_and_sisdr_wave_backward(se):
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(1)
    B, T = 5, 3000
    src = torch.randn(B, T, generator=g, dtype=torch.float64)
    tar = 0.6 * src + 0.4 * torch.randn(B, T, generator=g, dtype=torch.float64)
    tar[1] = 0.0                                                              # silent reference
    src[3] = 0.0                                                              # all-zero estimate
    lengths = torch.LongTensor([3000, 2000, 1500, 2500, 10])
    sisdr64, grad64 = wave_f64.wave_sisdr(src, tar, lengths)
    s = src.float().cuda().requires_grad_(True)
    crit = se.WaveSISDR()
    loss, _ = crit(wav_predicted=s, wav_tar=tar.float().cuda(), lengths=lengths.cuda())
    loss.backward()
    assert torch.isfinite(loss) and torch.isfinite(s.grad).all()
    assert loss.item() == pytest.approx(float(-sisdr64.mean()), rel=1e-4, abs=1e-4)
    gg = s.grad.double().cpu()
    assert (gg[:, 3000:] == 0).all() and (gg[2, 1500:] == 0).all()
    for b in range(B):
        scale = grad64[b].abs().max().item()
        assert (gg[b] - grad64[b]).abs().max().item() <= 2e-3 * scale + 1e-30, b
    # the finish kernel on K3-shaped sums: coefficients, mean, metric accumulators
    sums = torch.zeros(B, 6, dtype=torch.float64)
    for b, n in enumerate(lengths.tolist()):
        sums[b, :3] = torch.stack([(src[b, :n] * tar[b, :n]).sum(), (tar[b, :n] ** 2).sum(), (src[b, :n] ** 2).sum()])
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    lpu, lmean, coef = ops.wave_sisdr_finish(sums.cuda(), metric_acc=acc)
    torch.testing.assert_close(lpu.double().cpu(), -sisdr64, rtol=1e-5, atol=1e-4)
    assert float(lmean) == pytest.approx(float(lpu.double().mean()), rel=1e-6)
    a = acc.cpu()
    assert a[0].item() == pytest.approx(float(lpu.double().sum()), rel=1e-6) and a[1].item() == pytest.approx(-a[0].item())
    assert a[2].item() == B
    c = coef.double().cpu()
    for b, n in enumerate(lengths.tolist()):
        gb = c[b, 0] * src[b, :n] + c[b, 1] * tar[b, :n]
        assert (gb - grad64[b, :n]).abs().max().item() <= 1e-5 * grad64[b].abs().max().item() + 1e-30
    assert (c[1] == 0).all() and (c[3] == 0).all()


# ---------------------------------------------------------------------------------------------- the training routes
def _pre(se, n_fft, hop):
    n_freq, win_ms = {512: (257, 32), 400: (201, 25), 1024: (513, 64), 256: (129, 16)}[n_fft]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop // 16, n_freq=n_freq).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    return pre


def _linres(se, n_freq, device="cuda"):
    torch.manual_seed(11)
    return se.LinearResidual(n_freq, n_freq, precision=1).to(device)


def _oracle_wave_step(eng, lengths, wavs, make_mag):
    """The whole training step in float64 on the CPU: spectra by the oracle, make_mag(feats, linear_inp, |X|) -> the magnitude
    of the decoded spectrum (sqrt of the predicted power, recorded for autograd), istft(magnitude X / |X|) by torch.istft, -mean
    sisdr_eval.  Returns the loss."""
    n_fft, hop = eng.n_fft, eng.hop
    w = eng.pre._frame_window.double().cpu()
    x = wavs.double().cpu().numpy()
    T = x.shape[2]
    X = torch.from_numpy(stft_f64.stft(x[:, 0], n_fft, hop, w.numpy()))
    linear_inp = X.abs() ** 2
    feats = torch.log(linear_inp + eng.pre.eps)
    ax = X.abs()
    unit = torch.where(ax > 0, X / torch.where(ax > 0, ax, torch.ones_like(ax)), torch.ones_like(X))
    Y = make_mag(feats, linear_inp, ax) * unit
    wav = torch.istft(Y.transpose(1, 2), n_fft, hop, n_fft, w, center=True)
    wav = torch.nn.functional.pad(wav, (0, T - wav.shape[1]))
    clean = torch.from_numpy(x[:, 1])
    terms = []
    for b, n in enumerate(lengths.tolist()):
        s, t = wav[b, :n], clean[b, :n]
        a = (s * t).sum() / ((t * t).sum() + 1e-10)
        terms.append(-10.0 * torch.log10((a * t).pow(2).sum() / ((a * t - s).pow(2).sum() + 1e-10) + 1e-10))
    return torch.stack(terms).mean()


def _assert_close_to_f64(got, ref):
    for name, g64 in ref.items():
        g = got[name].double().cpu().flatten()
        g64 = g64.double().cpu().flatten()
        cos = torch.dot(g, g64) / (g.norm() * g64.norm())
        assert cos.item() > 0.9999, f"{name}: cosine {cos.item():.6f}"
        assert (g - g64).abs().max().item() < 1e-2 * g64.abs().max().item(), name


@gpu
@pytest.mark.parametrize("n_fft,hop,T", [(512, 256, 12000), (400, 160, 9000), (256, 64, 5000)])
def test_fused_linear_residual_step(se, n_fft, hop, T):
    tr = _tr()
    lengths, wavs = tr._ragged(3, T, hop, seed=n_fft + 3)
    pre = _pre(se, n_fft, hop)
    head = _linres(se, n_fft // 2 + 1)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = se.WaveSISDR()
    (l_f, g_f), (l_a, g_a) = [tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), crit, fused) for fused in (True, False)]
    assert np.isfinite(l_f) and l_f == pytest.approx(l_a, rel=2e-4, abs=2e-4)
    _assert_close_to_f64(g_f, g_a)
    W = head.linear.weight.detach().double().cpu().clone().requires_grad_(True)
    b = head.linear.bias.detach().double().cpu().clone().requires_grad_(True)
    loss64 = _oracle_wave_step(eng, lengths, wavs, lambda f, lin, ax: signal_path.linear_residual_head(
        f, lin, W, b, head.activation, head.cmvn, head.eps)[1].sqrt() * ax)
    loss64.backward()
    assert l_f == pytest.approx(loss64.item(), rel=1e-3, abs=1e-3)
    _assert_close_to_f64(g_f, {"linear.weight": W.grad, "linear.bias": b.grad})


@gpu
def test_fused_step_with_forced_generic_kernels(se):
    from speech_enhancement_by_s3prl_b200 import _lib
    tr = _tr()
    lengths, wavs = tr._ragged(3, 12000, 256, seed=41)
    pre = _pre(se, 512, 256)
    head = _linres(se, 257)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = se.WaveSISDR()
    ref = tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), crit, True)
    _lib.check(_lib.load().se_set_option(0, 1), "se_set_option")
    try:
        got = tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), crit, True)
    finally:
        _lib.check(_lib.load().se_set_option(0, 0), "se_set_option")
    assert got[0] == pytest.approx(ref[0], rel=1e-4, abs=1e-4)
    tr._assert_grads_agree(got[1], ref[1])


@gpu
@pytest.mark.parametrize("kind,bidir", [("Residual", False), ("LSTM", False), ("LSTM", True)])
def test_fused_recurrent_wave_step(se, monkeypatch, kind, bidir):
    tr = _tr()
    lengths, wavs = tr._ragged(3, 12000, 256, seed=19)
    pre = _pre(se, 512, 256)
    head = tr._head(se, kind, 257, 32, 2, bidir)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = se.WaveSISDR()
    (l_f, g_f), (l_a, g_a) = [tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), crit, fused) for fused in (True, False)]
    assert np.isfinite(l_f) and l_f == pytest.approx(l_a, rel=2e-4, abs=2e-4)
    state = {k: v.detach().double().cpu().clone().requires_grad_(k.startswith("scaling_layer")) for k, v in head.state_dict().items()}
    made = []

    class _Recorded(torch.nn.LSTM):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            made.append(self)

    monkeypatch.setattr(torch.nn, "LSTM", _Recorded)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        def mag(f, lin, ax):
            _, extra = signal_path.recurrent_head(kind, state, f, lin, bidirectional=bidir, activation=head.activation,
                                                  cmvn=getattr(head, "cmvn", False))
            return (extra["log_predicted"] / 2).exp() if kind == "LSTM" else extra["offset"].sqrt() * ax

        loss64 = _oracle_wave_step(eng, lengths, wavs, mag)
        loss64.backward()
    finally:
        torch.set_default_dtype(prev)
        monkeypatch.undo()
    ref = {"lstm." + n: p.grad for n, p in made[0].named_parameters()}
    ref.update({k: v.grad for k, v in state.items() if k.startswith("scaling_layer")})
    assert l_f == pytest.approx(loss64.item(), rel=1e-3, abs=1e-3)
    assert set(ref) == set(g_f)
    _assert_close_to_f64(g_f, ref)


@gpu
def test_route_check_by_kernel_names(se):
    tr = _tr()
    lengths, wavs = tr._ragged(4, 16000, 256, seed=3)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    pre = _pre(se, 512, 256)
    crit = se.WaveSISDR()
    for head in (_linres(se, 257), tr._head(se, "Residual", 257, 64, 2), tr._head(se, "LSTM", 257, 64, 2)):
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        opt = se.ClipAdam(head.parameters(), lr=1e-4)
        assert eng.fused_training_supported(crit, 4, 16000)
        names = tr._kernel_names(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0))
        has = lambda s: any(s in n for n in names)
        assert has("mask_istft_bwd_kernel") and has("linear_head_bwd_tma_kernel") and has("wave_sisdr_finish_kernel"), names
        assert has("adam_update_kernel") and not any("Adam" in n and "AdamArgs" not in n for n in names), names
        assert not any(has(k) for k in ("sisdr_mask", "wsd_", "l1_mask", "l1_logspec", "sisdr_spec")), names
    # a pair without a fused route (Linear) takes the autograd route through ops.istft's backward and still trains
    torch.manual_seed(5)
    head = se.Linear(257, 257, precision=1).cuda()
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    assert not eng.fused_training_supported(crit, 4, 16000)
    opt = torch.optim.Adam(head.parameters(), lr=1e-3)
    w0 = head.linear.weight.detach().clone()
    names = tr._kernel_names(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0))
    assert any("istft_bwd_kernel" in n for n in names) and any("wave_sisdr_bwd_kernel" in n for n in names)
    assert (head.linear.weight - w0).abs().max().item() > 0


@gpu
def test_train_step_graph_follows_eager_fused_steps(se):
    tr = _tr()
    lengths, wavs = tr._ragged(4, 16000, 256, seed=31)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    bad = wavs.clone()
    bad[1, 0, 100] = float("nan")                                    # a batch whose gradient norm is NaN: skipped on the device
    pre = _pre(se, 512, 256)
    crit = se.WaveSISDR()
    finals = []
    for graph in (False, True):
        head = _linres(se, 257)
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        opt = se.ClipAdam(head.parameters(), lr=1e-3)
        p0 = [p.detach().clone() for p in head.parameters()]
        step = (lambda x: eng.train_step_graph(lengths, x, crit, opt, 1.0)) if graph else (lambda x: eng.train_step(lengths, x, crit, opt, 1.0))
        batches = [wavs] * (3 if graph else 6) + [bad, wavs, wavs]   # graph: 3 eager warm-ups inside capture_train
        for x in batches:
            loss = step(x)
        torch.cuda.synchronize()
        assert opt.steps_taken() == [8] and opt.steps_skipped() == [1]
        finals.append((loss.item(), [p.detach().clone() for p in head.parameters()], p0))
    (l_e, p_e, p0), (l_g, p_g, _) = finals
    assert max((a - b).abs().max().item() for a, b in zip(p_e, p0)) > 1e-3
    assert l_g == pytest.approx(l_e, rel=1e-4, abs=1e-4)
    for a, b in zip(p_e, p_g):
        assert (a - b).abs().max().item() < 1e-4


@gpu
def test_eval_step_reports_minus_sisdr(se):
    tr = _tr()
    lengths, wavs = tr._ragged(4, 16000, 256, seed=7)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    pre = _pre(se, 512, 256)
    for head in (_linres(se, 257), tr._head(se, "LSTM", 257, 64, 2)):
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        acc = torch.zeros(3, dtype=torch.float64, device="cuda")
        out = eng.eval_step(lengths, wavs, metric_acc=acc, criterion=se.WaveSISDR())
        torch.cuda.synchronize()
        assert torch.equal(out["loss_per_utt"], -out["sisdr"])
        assert acc[0].item() == pytest.approx(-acc[1].item(), rel=1e-6) and acc[2].item() == 4
        assert acc[0].item() == pytest.approx(float(out["loss_per_utt"].double().sum()), rel=1e-6)
        st = eng.eval_step_graph(lengths, wavs, criterion=se.WaveSISDR())
        torch.cuda.synchronize()
        assert torch.equal(st["loss_per_utt"], -st["sisdr"]) and torch.equal(st["sisdr"], out["sisdr"])


def _dp_worker(rank, world_size, port, ret):
    import sys
    sys.path.insert(0, HERE)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp
    tr = _tr()
    lengths, wavs = tr._ragged(4, 12000, 256, seed=23)
    lengths, wavs = dp.shard_batch(lengths, wavs, rank, world_size)                  # 2 / 2 utterances
    pre = _pre(se, 512, 256)
    head = _linres(se, 257)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    loss, grads = tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), se.WaveSISDR(), True)
    ret[rank] = (loss, {n: g.cpu() for n, g in grads.items()})
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_two_ranks_give_the_single_process_gradient(se):
    import torch.multiprocessing as mp
    tr = _tr()
    world_size = 2
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(world_size, tr._free_port(), ret), nprocs=world_size, join=True)
    lengths, wavs = tr._ragged(4, 12000, 256, seed=23)
    head = _linres(se, 257)
    eng = se.EnhancementEngine(_pre(se, 512, 256), head, log_features=True, precision=1)
    loss, ref = tr._grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), se.WaveSISDR(), True)
    assert (ret[0][0] + ret[1][0]) / 2 == pytest.approx(loss, rel=1e-4, abs=1e-4)
    for name, g in ref.items():
        assert torch.equal(ret[0][1][name], ret[1][1][name])
    tr._assert_grads_agree({n: g for n, g in ret[0][1].items()}, {n: g.cpu() for n, g in ref.items()})
