"""The evaluation metric sums of the fused mask -> iSTFT kernel (K3, se_mask_istft_ex), their epilogue (K3',
se_finalize_metrics_acc) and the waveform helpers (se_sisdr_wave, se_masked_normalize_db) against float64 restatements.

Reference of K3 (direct DFT of oracle/stft_f64.py, no FFT library), per row with n = min(max(len, 0), T):
  X = stft(noisy), C = stft(clean) over the whole padded row; Y = X sqrt(mask) (power mode: sqrt(P) X / |X|, sqrt(P)
  where X = 0); y = istft(Y), zero beyond hop (F - 1);
  YC, CC, YY = sums over t < n;  ST, TT, SS = sums over frames f < min(F, n // hop + 1) of sqrt(relu(pred) tar), tar,
  relu(pred) with pred = mask |X|^2 (power mode: P) and tar = |C|^2.

Every boundary case is built so that an off-by-one shows: the rows are NOT zeroed past their length (the sums run over
t < len whatever the data), a loud burst covers the last hop before the length and the first one after it, and the
mask is large on the frames around the boundary.  ``assert_sensitive`` checks, for each row, that the reference with one
frame more or fewer, or one sample more or fewer, lies at least SENSITIVITY times outside the tolerance the kernel is held
to -- so the tolerances below are tight enough to see every such mistake.

Measured on one B200 (1000 W power limit), largest error of the fp32 kernels against float64 over every case of this
file, both routes, mask and power mode:
  the six K3 sums, relative to each sum          5.0e-7  (n_fft 400 / hop 160, 200 rows of 700 samples; 1.3e-7 .. 4.1e-7
                                                          at the other geometries)  -> SUM_RTOL 2e-6
  K3 waveform, relative to the row's max |y|     4.7e-7  (n_fft 512 / hop 256, T = 300)  -> WAV_RTOL 2e-6
  se_sisdr_wave                                  6.4e-6 dB  -> 3e-5 dB
  se_masked_normalize_db, relative to the row    1.1e-7  -> 5e-7
At these tolerances the smallest sensitivity margin is about 1800 tolerances (n_fft 2048 / hop 512).
"""
import math

import numpy as np
import pytest
import torch

from oracle import signal_path as sp
from oracle import stft_f64

gpu = pytest.mark.gpu

# tolerances of the fp32 kernels against float64 (a few times the maximum observed on a B200)
SUM_RTOL = 2e-6            # each of the six sums, relative to its reference value
SUM_ATOL = 1e-12
WAV_RTOL = 2e-6            # |wav - y| relative to max |y| of the row
SENSITIVITY = 10.0         # an off-by-one frame or sample must miss the reference by this many tolerances

# name -> (n_fft, hop, win_ms, hop_ms)
GEOS = {"512/256": (512, 256, 32, 16), "1024/256": (1024, 256, 64, 16), "400/160": (400, 160, 25, 10),
        "256/128": (256, 128, 16, 8), "512/160": (512, 160, 32, 10), "2048/512": (2048, 512, 128, 32)}


def boundary_lengths(n_fft, hop, T):
    """T, T - 1, k hop - 1, k hop, k hop + 1 (interior k), n_fft/2 + 1, 1 and a length beyond T (clamped to T)."""
    k = max(1, (T // hop) // 2)
    return [T, T - 1, k * hop - 1, k * hop, k * hop + 1, n_fft // 2 + 1, 1, T + 7]


def _cases():
    cases = []
    for geo, (n_fft, hop, _, _) in GEOS.items():
        for kind, T in (("mult", 48 * hop), ("nonmult", 48 * hop + hop // 3 + 1)):
            cases.append(pytest.param(geo, T, boundary_lengths(n_fft, hop, T), id=f"{geo}-{kind}"))
    # batches that fall back: fewer than six frames (the register-resident n_fft 1024 / 400 kernels need six) and the
    # two-frame minimum of the n_fft 512 kernel, 200 tiny rows
    for geo, T in (("1024/256", 1100), ("400/160", 700), ("512/256", 300)):
        n_fft, hop = GEOS[geo][:2]
        base = boundary_lengths(n_fft, hop, T)
        cases.append(pytest.param(geo, T, [base[i % len(base)] for i in range(200)], id=f"{geo}-tiny200"))
    # one long row (30 s and more): thousands of runs per row in the fast paths
    for geo in ("512/256", "400/160", "1024/256"):
        n_fft, hop = GEOS[geo][:2]
        T = 480000 + hop // 2 + 3
        k = (T // hop) // 2 + 3
        cases.append(pytest.param(geo, T, [T, k * hop, k * hop + 1], id=f"{geo}-long"))
    return cases


CASES = _cases()


def window_of(geo):
    from speech_enhancement_by_s3prl_b200.preprocessor import OnlinePreprocessor
    n_fft, hop, win_ms, hop_ms = GEOS[geo]
    pre = OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_fft // 2 + 1)
    assert pre._win_args["hop_length"] == hop and pre._frame_window.shape == (n_fft,)
    return pre._frame_window


def power_target(wavs, mask, n_fft, hop, window):
    """The power-mode input P = mask |X|^2 (float64 |X|, rounded to float32): sqrt(P) X / |X| keeps the noisy phase, and
    a bin whose phase is rounding noise (|X| near 0) also has a magnitude near 0, so the float64 comparison stays well
    conditioned.  (A random P would give such bins magnitudes of order one and a phase no fp32 transform can pin.)"""
    X = stft_f64.stft(wavs[:, 0].astype(np.float64), n_fft, hop, np.asarray(window, dtype=np.float64))
    return (mask.astype(np.float64) * np.abs(X) ** 2).astype(np.float32)


def make_case(n_fft, hop, T, lengths, seed):
    """(B, 3, T) float32 [noisy, clean, noise] and a (B, F, K) float32 mask; every row has a burst of |x| >= 0.5 over
    [n - hop, n + hop) around its clamped length n (|x| >= 1 at n - 1 and n), the mask is in [2, 4) on frames n // hop - 1 .. n // hop + 1 and in
    [0.05, 1) elsewhere; noise of every channel everywhere else, also past the length."""
    g = np.random.default_rng(seed)
    B, F, K = len(lengths), T // hop + 1, n_fft // 2 + 1
    clean = 0.02 * g.standard_normal((B, T))
    noise = 0.01 * g.standard_normal((B, T))
    mask = g.uniform(0.05, 1.0, (B, F, K))
    for b, n in enumerate(min(max(v, 0), T) for v in lengths):
        lo, hi = max(0, n - hop), min(T, n + hop)
        clean[b, lo:hi] = g.choice([-1.0, 1.0], hi - lo) * g.uniform(0.5, 1.0, hi - lo)
        edge = slice(max(0, n - 1), min(T, n + 1))                  # the last sample counted and the first one not
        clean[b, edge] *= 2.0
        k = n // hop
        f0, f1 = max(0, k - 1), min(F, k + 2)
        mask[b, f0:f1] = g.uniform(2.0, 4.0, (f1 - f0, K))
    wavs = np.stack([clean + noise, clean, noise], 1).astype(np.float32)
    return wavs, mask.astype(np.float32)


class Reference:
    """float64 K3 of one batch: the waveform y and prefix sums over samples and frames, so that the sums for any
    (samples, frames) count are O(1)."""

    def __init__(self, wavs, mask, n_fft, hop, window, power=False):
        noisy, clean = wavs[:, 0].astype(np.float64), wavs[:, 1].astype(np.float64)
        w = np.asarray(window, dtype=np.float64)
        X = stft_f64.stft(noisy, n_fft, hop, w)
        C = stft_f64.stft(clean, n_fft, hop, w)
        X[..., 0] = X[..., 0].real                   # a real signal's DC and Nyquist bins are real: drop the DFT's residue
        X[..., -1] = X[..., -1].real
        m = mask.astype(np.float64)
        ax2 = np.abs(X) ** 2
        if power:
            ax = np.sqrt(ax2)
            unit = np.where(ax > 0, X / np.where(ax > 0, ax, 1.0), 1.0)
            Y, pred = np.sqrt(m) * unit, m
        else:
            Y, pred = X * np.sqrt(m), m * ax2
        self.y = stft_f64.istft(Y, n_fft, hop, w)                 # (B, hop (F - 1))
        self.T, self.F, self.hop = wavs.shape[-1], X.shape[1], hop
        B, L = self.y.shape
        yfull = np.zeros((B, self.T))
        yfull[:, :L] = self.y
        z = np.zeros((B, 1))
        self.cw = [np.concatenate([z, np.cumsum(v, axis=1)], 1) for v in (yfull * clean, clean * clean, yfull * yfull)]
        rp, tar = np.maximum(pred, 0.0), np.abs(C) ** 2
        self.cs = [np.concatenate([z, np.cumsum(v.sum(-1), axis=1)], 1) for v in (np.sqrt(rp * tar), tar, rp)]

    def sums(self, b, samples, frames):
        return np.array([c[b, samples] for c in self.cw] + [c[b, frames] for c in self.cs])

    def counts(self, length):
        n = self.T if length is None else min(max(int(length), 0), self.T)
        return n, min(self.F, n // self.hop + 1)

    def batch_sums(self, lengths):
        return np.stack([self.sums(b, *self.counts(None if lengths is None else lengths[b])) for b in range(self.y.shape[0])])


def sum_tol(ref_sums):
    return SUM_RTOL * np.abs(ref_sums) + SUM_ATOL


def assert_sensitive(ref, lengths):
    """Each row's reference with one sample / one frame more or fewer lies >= SENSITIVITY tolerances away.
    Returns the smallest margin (in tolerances) over the rows and the four perturbations."""
    worst = math.inf
    for b in range(ref.y.shape[0]):
        ns, nf = ref.counts(None if lengths is None else lengths[b])
        r = ref.sums(b, ns, nf)
        tol = sum_tol(r)
        for ns2, nf2 in ((ns - 1, nf), (ns + 1, nf), (ns, nf - 1), (ns, nf + 1)):
            if not (0 <= ns2 <= ref.T and 0 <= nf2 <= ref.F):
                continue                                              # no such count: the kernels clamp to the row
            margin = float(np.max(np.abs(ref.sums(b, ns2, nf2) - r) / tol))
            assert margin >= SENSITIVITY, (f"row {b} (len {lengths[b] if lengths else None}): samples {ns}->{ns2}, frames "
                                           f"{nf}->{nf2} is only {margin:.1f} tolerances away")
            worst = min(worst, margin)
    return worst


def sisdr_from_sums64(st, tt, ss, eps=1e-10):
    """The epilogue's SI-SDR from <s,t>, <t,t>, <s,s> (evaluation.py:5-10 expanded), in float64."""
    a = st / (tt + eps)
    den = max(a * a * tt - 2.0 * a * st + ss, 0.0)
    return 10.0 * math.log10(a * a * tt / (den + eps) + eps)


# ------------------------------------------------------------------------------ CPU: the reference itself
def test_reference_matches_the_torch_oracle_and_the_metric_formulas():
    """The float64 K3 reference against the torch oracle preprocessor (stft / istft), oracle.signal_path.sisdr_spectral
    (objective.SISDR's per-utterance term) and decode_wav + sisdr_eval (level normalisation + waveform SI-SDR)."""
    from oracle.preprocessor import OnlinePreprocessor as OraclePre
    n_fft, hop = 512, 256
    T = 20 * hop + 77
    lengths = [T, 11 * hop, 11 * hop + 1, 300]
    wavs, mask = make_case(n_fft, hop, T, lengths, seed=5)
    window = window_of("512/256")
    ref = Reference(wavs, mask, n_fft, hop, window)
    ora = OraclePre(win_ms=32, hop_ms=16, n_freq=257)
    c = ora.get_feat_config
    lin, ph = ora(torch.from_numpy(wavs), [c("linear", 0), c("phase", 0)])
    y_ora = ora.istft(lin * torch.from_numpy(mask), ph).double().numpy()
    assert np.abs(ref.y - y_ora).max() < 1e-5 * np.abs(ref.y).max()
    X = stft_f64.stft(wavs[:, 0].astype(np.float64), n_fft, hop, window.double().numpy())
    Cs = stft_f64.stft(wavs[:, 1].astype(np.float64), n_fft, hop, window.double().numpy())
    assert np.abs(np.abs(X) ** 2 - lin.double().numpy()).max() < 1e-5 * (np.abs(X) ** 2).max()
    L = torch.tensor(lengths)
    sums = ref.batch_sums(lengths)
    # spectral term: objective.py:86-100 on predicted = mask |X|^2, the frames of runner.py:455
    frames = sp.length_masks(sp.stft_lengths(L, hop))
    frames = torch.cat([frames, frames.new_zeros(len(lengths), ref.F - frames.shape[1])], 1).double()
    pred = torch.from_numpy(mask.astype(np.float64) * np.abs(X) ** 2)
    _, per_utt = sp.sisdr_spectral(pred, torch.from_numpy(np.abs(Cs) ** 2), frames)
    ours = [-sisdr_from_sums64(*s[3:]) for s in sums]
    np.testing.assert_allclose(ours, per_utt.numpy(), rtol=0, atol=1e-9)
    # waveform: masked_normalize_decibel against the clean level, then sisdr_eval over the first len samples
    y = np.zeros((len(lengths), T))
    y[:, :ref.y.shape[1]] = ref.y
    clean = torch.from_numpy(wavs[:, 1].astype(np.float64))
    scaled = sp.masked_normalize_decibel(torch.from_numpy(y), clean, sp.length_masks(L).double())
    for b, n in enumerate(lengths):
        yc, cc, yy = sums[b, :3]
        np.testing.assert_allclose(sums[b, :3], [y[b, :n] @ wavs[b, 1, :n], clean[b, :n] @ clean[b, :n], y[b, :n] @ y[b, :n]],
                                   rtol=1e-12)
        gain = math.sqrt((cc / (n + 1e-8)) / (yy / (n + 1e-8) + 1e-8))
        assert sisdr_from_sums64(gain * yc, cc, gain * gain * yy) == pytest.approx(sp.sisdr_eval(scaled[b, :n], clean[b, :n]),
                                                                                 abs=1e-9)
    # the power-mode reference keeps the noisy phase: a target spectrum equal to |X|^2 mask reproduces the mask mode
    pw = Reference(wavs, (mask.astype(np.float64) * np.abs(X) ** 2), n_fft, hop, window, power=True)
    assert np.abs(pw.y - ref.y).max() < 1e-12 * np.abs(ref.y).max()
    np.testing.assert_allclose(pw.batch_sums(lengths), sums, rtol=1e-12)


@pytest.mark.parametrize("geo,T,lengths", CASES)
def test_reference_sees_one_frame_and_one_sample(geo, T, lengths):
    """The boundary cases of the GPU tests below are sensitive at the tolerances used (see assert_sensitive)."""
    n_fft, hop = GEOS[geo][:2]
    wavs, mask = make_case(n_fft, hop, T, lengths, seed=T + len(lengths))
    window = window_of(geo)
    assert_sensitive(Reference(wavs, mask, n_fft, hop, window), lengths)
    assert_sensitive(Reference(wavs, power_target(wavs, mask, n_fft, hop, window), n_fft, hop, window, power=True), lengths)


# ------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def run_k3(wavs_d, mask_d, lengths_d, n_fft, hop, window_d, generic, clean=True, **kw):
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    lib = _lib.load()
    if generic:
        lib.se_set_option(0, 1)                                  # SE_OPT_FORCE_GENERIC
    try:
        wav, sums = ops.mask_istft(wavs_d, 0, 1 if clean else None, mask_d, lengths_d, n_fft, hop, window_d, **kw)
        torch.cuda.synchronize()
    finally:
        if generic:
            lib.se_set_option(0, 0)
    return wav.double().cpu().numpy(), sums.cpu().numpy()


def check_wav(wav, ref, label):
    """wav within WAV_RTOL of the row's largest |y| up to hop (F - 1), exactly zero from there to the width."""
    L = ref.y.shape[1]
    err = float((np.abs(wav[:, :L] - ref.y) / np.abs(ref.y).max(axis=1, keepdims=True)).max())
    assert err <= WAV_RTOL, f"{label}: waveform error {err:.3g} of the row maximum > {WAV_RTOL}"
    assert (wav[:, L:] == 0).all(), f"{label}: samples past hop * (F - 1) are not zero"


def check_sums(got, want, label):
    bad = np.abs(got - want) > sum_tol(want)
    assert not bad.any(), (f"{label}: sums differ from float64 at (row, sum) {np.argwhere(bad)[:6].tolist()}: "
                           f"got {got[bad][:6]}, want {want[bad][:6]}")


@gpu
@pytest.mark.parametrize("geo,T,lengths", CASES)
def test_mask_istft_sums_match_float64(se, geo, T, lengths):
    """All six sums and the waveform of se_mask_istft_ex against the float64 reference: default and forced-generic
    route, mask and power modes, want_spec off (spectral sums exactly 0), no clean channel (only YY), a padded mask with
    NaN pad columns, pad_to beyond hop (F - 1), ragged lengths including 1, n_fft/2 + 1 and one beyond T."""
    n_fft, hop = GEOS[geo][:2]
    K, F = n_fft // 2 + 1, T // hop + 1
    wavs, mask = make_case(n_fft, hop, T, lengths, seed=T + len(lengths))
    window = window_of(geo)
    P = power_target(wavs, mask, n_fft, hop, window)
    refs = {False: Reference(wavs, mask, n_fft, hop, window), True: Reference(wavs, P, n_fft, hop, window, power=True)}
    for ref in refs.values():
        assert_sensitive(ref, lengths)
    want = {p: r.batch_sums(lengths) for p, r in refs.items()}
    wavs_d, mask_d, win_d = torch.from_numpy(wavs).cuda(), torch.from_numpy(mask).cuda(), window.cuda()
    inputs = {False: mask_d, True: torch.from_numpy(P).cuda()}
    len_d = torch.tensor(lengths, dtype=torch.int64, device="cuda")
    LD = (K + 3) // 4 * 4 + 4
    mask_nan = torch.full((len(lengths), F, LD), float("nan"), device="cuda")
    mask_nan[..., :K] = mask_d
    pad_to = max(T, hop * (F - 1)) + hop + 3
    for generic in (False, True):
        route = "generic" if generic else "default"
        for power in (False, True):
            label = f"{geo} T={T} {route} {'power' if power else 'mask'}"
            wav, sums = run_k3(wavs_d, inputs[power], len_d, n_fft, hop, win_d, generic, pad_to=T, mask_is_power=power)
            check_sums(sums, want[power], label)
            check_wav(wav, refs[power], label)
        # want_spec off: the waveform sums as before, the spectral sums exactly zero
        wav, sums = run_k3(wavs_d, mask_d, len_d, n_fft, hop, win_d, generic, pad_to=T, want_spec=False)
        check_sums(sums[:, :3], want[False][:, :3], f"{geo} {route} want_spec=0")
        assert (sums[:, 3:] == 0).all(), f"{geo} {route}: want_spec=0 left spectral sums"
        # no clean channel: only YY is defined
        wav, sums = run_k3(wavs_d, mask_d, len_d, n_fft, hop, win_d, generic, clean=False, pad_to=T)
        check_sums(sums[:, 2:3], want[False][:, 2:3], f"{geo} {route} clean=None")
        assert (sums[:, [0, 1, 3, 4, 5]] == 0).all(), f"{geo} {route}: clean=None produced sums other than YY"
        check_wav(wav, refs[False], f"{geo} {route} clean=None")
        # padded mask rows with NaN pad columns, output zero-filled beyond hop (F - 1) up to pad_to
        wav, sums = run_k3(wavs_d, mask_nan, len_d, n_fft, hop, win_d, generic, pad_to=pad_to, mask_padded=True)
        assert wav.shape == (len(lengths), pad_to) and np.isfinite(wav).all() and np.isfinite(sums).all()
        check_sums(sums, want[False], f"{geo} {route} padded mask")
        check_wav(wav, refs[False], f"{geo} {route} padded mask")


@gpu
@pytest.mark.parametrize("geo", list(GEOS))
def test_mask_istft_sums_without_lengths_match_float64(se, geo):
    """lengths=None: every row is summed over all T samples and all F frames."""
    n_fft, hop = GEOS[geo][:2]
    T = 40 * hop + hop // 2 + 1
    wavs, mask = make_case(n_fft, hop, T, [T, T, T], seed=7)
    window = window_of(geo)
    ref = Reference(wavs, mask, n_fft, hop, window)
    assert_sensitive(ref, None)
    for generic in (False, True):
        wav, sums = run_k3(torch.from_numpy(wavs).cuda(), torch.from_numpy(mask).cuda(), None, n_fft, hop, window.cuda(),
                           generic, pad_to=T)
        check_sums(sums, ref.batch_sums(None), f"{geo} lengths=None generic={generic}")
        check_wav(wav, ref, f"{geo} lengths=None generic={generic}")


# ------------------------------------------------------------------------------ GPU: the epilogue in isolation
def epilogue64(sums, lengths, T, target_db=None):
    """gain, waveform SI-SDR and loss term of finalize_metrics from the same sums, in float64; lengths clamped to [0, T]."""
    out = []
    for b, s in enumerate(sums):
        n = T if lengths is None else min(max(int(lengths[b]), 0), T)
        level = s[1] / (n + 1e-8) if target_db is None else 10.0 ** (target_db / 10.0)
        g = math.sqrt(level / (s[2] / (n + 1e-8) + 1e-8))
        out.append((g, sisdr_from_sums64(g * s[0], s[1], g * g * s[2]), -sisdr_from_sums64(s[3], s[4], s[5])))
    return np.array(out)


@gpu
@pytest.mark.parametrize("target_db", [None, -25.0])
def test_finalize_metrics_matches_float64_formulas(se, target_db):
    """finalize_metrics on K3's own sums: float rounding only against float64 formulas on the same sums.  A length
    beyond T is clamped to T, as K3 clamps it for the sums (its gain equals that of length T on the same sums)."""
    from speech_enhancement_by_s3prl_b200 import ops
    n_fft, hop = 512, 256
    T = 30 * hop + 100
    lengths = boundary_lengths(n_fft, hop, T)
    wavs, mask = make_case(n_fft, hop, T, lengths, seed=3)
    len_d = torch.tensor(lengths, device="cuda")
    _, sums = ops.mask_istft(torch.from_numpy(wavs).cuda(), 0, 1, torch.from_numpy(mask).cuda(), len_d, n_fft, hop,
                             window_of("512/256").cuda(), pad_to=T)
    gain, sisdr, loss = ops.finalize_metrics(sums, len_d, T, target_db=target_db)
    want = epilogue64(sums.cpu().numpy(), lengths, T, target_db)
    np.testing.assert_allclose(gain.double().cpu().numpy(), want[:, 0], rtol=2.0 ** -23, atol=0)
    np.testing.assert_allclose(sisdr.double().cpu().numpy(), want[:, 1], rtol=0, atol=1e-5)
    np.testing.assert_allclose(loss.double().cpu().numpy(), want[:, 2], rtol=0, atol=1e-5)
    # the row of length T + 7 and a copy of it with length T give the same gain
    same = sums[[0, -1]].clone()
    same[1] = same[0]
    g2, _, _ = ops.finalize_metrics(same, torch.tensor([T, T + 7], device="cuda"), T, target_db=target_db)
    assert g2[0].item() == g2[1].item()
    # lengths=None = T
    g3, s3, l3 = ops.finalize_metrics(sums, None, T, target_db=target_db)
    want3 = epilogue64(sums.cpu().numpy(), None, T, target_db)
    np.testing.assert_allclose(g3.double().cpu().numpy(), want3[:, 0], rtol=2.0 ** -23, atol=0)
    np.testing.assert_allclose(s3.double().cpu().numpy(), want3[:, 1], rtol=0, atol=1e-5)


def _synthetic_sums(B, seed):
    g = torch.Generator().manual_seed(seed)
    s = torch.rand(B, 6, generator=g, dtype=torch.float64) * 100 + 1
    s[:, 0] = s[:, 0] - 50                                        # <y, c> of either sign
    s[:, 3] = torch.sqrt(s[:, 4] * s[:, 5]) * torch.rand(B, generator=g, dtype=torch.float64)
    return s.cuda()


@gpu
@pytest.mark.parametrize("B,W,layout", [(5, 16000, "aligned"), (5, 16000, "unaligned"), (7, 9999, "aligned"),
                                        (7, 9999, "unaligned"), (3, 4097, "aligned"), (1, 300001, "aligned"),
                                        (1, 480003, "unaligned"), (300, 1003, "aligned")])
def test_finalize_metrics_scales_every_sample_exactly_once(se, B, W, layout):
    """In-place scaling is wav_before * gain[u] bitwise over [0, width): 16-byte aligned rows (vector path, with a
    tail when width % 4 != 0), unaligned rows (a view of a (B, W + 1) buffer: the scalar path) and one row of 300k+
    samples (split over many CTAs).  Nothing outside the view is touched."""
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(W)
    if layout == "aligned":                                      # every row 16-byte aligned, spare columns past width
        stride, off = (W + 3) // 4 * 4 + 4, 0
    else:                                                        # rows start one float past a (B, W + 1) buffer's rows
        stride, off = W + 1, 1
    buf = torch.randn(B, stride, generator=g).cuda()
    wav = buf[:, off:off + W]
    assert (wav.data_ptr() % 16 == 0 and wav.stride(0) % 4 == 0) == (layout == "aligned")
    before = buf.clone()
    sums = _synthetic_sums(B, W)
    lengths = torch.randint(1, W + 1, (B,), generator=g).cuda()
    gain, _, _ = ops.finalize_metrics(sums, lengths, W, wav=wav)
    torch.cuda.synchronize()
    assert torch.equal(wav, before[:, off:off + W] * gain[:, None]), "scaled samples differ from wav * gain"
    outside = torch.ones(B, stride, dtype=torch.bool, device="cuda")
    outside[:, off:off + W] = False
    assert torch.equal(buf[outside], before[outside]), "samples outside [0, width) were written"
    np.testing.assert_allclose(gain.double().cpu().numpy(), epilogue64(sums.cpu().numpy(), lengths.tolist(), W)[:, 0],
                               rtol=2.0 ** -23, atol=0)


@gpu
def test_finalize_metrics_accumulates_only_what_it_produces(se):
    """metric_acc over three calls equals the float64 sum of the returned terms and the utterance count; a call without
    the loss (or without SI-SDR) leaves that running sum alone and still counts its utterances."""
    from speech_enhancement_by_s3prl_b200 import ops
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    loss_sum = sisdr_sum = 0.0
    count = 0
    for i, B in enumerate((4, 1, 37)):
        sums = _synthetic_sums(B, i)
        lengths = torch.randint(1, 5000, (B,)).cuda()
        _, sisdr, loss = ops.finalize_metrics(sums, lengths, 5000, metric_acc=acc)
        loss_sum += float(loss.double().sum())
        sisdr_sum += float(sisdr.double().sum())
        count += B
    np.testing.assert_allclose(acc.cpu().numpy(), [loss_sum, sisdr_sum, count], rtol=1e-12)
    before = acc.clone()
    _, sisdr, loss = ops.finalize_metrics(_synthetic_sums(6, 9), None, 5000, want_loss=False, metric_acc=acc)
    assert loss is None
    assert acc[0].item() == before[0].item() and acc[2].item() == before[2].item() + 6
    assert acc[1].item() == pytest.approx(before[1].item() + float(sisdr.double().sum()), rel=1e-12)
    before = acc.clone()
    ops.finalize_metrics(_synthetic_sums(2, 10), None, 5000, want_sisdr=False, want_gain=False, metric_acc=acc)
    assert acc[1].item() == before[1].item() and acc[2].item() == before[2].item() + 2 and acc[0].item() != before[0].item()


@gpu
@pytest.mark.parametrize("precision", [1, 0])
def test_eval_step_without_the_loss_leaves_the_loss_sum_alone(se, precision):
    """eval_step(want_spec_loss=False) returns no loss and adds only SI-SDR and the count to metric_acc; the default
    call adds the mean's numerator of its returned losses, as before."""
    torch.manual_seed(1)
    pre = se.OnlinePreprocessor(win_ms=32, hop_ms=16, n_freq=257).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    eng = se.EnhancementEngine(pre, head, precision=precision)
    T = 16000
    wavs, _ = make_case(512, 256, T, [T, 12000, 9001, 4000], seed=11)
    lengths = torch.tensor([T, 12000, 9001, 4000], device="cuda")
    wavs = torch.from_numpy(wavs).cuda()
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    full = eng.eval_step(lengths, wavs, metric_acc=acc)
    torch.cuda.synchronize()
    np.testing.assert_allclose(acc.cpu().numpy(), [float(full["loss_per_utt"].double().sum()),
                                                   float(full["sisdr"].double().sum()), 4], rtol=1e-12)
    before = acc.clone()
    part = eng.eval_step(lengths, wavs, want_spec_loss=False, metric_acc=acc)
    torch.cuda.synchronize()
    assert part["loss_per_utt"] is None
    assert acc[0].item() == before[0].item() and acc[2].item() == 8
    assert acc[1].item() == pytest.approx(before[1].item() + float(part["sisdr"].double().sum()), rel=1e-12)
    np.testing.assert_allclose(part["sisdr"].cpu().numpy(), full["sisdr"].cpu().numpy(), rtol=0, atol=1e-4)
    np.testing.assert_allclose(part["gain"].cpu().numpy(), full["gain"].cpu().numpy(), rtol=1e-5)


# ------------------------------------------------------------------------------ GPU: waveform helpers
def _wave_batch(B, W, lengths, seed):
    g = np.random.default_rng(seed)
    tar = 0.1 * g.standard_normal((B, W))
    src = 0.8 * tar + 0.05 * g.standard_normal((B, W))
    # length-1 rows hold values whose float32 products are exact: their SI-SDR (src a multiple of tar) is decided by eps
    for b, n in enumerate(lengths):
        if n == 1:
            tar[b, 0], src[b, 0] = 0.25, 0.375
    return src.astype(np.float32), tar.astype(np.float32)


WAVE_CASES = [pytest.param(4, 5000, [1, 5000, 6000, 2345], id="1-width-beyond-mixed"),
              pytest.param(1, 480000, [479999], id="1x480000"),
              pytest.param(1000, 700, None, id="1000x700")]


def _lengths(spec, B, W, seed):
    if spec is not None:
        return spec
    g = np.random.default_rng(seed)
    out = g.integers(1, W + 50, B).tolist()
    out[:3] = [1, W, W + 9]
    return out


@gpu
@pytest.mark.parametrize("B,W,lengths", WAVE_CASES)
def test_sisdr_wave_matches_float64(se, B, W, lengths):
    """se_sisdr_wave against oracle sisdr_eval in float64 over the first min(len, width) samples."""
    from speech_enhancement_by_s3prl_b200 import ops
    lengths = _lengths(lengths, B, W, 1)
    src, tar = _wave_batch(B, W, lengths, seed=W)
    got = ops.sisdr_wave(torch.from_numpy(src).cuda(), torch.from_numpy(tar).cuda(), torch.tensor(lengths).cuda())
    s64, t64 = torch.from_numpy(src).double(), torch.from_numpy(tar).double()
    want = [sp.sisdr_eval(s64[b, :min(n, W)], t64[b, :min(n, W)]) for b, n in enumerate(lengths)]
    err = np.abs(got.double().cpu().numpy() - want)
    assert err.max() < 3e-5, f"max SI-SDR error {err.max():.3g} dB"


def _normalize64(audio, lengths, target_db=None, ref=None, eps=1e-8):
    B, W = audio.shape
    masks = torch.from_numpy((np.arange(W)[None, :] < np.minimum(np.asarray(lengths), W)[:, None]).astype(np.float64))
    a = torch.from_numpy(audio).double()
    target = torch.from_numpy(target_db).double() if ref is None else torch.from_numpy(ref).double()[:, :W]
    return sp.masked_normalize_decibel(a, target, masks, eps=eps).numpy()


@gpu
@pytest.mark.parametrize("B,W,lengths", WAVE_CASES)
@pytest.mark.parametrize("form", ["target_db", "ref", "ref_in_place"])
def test_masked_normalize_db_matches_float64(se, B, W, lengths, form):
    """se_masked_normalize_db against oracle masked_normalize_decibel in float64: per-row dB targets or a reference
    waveform's masked level (ref wider than the audio), out a new tensor or the audio itself."""
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    lengths = _lengths(lengths, B, W, 2)
    audio, ref = _wave_batch(B, W + 5, lengths, seed=W + 1)
    audio = np.ascontiguousarray(audio[:, :W])
    tdb = np.linspace(-35.0, -15.0, B).astype(np.float32)
    len_d = torch.tensor(lengths).cuda()
    a_d = torch.from_numpy(audio).cuda()
    if form == "target_db":
        got = ops.masked_normalize_db(a_d, len_d, target_db=torch.from_numpy(tdb).cuda())
        want = _normalize64(audio, lengths, target_db=tdb)
    elif form == "ref":
        got = ops.masked_normalize_db(a_d, len_d, ref=torch.from_numpy(ref).cuda())
        want = _normalize64(audio, lengths, ref=ref)
    else:
        ref_d = torch.from_numpy(ref).cuda()
        ws = torch.empty(B, 3, dtype=torch.float64, device="cuda")
        rc = _lib.load().se_masked_normalize_db(a_d.data_ptr(), W, len_d.data_ptr(), B, W, None, ref_d.data_ptr(), W + 5,
                                                1e-8, ws.data_ptr(), a_d.data_ptr(), W, torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "se_masked_normalize_db")
        got = a_d
        want = _normalize64(audio, lengths, ref=ref)
    got = got.double().cpu().numpy()
    err = np.abs(got - want).max(axis=1) / np.maximum(np.abs(want).max(axis=1), 1e-30)
    assert err.max() < 5e-7, f"max relative error {err.max():.3g}"


@gpu
def test_masked_normalize_db_eps_enters_only_the_gain(se):
    """A non-default eps at length 1: the masked means divide by len + 1e-8 as the reference's masked_mean does, and
    eps is added to the mean square only in the gain's denominator."""
    from speech_enhancement_by_s3prl_b200 import ops
    audio = np.array([[0.1, 3.0, -2.0, 5.0], [0.05, 0.07, 0.2, -0.3]], dtype=np.float32)
    ref = np.array([[0.2, 1.0, 1.0, 1.0], [0.5, 0.01, 0.02, 0.03]], dtype=np.float32)
    lengths = [1, 3]
    for form in ("target_db", "ref"):
        kw = dict(target_db=torch.tensor([-20.0, -31.0]).cuda()) if form == "target_db" else dict(ref=torch.from_numpy(ref).cuda())
        got = ops.masked_normalize_db(torch.from_numpy(audio).cuda(), torch.tensor(lengths).cuda(), eps=1e-3, **kw)
        want = _normalize64(audio, lengths, target_db=np.array([-20.0, -31.0]) if form == "target_db" else None,
                            ref=ref if form == "ref" else None, eps=1e-3)
        np.testing.assert_allclose(got.double().cpu().numpy(), want, rtol=1e-6, atol=0)
