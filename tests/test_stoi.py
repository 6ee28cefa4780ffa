"""STOI / ESTOI (se_stoi, ops.stoi, evaluation.stoi_eval / estoi_eval, EnhancementEngine.eval_step(want_stoi=True))
against the float64 restatement of pystoi 0.3.x in oracle/stoi_f64.py.

The CPU tests pin the oracle itself: its resampler against scipy.signal.resample_poly, its window and band table, the
properties of the metric (STOI(x, c x) = 1, gain invariance in y, zero signals, the 30-frame minimum on both sides of
the dropped-last-frame rule), and that every pystoi quirk the kernels reproduce moves the result on at least one case of
this file by SENSITIVITY tolerances, so the GPU tests would see the kernels miss it.

The GPU tests run ragged batches at 16, 8 and 10 kHz and one at 48 kHz.  Each batch has the lengths T, T - 1, 0, one
beyond T (clamped), one with fewer than 256 samples at 10 kHz, one whose 10 kHz length minus 256 is a multiple of 128, and
the pair with 30 / 31 frames and no silence (29 / 30 STFT frames).  The signals have a -60 dB gap in mid-row (frames are
removed, so the kept-frame list joins distant frames) and a loud burst at the end; y is a filtered, noisy, gain-changed x.
The kept-frame counts must match exactly: inputs are drawn so that no frame energy lies within MARGIN_DB of its threshold.

Measured on one B200 (1000 W power limit), largest |GPU - float64| per utterance over every case of this file:
  STOI   3.9e-8  (8 kHz; 2.7e-8 at 16 kHz, 2.3e-8 at 10 kHz, 3.3e-8 at 48 kHz)
  ESTOI  1.1e-7  (10 kHz; 4.5e-8 at 16 kHz, 1.9e-8 at 8 kHz, 6.1e-8 at 48 kHz)    -> TOL 5e-7 for both
"""
import functools

import numpy as np
import pytest
import torch

from oracle import stoi_f64 as ref

gpu = pytest.mark.gpu

TOL = 5e-7                 # per-utterance |STOI - oracle| and |ESTOI - oracle| (a few times the B200 maximum)
SENSITIVITY = 10.0         # each pystoi quirk must move the oracle by this many tolerances on some case of the file
MARGIN_DB = 1e-3           # no frame energy this close to its keep threshold


def len_for(n10, fs):
    """Shortest length whose 10 kHz length is n10."""
    p, q = ref.rates(fs)
    n = (n10 * q) // p
    while -(-n * p // q) > n10:
        n -= 1
    while -(-n * p // q) < n10:
        n += 1
    return n


def ragged_lengths(fs, T):
    return [T, T - 1, 0, T + 7, len_for(200, fs), len_for(256 + 128 * 40, fs), len_for(4096, fs), len_for(4224, fs)]


def make_batch(lengths, T, fs, seed):
    """x: amplitude-modulated noise, -60 dB in [0.4 T, 0.5 T), x4 over the 1500 samples before each row's end;
    y: FIR-filtered x, scaled by 0.37, plus noise.  Rows are not zeroed past their lengths."""
    rng = np.random.default_rng(seed)
    B = len(lengths)
    t = np.arange(T) / fs
    x = rng.standard_normal((B, T)) * (0.6 + 0.4 * np.sin(2 * np.pi * 3.1 * t + rng.uniform(0, 6, (B, 1))))
    x[:, int(0.4 * T):int(0.5 * T)] *= 1e-3
    for b, n in enumerate(lengths):
        n = min(max(n, 0), T)
        x[b, max(0, n - 1500):n] *= 4.0
    y = np.stack([np.convolve(r, [0.6, 0.3, -0.1], mode="same") for r in x]) * 0.37
    y += 0.15 * rng.standard_normal((B, T)) * np.abs(x).mean(axis=1, keepdims=True)
    return y.astype(np.float32), x.astype(np.float32)


CASES = {"16k": (16000, 32000), "8k": (8000, 16000), "10k": (10000, 20000)}


@functools.lru_cache(maxsize=None)
def case(name, variant=None):
    """-> (est, clean, lengths, fs, oracle dict); re-drawn until every decision is MARGIN_DB away from its threshold."""
    if name == "48k":
        fs, T = 48000, 96000
        lengths = [T, T - 5, len_for(256 + 128 * 50, fs), len_for(4224, fs)]
    else:
        fs, T = CASES[name]
        lengths = ragged_lengths(fs, T)
    for seed in range(100):
        est, clean = make_batch(lengths, T, fs, seed)
        o = ref.batch(est, clean, lengths, fs)
        if np.all(o["margin_db"] > MARGIN_DB):
            break
    else:
        raise AssertionError("no draw kept every frame energy away from its threshold")
    if variant is not None:
        o = ref.batch(est, clean, lengths, fs, variant=variant)
    return est, clean, lengths, fs, o


ALL_CASES = ("16k", "8k", "10k", "48k")


# ------------------------------------------------------------------ CPU: the oracle
def test_oracle_resampler_matches_scipy():
    signal = pytest.importorskip("scipy.signal")
    rng = np.random.default_rng(0)
    for fs in (8000, 16000, 48000):
        p, q = ref.rates(fs)
        h, _ = ref.resample_filter(p, q)
        for n in (777, 16001, 16003):
            x = rng.standard_normal(n)
            want = signal.resample_poly(x, p, q, window=h)
            got = ref.resample(x, p, q)
            assert got.shape == want.shape
            assert np.max(np.abs(got - want)) < 1e-13 * max(1.0, np.max(np.abs(want)))


def test_oracle_window_and_bands():
    assert np.allclose(ref.window(), np.hanning(258)[1:-1], rtol=0, atol=1e-15)
    assert ref.third_octave_bins() == ref.BANDS
    assert ref.rates(16000) == (5, 8) and ref.resample_filter(5, 8)[1] == 290
    x = np.random.default_rng(3).standard_normal(1001)
    assert np.max(np.abs(ref.resample(x, 1, 1) - x)) < 1e-14           # 10 kHz: the filter is a unit impulse


def test_oracle_properties():
    rng = np.random.default_rng(1)
    n = 24000
    x = rng.standard_normal(n) * (0.5 + 0.5 * np.sin(np.arange(n) / 900.0) ** 2)
    y = np.convolve(x, [0.5, 0.4, 0.2], mode="same") + 0.3 * rng.standard_normal(n)
    for c in (0.01, 1.0, 7.0):
        r = ref.stoi_estoi(x, c * x, 16000)
        assert abs(r["stoi"] - 1) < 1e-9 and abs(r["estoi"] - 1) < 1e-9
    a, b = ref.stoi_estoi(x, y, 16000), ref.stoi_estoi(x, 5.5 * y, 16000)
    assert 0.2 < a["stoi"] < 0.99 and abs(a["stoi"] - b["stoi"]) < 1e-9 and abs(a["estoi"] - b["estoi"]) < 1e-9
    for xx, yy in ((x, 0 * x), (0 * x, y)):
        r = ref.stoi_estoi(xx, yy, 16000)
        assert r["stoi"] == 0 and r["estoi"] == 0
    for m in (0, 100, 400, 4000):                                    # fewer than 30 STFT frames
        r = ref.stoi_estoi(x[:m], y[:m], 16000)
        assert r["stoi"] == 1e-5 and r["estoi"] == 1e-5


def test_oracle_thirty_frame_boundary():
    """No silence: 6553 samples at 16 kHz are 4096 at 10 kHz, 30 frames (4096 - 256 is a multiple of 128, so the last full
    frame is dropped), 29 STFT frames -> 1e-5; 6757 are 4224 at 10 kHz, 31 frames, 30 STFT frames -> a real value."""
    rng = np.random.default_rng(2)
    for n, kept in ((6553, 30), (6757, 31)):
        x = rng.standard_normal(n)
        r = ref.stoi_estoi(x, x + 0.5 * rng.standard_normal(n), 16000)
        assert r["n_kept"] == kept
        assert (r["stoi"] == 1e-5) == (kept == 30) and (r["estoi"] == 1e-5) == (kept == 30)
        if kept == 31:
            assert 0.1 < r["stoi"] < 1 and 0.05 < r["estoi"] < 1


@pytest.mark.parametrize("variant", ref.VARIANTS)
def test_each_quirk_is_visible_at_the_tolerance(variant):
    worst = 0.0
    for name in ALL_CASES:
        o, v = case(name)[4], case(name, variant)[4]
        worst = max(worst, float(np.max(np.abs(v["stoi"] - o["stoi"]))), float(np.max(np.abs(v["estoi"] - o["estoi"]))))
    assert worst >= SENSITIVITY * TOL, f"{variant}: the oracle moves by only {worst:.2e}"


# ------------------------------------------------------------------ GPU
def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_case(name, **kw):
    from speech_enhancement_by_s3prl_b200 import ops
    est, clean, lengths, fs, o = case(name)
    nk = torch.empty(len(lengths), dtype=torch.int32, device="cuda")
    s, e = ops.stoi(_dev(est), _dev(clean), _dev(np.array(lengths, np.int64)), fs=fs, n_kept=nk, **kw)
    return s, e, nk, o


@gpu
@pytest.mark.parametrize("name", ALL_CASES)
def test_stoi_matches_oracle(name):
    s, e, nk, o = run_case(name)
    assert nk.cpu().numpy().tolist() == o["n_kept"].astype(int).tolist()
    ds = np.abs(s.cpu().double().numpy() - o["stoi"])
    de = np.abs(e.cpu().double().numpy() - o["estoi"])
    print(f"\n{name}: max |dSTOI| {ds.max():.2e}  max |dESTOI| {de.max():.2e}  stoi {np.round(o['stoi'], 4).tolist()}")
    assert ds.max() <= TOL and de.max() <= TOL
    short = o["n_kept"] <= 30
    assert np.all(s.cpu().numpy()[short] == np.float32(1e-5)) and np.all(e.cpu().numpy()[short] == np.float32(1e-5))


@gpu
def test_properties_on_gpu():
    from speech_enhancement_by_s3prl_b200 import ops
    est, clean, lengths, fs, _ = case("16k")
    x = _dev(clean)
    L = _dev(np.array(lengths, np.int64))
    s, e = ops.stoi(3.0 * x, x, L, fs=fs)
    valid = torch.tensor([n > 7000 for n in lengths])
    assert torch.all((s.cpu()[valid] - 1).abs() < 1e-5) and torch.all((e.cpu()[valid] - 1).abs() < 1e-5)
    s, e = ops.stoi(torch.zeros_like(x), x, L, fs=fs)
    assert torch.all(s.cpu()[valid] == 0) and torch.all(e.cpu()[valid] == 0)
    s, e = ops.stoi(x, torch.zeros_like(x), L, fs=fs)
    assert torch.all(s.cpu()[valid] == 0) and torch.all(e.cpu()[valid] == 0)


@gpu
def test_deterministic_and_acc():
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    s1, e1, _, _ = run_case("16k", acc=acc)
    s2, e2, _, _ = run_case("16k", acc=acc)
    assert torch.equal(s1, s2) and torch.equal(e1, e2)
    want = torch.tensor([2 * s1.double().sum().item(), 2 * e1.double().sum().item(), 2.0 * len(s1)], dtype=torch.float64)
    assert torch.allclose(acc.cpu(), want, rtol=1e-12, atol=0)
    from speech_enhancement_by_s3prl_b200 import ops
    est, clean, lengths, fs, _ = case("16k")
    acc.zero_()
    s, e = ops.stoi(_dev(est), _dev(clean), _dev(np.array(lengths, np.int64)), fs=fs, want_stoi=False, acc=acc)
    assert s is None and torch.equal(e, e1)
    assert acc[0].item() == 0 and abs(acc[1].item() - e1.double().sum().item()) < 1e-12 and acc[2].item() == len(lengths)


@gpu
def test_strided_clean_channel():
    from speech_enhancement_by_s3prl_b200 import ops
    est, clean, lengths, fs, _ = case("16k")
    B, T = est.shape
    wavs = torch.randn(B, 3, T, device="cuda")
    wavs[:, 0] = _dev(est)
    wavs[:, 1] = _dev(clean)
    L = _dev(np.array(lengths, np.int64))
    s1, e1 = ops.stoi(wavs[:, 0], wavs[:, 1], L, fs=fs)
    assert wavs[:, 1].stride(0) == 3 * T
    s2, e2 = ops.stoi(wavs[:, 0].contiguous(), wavs[:, 1].contiguous(), L, fs=fs)
    assert torch.equal(s1, s2) and torch.equal(e1, e2)


@gpu
def test_drop_ins_and_errors():
    from speech_enhancement_by_s3prl_b200 import evaluation, ops
    est, clean, lengths, fs, _ = case("16k")
    s, e, _, _ = run_case("16k")
    for b, n in enumerate(lengths):
        n = min(n, est.shape[1])
        if n < 1000:
            continue
        src, tar = torch.from_numpy(est[b, :n]), torch.from_numpy(clean[b, :n])
        assert abs(evaluation.stoi_eval(src, tar, sr=fs) - s[b].item()) <= 1e-6
        assert abs(evaluation.estoi_eval(src, tar, sr=fs) - e[b].item()) <= 1e-6
    bs, be = evaluation.stoi_eval_batch(_dev(est), _dev(clean), _dev(np.array(lengths, np.int64)), sr=fs)
    assert torch.equal(bs, s) and torch.equal(be, e)
    with pytest.raises(RuntimeError):
        ops.stoi(_dev(est), _dev(clean), fs=44100)
    from speech_enhancement_by_s3prl_b200 import _lib
    assert _lib.load().se_stoi_workspace(4, 16000, 44100) <= 0 and _lib.load().se_stoi_workspace(4, 16000, 16000) > 0


def _engine():
    import speech_enhancement_by_s3prl_b200 as se
    pre = se.OnlinePreprocessor(win_ms=32, hop_ms=16, n_freq=257).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    return se.EnhancementEngine(pre, head, precision=1)


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted(ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA and "Memcpy" not in ev.name)


@gpu
def test_engine_eval_step_stoi():
    from speech_enhancement_by_s3prl_b200 import ops
    est, clean, lengths, fs, _ = case("16k")
    B, T = est.shape
    wavs = torch.stack([_dev(clean) + 0.3 * _dev(est), _dev(clean), _dev(est)], 1).contiguous()
    L = _dev(np.minimum(np.array(lengths, np.int64), T))
    eng = _engine()
    plain = eng.eval_step(L, wavs)
    n_plain = eng.launches_per_step
    off = eng.eval_step(L, wavs, want_stoi=False)
    assert set(off) == set(plain) and "stoi" not in off and eng.launches_per_step == n_plain
    acc = torch.zeros(3, dtype=torch.float64, device="cuda")
    out = eng.eval_step(L, wavs, want_stoi=True, stoi_acc=acc)
    assert set(out) == set(plain) | {"stoi", "estoi"}
    s, e = ops.stoi(out["wav_predicted"], wavs[:, 1], L, fs=16000)
    assert torch.equal(out["stoi"], s) and torch.equal(out["estoi"], e)
    assert acc[2].item() == B and abs(acc[0].item() - s.double().sum().item()) < 1e-9
    k_default = _kernels(lambda: eng.eval_step(L, wavs))
    k_off = _kernels(lambda: eng.eval_step(L, wavs, want_stoi=False))
    k_on = _kernels(lambda: eng.eval_step(L, wavs, want_stoi=True))
    assert k_off == k_default and not any("stoi" in k for k in k_default)
    extra = list(k_on)
    for k in k_default:
        extra.remove(k)
    assert sorted(extra) == sorted(["stoi_taps_kernel", "stoi_resample_kernel", "stoi_frames_kernel", "stoi_bands_kernel",
                                    "stoi_segments_kernel", "stoi_finish_kernel"]) or all("stoi_" in k for k in extra), extra
    # a captured step carries the metrics; each replay adds to the accumulator
    wavs_s, L_s = wavs.clone(), L.clone()
    acc_g = torch.zeros(3, dtype=torch.float64, device="cuda")
    st = eng.capture_bound(L_s, wavs_s, want_stoi=True, stoi_acc=acc_g)
    st["graph"].replay()
    st["graph"].replay()
    torch.cuda.synchronize()
    assert torch.equal(st["stoi"], out["stoi"]) and torch.equal(st["estoi"], out["estoi"])
    assert acc_g[2].item() == 2 * B and abs(acc_g[1].item() - 2 * e.double().sum().item()) < 1e-9
