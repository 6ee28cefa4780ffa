"""Float64 restatement of STOI and ESTOI as pystoi 0.3.x computes them (NumPy only).

TEST INFRASTRUCTURE -- see ``oracle/__init__.py``.  Parity with pystoi itself is UNPINNED (pystoi is not a
dependency of this project); the definition is the contract below, written from pystoi's source:

  1. resample to 10 kHz unless fs == 10000: p / q = 10000 / fs reduced, Octave-style Kaiser filter h (``resample_filter``),
     y[m] = p sum_n x[n] h[L + m q - n p], m < ceil(n p / q)   (== scipy.signal.resample_poly(x, p, q, window=h))
  2. silent frames: frames i*128 .. i*128+255 for i in range(0, n10 - 256, 128) (the last full frame is dropped when
     n10 - 256 is a multiple of 128), windowed by w = hanning(258)[1:-1]; frame i is kept iff max_j e_j - 40 - e_i < 0,
     e = 20 log10(|w x_i| + EPS) of the CLEAN signal; kept frames of both signals are overlap-added at hop 128
  3. STFT of the result with the same framing rule, window w again, rfft n = 512
  4. 15 one-third-octave bands (BANDS, upper edge exclusive): tob = sqrt(sum |X|^2)
  5. fewer than N = 30 STFT frames -> 1e-5
  6. segments of 30 frames: STOI (clipped, centred, normalised correlations per band) and ESTOI (row then column
     normalisation; pystoi's EPS noise dropped, zero norms contribute 0)

``variant`` switches one pystoi quirk off, to show that the GPU tests would see the mistake:
  "keep_last_vad"  the last full frame is not dropped in step 2      "keep_last_stft"  ... nor in step 3
  "band_inclusive" band upper edges inclusive                         "one_window"      no second window in step 3
  "N29" / "N31"    segments of 29 / 31 frames
Resampling at 10 kHz is no such quirk: at p = q = 1 the filter taps sample the sinc at integers, so h is a unit impulse
and the signal passes unchanged (``resample(x, 1, 1) == x``, pinned by the tests).
"""
import math

import numpy as np

FS = 10000
N_FRAME = 256
HOP = 128
NFFT = 512
NUM_BAND = 15
MIN_FREQ = 150
N = 30
BETA = -15.0
DYN_RANGE = 40.0
EPS = float(np.finfo(float).eps)
BANDS = ((7, 9), (9, 11), (11, 14), (14, 17), (17, 22), (22, 27), (27, 34), (34, 43), (43, 55), (55, 69), (69, 87),
         (87, 109), (109, 138), (138, 174), (174, 219))
VARIANTS = ("keep_last_vad", "keep_last_stft", "band_inclusive", "one_window", "N29", "N31")


def window():
    r = np.arange(N_FRAME)
    return 0.5 - 0.5 * np.cos(2.0 * np.pi * (r + 1) / (N_FRAME + 1))


def third_octave_bins(fs=FS, nfft=NFFT, num_bands=NUM_BAND, min_freq=MIN_FREQ):
    """(lo, hi) bin edges of pystoi's thirdoct: band centres 150 * 2^(k/3), edges matched to the nearest bin."""
    f = np.linspace(0, fs, nfft + 1)[:nfft // 2 + 1]
    k = np.arange(num_bands, dtype=float)
    lo = min_freq * 2.0 ** ((2 * k - 1) / 6)
    hi = min_freq * 2.0 ** ((2 * k + 1) / 6)
    return tuple((int(np.argmin((f - a) ** 2)), int(np.argmin((f - b) ** 2))) for a, b in zip(lo, hi))


def rates(fs):
    g = math.gcd(int(fs), FS)
    return FS // g, int(fs) // g


def resample_filter(p, q):
    """pystoi's resample_oct filter for the reduced ratio p / q: (h normalised to sum 1, L)."""
    stop = 1.0 / (2 * max(p, q))
    roll = stop / 10
    L = int(math.ceil((60.0 - 8) / (28.714 * roll)))
    t = np.arange(-L, L + 1)
    h = np.kaiser(2 * L + 1, 0.1102 * (60.0 - 8.7)) * 2 * p * stop * np.sinc(2 * stop * t)
    return h / np.sum(h), L


def resample(x, p, q):
    """y[m] = p sum_n x[n] h[L + m q - n p] for m < ceil(n p / q) (direct polyphase form, no scipy)."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    h, L = resample_filter(p, q)
    n_out = -(-n * p // q)
    K = (2 * L) // p + 1
    k = np.arange(K)
    y = np.empty(n_out)
    for m0 in range(0, n_out, 4096):
        m = np.arange(m0, min(n_out, m0 + 4096))
        t = L + m * q
        n_hi = t // p
        ih = (t - n_hi * p)[:, None] + k * p
        ix = n_hi[:, None] - k
        ok = (ih <= 2 * L) & (ix >= 0) & (ix < n)
        y[m] = p * np.sum(np.where(ok, x[np.clip(ix, 0, max(n - 1, 0))] * h[np.clip(ih, 0, 2 * L)], 0.0), axis=1) if n else 0.0
    return y


def _frame_starts(n, keep_last):
    return range(0, n - N_FRAME + (1 if keep_last else 0), HOP)


def remove_silent_frames(x, y, keep_last=False):
    """-> (s_x, s_y, n_kept, margin_db): margin_db = min_i |max_j e_j - 40 - e_i| (inf without frames)."""
    w = window()
    starts = list(_frame_starts(len(x), keep_last))
    if not starts:
        return np.zeros(0), np.zeros(0), 0, math.inf
    xf = np.array([w * x[i:i + N_FRAME] for i in starts])
    yf = np.array([w * y[i:i + N_FRAME] for i in starts])
    e = 20 * np.log10(np.linalg.norm(xf, axis=1) + EPS)
    d = np.max(e) - DYN_RANGE - e
    keep = d < 0
    margin = float(np.min(np.abs(d)))
    xf, yf = xf[keep], yf[keep]
    nk = len(xf)
    sx, sy = np.zeros((nk - 1) * HOP + N_FRAME), np.zeros((nk - 1) * HOP + N_FRAME)
    for i in range(nk):
        sx[i * HOP:i * HOP + N_FRAME] += xf[i]
        sy[i * HOP:i * HOP + N_FRAME] += yf[i]
    return sx, sy, nk, margin


def band_envelopes(s, keep_last=False, second_window=True, inclusive=False):
    """(15, F) one-third-octave magnitudes of the STFT of s."""
    w = window() if second_window else np.ones(N_FRAME)
    starts = list(_frame_starts(len(s), keep_last))
    if not starts:
        return np.zeros((NUM_BAND, 0))
    X = np.fft.rfft(np.array([w * s[i:i + N_FRAME] for i in starts]), n=NFFT, axis=1)
    P = np.abs(X) ** 2
    return np.array([np.sqrt(np.sum(P[:, lo:hi + (1 if inclusive else 0)], axis=1)) for lo, hi in BANDS])


def _stoi_segments(xs, ys):
    """xs, ys: (J, 15, N) -> sum of the per-band correlations over every segment and band."""
    alpha = np.linalg.norm(xs, axis=2, keepdims=True) / (np.linalg.norm(ys, axis=2, keepdims=True) + EPS)
    yp = np.minimum(ys * alpha, xs * (1 + 10 ** (-BETA / 20)))
    yp = yp - np.mean(yp, axis=2, keepdims=True)
    xc = xs - np.mean(xs, axis=2, keepdims=True)
    yp = yp / (np.linalg.norm(yp, axis=2, keepdims=True) + EPS)
    xc = xc / (np.linalg.norm(xc, axis=2, keepdims=True) + EPS)
    return float(np.sum(yp * xc))


def _normalize(v, axis):
    v = v - np.mean(v, axis=axis, keepdims=True)
    nrm = np.linalg.norm(v, axis=axis, keepdims=True)
    return np.divide(v, nrm, out=np.zeros_like(v), where=nrm > 0)


def _estoi_segments(xs, ys):
    xn = _normalize(_normalize(xs, 2), 1)
    yn = _normalize(_normalize(ys, 2), 1)
    return float(np.sum(xn * yn))


def stoi_estoi(x, y, fs, variant=None):
    """x: clean reference, y: processed (1-D).  -> dict(stoi, estoi, n_kept, margin_db)."""
    assert variant is None or variant in VARIANTS, variant
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    assert x.shape == y.shape and x.ndim == 1
    p, q = rates(fs)
    if (p, q) != (1, 1):
        x, y = resample(x, p, q), resample(y, p, q)
    sx, sy, nk, margin = remove_silent_frames(x, y, keep_last=variant == "keep_last_vad")
    n_seg = {"N29": 29, "N31": 31}.get(variant, N)
    kw = dict(keep_last=variant == "keep_last_stft", second_window=variant != "one_window", inclusive=variant == "band_inclusive")
    out = dict(stoi=1e-5, estoi=1e-5, n_kept=nk, margin_db=margin)
    if nk == 0:
        return out
    xt, yt = band_envelopes(sx, **kw), band_envelopes(sy, **kw)
    F = xt.shape[1]
    if F < n_seg:
        return out
    xs = np.array([xt[:, m - n_seg:m] for m in range(n_seg, F + 1)])
    ys = np.array([yt[:, m - n_seg:m] for m in range(n_seg, F + 1)])
    J = xs.shape[0]
    out["stoi"] = _stoi_segments(xs, ys) / (NUM_BAND * J)
    out["estoi"] = _estoi_segments(xs, ys) / (n_seg * J)
    return out


def batch(est, ref, lengths, fs, variant=None):
    """Rows of (B, T) arrays cut to their lengths (clamped to [0, T]); est = processed, ref = clean (pystoi's x)."""
    est, ref = np.asarray(est, np.float64), np.asarray(ref, np.float64)
    T = est.shape[1]
    res = [stoi_estoi(ref[b, :min(max(int(n), 0), T)], est[b, :min(max(int(n), 0), T)], fs, variant) for b, n in enumerate(lengths)]
    return {k: np.array([r[k] for r in res]) for k in ("stoi", "estoi", "n_kept", "margin_db")}
