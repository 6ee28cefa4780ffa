// Tile bodies of the STFT / iSTFT / fused mask->iSTFT kernels (generic path).
//
// Each body processes one tile of one utterance and is written against an
// "executor" (Exec) that supplies the thread loop, the block barrier and the
// block reduction.  On the GPU the executor is the CTA (BlockExec in
// signal_kernels.cu); in tests/test_fft_core.py a serial HostExec runs the very
// same code under g++ so that indexing, padding, twiddles and overlap-add can be
// checked against numpy without a GPU.  No state lives in registers across an
// ex.sync(): everything that crosses a barrier is in the tile's shared memory.
//
// Reference behaviour being reproduced (see oracle/preprocessor.py, oracle/stft_f64.py):
//   STFT   S3PRL OnlinePreprocessor.forward  -> call sites runner.py:433,558; sampler.py:60,226
//   iSTFT  OnlinePreprocessor.istft          -> call site  runner.py:267
#pragma once
#include "fft_core.cuh"

namespace sekern {
using namespace sefft;

// Per-n_fft tile configuration: G = frames transformed concurrently by one CTA.
template <int N> struct Cfg;
template <> struct Cfg<256>  { static constexpr int G = 16, THREADS = 256; };
template <> struct Cfg<400>  { static constexpr int G = 16, THREADS = 256; };
template <> struct Cfg<512>  { static constexpr int G = 16, THREADS = 256; };
template <> struct Cfg<1024> { static constexpr int G = 8,  THREADS = 256; };
template <> struct Cfg<2048> { static constexpr int G = 4,  THREADS = 256; };

struct Tables {
    const float* window;   // [N]   analysis/synthesis window, already centred in the frame
    const float2* twM;     // [M]   exp(-2*pi*i*j/M)
    const float2* twN;     // [M+1] exp(-2*pi*i*k/N)
};

struct StftArgs {
    const float* wav;          // row u starts at wav + u*utt_stride, T samples
    long long utt_stride;
    int n_utt, T, hop, n_frames;
    Tables tab;
    float* power;              // (n_utt, n_frames, K) or null
    float* phase;              // idem or null
    float* logp;               // log(power + log_eps), idem or null
    float log_eps;
    long long spec_stride;     // floats between consecutive frames of an output (>= K; K = dense)
    double* stat_sums;         // (n_utt, ld_stats, 2) += [sum x, sum x^2] over frames of the feature written, or null
    long long ld_stats;
    unsigned long long* trace; // CTA timeline buffer (se_set_trace) or null
    double* zero_ptr;          // SE_FLAG_WS_SELF_CLEAN: doubles this kernel zeroes for the step's next replay (or null)
    long long zero_count;
    // pair mode (se_stft_features_pair; register-resident geo kernels only): n_utt counts BOTH channels' rows; row v >= n_real is
    // row v - n_real of the second channel, chan_step floats further into the utterance; only `power` is written for it
    int n_real;                // 0: plain mode
    long long chan_step;
};

struct IstftArgs {
    const float* power;        // (n_utt, n_frames, K) power spectrum
    const float* phase;        // (n_utt, n_frames, K)
    int n_utt, n_frames, hop;
    Tables tab;
    float* wav_out;            // row u at wav_out + u*out_stride
    long long out_stride;
    int out_len;               // hop * (n_frames - 1): samples torch.istft returns
    int pad_to;                // zero-fill [out_len, pad_to)  (runner.py:268)
    int tile_len;              // output samples per tile
};

// sums accumulated per utterance by the fused kernel (double precision)
enum { SUM_YC = 0, SUM_CC = 1, SUM_YY = 2, SUM_SPEC_ST = 3, SUM_SPEC_TT = 4, SUM_SPEC_SS = 5, NSUMS = 6 };

struct MaskIstftArgs {
    const float* noisy;        // row u at noisy + u*utt_stride, T samples
    const float* clean;        // same layout, or null (no metrics)
    long long utt_stride;
    const float* mask;         // (n_utt, n_frames, K) head output ("offset"), applied to the power spectrum
    const long long* lengths;  // (n_utt,) true sample counts, or null (= T)
    int n_utt, T, hop, n_frames;
    Tables tab;
    float* wav_out;
    long long out_stride;
    int out_len, pad_to, tile_len;
    double* sums;              // (n_utt, NSUMS) or null
    int want_spec;             // also accumulate the spectral SI-SDR sums (needs clean)
    long long mask_stride;     // floats between consecutive frames of mask (>= K)
    unsigned long long* trace; // CTA timeline buffer (se_set_trace) or null
    double* zero_ptr;          // SE_FLAG_WS_SELF_CLEAN: doubles zeroed after the upstream kernel has completed (or null)
    long long zero_count;
    int mask_is_power;         // `mask` holds the TARGET power spectrum: output = iSTFT(sqrt(mask) e^{i phase(noisy)}) (runner.py:266-281)
    float* wsd_terms;          // se_mask_istft_wsd (fastgeo.cu only): (n_utt, n_frames) float2 {E_f, D_f}, or null
    float* wsd_max;            // idem: the batch's largest E_f (1 float, at rest 0.0f)
};

SE_HD int imin(int a, int b) { return a < b ? a : b; }
SE_HD int imax(int a, int b) { return a > b ? a : b; }
SE_HD int floordiv(int a, int b) { int q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; }

// ------------------------------------------------------------------ shared-memory carve-up
template <int N> struct Smem {
    static constexpr int M = N / 2;
    static constexpr int PAD = Padded<M>::SIZE;
    static constexpr int G = Cfg<N>::G;
    float2* twM; float2* twN; float* win; float2* bx; float2* by; float* seg; float* aux;
    // seg_floats: capacity of the waveform segment; aux_floats: extra scratch
    SE_HD static size_t bytes(int seg_floats, int aux_floats) {
        return sizeof(float2) * (size_t)(M + (M + 2) + 2 * G * PAD) + sizeof(float) * (size_t)(N + seg_floats + aux_floats) + 16;
    }
    SE_HD Smem(unsigned char* raw, int seg_floats) {
        float2* p = reinterpret_cast<float2*>(raw);
        twM = p; p += M;
        twN = p; p += M + 2;
        bx = p; p += G * PAD;
        by = p; p += G * PAD;
        win = reinterpret_cast<float*>(p);
        seg = win + N;
        aux = seg + seg_floats;
    }
};

template <int N, class Exec> SE_HD void load_tables(Exec& ex, const Tables& t, Smem<N>& s) {
    constexpr int M = N / 2;
    ex.foreach(M, [&](int i) { s.twM[i] = t.twM[i]; });
    ex.foreach(M + 1, [&](int i) { s.twN[i] = t.twN[i]; });
    ex.foreach(N, [&](int i) { s.win[i] = t.window[i]; });
}

// reflect-padded gather of `count` samples starting at original coordinate t0 (center=True framing)
template <class Exec> SE_HD void load_segment(Exec& ex, const float* row, int T, int t0, int count, float* dst) {
    ex.foreach(count, [&](int i) {
        int t = t0 + i;
        if (t < 0) t = -t;
        if (t >= T) t = 2 * (T - 1) - t;
        dst[i] = row[t];
    });
}

// ------------------------------------------------------------------ batched Stockham FFT
template <int M, int R, int NS, int DIR, class Exec, class Load>
SE_HD void run_stage(Exec& ex, int nfft, Load load, float2* out, const float2* twM) {
    constexpr int ITEMS = M / R;
    constexpr int PAD = Padded<M>::SIZE;
    ex.foreach(nfft * ITEMS, [&](int w) {
        const int g = w / ITEMS;
        const int j = w - g * ITEMS;
        float2* o = out + g * PAD;
        stockham_item<M, R, NS, DIR>(
            j, [&](int i) { return load(g, i); }, [&](int i, float2 v) { o[phys(i)] = v; }, twM);
    });
    ex.sync();
}

struct BufLoad {
    const float2* buf; int pad;
    SE_HD float2 operator()(int g, int i) const { return buf[g * pad + phys(i)]; }
};

// Transforms nfft sequences.  Stage 0 reads through load0(g, i); results end in the returned
// buffer (bx or by) at [g*PAD + phys(k)], natural order.  bx may be the source of load0.
template <class P, int DIR, class Exec, class Load0>
SE_HD float2* fft_run(Exec& ex, int nfft, Load0 load0, float2* bx, float2* by, const float2* twM) {
    constexpr int M = P::M;
    constexpr int PAD = Padded<M>::SIZE;
    run_stage<M, P::R0, 1, DIR>(ex, nfft, load0, by, twM);
    if constexpr (P::R1 == 1) {
        return by;
    } else {
        run_stage<M, P::R1, P::R0, DIR>(ex, nfft, BufLoad{by, PAD}, bx, twM);
        if constexpr (P::R2 == 1) {
            return bx;
        } else {
            run_stage<M, P::R2, P::R0 * P::R1, DIR>(ex, nfft, BufLoad{bx, PAD}, by, twM);
            if constexpr (P::R3 == 1) {
                return by;
            } else {
                run_stage<M, P::R3, P::R0 * P::R1 * P::R2, DIR>(ex, nfft, BufLoad{by, PAD}, bx, twM);
                return bx;
            }
        }
    }
}

// ------------------------------------------------------------------ forward STFT tile
// tile covers frames [tile*G, tile*G + G) of utterance utt
template <int N, class Exec>
SE_HD void stft_tile(Exec& ex, const StftArgs& a, int utt, int tile, unsigned char* smem_raw) {
    constexpr int M = N / 2, K = M + 1, G = Cfg<N>::G;
    constexpr int PAD = Padded<M>::SIZE;
    using P = Plan<M>;
    const int seg_cap = (G - 1) * a.hop + N;
    Smem<N> s(smem_raw, seg_cap);
    const int f0 = tile * G;
    const int nf = imin(G, a.n_frames - f0);
    if (nf <= 0) return;
    load_tables<N>(ex, a.tab, s);
    const float* row = a.wav + (long long)utt * a.utt_stride;
    load_segment(ex, row, a.T, f0 * a.hop - N / 2, (nf - 1) * a.hop + N, s.seg);
    ex.sync();
    const int hop = a.hop;
    const float* seg = s.seg;
    const float* win = s.win;
    auto load0 = [=](int g, int i) {
        const float* fr = seg + g * hop;
        return make_float2(fr[2 * i] * win[2 * i], fr[2 * i + 1] * win[2 * i + 1]);
    };
    const float2* Z = fft_run<P, -1>(ex, nf, load0, s.bx, s.by, s.twM);
    const long long out0 = ((long long)utt * a.n_frames + f0) * a.spec_stride;
    ex.foreach(nf * K, [&](int w0) {
        const int g = w0 / K;
        const int k = w0 - g * K;
        const long long w = (long long)g * a.spec_stride + k;
        const float2* z = Z + g * PAD;
        const float2 zk = z[phys(k == M ? 0 : k)];
        const float2 zmk = z[phys(k == 0 ? 0 : M - k)];
        float2 x = rfft_split(zk, zmk, s.twN[k]);
        if (k == 0 || k == M) x.y = 0.0f;               // DC / Nyquist of a real signal
        const float pw = x.x * x.x + x.y * x.y;
        if (a.power) a.power[out0 + w] = pw;
        if (a.phase) a.phase[out0 + w] = atan2f(x.y, x.x);
        if (a.logp) a.logp[out0 + w] = logf(pw + a.log_eps);
    });
}

// frames whose window touches padded range [p_lo, p_hi): f*hop + N > p_lo  and  f*hop < p_hi
SE_HD void covering_frames(int p_lo, int p_hi, int N, int hop, int n_frames, int& f_lo, int& f_hi) {
    f_lo = imax(0, floordiv(p_lo - N, hop) + 1);
    f_hi = imin(n_frames - 1, floordiv(p_hi - 1, hop));
}

// windowed overlap-add of the inverse transforms in `z` (frames f_lo..f_lo+nf-1) for sample p
template <int N> SE_HD float ola_sample(const float2* z, const float* win, int p, int f_lo, int nf, int hop) {
    constexpr int M = N / 2;
    constexpr int PAD = Padded<M>::SIZE;
    int fa = imax(f_lo, floordiv(p - N, hop) + 1);
    int fb = imin(f_lo + nf - 1, floordiv(p, hop));
    float acc = 0.0f, env = 0.0f;
    for (int f = fa; f <= fb; ++f) {
        const int n = p - f * hop;
        const float2 v = z[(f - f_lo) * PAD + phys(n >> 1)];
        const float w = win[n];
        acc += w * ((n & 1) ? v.y : v.x);
        env += w * w;
    }
    return acc * (1.0f / M) / env;
}

// ------------------------------------------------------------------ inverse STFT tile (power, phase)
template <int N, class Exec>
SE_HD void istft_tile(Exec& ex, const IstftArgs& a, int utt, int tile, unsigned char* smem_raw) {
    constexpr int M = N / 2, K = M + 1;
    constexpr int PAD = Padded<M>::SIZE;
    using P = Plan<M>;
    Smem<N> s(smem_raw, 0);
    const int t_lo = tile * a.tile_len;
    const int t_end = imax(a.out_len, a.pad_to);
    const int t_hi = imin(t_lo + a.tile_len, t_end);
    if (t_lo >= t_end) return;
    float* orow = a.wav_out + (long long)utt * a.out_stride;
    int f_lo, f_hi;
    covering_frames(t_lo + N / 2, imin(t_hi, a.out_len) + N / 2, N, a.hop, a.n_frames, f_lo, f_hi);
    const int nf = (t_lo < a.out_len) ? (f_hi - f_lo + 1) : 0;       // <= G by construction of tile_len
    if (nf > 0) {
        load_tables<N>(ex, a.tab, s);
        // spectrum -> bx[g][phys(k)], k = 0..M
        const long long in0 = ((long long)utt * a.n_frames + f_lo) * K;
        ex.foreach(nf * K, [&](int w) {
            const int g = w / K;
            const int k = w - g * K;
            const float mag = sqrtf(a.power[in0 + w]);
            float sn, cs;
            sincosf(a.phase[in0 + w], &sn, &cs);
            float2 x = make_float2(mag * cs, mag * sn);
            if (k == 0 || k == M) x.y = 0.0f;           // c2r transforms ignore these
            s.bx[g * PAD + phys(k)] = x;
        });
        ex.sync();
        // merge pairs (k, M-k) in place -> Z[k], k < M
        ex.foreach(nf * (M / 2 + 1), [&](int w) {
            const int g = w / (M / 2 + 1);
            const int k = w - g * (M / 2 + 1);
            float2* x = s.bx + g * PAD;
            const float2 xa = x[phys(k)], xb = x[phys(M - k)];
            const float2 za = irfft_merge(xa, xb, s.twN[k]);
            if (k > 0 && k < M - k) x[phys(M - k)] = irfft_merge(xb, xa, s.twN[M - k]);
            x[phys(k)] = za;
        });
        ex.sync();
        const float2* z = fft_run<P, +1>(ex, nf, BufLoad{s.bx, PAD}, s.bx, s.by, s.twM);
        ex.foreach(imin(t_hi, a.out_len) - t_lo, [&](int i) {
            orow[t_lo + i] = ola_sample<N>(z, s.win, t_lo + i + N / 2, f_lo, nf, a.hop);
        });
    }
    const int z_lo = imax(t_lo, a.out_len);
    if (t_hi > z_lo) ex.foreach(t_hi - z_lo, [&](int i) { orow[z_lo + i] = 0.0f; });
}

// ------------------------------------------------------------------ fused mask -> iSTFT (+ metric sums)
// wav_out = iSTFT( sqrt(mask) * STFT(noisy) ), i.e. runner.py:569-570 (predicted = linears*offset;
// istft(predicted, phase_inp)) without materialising the spectrum, `predicted` or the phase.
// Optionally accumulates, per utterance, the sums needed by masked_normalize_decibel
// (utils.py:31-46), sisdr_eval (evaluation.py:5-10) and the spectral SISDR (objective.py:86-100).
template <int N, class Exec>
SE_HD void mask_istft_tile(Exec& ex, const MaskIstftArgs& a, int utt, int tile, unsigned char* smem_raw) {
    constexpr int M = N / 2, K = M + 1, G = Cfg<N>::G;
    constexpr int PAD = Padded<M>::SIZE;
    using P = Plan<M>;
    const int seg_cap = (G - 1) * a.hop + N;
    Smem<N> s(smem_raw, seg_cap);
    const int t_lo = tile * a.tile_len;
    const int t_end = imax(a.out_len, a.pad_to);
    const int t_hi = imin(t_lo + a.tile_len, t_end);
    float* orow = a.wav_out + (long long)utt * a.out_stride;
    const float* nrow = a.noisy + (long long)utt * a.utt_stride;
    const float* crow = a.clean ? a.clean + (long long)utt * a.utt_stride : nullptr;
    const long long len_raw = a.lengths ? a.lengths[utt] : (long long)a.T;
    const int len = (int)(len_raw < 0 ? 0 : (len_raw > a.T ? a.T : len_raw));          // clamped to the padded row
    int f_lo, f_hi;
    covering_frames(t_lo + N / 2, imin(t_hi, a.out_len) + N / 2, N, a.hop, a.n_frames, f_lo, f_hi);
    const bool spec = a.want_spec && crow && a.sums;
    // frames this tile owns for the spectral sums: f*hop in [t_lo, t_lo + tile_len)
    const int own_lo = (t_lo + a.hop - 1) / a.hop;
    const int own_hi = imin(a.n_frames, imin((t_lo + a.tile_len + a.hop - 1) / a.hop, len / a.hop + 1));
    if (t_lo >= a.out_len) {               // only the extra last frame and/or zero fill
        f_lo = own_lo;
        f_hi = (spec && own_lo < own_hi) ? own_hi - 1 : f_lo - 1;
    } else if (spec) {
        f_hi = imax(f_hi, own_hi - 1);
    }
    const int nf = f_hi - f_lo + 1;
    float acc[NSUMS];
    for (int i = 0; i < NSUMS; ++i) acc[i] = 0.0f;
    if (nf > 0) {
        load_tables<N>(ex, a.tab, s);
        const int hop = a.hop;
        const float* seg = s.seg;
        const float* win = s.win;
        auto load0 = [=](int g, int i) {
            const float* fr = seg + g * hop;
            return make_float2(fr[2 * i] * win[2 * i], fr[2 * i + 1] * win[2 * i + 1]);
        };
        float* ptar = s.aux;                // [G][K] clean power spectrum (spec only)
        if (spec) {
            load_segment(ex, crow, a.T, f_lo * hop - N / 2, (nf - 1) * hop + N, s.seg);
            ex.sync();
            const float2* Zc = fft_run<P, -1>(ex, nf, load0, s.bx, s.by, s.twM);
            ex.foreach(nf * K, [&](int w) {
                const int g = w / K;
                const int k = w - g * K;
                const float2* z = Zc + g * PAD;
                float2 x = rfft_split(z[phys(k == M ? 0 : k)], z[phys(k == 0 ? 0 : M - k)], s.twN[k]);
                if (k == 0 || k == M) x.y = 0.0f;
                ptar[w] = x.x * x.x + x.y * x.y;
            });
            ex.sync();
        }
        load_segment(ex, nrow, a.T, f_lo * hop - N / 2, (nf - 1) * hop + N, s.seg);
        ex.sync();
        float2* Zn = fft_run<P, -1>(ex, nf, load0, s.bx, s.by, s.twM);
        float2* other = (Zn == s.bx) ? s.by : s.bx;
        const long long m0 = ((long long)utt * a.n_frames + f_lo) * a.mask_stride;
        // split -> mask -> merge, pairwise in place
        ex.foreach(nf * (M / 2 + 1), [&](int w) {
            const int g = w / (M / 2 + 1);
            const int k = w - g * (M / 2 + 1);
            const int k2 = M - k;
            float2* z = Zn + g * PAD;
            const float* mk = a.mask + m0 + (long long)g * a.mask_stride;
            const float2 za = z[phys(k)], zb = z[phys(k2 == M ? 0 : k2)];
            float2 xa = rfft_split(za, zb, s.twN[k]);
            float2 xb = rfft_split(zb, za, s.twN[k2]);
            if (k == 0) { xa.y = 0.0f; xb.y = 0.0f; }
            const float ga = mk[k], gb = mk[k2];
            float2 ya, yb;
            if (a.mask_is_power) {            // polar(sqrt(power), phase(X)); phase(0) = 0
                const float qa = xa.x * xa.x + xa.y * xa.y, qb = xb.x * xb.x + xb.y * xb.y;
                ya = qa > 0.0f ? cscale(xa, sqrtf(ga) / sqrtf(qa)) : make_float2(sqrtf(ga), 0.0f);
                yb = qb > 0.0f ? cscale(xb, sqrtf(gb) / sqrtf(qb)) : make_float2(sqrtf(gb), 0.0f);
            } else {
                ya = cscale(xa, sqrtf(ga));
                yb = cscale(xb, sqrtf(gb));
            }
            if (spec) {
                const int f = f_lo + g;
                if (f >= own_lo && f < own_hi) {
                    const float pa = a.mask_is_power ? ga : ga * (xa.x * xa.x + xa.y * xa.y), ta = ptar[g * K + k];
                    const float ra = pa > 0.0f ? pa : 0.0f;            // relu, objective.py:89
                    acc[SUM_SPEC_ST] += sqrtf(ra * ta); acc[SUM_SPEC_TT] += ta; acc[SUM_SPEC_SS] += ra;
                    if (k2 != k) {
                        const float pb = a.mask_is_power ? gb : gb * (xb.x * xb.x + xb.y * xb.y), tb = ptar[g * K + k2];
                        const float rb = pb > 0.0f ? pb : 0.0f;
                        acc[SUM_SPEC_ST] += sqrtf(rb * tb); acc[SUM_SPEC_TT] += tb; acc[SUM_SPEC_SS] += rb;
                    }
                }
            }
            const float2 qa = irfft_merge(ya, yb, s.twN[k]);
            if (k > 0 && k < k2) z[phys(k2)] = irfft_merge(yb, ya, s.twN[k2]);
            z[phys(k)] = qa;
        });
        ex.sync();
        const float2* y = fft_run<P, +1>(ex, nf, BufLoad{Zn, PAD}, Zn, other, s.twM);
        const int n_out = imin(t_hi, a.out_len) - t_lo;
        if (n_out > 0) {
            ex.foreach(n_out, [&](int i) {
                const int t = t_lo + i;
                const float v = ola_sample<N>(y, s.win, t + N / 2, f_lo, nf, hop);
                orow[t] = v;
                if (a.sums && t < len) {
                    acc[SUM_YY] += v * v;
                    if (crow) { const float c = crow[t]; acc[SUM_YC] += v * c; acc[SUM_CC] += c * c; }
                }
            });
        }
    }
    const int z_lo = imax(t_lo, a.out_len);
    if (t_hi > z_lo) {
        ex.foreach(t_hi - z_lo, [&](int i) {
            const int t = z_lo + i;
            orow[t] = 0.0f;
            if (a.sums && crow && t < len) { const float c = crow[t]; acc[SUM_CC] += c * c; }
        });
    }
    if (a.sums) ex.template block_accumulate<NSUMS>(acc, a.sums + (long long)utt * NSUMS);
}

}  // namespace sekern
