// STOI and ESTOI (pystoi 0.3.x semantics, oracle/stoi_f64.py) for a batch of ragged utterances: se_stoi_workspace, se_stoi.
//
// Six launches, no host synchronisation and no allocation (capturable):
//   taps      the Octave-style Kaiser resampling filter, built in double and stored in fp32 polyphase order
//   resample  both channels to 10 kHz (skipped at fs = 10000), polyphase direct form from shared memory
//   frames    per utterance: windowed frame energies of the clean signal, the 40 dB keep decision and the ordered
//             list of kept frames (a block scan)
//   bands     STFT frame j of the overlap-added kept frames is built from kept frames j-1, j, j+1, windowed again,
//             transformed (512-point real FFT of fft_core.cuh) and reduced to the 15 one-third-octave magnitudes
//   segments  one warp per 30-frame segment: the STOI correlation summed over the bands and the ESTOI row / column
//             normalised correlation summed over the frames
//   finish    per utterance, a fixed-order double sum over the segments (bitwise reproducible), and acc += totals
#include <algorithm>
#include <cmath>
#include "se_common.cuh"
#include "tile_kernels.cuh"

namespace {
using namespace sefft;

constexpr int kFrame = 256, kHop = 128, kNfft = 512, kBands = 15, kSeg = 30;
constexpr int kMaxRatio = 48;                  // p, q <= 48 after reduction (fs = 8, 16, 32, 48 kHz: q = 4, 8, 16, 24)
constexpr int kR = 3;                          // resampler: outputs of one phase per thread (R q = 24 words: thread groups fall on different banks at 16 kHz)
constexpr int kSpanCap = 8192;                 // resampler: input samples per CTA (with the taps, < 48 KB of shared memory)
constexpr int kBandFrames = 4;                 // bands: STFT frames per CTA (x 2 channels = 8 transforms)
constexpr float kEps = 2.220446049250313e-16f; // np.finfo(float).eps, as pystoi adds it
__constant__ int kBandLo[kBands] = {7, 9, 11, 14, 17, 22, 27, 34, 43, 55, 69, 87, 109, 138, 174};
__constant__ int kBandHi[kBands] = {9, 11, 14, 17, 22, 27, 34, 43, 55, 69, 87, 109, 138, 174, 219};

struct Geo {
    int p = 1, q = 1, L = 0, K = 0, W = 0;     // ratio, filter half-length, taps per phase, thread groups per resampler CTA
    long long T10 = 0, NF = 0, NS = 0, NJ = 0; // samples / VAD frames / STFT frames / segments per utterance (caps)
    size_t off_taps = 0, off_sig = 0, off_energy = 0, off_kept = 0, off_nk = 0, off_tob = 0, off_seg = 0, bytes = 0;
    __host__ __device__ bool resample() const { return p != 1 || q != 1; }
    __host__ __device__ int tile() const { return p * kR * W; }
    __host__ __device__ int span() const { return (int)(((long long)tile() - 1) * q / p) + K + 2; }
};

long long gcd_ll(long long a, long long b) { while (b) { long long t = a % b; a = b; b = t; } return a; }

// false: unsupported rate or shape
bool plan(long long n_utt, long long T, int fs, Geo& g) {
    if (n_utt <= 0 || n_utt > 65535 || T <= 0 || fs <= 0) return false;
    const long long d = gcd_ll(fs, 10000);
    g.p = (int)(10000 / d);
    g.q = (int)(fs / d);
    if (g.p > kMaxRatio || g.q > kMaxRatio) return false;
    if (g.resample()) {
        const double stop = 1.0 / (2 * std::max(g.p, g.q)), roll = stop / 10;
        g.L = (int)std::ceil((60.0 - 8) / (28.714 * roll));
        g.K = 2 * g.L / g.p + 1;
        g.W = std::min(256 / g.p, (kSpanCap - g.K - 2) / (kR * g.q));
        g.T10 = (T * g.p + g.q - 1) / g.q;
    } else {
        g.T10 = T;
    }
    g.NF = g.T10 > kFrame ? (g.T10 - kFrame + kHop - 1) / kHop : 0;
    g.NS = std::max(g.NF - 1, 0LL);
    g.NJ = std::max(g.NS - (kSeg - 1), 0LL);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    g.off_taps = take(g.resample() ? sizeof(float) * g.K * g.p : 0);
    g.off_sig = take(g.resample() ? sizeof(float) * 2 * n_utt * g.T10 : 0);
    g.off_energy = take(sizeof(float) * n_utt * g.NF);
    g.off_kept = take(sizeof(int) * n_utt * g.NF);
    g.off_nk = take(sizeof(int) * n_utt);
    g.off_tob = take(sizeof(float) * n_utt * g.NS * 2 * 16);
    g.off_seg = take(sizeof(float) * n_utt * g.NJ * 2);
    g.bytes = std::max<size_t>(off, 256);
    return true;
}

__device__ __forceinline__ int clamp_len(const long long* lengths, int u, long long T) {
    long long n = lengths ? lengths[u] : T;
    return (int)(n < 0 ? 0 : (n > T ? T : n));
}

// 10 kHz length of an utterance of n samples
__device__ __forceinline__ int len10(int n, int p, int q) { return (int)(((long long)n * p + q - 1) / q); }

__device__ __forceinline__ float hann258(int r) { return (float)(0.5 - 0.5 * cospi(2.0 * (r + 1) / 257.0)); }

// taps[k p + phase] = p h[phase + k p] (0 beyond 2L), h = kaiser(2L+1, 5.65) * sinc(2 stop (i - L)) / sum
__device__ __forceinline__ double filter_tap(int i, int L, double stop) {
    const double beta = 0.1102 * (60.0 - 8.7);
    const double r = (double)i / L - 1.0;
    const double kai = cyl_bessel_i0(beta * sqrt(fmax(0.0, 1.0 - r * r))) / cyl_bessel_i0(beta);
    const double t = 2 * stop * (i - L);
    return kai * (t == 0.0 ? 1.0 : sinpi(t) / (M_PI * t));
}

__global__ void __launch_bounds__(512) stoi_taps_kernel(int p, int q, int L, int K, float* __restrict__ taps) {
    __shared__ double part[512];
    const double stop = 1.0 / (2 * max(p, q));
    double s = 0.0;
    for (int i = threadIdx.x; i <= 2 * L; i += blockDim.x) s += filter_tap(i, L, stop);
    part[threadIdx.x] = s;
    __syncthreads();
    for (int h = 256; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) part[threadIdx.x] += part[threadIdx.x + h];
        __syncthreads();
    }
    const double scale = p / part[0];
    for (int idx = threadIdx.x; idx < K * p; idx += blockDim.x) {
        const int i = idx % p + (idx / p) * p;
        taps[idx] = i <= 2 * L ? (float)(filter_tap(i, L, stop) * scale) : 0.0f;
    }
}

// grid (tiles, n_utt, 2 channels): channel 0 = ref (x), 1 = est (y) -> sig[c][u][T10]
__global__ void __launch_bounds__(256) stoi_resample_kernel(const float* __restrict__ est, long long est_stride,
                                                             const float* __restrict__ ref, long long ref_stride,
                                                             const long long* __restrict__ lengths, long long T, Geo g,
                                                             const float* __restrict__ taps, float* __restrict__ sig) {
    extern __shared__ __align__(16) float smem[];
    const int u = blockIdx.y, c = blockIdx.z;
    const int n = clamp_len(lengths, u, T);
    const int n10 = len10(n, g.p, g.q);
    const int tile = g.tile();
    const long long m0 = (long long)blockIdx.x * tile;
    if (m0 >= n10) return;
    const int p = g.p, q = g.q, K = g.K;
    float* tp = smem;
    float* xs = smem + K * p;
    const float* row = c == 0 ? ref + u * ref_stride : est + u * est_stride;
    const long long lo = (g.L + m0 * q) / p - (K - 1);
    const int span = (int)((g.L + (m0 + tile - 1) * q) / p - lo + 1);
    for (int i = threadIdx.x; i < K * p; i += blockDim.x) tp[i] = taps[i];
    for (int i = threadIdx.x; i < span; i += blockDim.x) {
        const long long t = lo + i;
        xs[i] = (t >= 0 && t < n) ? row[t] : 0.0f;
    }
    __syncthreads();
    const int grp = threadIdx.x / p, phi = threadIdx.x - grp * p;
    if (grp >= g.W) return;
    const long long mb = m0 + (long long)grp * p * kR + phi;        // outputs mb + j p, j < kR: one phase
    const int ph = (int)((g.L + mb * q) % p);
    int base[kR];
    float acc[kR];
#pragma unroll
    for (int j = 0; j < kR; ++j) {
        base[j] = (int)((g.L + (mb + (long long)j * p) * q) / p - lo);
        acc[j] = 0.0f;
    }
    for (int k = 0; k < K; ++k) {
        const float h = tp[k * p + ph];
#pragma unroll
        for (int j = 0; j < kR; ++j) acc[j] = fmaf(h, xs[base[j] - k], acc[j]);
    }
    float* out = sig + ((long long)c * gridDim.y + u) * g.T10;
#pragma unroll
    for (int j = 0; j < kR; ++j) {
        const long long m = mb + (long long)j * p;
        if (m < n10) out[m] = acc[j];
    }
}

// 10 kHz row of channel c (0 = x, 1 = y) of utterance u
__device__ __forceinline__ const float* row10(const Geo& g, const float* sig, const float* est, long long est_stride,
                                              const float* ref, long long ref_stride, int n_utt, int u, int c) {
    if (g.resample()) return sig + ((long long)c * n_utt + u) * g.T10;
    return c == 0 ? ref + u * ref_stride : est + u * est_stride;
}

// one CTA per utterance: energies, keep flags (step 2 of the contract) and the ordered kept-frame list
__global__ void __launch_bounds__(256) stoi_frames_kernel(const float* __restrict__ est, long long est_stride,
                                                           const float* __restrict__ ref, long long ref_stride,
                                                           const long long* __restrict__ lengths, long long T, Geo g,
                                                           const float* __restrict__ sig, float* __restrict__ energy,
                                                           int* __restrict__ kept, int* __restrict__ nk, int* __restrict__ n_kept_out) {
    __shared__ float win[kFrame];
    __shared__ float wmax[8];
    __shared__ int wcount[8];
    const int u = blockIdx.x, n_utt = gridDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n10 = g.resample() ? len10(clamp_len(lengths, u, T), g.p, g.q) : clamp_len(lengths, u, T);
    const int nf = n10 > kFrame ? (n10 - kFrame + kHop - 1) / kHop : 0;       // range(0, n10 - 256, 128)
    const float* x = row10(g, sig, est, est_stride, ref, ref_stride, n_utt, u, 0);
    float* e = energy + (long long)u * g.NF;
    int* kp = kept + (long long)u * g.NF;
    win[threadIdx.x] = hann258(threadIdx.x);
    __syncthreads();
    float mx = -INFINITY;
    for (int f = warp; f < nf; f += 8) {
        const float* fr = x + (long long)f * kHop;
        float s = 0.0f;
#pragma unroll
        for (int i = 0; i < kFrame / 32; ++i) {
            const float v = win[lane + 32 * i] * fr[lane + 32 * i];
            s = fmaf(v, v, s);
        }
        s = secommon::warp_sum(s);
        const float db = 20.0f * log10f(sqrtf(s) + kEps);
        if (lane == 0) e[f] = db;
        mx = fmaxf(mx, db);
    }
    if (lane == 0) wmax[warp] = mx;
    __syncthreads();
    float emax = wmax[0];
    for (int w = 1; w < 8; ++w) emax = fmaxf(emax, wmax[w]);
    const float thr = emax - 40.0f;
    int running = 0;
    for (int f0 = 0; f0 < nf; f0 += 256) {
        const int f = f0 + threadIdx.x;
        const bool keep = f < nf && thr - e[f] < 0.0f;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) wcount[warp] = __popc(bal);
        __syncthreads();
        int before = running, total = 0;
        for (int w = 0; w < 8; ++w) {
            if (w < warp) before += wcount[w];
            total += wcount[w];
        }
        if (keep) kp[before + __popc(bal & ((1u << lane) - 1))] = f;
        running += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        nk[u] = running;
        if (n_kept_out) n_kept_out[u] = running;
    }
}

struct StoiExec {
    template <class F> __device__ __forceinline__ void foreach(int n, F f) {
        for (int w = threadIdx.x; w < n; w += blockDim.x) f(w);
    }
    __device__ __forceinline__ void sync() { __syncthreads(); }
};

// grid (tiles of kBandFrames STFT frames, n_utt): tob[u][j][c][16] = one-third-octave magnitudes of STFT frame j
__global__ void __launch_bounds__(128) stoi_bands_kernel(const float* __restrict__ est, long long est_stride,
                                                          const float* __restrict__ ref, long long ref_stride, Geo g,
                                                          const float* __restrict__ sig, const int* __restrict__ kept,
                                                          const int* __restrict__ nk, float* __restrict__ tob) {
    constexpr int M = kNfft / 2, PAD = Padded<M>::SIZE, G = kBandFrames;
    __shared__ float2 twM[M], twN[M + 1];
    __shared__ float win[kFrame];
    __shared__ int ids[G + 2];
    __shared__ float2 bx[2 * G * PAD], by[2 * G * PAD];
    const int u = blockIdx.y, n_utt = gridDim.y;
    const int F = nk[u] - 1;                                   // STFT frames of the overlap-added signal
    const int j0 = blockIdx.x * G;
    if (F < kSeg || j0 >= F) return;                           // fewer than 30 frames: the result is 1e-5 anyway
    for (int i = threadIdx.x; i <= M; i += blockDim.x) {
        float s, c;
        if (i < M) { sincospif(-2.0f * i / M, &s, &c); twM[i] = make_float2(c, s); }
        sincospif(-2.0f * i / kNfft, &s, &c);
        twN[i] = make_float2(c, s);
    }
    for (int i = threadIdx.x; i < kFrame; i += blockDim.x) win[i] = hann258(i);
    const int* kp = kept + (long long)u * g.NF;
    if (threadIdx.x < G + 2) {
        const int j = j0 - 1 + (int)threadIdx.x;               // kept frames j0-1 .. j0+G
        ids[threadIdx.x] = (j >= 0 && j <= F) ? kp[j] : -1;
    }
    __syncthreads();
    const float* row_x = row10(g, sig, est, est_stride, ref, ref_stride, n_utt, u, 0);
    const float* row_y = row10(g, sig, est, est_stride, ref, ref_stride, n_utt, u, 1);
    const int ng = min(G, F - j0);
    // sample r of STFT frame j0+g: w[r] * (overlap-add of the windowed kept frames j-1, j, j+1 at hop 128)
    auto sample = [&](int gi, int r) -> float {
        const int g0 = gi >> 1;
        if (g0 >= ng || r >= kFrame) return 0.0f;
        const float* x = (gi & 1) ? row_y : row_x;
        const int cur = ids[g0 + 1];
        float v = win[r] * x[(long long)cur * kHop + r];
        if (r < kHop) {
            const int prev = ids[g0];
            if (prev >= 0) v = fmaf(win[r + kHop], x[(long long)prev * kHop + r + kHop], v);
        } else {
            v = fmaf(win[r - kHop], x[(long long)ids[g0 + 2] * kHop + r - kHop], v);
        }
        return win[r] * v;
    };
    auto load0 = [&](int gi, int i) { return make_float2(sample(gi, 2 * i), sample(gi, 2 * i + 1)); };
    StoiExec ex;
    const float2* Z = sekern::fft_run<Plan<M>, -1>(ex, 2 * G, load0, bx, by, twM);
    if (threadIdx.x < 2 * ng * kBands) {
        const int gi = threadIdx.x / kBands, b = threadIdx.x - gi * kBands;
        const float2* z = Z + gi * PAD;
        float s = 0.0f;
        for (int k = kBandLo[b]; k < kBandHi[b]; ++k) {
            const float2 X = rfft_split(z[phys(k)], z[phys(M - k)], twN[k]);
            s = fmaf(X.x, X.x, fmaf(X.y, X.y, s));
        }
        tob[(((long long)u * g.NS + j0 + (gi >> 1)) * 2 + (gi & 1)) * 16 + b] = sqrtf(s);
    }
}

// grid (ceil(NJ / 8), n_utt), one warp per segment s (STFT frames s .. s+29): seg[u][s] = {sum_b STOI corr, sum_f ESTOI corr}
__global__ void __launch_bounds__(256) stoi_segments_kernel(Geo g, const int* __restrict__ nk, const float* __restrict__ tob,
                                                             float* __restrict__ seg) {
    __shared__ float xn[8][kBands][kSeg + 1], yn[8][kBands][kSeg + 1];
    const int u = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int J = nk[u] - 1 - (kSeg - 1);
    const int s = blockIdx.x * 8 + warp;
    if (s >= J) return;
    float stoi_t = 0.0f, estoi_t = 0.0f;
    if (lane < kBands) {
        const float* t = tob + ((long long)u * g.NS + s) * 32 + lane;
        float xv[kSeg], yv[kSeg];
        float sxx = 0.0f, syy = 0.0f, mx = 0.0f, my = 0.0f;
#pragma unroll
        for (int i = 0; i < kSeg; ++i) {
            xv[i] = t[i * 32];
            yv[i] = t[i * 32 + 16];
            sxx = fmaf(xv[i], xv[i], sxx);
            syy = fmaf(yv[i], yv[i], syy);
            mx += xv[i];
            my += yv[i];
        }
        mx *= 1.0f / kSeg;
        my *= 1.0f / kSeg;
        // STOI: scale y to x's energy, clip at BETA = -15 dB, correlate
        const float alpha = sqrtf(sxx) / (sqrtf(syy) + kEps);
        const float clip = 1.0f + 5.6234132519034912f;                         // 1 + 10^(15/20)
        float yp[kSeg], mp = 0.0f;
#pragma unroll
        for (int i = 0; i < kSeg; ++i) {
            yp[i] = fminf(alpha * yv[i], xv[i] * clip);
            mp += yp[i];
        }
        mp *= 1.0f / kSeg;
        float cxx = 0.0f, cpp = 0.0f, cxp = 0.0f, ryy = 0.0f;
#pragma unroll
        for (int i = 0; i < kSeg; ++i) {
            const float a = xv[i] - mx, b = yp[i] - mp, c = yv[i] - my;
            cxx = fmaf(a, a, cxx);
            cpp = fmaf(b, b, cpp);
            cxp = fmaf(a, b, cxp);
            ryy = fmaf(c, c, ryy);
        }
        stoi_t = cxp / ((sqrtf(cxx) + kEps) * (sqrtf(cpp) + kEps));
        // ESTOI, first half: mean and norm over the 30 frames of each band row
        const float ix = cxx > 0.0f ? 1.0f / sqrtf(cxx) : 0.0f, iy = ryy > 0.0f ? 1.0f / sqrtf(ryy) : 0.0f;
#pragma unroll
        for (int i = 0; i < kSeg; ++i) {
            xn[warp][lane][i] = (xv[i] - mx) * ix;
            yn[warp][lane][i] = (yv[i] - my) * iy;
        }
    }
    __syncwarp();
    if (lane < kSeg) {
        // ESTOI, second half: mean and norm over the 15 bands of each frame column
        float mx = 0.0f, my = 0.0f;
        for (int b = 0; b < kBands; ++b) { mx += xn[warp][b][lane]; my += yn[warp][b][lane]; }
        mx *= 1.0f / kBands;
        my *= 1.0f / kBands;
        float sxx = 0.0f, syy = 0.0f, sxy = 0.0f;
        for (int b = 0; b < kBands; ++b) {
            const float a = xn[warp][b][lane] - mx, c = yn[warp][b][lane] - my;
            sxx = fmaf(a, a, sxx);
            syy = fmaf(c, c, syy);
            sxy = fmaf(a, c, sxy);
        }
        estoi_t = (sxx > 0.0f && syy > 0.0f) ? sxy / (sqrtf(sxx) * sqrtf(syy)) : 0.0f;
    }
    stoi_t = secommon::warp_sum(stoi_t);
    estoi_t = secommon::warp_sum(estoi_t);
    if (lane == 0) {
        seg[((long long)u * g.NJ + s) * 2] = stoi_t;
        seg[((long long)u * g.NJ + s) * 2 + 1] = estoi_t;
    }
}

// one CTA per utterance: fixed-order double sums over the segments
__global__ void __launch_bounds__(256) stoi_finish_kernel(Geo g, const int* __restrict__ nk, const float* __restrict__ seg,
                                                           float* __restrict__ stoi, float* __restrict__ estoi, double* __restrict__ acc) {
    __shared__ double ps[256], pe[256];
    const int u = blockIdx.x;
    const int J = nk[u] - 1 - (kSeg - 1);
    double a = 0.0, b = 0.0;
    for (int s = threadIdx.x; s < J; s += blockDim.x) {
        a += seg[((long long)u * g.NJ + s) * 2];
        b += seg[((long long)u * g.NJ + s) * 2 + 1];
    }
    ps[threadIdx.x] = a;
    pe[threadIdx.x] = b;
    __syncthreads();
    for (int h = 128; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) { ps[threadIdx.x] += ps[threadIdx.x + h]; pe[threadIdx.x] += pe[threadIdx.x + h]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float d1 = J >= 1 ? (float)(ps[0] / (kBands * (double)J)) : 1e-5f;
        const float d2 = J >= 1 ? (float)(pe[0] / (kSeg * (double)J)) : 1e-5f;
        if (stoi) stoi[u] = d1;
        if (estoi) estoi[u] = d2;
        if (acc) {
            if (stoi) atomicAdd(acc, (double)d1);
            if (estoi) atomicAdd(acc + 1, (double)d2);
            atomicAdd(acc + 2, 1.0);
        }
    }
}

}  // namespace

extern "C" {

int64_t se_stoi_workspace(int64_t n_utt, int64_t T, int fs) {
    Geo g;
    if (!plan(n_utt, T, fs, g)) return 0;
    return (int64_t)g.bytes;
}

int se_stoi(const float* est, int64_t est_stride, const float* ref, int64_t ref_stride, const int64_t* lengths, int64_t n_utt,
            int64_t T, int fs, void* ws, int64_t ws_bytes, float* stoi, float* estoi, int32_t* n_kept, double* acc, void* stream) {
    SE_REQUIRE(est && ref && ws && n_utt > 0 && T > 0, "se_stoi: bad argument");
    SE_REQUIRE(stoi || estoi, "se_stoi: neither stoi nor estoi requested");
    Geo g;
    if (!plan(n_utt, T, fs, g))
        return secommon::fail(SE_ERR_UNSUPPORTED, "se_stoi: unsupported sample rate %d or shape (10000 / fs reduced to p / q needs "
                              "p, q <= %d; n_utt <= 65535)", fs, kMaxRatio);
    SE_REQUIRE(ws_bytes >= (int64_t)g.bytes, "se_stoi: workspace of %lld bytes, %lld needed", (long long)ws_bytes, (long long)g.bytes);
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* w = (unsigned char*)ws;
    float* taps = (float*)(w + g.off_taps);
    float* sig = (float*)(w + g.off_sig);
    float* energy = (float*)(w + g.off_energy);
    int* kept = (int*)(w + g.off_kept);
    int* nk = (int*)(w + g.off_nk);
    float* tob = (float*)(w + g.off_tob);
    float* seg = (float*)(w + g.off_seg);
    const long long* len = (const long long*)lengths;
    const unsigned U = (unsigned)n_utt;
    int rc;
    if (g.resample()) {
        stoi_taps_kernel<<<1, 512, 0, st>>>(g.p, g.q, g.L, g.K, taps);
        if ((rc = secommon::check_launch("stoi_taps_kernel")) != SE_OK) return rc;
        const unsigned tiles = (unsigned)((g.T10 + g.tile() - 1) / g.tile());
        const size_t smem = sizeof(float) * ((size_t)g.K * g.p + g.span());
        stoi_resample_kernel<<<dim3(tiles, U, 2), 256, smem, st>>>(est, est_stride, ref, ref_stride, len, T, g, taps, sig);
        if ((rc = secommon::check_launch("stoi_resample_kernel")) != SE_OK) return rc;
    }
    stoi_frames_kernel<<<U, 256, 0, st>>>(est, est_stride, ref, ref_stride, len, T, g, sig, energy, kept, nk, n_kept);
    if ((rc = secommon::check_launch("stoi_frames_kernel")) != SE_OK) return rc;
    if (g.NJ > 0) {
        const unsigned band_tiles = (unsigned)((g.NS + kBandFrames - 1) / kBandFrames);
        stoi_bands_kernel<<<dim3(band_tiles, U), 128, 0, st>>>(est, est_stride, ref, ref_stride, g, sig, kept, nk, tob);
        if ((rc = secommon::check_launch("stoi_bands_kernel")) != SE_OK) return rc;
        stoi_segments_kernel<<<dim3((unsigned)((g.NJ + 7) / 8), U), 256, 0, st>>>(g, nk, tob, seg);
        if ((rc = secommon::check_launch("stoi_segments_kernel")) != SE_OK) return rc;
    }
    stoi_finish_kernel<<<U, 256, 0, st>>>(g, nk, seg, stoi, estoi, acc);
    return secommon::check_launch("stoi_finish_kernel");
}

}  // extern "C"
