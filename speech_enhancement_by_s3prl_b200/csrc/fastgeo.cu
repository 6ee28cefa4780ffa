// libse_b200.so -- register-resident fast paths, one kernel template over three geometries:
//
//   Geo512    n_fft 512  / hop 256   (BASELINE configs[1], the headline)      one frame per group of 16 lanes, 2 groups per warp
//   Geo1024   n_fft 1024 / hop 256   (BASELINE configs[3], long-form)        one frame per WARP
//   Geo400    n_fft 400  / hop 160   (the reference's default 25 ms / 10 ms, pretrain_sample.yaml:46-48; configs[2], [4])
//                                                                             one frame per group of 10 lanes, 3 groups per warp
//
//   stft_run_kernel         K1: frame -> window -> rFFT -> power / phase / log-power (+ CMVN sums)
//   mask_istft_run_kernel   K3: frame -> rFFT -> x sqrt(mask) -> irFFT -> window -> overlap-add in registers along a run of
//                               consecutive frames -> / envelope -> wav, plus the per-utterance metric sums
//
// A lane group owns a RUN of consecutive frames, FFT values live in registers, only the transposes of the FFT go through
// shared memory, and there is no block-level barrier in the frame loops.  All groups of a warp run in lock-step, so every
// shuffle and __syncwarp uses the full warp mask.  The geometries differ in two places:
//
//   * FFT cores.  Geo512: the 256-point complex transform of a frame is one 16-lane transform (fft256_warp.cuh).
//     Geo1024: the 512-point complex transform of a frame is two 256-point 16-lane transforms
//     (fft256_warp.cuh) plus ONE radix-2 exchange between the halves (16 shuffles): decimation in time on the way
//     forward (strided "time" layout in, blocked "spectral" layout out), decimation in frequency on the way back
//     (blocked in, strided out), so neither direction needs a second transpose.  Geo400: 200 = 20 x 10 -- a
//     prime-factor (Good-Thomas, twiddle-free) 20-point DFT in registers, one transpose through shared memory, the
//     twiddles, then two prime-factor 10-point DFTs; lane j holds element j + 10 s before and after.
//     tools/lane_model.py is the lane-level numpy model these index maps were checked with.
//   * Overlap-add (512/256: 2 frames cover a sample; 1024/256: 4; 400/160: 2 or 3).  Frame f EMITS the window of
//     hop samples [f hop - N/2, f hop - N/2 + hop) that no later frame touches; the rest of its windowed inverse
//     transform stays in the register carry.  A run that owns emit windows e0..e1 walks frames e0 - halo .. e1
//     (halo = ceil(N / hop) - 1 frames recomputed at the start of every run) and, past the last frame of the
//     utterance, "virtual" frames that only flush the carry.  The first / last N/2 - hop samples of an utterance are
//     covered by fewer frames than the interior: there the folded 1 / envelope is corrected per sample.
//
// Reference behaviour: torch.stft / torch.istft as called by S3PRL's OnlinePreprocessor (oracle/preprocessor.py;
// call sites runner.py:433,558,267), objective.py:86-100, evaluation.py:5-10, utils.py:31-46.
#include "se_common.cuh"
#include "fft256_warp.cuh"
#include "fast_common.cuh"
#include "tile_kernels.cuh"

using namespace fastc;
using sekern::StftArgs;
using sekern::MaskIstftArgs;
using sekern::Tables;

namespace {

constexpr unsigned kFull = 0xffffffffu;

struct Geo512  { enum { N = 512,  M = 256, H = 256, G = 16, V = 16, GPW = 2, IDLE = 0, NB = 2, HB = 1, VB = 8, NP = 8,  XBUF = 2048 }; };
struct Geo1024 { enum { N = 1024, M = 512, H = 256, G = 32, V = 16, GPW = 1, IDLE = 0, NB = 4, HB = 1, VB = 4, NP = 8, XBUF = 4224 }; };
struct Geo400  { enum { N = 400,  M = 200, H = 160, G = 10, V = 20, GPW = 3, IDLE = 1, NB = 5, HB = 2, VB = 4, NP = 10, XBUF = 1792 }; };

__device__ __forceinline__ float2 shfl2(float2 v, int src) {
    return make_float2(__shfl_sync(kFull, v.x, src), __shfl_sync(kFull, v.y, src));
}
__device__ __forceinline__ float2 shfl2_xor(float2 v, int m) {
    return make_float2(__shfl_xor_sync(kFull, v.x, m), __shfl_xor_sync(kFull, v.y, m));
}
__device__ __forceinline__ float2 sel2(bool c, float2 a, float2 b) { return make_float2(c ? a.x : b.x, c ? a.y : b.y); }

// ------------------------------------------------------------------ prime-factor DFTs (forward), in place, natural order
// 20 = 4 x 5: n = (5 n1 + 4 n2) mod 20, k = (5 k1 + 16 k2) mod 20; 10 = 2 x 5: n = (5 n1 + 2 n2) mod 10, k = (5 k1 + 6 k2) mod 10
__device__ __forceinline__ void pfa20(float2 (&x)[20]) {
    float2 t[4][5];
#pragma unroll
    for (int n2 = 0; n2 < 5; ++n2) {
        float2 a0 = x[(4 * n2) % 20], a1 = x[(5 + 4 * n2) % 20], a2 = x[(10 + 4 * n2) % 20], a3 = x[(15 + 4 * n2) % 20];
        bfly4<-1>(a0, a1, a2, a3);
        t[0][n2] = a0; t[1][n2] = a1; t[2][n2] = a2; t[3][n2] = a3;
    }
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
        bfly5<-1>(t[k1][0], t[k1][1], t[k1][2], t[k1][3], t[k1][4]);
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) x[(5 * k1 + 16 * k2) % 20] = t[k1][k2];
    }
}
__device__ __forceinline__ void pfa10(float2 (&x)[10]) {
    float2 t[2][5];
#pragma unroll
    for (int n2 = 0; n2 < 5; ++n2) {
        const float2 a = x[(2 * n2) % 10], b = x[(5 + 2 * n2) % 10];
        t[0][n2] = cadd(a, b);
        t[1][n2] = csub(a, b);
    }
#pragma unroll
    for (int k1 = 0; k1 < 2; ++k1) {
        bfly5<-1>(t[k1][0], t[k1][1], t[k1][2], t[k1][3], t[k1][4]);
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) x[(5 * k1 + 6 * k2) % 10] = t[k1][k2];
    }
}

// ------------------------------------------------------------------ FFT cores
// Layouts.  "time": lane holds complex element tidx + G r in slot r (element m = samples 2m, 2m+1 of the frame).
// "spectral": what fft() + post_forward() leave: pair q < NP of the lane is (bin k = pair_bin(q) in slot q, its mirror
// M - k somewhere else); fetch_mirror() brings Z[M - k] next to Z[k], scatter_mirror() is its inverse.  The self-paired
// bin M/2 sits in slot V/2 of the group's leader lane, whose pair 0 is (DC, Nyquist).
template <class Geo> struct Core;

template <> struct Core<Geo512> {
    float2 tw[15], twn[8];
    float2* xbuf;
    int j, tidx, ln;
    bool leader, active;
    __device__ __forceinline__ void init(int lane, unsigned char* region, const Tables& tab) {
        j = lane & 15; tidx = j; ln = lane;                                             // group lane >> 4, its own region
        leader = j == 0; active = true;
        xbuf = reinterpret_cast<float2*>(region);
        fft256w::load_lane_constants(j, tab.twM, tab.twN, tw, twn);
    }
    static __device__ __forceinline__ int group_of(int lane) { return lane >> 4; }
    static __device__ __forceinline__ int lane_in_group(int lane) { return lane & 15; }
    __device__ __forceinline__ int pair_bin(int q) const { return j + 16 * q; }
    __device__ __forceinline__ void fft(float2 (&v)[16]) { fft256w::fft256<-1>(v, xbuf, j, tw); }
    __device__ __forceinline__ void post_forward(float2 (&)[16]) {}
    __device__ __forceinline__ void pre_inverse(float2 (&)[16]) {}
    __device__ __forceinline__ void fetch_mirror(const float2 (&v)[16], float2 (&zm)[8], int lane) const { fft256w::fetch_mirror(v, lane, zm); }
    __device__ __forceinline__ void scatter_mirror(const float2 (&ca)[8], const float2 (&cb)[8], float2 cmid, float2 (&v)[16]) const {
        fft256w::scatter_mirror(ca, cb, cmid, ln, v);
    }
};

template <> struct Core<Geo1024> {
    float2 tw[15], tc[8], twn[8];
    float2* xbuf;
    int j, h, src, tidx;
    bool leader, active;
    __device__ __forceinline__ void init(int lane, unsigned char* region, const Tables& tab) {
        // half h = lane & 1 transforms the complex samples of parity h: time index = lane, consecutive lanes touch
        // consecutive elements (coalesced, conflict-free); the halves' transpose buffers sit 16 banks apart
        j = lane >> 1; h = lane & 1; tidx = lane;
        leader = lane == 0; active = true;
        src = (((16 - j) & 15) << 1) | (h ^ 1);
        xbuf = reinterpret_cast<float2*>(region + h * 2112);
#pragma unroll
        for (int r = 1; r < 16; ++r) tw[r - 1] = tab.twM[2 * r * j];                  // W_256^(r j)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int k = j + 16 * (q + 8 * h);
            tc[q] = tab.twM[k];                                                        // W_512^k
            twn[q] = tab.twN[k];                                                       // W_1024^k
        }
    }
    static __device__ __forceinline__ int group_of(int) { return 0; }
    static __device__ __forceinline__ int lane_in_group(int lane) { return lane; }
    __device__ __forceinline__ int pair_bin(int q) const { return j + 16 * (q + 8 * h); }
    __device__ __forceinline__ void fft(float2 (&v)[16]) { fft256w::fft256<-1>(v, xbuf, j, tw); }
    // decimation in time: Z[k] = E[k] + W^k O[k], Z[k + 256] = E[k] - W^k O[k]; half h keeps k = j + 16 (q + 8 h)
    __device__ __forceinline__ void post_forward(float2 (&v)[16]) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float2 recv = shfl2_xor(sel2(h, v[q], v[8 + q]), 1);
            const float2 E = sel2(h, recv, v[q]);
            const float2 t = cmul(sel2(h, v[8 + q], recv), tc[q]);
            v[q] = cadd(E, t);
            v[8 + q] = csub(E, t);
        }
    }
    // decimation in frequency: half 0 transforms a[k] = C[k] + C[k + 256], half 1 b[k] = (C[k] - C[k + 256]) W^k
    __device__ __forceinline__ void pre_inverse(float2 (&v)[16]) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float2 a = cadd(v[q], v[8 + q]);
            const float2 b = cmul(csub(v[q], v[8 + q]), tc[q]);
            const float2 recv = shfl2_xor(sel2(h, a, b), 1);
            v[q] = sel2(h, recv, a);
            v[8 + q] = sel2(h, b, recv);
        }
    }
    __device__ __forceinline__ void fetch_mirror(const float2 (&v)[16], float2 (&zm)[8], int lane) const {
        zm[0] = shfl2(j == 0 ? (h ? v[8] : v[0]) : v[15], j == 0 ? lane : src);
#pragma unroll
        for (int q = 1; q < 8; ++q) zm[q] = shfl2(j == 0 ? v[16 - q] : v[15 - q], src);
    }
    __device__ __forceinline__ void scatter_mirror(const float2 (&ca)[8], const float2 (&cb)[8], float2 cmid, float2 (&v)[16]) const {
        float2 rcv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { rcv[q] = shfl2(cb[q], src); v[q] = ca[q]; }
        v[8] = j == 0 ? (h ? cb[0] : cmid) : rcv[7];
#pragma unroll
        for (int p = 1; p < 8; ++p) v[8 + p] = j == 0 ? rcv[8 - p] : rcv[7 - p];
    }
};

template <> struct Core<Geo400> {
    float2 twa[9], twb[9], twn[10];
    float2* xbuf;
    int j, src, tidx;
    bool leader, active;
    static constexpr int ROW = 22;                                                      // float2 per transpose row: conflict-free STS.128
    __device__ __forceinline__ void init(int lane, unsigned char* region, const Tables& tab) {
        const int grp = lane / 10;
        j = lane - 10 * grp; tidx = j;
        active = grp < 3;                                                               // lanes 30, 31 idle along (own scratch region)
        leader = active && j == 0;
        src = active ? grp * 10 + (10 - j) % 10 : lane;
        xbuf = reinterpret_cast<float2*>(region);
#pragma unroll
        for (int i = 1; i < 10; ++i) { twa[i - 1] = tab.twM[i * j]; twb[i - 1] = tab.twM[i * (j + 10)]; }
#pragma unroll
        for (int q = 0; q < 10; ++q) twn[q] = tab.twN[j + 10 * q];
    }
    static __device__ __forceinline__ int group_of(int lane) { return lane / 10; }
    static __device__ __forceinline__ int lane_in_group(int lane) { return lane % 10; }
    __device__ __forceinline__ int pair_bin(int q) const { return j + 10 * q; }
    // lane j: z[j + 10 r] -> Z[j + 10 s]
    __device__ __forceinline__ void fft(float2 (&v)[20]) {
        pfa20(v);                                                                       // A[j][q], q < 20
        float4* row = reinterpret_cast<float4*>(xbuf + j * ROW);
#pragma unroll
        for (int c = 0; c < 10; ++c) row[c] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
        __syncwarp();
        float2 a[10], b[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) { a[i] = xbuf[i * ROW + j]; b[i] = xbuf[i * ROW + j + 10]; }
        __syncwarp();
#pragma unroll
        for (int i = 1; i < 10; ++i) { a[i] = cmul(a[i], twa[i - 1]); b[i] = cmul(b[i], twb[i - 1]); }
        pfa10(a);                                                                       // Z[j + 20 p]
        pfa10(b);                                                                       // Z[j + 10 + 20 p]
#pragma unroll
        for (int p = 0; p < 10; ++p) { v[2 * p] = a[p]; v[2 * p + 1] = b[p]; }
    }
    __device__ __forceinline__ void post_forward(float2 (&)[20]) {}
    __device__ __forceinline__ void pre_inverse(float2 (&)[20]) {}
    __device__ __forceinline__ void fetch_mirror(const float2 (&v)[20], float2 (&zm)[10], int) const {
#pragma unroll
        for (int q = 0; q < 10; ++q) zm[q] = shfl2(j == 0 ? v[(20 - q) % 20] : v[19 - q], src);
    }
    __device__ __forceinline__ void scatter_mirror(const float2 (&ca)[10], const float2 (&cb)[10], float2 cmid, float2 (&v)[20]) const {
        float2 rcv[10];
#pragma unroll
        for (int q = 0; q < 10; ++q) { rcv[q] = shfl2(cb[q], src); v[q] = ca[q]; }
#pragma unroll
        for (int q = 0; q < 9; ++q) v[19 - q] = j == 0 ? rcv[q + 1] : rcv[q];
        v[10] = j == 0 ? cmid : rcv[9];
    }
};

// ------------------------------------------------------------------ shared sizes
template <class Geo> struct Sz {
    static constexpr int N = Geo::N, M = Geo::M, H = Geo::H, G = Geo::G, V = Geo::V, NP = Geo::NP;
    static constexpr int K = M + 1;
    static constexpr int Bs = N / Geo::NB;                          // floats per staging block
    static constexpr int RB = Geo::NB + Geo::HB;                    // ring blocks: a frame + the incoming hop
    static constexpr int HS = Geo::HB * Geo::VB;                    // register slots per hop
    static constexpr int HALO = (N + H - 1) / H - 1;                // frames recomputed at the start of a run
    static constexpr int EDGE = N / 2 - H;                          // samples at either end covered by fewer frames
    static constexpr int E_MIN = EDGE / H + 1;                      // first emit window that reaches t >= 0
    static constexpr int NV = (EDGE + H - 1) / H;                   // virtual frames past the last one
    static constexpr int MROW = (K + 16 * (K >> 7) + 3) / 4 * 4;    // skewed mask row (bins 128 apart land 16 banks apart)
    static constexpr int TAB_BYTES = (2 * M * 8 + 127) / 128 * 128; // s_win2 | s_bw2
};
// position of bin k in the staged mask row.  Geo1024: the two halves of a warp read bins 128 apart in the same instruction, so
// every 128 bins are skewed by 16 floats (16 banks); Geo400: plain; Geo512: plain, each group reads 16 consecutive bins of its
// own row, and the two rows of a warp sit 16 banks apart (K3Sz::GSTRIDE).
template <class Geo> __device__ __forceinline__ int mpos(int k) { return Geo::G == 32 ? k + ((k >> 7) << 4) : k; }

// stage one block of Bs floats starting at original coordinate t0 (reflect outside [0, T)); jg = lane in group
template <class Geo>
__device__ __forceinline__ void stage_block(float* __restrict__ dst, const float* __restrict__ row, int T, int t0, int jg) {
    constexpr int Bs = Sz<Geo>::Bs, G = Geo::G;
    const float* src = row + t0;
    if (t0 >= 0 && t0 + Bs <= T && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
#pragma unroll
        for (int c = 0; c < Bs / 4 / G; ++c) cp_async16(dst + 4 * (jg + G * c), src + 4 * (jg + G * c));
    } else {
#pragma unroll 4
        for (int i = jg; i < Bs; i += G) {
            int t = t0 + i;
            t = t < 0 ? -t : t;
            t = t >= T ? 2 * (T - 1) - t : t;
            cp_async4(dst + i, row + t);
        }
    }
}
template <class Geo>
__device__ __forceinline__ void stage_mask_row(float* __restrict__ dst, const float* __restrict__ src, bool padded, int jg) {
    constexpr int K = Sz<Geo>::K, G = Geo::G;
    if (padded && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        if (Geo::G == 32) {
            // chunk c = jg + 32 i holds bins 4 c .. 4 c + 3 = 128 i + 4 jg ..: destination 4 jg + 144 i (immediate offsets)
#pragma unroll
            for (int i = 0; i < (K + 3) / 4 / 32; ++i) cp_async16(dst + 4 * jg + 144 * i, src + 4 * jg + 128 * i);
            if (jg < (K + 3) / 4 % 32) cp_async16(dst + 4 * jg + 144 * ((K + 3) / 4 / 32), src + 4 * jg + 128 * ((K + 3) / 4 / 32));
        } else {
            for (int c = jg; c < (K + 3) / 4; c += G) cp_async16(dst + 4 * c, src + 4 * c);
        }
    } else {
        for (int k = jg; k < K; k += G) cp_async4(dst + mpos<Geo>(k), src + k);
    }
}
// v[r] = (x[2m], x[2m+1]) * win2[m], m = tidx + G r, from the ring (block 0 of the frame in ring slot `slot0`)
template <class Geo>
__device__ __forceinline__ void frame_from_ring(const float* __restrict__ ring, int slot0, int tidx, const float2* __restrict__ win2,
                                                float2 (&v)[Geo::V]) {
    constexpr int Bs = Sz<Geo>::Bs, RB = Sz<Geo>::RB, G = Geo::G, VB = Geo::VB;
#pragma unroll
    for (int b = 0; b < Geo::NB; ++b) {
        int slot = slot0 + b;
        slot = slot >= RB ? slot - RB : slot;
        const float2* p = reinterpret_cast<const float2*>(ring + slot * Bs) + tidx;
#pragma unroll
        for (int i = 0; i < VB; ++i) v[b * VB + i] = pmul(p[G * i], win2[tidx + G * (b * VB + i)]);
    }
}

// interior envelope / envelope over the frames that exist, for original sample t (first / last N/2 - hop samples)
__device__ __forceinline__ float edge_scale(const float* __restrict__ w, int t, int N, int H, int F) {
    float ei = 0.0f, ee = 0.0f;
    for (int n = (t + N / 2) % H; n < N; n += H) {
        const float ww = __ldg(w + n) * __ldg(w + n);
        const int g = (t + N / 2 - n) / H;
        ei += ww;
        if (g >= 0 && g <= F - 1) ee += ww;
    }
    return ei / ee;
}

// se_set_trace: one TraceScope record per CTA (kernel id 1 = K1, 3 = K3), from the TRACE instantiations that the launchers
// pick when a trace buffer is set, so that the kernels without it are unchanged.  Thread 0 parks the start time in the last 8
// bytes of the dynamic shared memory: a register would stay live across the frame loops.
__device__ __forceinline__ void trace_begin(unsigned char* smem_end) {
    if (threadIdx.x == 0) reinterpret_cast<unsigned long long*>(smem_end)[-1] = secommon::TraceScope::now();
}
__device__ __forceinline__ void trace_end(unsigned long long* buf, int kernel_id, const unsigned char* smem_end) {
    __syncthreads();
    secommon::TraceScope trace(buf, kernel_id);
    trace.t0 = reinterpret_cast<const unsigned long long*>(smem_end)[-1];
    trace.finish();
}

struct GeoRunPlan { int per_utt; int runs_per_utt; long long total_runs; };      // per_utt frames (K1) / emit windows (K3)
// run ri of `rpu` over `n` items: n / rpu each, the first n % rpu runs one more
__device__ __forceinline__ void run_range(int ri, int n, int rpu, int& first, int& len) {
    const int base = n / rpu, rem = n - base * rpu;
    first = ri * base + (ri < rem ? ri : rem);
    len = base + (ri < rem ? 1 : 0);
}

// ------------------------------------------------------------------ K1
template <class Geo> struct K1Cfg;
// Geo512: small CTAs (2 warps, four per SM at up to 255 registers per thread): with two steps in flight the other step's
// kernels get SMs back in finer grains (8-warp CTAs: +1.4 us per step at 64 x 4 s, round 2)
template <> struct K1Cfg<Geo512>  { static constexpr int WARPS = 2, MIN_BLOCKS = 4; };
template <> struct K1Cfg<Geo1024> { static constexpr int WARPS = 4, MIN_BLOCKS = 2; };
template <> struct K1Cfg<Geo400>  { static constexpr int WARPS = 4, MIN_BLOCKS = 2; };
template <class Geo> struct K1Sz {
    static constexpr int ACC_BYTES = (Geo::M + 2) * 8;
    static constexpr int GROUP_BYTES = Geo::XBUF + ACC_BYTES;       // XBUF keeps groups 20 banks apart (Geo400: 1792 % 128 = 0 ...
    static constexpr int GSTRIDE = (GROUP_BYTES + 127) / 128 * 128 + (Geo::G == 10 ? 80 : 0);   // ... + 80 -> conflict-free column reads)
    static constexpr int WARP_BYTES = (Geo::GPW + Geo::IDLE) * GSTRIDE;
    static constexpr int GROUPS = K1Cfg<Geo>::WARPS * Geo::GPW;
    static constexpr size_t SMEM = Sz<Geo>::TAB_BYTES + (size_t)K1Cfg<Geo>::WARPS * WARP_BYTES + GROUPS * 4 + 16;   // + trace start
};

// x[r] = raw samples (2m, 2m+1), m = tidx + G r, of the frame starting at original coordinate t0
template <class Geo>
__device__ __forceinline__ void load_frame(float2 (&x)[Geo::V], const float* __restrict__ row, int T, int t0, int tidx) {
    constexpr int N = Geo::N, G = Geo::G, V = Geo::V;
    const float* src = row + t0;
    if (t0 >= 0 && t0 + N <= T && (reinterpret_cast<uintptr_t>(src) & 7) == 0) {
        const float2* s2 = reinterpret_cast<const float2*>(src) + tidx;
#pragma unroll
        for (int r = 0; r < V; ++r) x[r] = __ldg(s2 + G * r);
    } else {
#pragma unroll
        for (int r = 0; r < V; ++r) {
            int ta = t0 + 2 * (tidx + G * r), tb = ta + 1;
            ta = ta < 0 ? -ta : ta; ta = ta >= T ? 2 * (T - 1) - ta : ta;
            tb = tb < 0 ? -tb : tb; tb = tb >= T ? 2 * (T - 1) - tb : tb;
            x[r] = make_float2(__ldg(row + ta), __ldg(row + tb));
        }
    }
}

template <class Geo, bool PHASE, bool STATS, bool TRACE>
__global__ void __launch_bounds__(K1Cfg<Geo>::WARPS * 32, K1Cfg<Geo>::MIN_BLOCKS) stft_run_kernel(StftArgs a, GeoRunPlan plan) {
    extern __shared__ __align__(128) unsigned char smem[];
    if (TRACE) trace_begin(smem + K1Sz<Geo>::SMEM);
    using S = Sz<Geo>;
    constexpr int M = S::M, H = S::H, G = S::G, V = S::V, NP = S::NP, N = S::N;
    constexpr int WARPS = K1Cfg<Geo>::WARPS, THREADS = WARPS * 32, GROUPS = K1Sz<Geo>::GROUPS;
    float2* s_win2 = reinterpret_cast<float2*>(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = Core<Geo>::group_of(lane), jg = Core<Geo>::lane_in_group(lane);
    unsigned char* region = smem + S::TAB_BYTES + (size_t)warp * K1Sz<Geo>::WARP_BYTES + (size_t)grp * K1Sz<Geo>::GSTRIDE;
    int* s_utt = reinterpret_cast<int*>(smem + S::TAB_BYTES + (size_t)WARPS * K1Sz<Geo>::WARP_BYTES);
    if (a.zero_ptr)                                                                 // SE_FLAG_WS_SELF_CLEAN: K3's sums of this step
        for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < a.zero_count; i += (long long)gridDim.x * THREADS)
            a.zero_ptr[i] = 0.0;
    Core<Geo> core;
    core.init(lane, region, a.tab);
    float2* acc = reinterpret_cast<float2*>(region + Geo::XBUF);
    const int gslot = warp * Geo::GPW + grp;                                        // group index in the CTA (idle lanes: unused)
    const long long unit = (long long)blockIdx.x * GROUPS + gslot;
    const bool active = core.active && unit < plan.total_runs;
    const int u = active ? (int)(unit / plan.runs_per_utt) : -1;
    int fa = 0, len = 0;
    const float* row = a.wav;
    float2 x[V];
#pragma unroll
    for (int r = 0; r < V; ++r) x[r] = make_float2(0.0f, 0.0f);
    if (active) {
        run_range((int)(unit - (long long)u * plan.runs_per_utt), a.n_frames, plan.runs_per_utt, fa, len);
        row = (a.n_real > 0 && u >= a.n_real) ? a.wav + (long long)(u - a.n_real) * a.utt_stride + a.chan_step
                                               : a.wav + (long long)u * a.utt_stride;
        if (len > 0) load_frame<Geo>(x, row, a.T, fa * H - N / 2, core.tidx);       // first loads in flight before the tables
    }
    const bool second = a.n_real > 0 && u >= a.n_real;                              // pair mode, second channel: power only
    for (int i = threadIdx.x; i < M; i += THREADS)
        s_win2[i] = make_float2(0.5f * a.tab.window[2 * i], 0.5f * a.tab.window[2 * i + 1]);
    if (STATS && core.active && jg == 0) s_utt[gslot] = (active && len > 0 && !second) ? u : -1;
    float2 sacc[2 * NP + 1];
#pragma unroll
    for (int i = 0; i < 2 * NP + 1; ++i) sacc[i] = make_float2(0.0f, 0.0f);
    __syncthreads();
    griddep_launch();
    const int n_iter = __reduce_max_sync(kFull, len);
    const int F = a.n_frames;
    const bool want_pw = a.power != nullptr, want_lg = a.logp != nullptr && !second;
#pragma unroll 1
    for (int it = 0; it < n_iter; ++it) {
        const bool live = it < len;
        const int f = fa + it;
        float2 v[V];
#pragma unroll
        for (int r = 0; r < V; ++r) v[r] = pmul(x[r], s_win2[core.tidx + G * r]);
        if (it + 1 < len) load_frame<Geo>(x, row, a.T, (f + 1) * H - N / 2, core.tidx);   // lands behind this frame's transform
        core.fft(v);
        core.post_forward(v);
        float2 zm[NP];
        core.fetch_mirror(v, zm, lane);
        if (live) {
            const long long o = ((long long)u * F + f) * a.spec_stride;
            float* pw = want_pw ? a.power + o : nullptr;
            float* lg = want_lg ? a.logp + o : nullptr;
            float* ph = PHASE ? a.phase + o : nullptr;
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                const int k = core.pair_bin(q);
                float2 xa, xb;
                split_pair(v[q], zm[q], core.twn[q], xa, xb);
                const float pa = xa.x * xa.x + xa.y * xa.y, pb = xb.x * xb.x + xb.y * xb.y;
                float la = 0.f, lb = 0.f;
                if (want_pw) { pw[k] = pa; pw[M - k] = pb; }
                if (want_lg) { la = fast_log(pa + a.log_eps); lb = fast_log(pb + a.log_eps); lg[k] = la; lg[M - k] = lb; }
                if (PHASE) { ph[k] = atan2f(k == 0 ? 0.0f : xa.y, xa.x); ph[M - k] = atan2f(k == 0 ? 0.0f : xb.y, xb.x); }
                if (STATS) {
                    const float sa = want_lg ? la : pa, sb = want_lg ? lb : pb;
                    sacc[q] = pfma(make_float2(sa, sa), make_float2(1.0f, sa), sacc[q]);
                    sacc[NP + q] = pfma(make_float2(sb, sb), make_float2(1.0f, sb), sacc[NP + q]);
                }
            }
            if (core.leader) {                                          // bin M/2 pairs with itself: X = 2 conj(Z[M/2])
                const float2 xm = make_float2(2.0f * v[V / 2].x, -2.0f * v[V / 2].y);
                const float p = xm.x * xm.x + xm.y * xm.y;
                float l = 0.f;
                if (want_pw) pw[M / 2] = p;
                if (want_lg) { l = fast_log(p + a.log_eps); lg[M / 2] = l; }
                if (PHASE) ph[M / 2] = atan2f(xm.y, xm.x);
                if (STATS) { const float s = want_lg ? l : p; sacc[2 * NP] = pfma(make_float2(s, s), make_float2(1.0f, s), sacc[2 * NP]); }
            }
        }
    }
    if (STATS) {
        if (core.active) {
#pragma unroll
            for (int q = 0; q < NP; ++q) {
                const int k = core.pair_bin(q);
                acc[k] = sacc[q];
                acc[M - k] = sacc[NP + q];
            }
            if (core.leader) acc[M / 2] = sacc[2 * NP];
        }
        __syncthreads();
        // thread t owns bins t, t + THREADS, ...; the CTA's runs are consecutive, so utterances are non-decreasing
        for (int bin = threadIdx.x; bin <= M; bin += THREADS) {
            double s1 = 0.0, s2 = 0.0;
            int cur = -1;
            for (int g = 0; g < GROUPS; ++g) {
                const int uh = s_utt[g];
                if (uh < 0) continue;
                if (uh != cur) {
                    if (cur >= 0) {
                        double* pdst = a.stat_sums + ((long long)cur * a.ld_stats + bin) * 2;
                        atomicAdd(pdst, s1);
                        atomicAdd(pdst + 1, s2);
                    }
                    cur = uh; s1 = 0.0; s2 = 0.0;
                }
                const int w = g / Geo::GPW, gi = g - w * Geo::GPW;
                const float2 t = reinterpret_cast<const float2*>(smem + S::TAB_BYTES + (size_t)w * K1Sz<Geo>::WARP_BYTES +
                                                                 (size_t)gi * K1Sz<Geo>::GSTRIDE + Geo::XBUF)[bin];
                s1 += (double)t.x;
                s2 += (double)t.y;
            }
            if (cur >= 0) {
                double* pdst = a.stat_sums + ((long long)cur * a.ld_stats + bin) * 2;
                atomicAdd(pdst, s1);
                atomicAdd(pdst + 1, s2);
            }
        }
    }
    if (TRACE) trace_end(a.trace, 1, smem + K1Sz<Geo>::SMEM);
}

// ------------------------------------------------------------------ K3
template <class Geo> struct K3Cfg;
// warps per CTA / CTAs per SM the register cap is set for (8 resident warps per SM either way; the occupancy sweeps of round 2
// -- 12 warps at a 168-register cap lose 30 % to spills -- are in DESIGN.md 4.2)
#ifndef SE_GEO512_K3_WARPS
#define SE_GEO512_K3_WARPS 4
#endif
#ifndef SE_GEO512_K3_MINB
#define SE_GEO512_K3_MINB 2
#endif
#ifndef SE_GEO1024_K3_WARPS
#define SE_GEO1024_K3_WARPS 4
#endif
#ifndef SE_GEO1024_K3_MINB
#define SE_GEO1024_K3_MINB 2
#endif
#ifndef SE_GEO400_K3_WARPS
#define SE_GEO400_K3_WARPS 8                 // one 8-warp CTA per SM: 103.0 vs 104.7 us per 64 x 4 s step (tools/sweep_lib_configs.sh)
#endif
#ifndef SE_GEO400_K3_MINB
#define SE_GEO400_K3_MINB 1
#endif
template <> struct K3Cfg<Geo512>  { static constexpr int WARPS = SE_GEO512_K3_WARPS, MIN_BLOCKS = SE_GEO512_K3_MINB; };
template <> struct K3Cfg<Geo1024> { static constexpr int WARPS = SE_GEO1024_K3_WARPS, MIN_BLOCKS = SE_GEO1024_K3_MINB; };
template <> struct K3Cfg<Geo400>  { static constexpr int WARPS = SE_GEO400_K3_WARPS, MIN_BLOCKS = SE_GEO400_K3_MINB; };
// MB: staged mask rows per group (2 in the WSD variant, which reads frame f's row again in pass 2 while f + 1's is in flight)
template <class Geo, int MB = 1> struct K3Sz {
    using S = Sz<Geo>;
    static constexpr int RING_BYTES = S::RB * S::Bs * 4;
    static constexpr int GROUP_BYTES = Geo::XBUF + 2 * RING_BYTES + MB * S::MROW * 4;
    // Geo400: + 80 -> conflict-free column reads; Geo512: + 64 -> the two groups' mask rows 16 banks apart
    static constexpr int GSTRIDE = (GROUP_BYTES + 127) / 128 * 128 + (Geo::G == 10 ? 80 : Geo::G == 16 ? 64 : 0);
    static constexpr int IDLE_BYTES = Geo::IDLE ? (Geo::XBUF + 127) / 128 * 128 : 0;      // idle lanes only need transpose scratch
    static constexpr int WARP_BYTES = Geo::GPW * GSTRIDE + IDLE_BYTES;
    static constexpr int GROUPS = K3Cfg<Geo>::WARPS * Geo::GPW;
    static constexpr size_t SMEM = S::TAB_BYTES + (size_t)K3Cfg<Geo>::WARPS * WARP_BYTES + 16;                 // + trace start
};

// sum of v over the lane group (every lane of the group gets it; all 32 lanes must call).  Geo400's groups of 10 lanes: pairs
// (j, j + 5), then the five pair sums, which lanes j and j + 5 both hold.
template <class Geo> __device__ __forceinline__ float2 group_sum(float2 v, int lane, int jg, bool active) {
    if constexpr (Geo::G == 10) {
        const int base = lane - jg;
        auto at = [&](int d) { return active ? base + (jg + d) % 10 : lane; };
        const float2 p = cadd(v, shfl2(v, at(5)));
        float2 s = cadd(p, shfl2(p, at(1)));
        s = cadd(s, shfl2(s, at(2)));
        return cadd(s, shfl2(p, at(4)));
    } else {
#pragma unroll
        for (int o = Geo::G / 2; o > 0; o >>= 1) v = cadd(v, shfl2_xor(v, o));
        return v;
    }
}

// WSD: the variant of K3 for objective.WSD (objective.py:127-153).  Pass 2 runs for every real frame the run owns (frames past an
// utterance's valid length included: the reference does not mask the energies) and writes per frame {E_f = sum_k S,
// D_f = sum_k (S - G S)^2 (0 past the valid length)} to a.wsd_terms; sum_k (G max(X - S, 0))^2 over valid frames goes to the
// SE_SUM_SPEC_ST slot of the sums, and the run's largest E_f to *a.wsd_max (float bits, atomicMax: energies are >= 0).
template <class Geo, bool PM, bool TRACE, bool WSD = false>
__global__ void __launch_bounds__(K3Cfg<Geo>::WARPS * 32, K3Cfg<Geo>::MIN_BLOCKS) mask_istft_run_kernel(MaskIstftArgs a, GeoRunPlan plan) {
    using Z = K3Sz<Geo, WSD ? 2 : 1>;
    extern __shared__ __align__(128) unsigned char smem[];
    if (TRACE) trace_begin(smem + Z::SMEM);
    using S = Sz<Geo>;
    constexpr int N = S::N, M = S::M, H = S::H, G = S::G, V = S::V, NP = S::NP, Bs = S::Bs, RB = S::RB, HS = S::HS;
    constexpr int WARPS = K3Cfg<Geo>::WARPS, THREADS = WARPS * 32, GROUPS = Z::GROUPS;
    float2* s_win2 = reinterpret_cast<float2*>(smem);
    float2* s_bw2 = s_win2 + M;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = Core<Geo>::group_of(lane), jg = Core<Geo>::lane_in_group(lane);
    unsigned char* region = smem + S::TAB_BYTES + (size_t)warp * Z::WARP_BYTES + (size_t)grp * Z::GSTRIDE;
    // idle lanes (Geo400: 30, 31) execute every load of the frame loop too: they read the last real group's staging
    // (same addresses as its lanes 0, 1: a broadcast) and own only scratch for the transposes
    const int dgrp = grp < Geo::GPW ? grp : Geo::GPW - 1;
    float* nring = reinterpret_cast<float*>(smem + S::TAB_BYTES + (size_t)warp * Z::WARP_BYTES + (size_t)dgrp * Z::GSTRIDE + Geo::XBUF);
    float* cring = nring + RB * Bs;
    float* mb = cring + RB * Bs;                                                    // WSD: two rows, frame f_first + it in row (it & 1)
    const bool lane_active = grp < Geo::GPW;
    const long long unit = (long long)blockIdx.x * GROUPS + warp * Geo::GPW + grp;
    const bool active = lane_active && unit < plan.total_runs;
    const int F = a.n_frames;
    int u = 0, ri = 0, e0 = 0, e1 = -1, f_first = 0, my_iters = 0;
    const float* nrow = a.noisy;
    if (active) {
        u = (int)(unit / plan.runs_per_utt);
        ri = (int)(unit - (long long)u * plan.runs_per_utt);
        int first, len;
        run_range(ri, plan.per_utt, plan.runs_per_utt, first, len);
        e0 = S::E_MIN + first;
        e1 = e0 + len - 1;
        f_first = e0 - S::HALO > 0 ? e0 - S::HALO : 0;
        my_iters = len > 0 ? e1 - f_first + 1 : 0;
        nrow = a.noisy + (long long)u * a.utt_stride;
        // the first frame's noisy samples are inputs of the step: requested before the tables and the upstream kernel's end
        if (my_iters > 0) {
#pragma unroll
            for (int b = 0; b < Geo::NB; ++b) stage_block<Geo>(nring + b * Bs, nrow, a.T, (f_first * Geo::HB + b) * Bs - N / 2, jg);
        }
    }
    for (int i = threadIdx.x; i < M; i += THREADS) {
        const float w0 = a.tab.window[2 * i], w1 = a.tab.window[2 * i + 1];
        s_win2[i] = make_float2(0.5f * w0, 0.5f * w1);
        float en0 = 0.0f, en1 = 0.0f;                                               // interior envelope: all frames that can cover the sample
        for (int n = (2 * i) % H; n < N; n += H) en0 += a.tab.window[n] * a.tab.window[n];
        for (int n = (2 * i + 1) % H; n < N; n += H) en1 += a.tab.window[n] * a.tab.window[n];
        s_bw2[i] = make_float2(w0 / (2.0f * M * en0), -w1 / (2.0f * M * en1));     // sign: conjugation of the forward-as-inverse FFT
    }
    Core<Geo> core;
    core.init(lane, region, a.tab);
    __syncthreads();
    griddep_launch();
    const int n_iter = __reduce_max_sync(kFull, my_iters);
    const float* crow = a.clean ? a.clean + (long long)u * a.utt_stride : nullptr;
    float* orow = a.wav_out + (long long)u * a.out_stride;
    const int len = a.lengths ? (int)min((long long)a.T, max(0LL, a.lengths[active ? u : 0])) : a.T;   // clamped to the padded row
    const int valid_frames = min(F, len / H + 1);                                   // runner.py:455
    const bool spec = a.want_spec && crow && a.sums;
    const bool need_clean = crow && a.sums;
    const bool out_aligned = (reinterpret_cast<uintptr_t>(orow) & 7) == 0;
    const bool mask_padded = (a.mask_stride & 3) == 0;
    const float* mrow0 = a.mask + (long long)u * F * a.mask_stride;
    const int tidx = core.tidx;
    // Geo1024: bins k = k0 + 16 q and M - k = (M - k0) - 16 q of pairs q >= 1 at constant offsets from two per-lane pointers
    const int k0 = core.pair_bin(0);
    const float* mlo = mb + mpos<Geo>(k0 + 16) - 16;
    const float* mhi = mb + mpos<Geo>(M - k0 - 16) + 16;
    float acc[sekern::NSUMS];
#pragma unroll
    for (int i = 0; i < sekern::NSUMS; ++i) acc[i] = 0.0f;
    float2 carry[V - HS];
#pragma unroll
    for (int i = 0; i < V - HS; ++i) carry[i] = make_float2(0.0f, 0.0f);
    float2 yy2 = make_float2(0.0f, 0.0f), yc2 = yy2, cc2 = yy2, st2 = yy2, tt2 = yy2, ss2 = yy2;   // WSD: st2 = residual noise
    float wmax = 0.0f;                                                              // WSD: largest frame energy of the run

    griddep_wait();                                                                 // the mask (and the zeroed sums) come from upstream kernels
    if (a.zero_ptr)                                                                 // SE_FLAG_WS_SELF_CLEAN: the CMVN sums the head has consumed
        for (long long i = (long long)blockIdx.x * THREADS + threadIdx.x; i < a.zero_count; i += (long long)gridDim.x * THREADS)
            a.zero_ptr[i] = 0.0;
    if (my_iters > 0 && need_clean) {
#pragma unroll
        for (int b = 0; b < Geo::NB; ++b) stage_block<Geo>(cring + b * Bs, crow, a.T, (f_first * Geo::HB + b) * Bs - N / 2, jg);
    }
    cp_async_commit();                                                              // group W(f_first)
    if (my_iters > 0 && f_first <= F - 1) stage_mask_row<Geo>(mb, mrow0 + (long long)f_first * a.mask_stride, mask_padded, jg);
    cp_async_commit();                                                              // group M(f_first)

    int slot0 = 0;                                                                  // ring slot of block 0 of the current frame
#pragma unroll 1
    for (int it = 0; it < n_iter; ++it) {
        const int f = f_first + it;
        const bool live = it < my_iters;
        const bool real = live && f <= F - 1;
        const bool emit = live && f >= e0;
        // WSD: own = every real frame of the run (energies), wval = the valid ones among them (loss terms)
        const bool own = WSD ? need_clean && real && (f >= e0 || ri == 0) : spec && real && f < valid_frames && (f >= e0 || ri == 0);
        const bool wval = WSD && own && f < valid_frames;
        const int moff = WSD ? (it & 1) * S::MROW : 0;
        const bool next_real = it + 1 < my_iters && f + 1 <= F - 1;
        if (next_real) {                                                            // the hop of frame f + 1 -> the free ring slots
#pragma unroll
            for (int b = 0; b < Geo::HB; ++b) {
                int slot = slot0 + Geo::NB + b;
                slot = slot >= RB ? slot - RB : slot;
                const int t0 = ((f + 1) * Geo::HB + Geo::NB - Geo::HB + b) * Bs - N / 2;
                stage_block<Geo>(nring + slot * Bs, nrow, a.T, t0, jg);
                if (need_clean) stage_block<Geo>(cring + slot * Bs, crow, a.T, t0, jg);
            }
        }
        cp_async_commit();                                                          // group W(f + 1)
        cp_async_wait<1>();                                                         // W(f) and M(f) have landed
        __syncwarp();
        float ra[NP], rb[NP], rmid = 0.0f;                                          // relu(mask |X|^2) of this frame (objective.py:89)
#pragma unroll
        for (int q = 0; q < NP; ++q) { ra[q] = 0.0f; rb[q] = 0.0f; }
        float2 v[V];
        bool mask_group_open = true;
#pragma unroll 1
        for (int pass = 0; pass < 3; ++pass) {
            // a pass runs if ANY group of the warp needs it (shuffles are warp-wide); the others compute and discard
            if (!__any_sync(kFull, pass == 0 ? real : pass == 1 ? live : own)) continue;
            if (pass == 0) frame_from_ring<Geo>(nring, slot0, tidx, s_win2, v);
            else if (pass == 2) frame_from_ring<Geo>(cring, slot0, tidx, s_win2, v);
            else if (!real) {                                                       // virtual frame (or idle): nothing to add
#pragma unroll
                for (int r = 0; r < V; ++r) v[r] = make_float2(0.0f, 0.0f);
            }
            core.fft(v);
            if (pass != 1) core.post_forward(v);
            if (pass == 0) {
                float2 zm[NP];
                core.fetch_mirror(v, zm, lane);
                float2 ca[NP], cbv[NP];
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    const int k = core.pair_bin(q);
                    float2 xa, xb;
                    split_pair(v[q], zm[q], core.twn[q], xa, xb);
                    // (Geo1024: q >= 1 keeps k and M - k inside one 128-bin skew block per lane: constant offsets from mlo / mhi)
                    const float ga = (Geo::G == 32 && q > 0) ? mlo[moff + 16 * q] : mb[moff + mpos<Geo>(k)];
                    const float gb = (Geo::G == 32 && q > 0) ? mhi[moff - 16 * q] : mb[moff + mpos<Geo>(M - k)];
                    mask_merge<PM, !WSD>(xa, xb, ga, gb, core.twn[q], WSD ? wval : own, ra[q], rb[q], ca[q], cbv[q]);
                }
                const float gmid = mb[moff + mpos<Geo>(M / 2)];
                const float2 xmid = make_float2(2.0f * v[V / 2].x, -2.0f * v[V / 2].y);   // bin M/2 pairs with itself: X = 2 conj(Z[M/2])
                if (WSD) { if (wval) rmid = gmid * (xmid.x * xmid.x + xmid.y * xmid.y); }
                else if (own) rmid = fmaxf(PM ? gmid : gmid * (xmid.x * xmid.x + xmid.y * xmid.y), 0.0f);
                __syncwarp();
                if (next_real) stage_mask_row<Geo>(mb + (S::MROW - moff) * WSD, mrow0 + (long long)(f + 1) * a.mask_stride, mask_padded, jg);
                cp_async_commit();                                                  // group M(f + 1)
                mask_group_open = false;
                float2 ymid;                                                        // 2 Y[M/2]: conj(Zinv[M/2]), same factor 2 as merge_pair_conj
                if (PM) { ymid = apply_gain<true>(xmid, gmid); ymid.x *= 2.0f; ymid.y *= 2.0f; }
                else { const float sm = 2.0f * fast_sqrt(gmid); ymid = make_float2(sm * xmid.x, sm * xmid.y); }
                core.scatter_mirror(ca, cbv, ymid, v);
                core.pre_inverse(v);
            } else if (pass == 1) {
                // v[r] = conj(z[m]) unnormalised, m = tidx + G r; signs, 1/M and the interior 1/envelope are in s_bw2
                float2 y[HS];
#pragma unroll
                for (int i = 0; i < HS; ++i) y[i] = pfma(s_bw2[tidx + G * i], v[i], carry[i]);
#pragma unroll
                for (int i = 0; i < V - HS; ++i) {
                    if (i < V - 2 * HS) carry[i] = pfma(s_bw2[tidx + G * (i + HS)], v[i + HS], carry[i + HS]);
                    else carry[i] = pmul(s_bw2[tidx + G * (i + HS)], v[i + HS]);
                }
                if (emit) {
                    const int t0 = f * H - N / 2;
                    // clean samples of the emit window = the first hop of the clean frame (ring blocks 0 .. HB-1 of the frame)
                    const bool interior = t0 >= S::EDGE && t0 + H <= a.out_len - S::EDGE;
                    if (interior && out_aligned && t0 >= 0 && (!a.sums || t0 + H <= len)) {
                        float2* o2 = reinterpret_cast<float2*>(orow + t0) + tidx;
#pragma unroll
                        for (int i = 0; i < HS; ++i) {
                            o2[G * i] = y[i];
                            if (a.sums) yy2 = pfma(y[i], y[i], yy2);
                            if (need_clean) {
                                int slot = slot0 + i / Geo::VB;
                                slot = slot >= RB ? slot - RB : slot;
                                const float2 c = (reinterpret_cast<const float2*>(cring + slot * Bs) + tidx)[G * (i % Geo::VB)];
                                yc2 = pfma(y[i], c, yc2);
                                cc2 = pfma(c, c, cc2);
                            }
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < HS; ++i) {
                            float2 c = make_float2(0.0f, 0.0f);
                            if (need_clean) {
                                int slot = slot0 + i / Geo::VB;
                                slot = slot >= RB ? slot - RB : slot;
                                c = (reinterpret_cast<const float2*>(cring + slot * Bs) + tidx)[G * (i % Geo::VB)];
                            }
                            const int t = t0 + 2 * (tidx + G * i);
#pragma unroll
                            for (int s = 0; s < 2; ++s) {
                                const int ts = t + s;
                                if (ts >= 0 && ts < a.out_len) {
                                    float ys = s ? y[i].y : y[i].x;
                                    if (ts < S::EDGE || ts >= a.out_len - S::EDGE) ys *= edge_scale(a.tab.window, ts, N, H, F);
                                    orow[ts] = ys;
                                    if (a.sums && ts < len) {
                                        const float cs = s ? c.y : c.x;
                                        acc[sekern::SUM_YY] += ys * ys;
                                        acc[sekern::SUM_YC] += ys * cs;
                                        acc[sekern::SUM_CC] += cs * cs;
                                    }
                                }
                            }
                        }
                    }
                }
            } else if (WSD) {
                // S = clean power, G re-read from the frame's mask row, ra / rb = G X: d = G X - G S is G (X - S), so the
                // residual-noise term (G max(X - S, 0))^2 is d^2 where G d > 0, for a mask of any sign
                float2 zm[NP];
                core.fetch_mirror(v, zm, lane);
                float2 ed = make_float2(0.0f, 0.0f);                                // (E_f, D_f) parts of this lane
                if (own) {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        const int k = core.pair_bin(q);
                        float2 xa, xb;
                        split_pair(v[q], zm[q], core.twn[q], xa, xb);
                        const float2 pt = make_float2(xa.x * xa.x + xa.y * xa.y, xb.x * xb.x + xb.y * xb.y);
                        ed.x += pt.x + pt.y;
                        if (wval) {
                            const float ga = (Geo::G == 32 && q > 0) ? mlo[moff + 16 * q] : mb[moff + mpos<Geo>(k)];
                            const float gb = (Geo::G == 32 && q > 0) ? mhi[moff - 16 * q] : mb[moff + mpos<Geo>(M - k)];
                            const float sa = pt.x - ga * pt.x, sb = pt.y - gb * pt.y;
                            ed.y += sa * sa + sb * sb;
                            const float da = ra[q] - ga * pt.x, db = rb[q] - gb * pt.y;
                            st2.x += ga * da > 0.0f ? da * da : 0.0f;
                            st2.y += gb * db > 0.0f ? db * db : 0.0f;
                        }
                    }
                    if (core.leader) {
                        const float ptm = 4.0f * (v[V / 2].x * v[V / 2].x + v[V / 2].y * v[V / 2].y);
                        ed.x += ptm;
                        if (wval) {
                            const float gmid = mb[moff + mpos<Geo>(M / 2)];
                            const float sm = ptm - gmid * ptm, dm = rmid - gmid * ptm;
                            ed.y += sm * sm;
                            acc[sekern::SUM_SPEC_ST] += gmid * dm > 0.0f ? dm * dm : 0.0f;
                        }
                    }
                }
                ed = group_sum<Geo>(ed, lane, jg, core.active);
                if (own && core.leader) {
                    reinterpret_cast<float2*>(a.wsd_terms)[(long long)u * F + f] = ed;
                    wmax = fmaxf(wmax, ed.x);
                }
            } else {
                float2 zm[NP];
                core.fetch_mirror(v, zm, lane);
                if (own) {
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        float2 xa, xb;
                        split_pair(v[q], zm[q], core.twn[q], xa, xb);
                        const float2 pt = make_float2(xa.x * xa.x + xa.y * xa.y, xb.x * xb.x + xb.y * xb.y);
                        const float2 r = make_float2(ra[q], rb[q]);
                        const float2 rt = pmul(r, pt);
                        st2 = cadd(st2, make_float2(fast_sqrt(rt.x), fast_sqrt(rt.y)));
                        tt2 = cadd(tt2, pt);
                        ss2 = cadd(ss2, r);
                    }
                    if (core.leader) {
                        const float ptm = 4.0f * (v[V / 2].x * v[V / 2].x + v[V / 2].y * v[V / 2].y);
                        acc[sekern::SUM_SPEC_ST] += fast_sqrt(rmid * ptm);
                        acc[sekern::SUM_SPEC_TT] += ptm;
                        acc[sekern::SUM_SPEC_SS] += rmid;
                    }
                }
            }
        }
        if (mask_group_open) cp_async_commit();                                     // keep the group count uniform
        __syncwarp();                                                               // the first hop's ring slots are dead now
        slot0 += Geo::HB;
        slot0 = slot0 >= RB ? slot0 - RB : slot0;
    }
    cp_async_wait<0>();
    // the last run of an utterance also zero-fills [out_len, pad_to) and finishes sum c^2 over [out_len, len)
    if (active && my_iters > 0 && e1 == S::E_MIN + plan.per_utt - 1) {
        const int hi = a.pad_to > len ? a.pad_to : len;
        for (int t = a.out_len + jg; t < hi; t += G) {
            if (t < a.pad_to) orow[t] = 0.0f;
            if (a.sums && crow && t < len) { const float c = __ldg(crow + t); acc[sekern::SUM_CC] += c * c; }
        }
    }
    if (a.sums) {
        acc[sekern::SUM_YY] += yy2.x + yy2.y;
        acc[sekern::SUM_YC] += yc2.x + yc2.y;
        acc[sekern::SUM_CC] += cc2.x + cc2.y;
        acc[sekern::SUM_SPEC_ST] += st2.x + st2.y;
        acc[sekern::SUM_SPEC_TT] += tt2.x + tt2.y;
        acc[sekern::SUM_SPEC_SS] += ss2.x + ss2.y;
        if (Geo::GPW == 1) {
#pragma unroll
            for (int i = 0; i < sekern::NSUMS; ++i) {
                float s = acc[i];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
                if (lane == 0 && active && s != 0.0f) atomicAdd(a.sums + (long long)u * sekern::NSUMS + i, (double)s);
            }
        } else {
            // groups of G lanes: through the group's (now idle) transpose buffer
            float* red = reinterpret_cast<float*>(region);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < sekern::NSUMS; ++i) red[i * G + jg] = acc[i];
            __syncwarp();
            if (active && jg < sekern::NSUMS) {
                float s = 0.0f;
                for (int l = 0; l < G; ++l) s += red[jg * G + l];
                if (s != 0.0f) atomicAdd(a.sums + (long long)u * sekern::NSUMS + jg, (double)s);
            }
        }
    }
    // one atomic per run; the buffer rests at 0.0f, and non-negative floats order as their bit patterns
    if (WSD && active && core.leader && wmax > 0.0f) atomicMax(reinterpret_cast<int*>(a.wsd_max), __float_as_int(wmax));
    if (TRACE) trace_end(a.trace, 3, smem + Z::SMEM);
}

template <class Geo> long long resident_groups(int warps, int min_blocks) {
    return (long long)secommon::device_sms() * min_blocks * warps * Geo::GPW;
}

template <class Geo, bool TRACE> int prepare_geo() {
#define SE_OPT(K, BYTES) SE_CUDA_CHECK(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES)))
    SE_OPT((stft_run_kernel<Geo, false, false, TRACE>), K1Sz<Geo>::SMEM);
    SE_OPT((stft_run_kernel<Geo, true, false, TRACE>), K1Sz<Geo>::SMEM);
    SE_OPT((stft_run_kernel<Geo, false, true, TRACE>), K1Sz<Geo>::SMEM);
    SE_OPT((mask_istft_run_kernel<Geo, false, TRACE>), K3Sz<Geo>::SMEM);
    SE_OPT((mask_istft_run_kernel<Geo, true, TRACE>), K3Sz<Geo>::SMEM);
    SE_OPT((mask_istft_run_kernel<Geo, false, TRACE, true>), (K3Sz<Geo, 2>::SMEM));
#undef SE_OPT
    return TRACE ? SE_OK : prepare_geo<Geo, true>();
}

template <class Geo, bool PHASE, bool STATS> void launch_stft_kernel(const StftArgs& a, const GeoRunPlan& plan, unsigned grid, cudaStream_t st) {
    constexpr int THREADS = K1Cfg<Geo>::WARPS * 32;
    constexpr size_t SMEM = K1Sz<Geo>::SMEM;
    if (a.trace) stft_run_kernel<Geo, PHASE, STATS, true><<<grid, THREADS, SMEM, st>>>(a, plan);
    else stft_run_kernel<Geo, PHASE, STATS, false><<<grid, THREADS, SMEM, st>>>(a, plan);
}

template <class Geo> int launch_stft_geo(const StftArgs& a, cudaStream_t st) {
    const long long total = (long long)a.n_utt * a.n_frames;
    if (total > 0x7fffff00LL) return secommon::fail(SE_ERR_BAD_ARG, "too many frames (%lld)", total);
    if (!a.power && !a.phase && !a.logp) return SE_OK;
    if (a.stat_sums && a.phase) return secommon::fail(SE_ERR_BAD_ARG, "statistics need power and / or logpower (no phase)");
    constexpr int WARPS = K1Cfg<Geo>::WARPS, GROUPS = K1Sz<Geo>::GROUPS;
    // runs: one balanced wave when the batch is small, runs of about 32 frames otherwise
    const long long slots = resident_groups<Geo>(WARPS, K1Cfg<Geo>::MIN_BLOCKS);
    long long rpu;
    if (total <= slots * 32) {
        rpu = slots / a.n_utt;
        if (rpu > a.n_frames) rpu = a.n_frames;
    } else rpu = (a.n_frames + 31) / 32;
    if (rpu < 1) rpu = 1;
    GeoRunPlan plan;
    plan.per_utt = a.n_frames;
    plan.runs_per_utt = (int)rpu;
    plan.total_runs = (long long)a.n_utt * rpu;
    const long long grid = (plan.total_runs + GROUPS - 1) / GROUPS;
    if (grid > 0x7fffffffLL) return secommon::fail(SE_ERR_BAD_ARG, "grid too large");
    if (a.stat_sums) launch_stft_kernel<Geo, false, true>(a, plan, (unsigned)grid, st);
    else if (a.phase) launch_stft_kernel<Geo, true, false>(a, plan, (unsigned)grid, st);
    else launch_stft_kernel<Geo, false, false>(a, plan, (unsigned)grid, st);
    return secommon::check_launch("stft_run_kernel");
}

template <class Geo> int launch_mask_istft_geo(const MaskIstftArgs& a, cudaStream_t st) {
    using S = Sz<Geo>;
    constexpr int WARPS = K3Cfg<Geo>::WARPS, GROUPS = K3Sz<Geo>::GROUPS;
    // emit windows E_MIN .. F - 1 + NV of every utterance are cut into runs_per_utt near-equal runs.  Small batches: as many
    // runs as there are resident lane groups (one balanced wave), but runs of at least 4 x halo windows (every run recomputes
    // `halo` frames); large batches: runs of about 64 windows.
    const int per_utt = a.n_frames - 1 + S::NV - S::E_MIN + 1;
    const long long slots = resident_groups<Geo>(WARPS, K3Cfg<Geo>::MIN_BLOCKS);
    long long rpu;
    if ((long long)a.n_utt * per_utt <= slots * 32) {
        rpu = slots / a.n_utt;
        const long long cap = per_utt / (4 * S::HALO);
        if (rpu > cap) rpu = cap;
    } else rpu = (per_utt + 63) / 64;                                 // (every run recomputes `halo` frames: 64 beats 32 by 3 % at 128 x 60 s)
    if (rpu < 1) rpu = 1;
    if (rpu > per_utt) rpu = per_utt;
    GeoRunPlan plan;
    plan.per_utt = per_utt;
    plan.runs_per_utt = (int)rpu;
    plan.total_runs = (long long)a.n_utt * rpu;
    const long long grid = (plan.total_runs + GROUPS - 1) / GROUPS;
    if (grid > 0x7fffffffLL) return secommon::fail(SE_ERR_BAD_ARG, "grid too large");
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(WARPS * 32);
    cfg.dynamicSmemBytes = a.wsd_terms ? K3Sz<Geo, 2>::SMEM : K3Sz<Geo>::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;       // prologue overlaps the upstream kernel's tail
    attr[0].val.programmaticStreamSerializationAllowed = (secommon::pdl_mask() & 2) ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    void (*kernel)(MaskIstftArgs, GeoRunPlan) =
        a.wsd_terms ? (a.trace ? mask_istft_run_kernel<Geo, false, true, true> : mask_istft_run_kernel<Geo, false, false, true>)
        : a.mask_is_power ? (a.trace ? mask_istft_run_kernel<Geo, true, true> : mask_istft_run_kernel<Geo, true, false>)
                          : (a.trace ? mask_istft_run_kernel<Geo, false, true> : mask_istft_run_kernel<Geo, false, false>);
    SE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, a, plan));
    return secommon::check_launch("mask_istft_run_kernel");
}

}  // namespace

namespace sefast {

bool geo_supported(int n_fft, int hop) {
    return (n_fft == 512 && hop == 256) || (n_fft == 1024 && hop == 256) || (n_fft == 400 && hop == 160);
}

int prepare_geo_kernels(int n_fft) {
    if (n_fft == 512) return prepare_geo<Geo512, false>();
    if (n_fft == 1024) return prepare_geo<Geo1024, false>();
    if (n_fft == 400) return prepare_geo<Geo400, false>();
    return SE_OK;
}

int launch_stft_run(const StftArgs& a, int n_fft, cudaStream_t st) {
    if (n_fft == 512) return launch_stft_geo<Geo512>(a, st);
    if (n_fft == 1024) return launch_stft_geo<Geo1024>(a, st);
    return launch_stft_geo<Geo400>(a, st);
}

int launch_mask_istft_run(const MaskIstftArgs& a, int n_fft, cudaStream_t st) {
    if (n_fft == 512) return launch_mask_istft_geo<Geo512>(a, st);
    if (n_fft == 1024) return launch_mask_istft_geo<Geo1024>(a, st);
    return launch_mask_istft_geo<Geo400>(a, st);
}

}  // namespace sefast
