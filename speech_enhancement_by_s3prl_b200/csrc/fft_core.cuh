// Radix butterflies and Stockham stages for the shared-memory FFT used by the
// STFT / iSTFT kernels.  Everything here is plain arithmetic on caller-provided
// arrays, marked SE_HD so that the same code is (a) inlined into the sm_100a
// kernels and (b) compiled by g++ into a host test harness (tests/test_fft_core.py)
// that checks indexing and twiddles against numpy without a GPU.
//
// Conventions
//   * complex numbers are float2 (x = re, y = im)
//   * DIR = -1 : forward transform  exp(-2*pi*i*k*n/M);  DIR = +1 : inverse (unnormalised)
//   * twM[i] = exp(-2*pi*i * i / M), i < M   (forward M-th roots; conjugated for DIR=+1)
//   * twN[k] = exp(-2*pi*i * k / N), k <= M, N = 2M (real-FFT split/merge twiddles)
//   * a real N-point transform is done as an M = N/2 point complex transform of
//     z[m] = x[2m] + i*x[2m+1] followed (forward) or preceded (inverse) by the
//     split/merge step below.
#pragma once

#if defined(__CUDACC__)
#define SE_HD __host__ __device__ __forceinline__
#else
#define SE_HD inline
#include <cmath>
struct float2 { float x, y; };
static inline float2 make_float2(float x, float y) { float2 r; r.x = x; r.y = y; return r; }
#endif

namespace sefft {

#if defined(__CUDA_ARCH__)
// sm_100 packed fp32 arithmetic: one FADD2 / FMUL2 / FFMA2 works on a (re, im) register pair, and ptxas folds some
// component shuffles into the operand selectors of those instructions (R.F32 broadcast, R.F32x2.HI_LO swap, .NP), so a
// complex add is ONE instruction.  Which shuffles fold depends on the operand: cmul is written as
//   a * b = (a.x, a.y) * (b.x, b.x) + (a.y, a.x) * (-b.y, b.y)
// (broadcast of b.x, swap of a, the sign pattern on the broadcast of b.y), which compiles to one FMUL2 + one FFMA2 also
// when b is a conjugated twiddle.  The textbook form (a.x, a.x) * (b.x, b.y) + (a.y, a.y) * (-b.y, b.x) does not fold:
// ptxas builds (-b.y, b.x) with a scalar FADD and a MOV per use (4 instructions per multiply; tools/sass_fastgeo.py).
// The rounding is that of the scalar forms with the usual mul+add contraction (re = fma(-a.y, b.y, a.x b.x),
// im = fma(a.x, b.y, a.y b.x)).
typedef unsigned long long se_u64;
__device__ __forceinline__ se_u64 pk2(float lo, float hi) { se_u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ float2 upk2(se_u64 v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r; }
__device__ __forceinline__ se_u64 add2(se_u64 a, se_u64 b) { se_u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ se_u64 sub2(se_u64 a, se_u64 b) { se_u64 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ se_u64 mul2(se_u64 a, se_u64 b) { se_u64 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ se_u64 fma2(se_u64 a, se_u64 b, se_u64 c) { se_u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return upk2(add2(pk2(a.x, a.y), pk2(b.x, b.y))); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return upk2(sub2(pk2(a.x, a.y), pk2(b.x, b.y))); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return upk2(fma2(pk2(a.y, a.x), pk2(-b.y, b.y), mul2(pk2(a.x, a.y), pk2(b.x, b.x))));
}
__device__ __forceinline__ float2 cscale(float2 a, float s) { return upk2(mul2(pk2(a.x, a.y), pk2(s, s))); }
// a * b + c (complex), and element-wise a * b / a * b + c on (x, y) pairs
__device__ __forceinline__ float2 cmadd(float2 a, float2 b, float2 c) {
    return upk2(fma2(pk2(a.y, a.x), pk2(-b.y, b.y), fma2(pk2(a.x, a.y), pk2(b.x, b.x), pk2(c.x, c.y))));
}
__device__ __forceinline__ float2 pmul(float2 a, float2 b) { return upk2(mul2(pk2(a.x, a.y), pk2(b.x, b.y))); }
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c) { return upk2(fma2(pk2(a.x, a.y), pk2(b.x, b.y), pk2(c.x, c.y))); }
#else
SE_HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
SE_HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
SE_HD float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
SE_HD float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
SE_HD float2 cmadd(float2 a, float2 b, float2 c) { return cadd(cmul(a, b), c); }
SE_HD float2 pmul(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
SE_HD float2 pfma(float2 a, float2 b, float2 c) { return make_float2(a.x * b.x + c.x, a.y * b.y + c.y); }
#endif
SE_HD float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
// multiply by DIR * i  (forward: by -i, inverse: by +i)
template <int DIR> SE_HD float2 mul_dir_i(float2 a) {
    return DIR < 0 ? make_float2(a.y, -a.x) : make_float2(-a.y, a.x);
}

template <int DIR> SE_HD void bfly2(float2& a, float2& b) {
    float2 t = csub(a, b);
    a = cadd(a, b);
    b = t;
}

// in-place DFT of (a0,a1,a2,a3), natural order out
template <int DIR> SE_HD void bfly4(float2& a0, float2& a1, float2& a2, float2& a3) {
    float2 t0 = cadd(a0, a2), t1 = csub(a0, a2);
    float2 t2 = cadd(a1, a3), t3 = mul_dir_i<DIR>(csub(a1, a3));
    a0 = cadd(t0, t2);
    a2 = csub(t0, t2);
    a1 = cadd(t1, t3);
    a3 = csub(t1, t3);
}

template <int DIR> SE_HD void bfly5(float2& a0, float2& a1, float2& a2, float2& a3, float2& a4) {
    const float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f;
    const float s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
    float2 t1 = cadd(a1, a4), t2 = cadd(a2, a3), t3 = csub(a1, a4), t4 = csub(a2, a3);
    float2 m1 = make_float2(a0.x + c1 * t1.x + c2 * t2.x, a0.y + c1 * t1.y + c2 * t2.y);
    float2 m2 = make_float2(a0.x + c2 * t1.x + c1 * t2.x, a0.y + c2 * t1.y + c1 * t2.y);
    float2 n1 = mul_dir_i<DIR>(make_float2(s1 * t3.x + s2 * t4.x, s1 * t3.y + s2 * t4.y));
    float2 n2 = mul_dir_i<DIR>(make_float2(s2 * t3.x - s1 * t4.x, s2 * t3.y - s1 * t4.y));
    a0 = make_float2(a0.x + t1.x + t2.x, a0.y + t1.y + t2.y);
    a1 = cadd(m1, n1);
    a4 = csub(m1, n1);
    a2 = cadd(m2, n2);
    a3 = csub(m2, n2);
}

// multiply by exp(DIR * 2*pi*i * q / 8), q = 1, 3  (q = 2 is mul_dir_i)
template <int DIR> SE_HD float2 mul_w8_1(float2 a) {
    const float h = 0.70710678118654752f;
    return cscale(cadd(a, mul_dir_i<DIR>(a)), h);            // (1 + DIR i) a / sqrt 2
}
template <int DIR> SE_HD float2 mul_w8_3(float2 a) {
    const float h = 0.70710678118654752f;
    return cscale(csub(a, mul_dir_i<DIR>(a)), -h);           // (-1 + DIR i) a / sqrt 2
}

// in-place 8-point DFT of v[0..7] (stride S in the array), natural order out
template <int DIR, int S> SE_HD void bfly8(float2* v) {
    bfly4<DIR>(v[0 * S], v[2 * S], v[4 * S], v[6 * S]);   // E[0..3] -> slots 0,2,4,6
    bfly4<DIR>(v[1 * S], v[3 * S], v[5 * S], v[7 * S]);   // O[0..3] -> slots 1,3,5,7
    float2 e0 = v[0 * S], e1 = v[2 * S], e2 = v[4 * S], e3 = v[6 * S];
    float2 o0 = v[1 * S], o1 = mul_w8_1<DIR>(v[3 * S]), o2 = mul_dir_i<DIR>(v[5 * S]), o3 = mul_w8_3<DIR>(v[7 * S]);
    v[0 * S] = cadd(e0, o0); v[4 * S] = csub(e0, o0);
    v[1 * S] = cadd(e1, o1); v[5 * S] = csub(e1, o1);
    v[2 * S] = cadd(e2, o2); v[6 * S] = csub(e2, o2);
    v[3 * S] = cadd(e3, o3); v[7 * S] = csub(e3, o3);
}

template <int DIR> SE_HD float2 mul_w16(float2 a, int q) {   // exp(DIR*2*pi*i*q/16), q = 1,3,5,7
    const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f;
    float wr, wi;
    switch (q) {
        case 1: wr = c1; wi = s1; break;
        case 3: wr = s1; wi = c1; break;
        case 5: wr = -s1; wi = c1; break;
        default: wr = -c1; wi = s1; break;
    }
    wi = DIR < 0 ? -wi : wi;
    return cmul(a, make_float2(wr, wi));
}

template <int DIR> SE_HD void bfly16(float2* v) {
    bfly8<DIR, 2>(v);        // evens -> E[k] in slot 2k
    bfly8<DIR, 2>(v + 1);    // odds  -> O[k] in slot 2k+1
    float2 e[8], o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { e[k] = v[2 * k]; o[k] = v[2 * k + 1]; }
    o[1] = mul_w16<DIR>(o[1], 1);
    o[2] = mul_w8_1<DIR>(o[2]);
    o[3] = mul_w16<DIR>(o[3], 3);
    o[4] = mul_dir_i<DIR>(o[4]);
    o[5] = mul_w16<DIR>(o[5], 5);
    o[6] = mul_w8_3<DIR>(o[6]);
    o[7] = mul_w16<DIR>(o[7], 7);
#pragma unroll
    for (int k = 0; k < 8; ++k) { v[k] = cadd(e[k], o[k]); v[k + 8] = csub(e[k], o[k]); }
}

template <int R, int DIR> struct Butterfly;
template <int DIR> struct Butterfly<2, DIR> { static SE_HD void run(float2* v) { bfly2<DIR>(v[0], v[1]); } };
template <int DIR> struct Butterfly<4, DIR> { static SE_HD void run(float2* v) { bfly4<DIR>(v[0], v[1], v[2], v[3]); } };
template <int DIR> struct Butterfly<5, DIR> { static SE_HD void run(float2* v) { bfly5<DIR>(v[0], v[1], v[2], v[3], v[4]); } };
template <int DIR> struct Butterfly<8, DIR> { static SE_HD void run(float2* v) { bfly8<DIR, 1>(v); } };
template <int DIR> struct Butterfly<16, DIR> { static SE_HD void run(float2* v) { bfly16<DIR>(v); } };

// One radix-R work item (index j in [0, M/R)) of a Stockham autosort stage.
// NS = product of the radices of the earlier stages.  `in(i)` returns logical element i of
// the stage input, `out(i, v)` stores logical element i of the stage output; after the last
// stage the output is in natural order.
template <int M, int R, int NS, int DIR, class In, class Out>
SE_HD void stockham_item(int j, In in, Out out, const float2* __restrict__ twM) {
    float2 v[R];
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = in(j + r * (M / R));
    const int k = (NS > 1) ? (j % NS) : 0;
    if (NS > 1) {
#pragma unroll
        for (int r = 1; r < R; ++r) {
            float2 w = twM[r * k * (M / (NS * R))];
            if (DIR > 0) w.y = -w.y;
            v[r] = cmul(v[r], w);
        }
    }
    Butterfly<R, DIR>::run(v);
    const int base = (j - k) * R + k;
#pragma unroll
    for (int r = 0; r < R; ++r) out(base + r * NS, v[r]);
}

// ---- real <-> half-size complex split / merge -------------------------------------
// forward: X[k] (k in [0, M]) of the real N-point signal from Z = FFT_M(z)
SE_HD float2 rfft_split(float2 zk, float2 zmk, float2 wN) {
    // zk = Z[k mod M], zmk = Z[(M-k) mod M], wN = exp(-2*pi*i*k/N)
    float2 e = make_float2(0.5f * (zk.x + zmk.x), 0.5f * (zk.y - zmk.y));
    float2 d = make_float2(0.5f * (zk.x - zmk.x), 0.5f * (zk.y + zmk.y));   // (Z[k]-conj(Z[M-k]))/2
    float2 o = make_float2(d.y, -d.x);                                          // * (-i)
    return cadd(e, cmul(o, wN));
}
// inverse: Z[k] (k in [0, M)) to feed the unnormalised inverse M-point FFT, from the
// one-sided spectrum X; the result of that FFT times 1/M is x[2m] + i*x[2m+1].
SE_HD float2 irfft_merge(float2 xk, float2 xmk, float2 wN) {
    // xk = X[k], xmk = X[M-k], wN = exp(-2*pi*i*k/N)
    float2 e = make_float2(0.5f * (xk.x + xmk.x), 0.5f * (xk.y - xmk.y));
    float2 d = make_float2(0.5f * (xk.x - xmk.x), 0.5f * (xk.y + xmk.y));
    float2 o = cmul(d, cconj(wN));
    return make_float2(e.x - o.y, e.y + o.x);                                   // e + i*o
}

// ---- compile-time plans -----------------------------------------------------------
// Plan<M>: radices R0..R3 (1 = unused) with R0*R1*R2*R3 == M.
template <int M_> struct Plan;
template <> struct Plan<128>  { static constexpr int M = 128,  R0 = 16, R1 = 8,  R2 = 1, R3 = 1; };
template <> struct Plan<200>  { static constexpr int M = 200,  R0 = 8,  R1 = 5,  R2 = 5, R3 = 1; };
template <> struct Plan<256>  { static constexpr int M = 256,  R0 = 16, R1 = 16, R2 = 1, R3 = 1; };
template <> struct Plan<512>  { static constexpr int M = 512,  R0 = 8,  R1 = 8,  R2 = 8, R3 = 1; };
template <> struct Plan<1024> { static constexpr int M = 1024, R0 = 16, R1 = 8,  R2 = 8, R3 = 1; };

// padded physical index of logical complex element i (one pad slot every 16 elements)
SE_HD int phys(int i) { return i + (i >> 4); }
template <int M> struct Padded { static constexpr int SIZE = M + (M >> 4) + 1; };

}  // namespace sefft
