// Device helpers of the register-resident fast paths (fastgeo.cu: n_fft 512 / hop 256, n_fft 1024 / hop 256 and n_fft 400 /
// hop 160): approximate transcendental wrappers, cp.async staging primitives, the real-input split /
// inverse merge of one pair of bins, the mask application and the programmatic-dependent-launch fences.
#pragma once
#include "fft_core.cuh"

namespace fastc {
using namespace sefft;

// sqrt.approx: no denormal / special-value fix-up path (2 ulp), keeps the kernels free of slow-path calls
__device__ __forceinline__ float fast_sqrt(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// log(x) for x >= log_eps > 0 (never denormal): lg2.approx * ln 2 without __logf's denormal range fix-up (4 of its 8 instructions)
__device__ __forceinline__ float fast_log(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r * 0.693147182464599609375f;
}

// ---- asynchronous staging (cp.async): the global loads of frame i+1 are in flight while frame i is
// transformed, so no lane group ever waits on a DRAM round trip between its transforms.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_PENDING> __device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N_PENDING) : "memory");
}


// One pair of bins (k, M-k) of the real-input split.  zk = Z[k], zm = Z[M-k] (of the 1/2-scaled frame),
// w = exp(-2*pi*i*k/N).  xa = X[k], xb = X[M-k].
__device__ __forceinline__ void split_pair(float2 zk, float2 zm, float2 w, float2& xa, float2& xb) {
    const float2 e = cadd(zk, make_float2(zm.x, -zm.y));
    const float2 o = cadd(make_float2(zk.y, -zk.x), make_float2(zm.y, zm.x));   // -i * (Z[k] - conj Z[M-k])
    const float2 t = cmul(o, w);
    xa = cadd(e, t);
    xb = cconj(csub(e, t));
}
// Inverse of split_pair up to a factor 2: from Y[k], Y[M-k] the values conj(Zinv[k]), conj(Zinv[M-k])
// that feed the forward FFT used as an inverse.
__device__ __forceinline__ void merge_pair_conj(float2 ya, float2 yb, float2 w, float2& ca, float2& cb) {
    const float2 ybc = make_float2(yb.x, -yb.y);
    const float2 e = cadd(ya, ybc);
    const float2 d = csub(ya, ybc);
    const float2 o = cmul(d, make_float2(w.x, -w.y));
    const float2 u = make_float2(-o.y, o.x);                                  // i * o
    ca = cconj(cadd(e, u));                                                   // conj(Zinv[k])   = conj(e + u)
    cb = csub(e, u);                                                          // conj(Zinv[M-k]) = e - u
}


__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// One masked pair of bins: spectral-loss terms (own) and the merged, conjugated inverse-FFT input
// PM ("power mode"): ga / gb are the target POWER of the bins, the output keeps the phase of X: Y = sqrt(g) X / |X|, and
// Y = sqrt(g) where X = 0 (atan2(0, 0) = 0) -- OnlinePreprocessor.istft(linears, phase_inp) without the phase (runner.py:266-281)
template <bool PM> __device__ __forceinline__ float2 apply_gain(float2 x, float g) {
    if (!PM) return cscale(x, fast_sqrt(g));
    const float p = x.x * x.x + x.y * x.y;
    return p > 0.0f ? cscale(x, fast_sqrt(g) * rsqrtf(p)) : make_float2(fast_sqrt(g), 0.0f);
}
// RELU = false (the WSD variant of K3): ra / rb keep the signed mask * |X|^2
template <bool PM, bool RELU = true>
__device__ __forceinline__ void mask_merge(float2 xa, float2 xb, float ga, float gb, float2 w, bool own, float& ra, float& rb,
                                           float2& ca, float2& cb) {
    if (own) {
        ra = PM ? ga : ga * (xa.x * xa.x + xa.y * xa.y);
        rb = PM ? gb : gb * (xb.x * xb.x + xb.y * xb.y);
        if (RELU) { ra = fmaxf(ra, 0.0f); rb = fmaxf(rb, 0.0f); }
    }
    merge_pair_conj(apply_gain<PM>(xa, ga), apply_gain<PM>(xb, gb), w, ca, cb);
}


}  // namespace fastc
