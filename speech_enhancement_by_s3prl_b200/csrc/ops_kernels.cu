// libse_b200.so -- objectives, metrics, level normalisation, length masks, feature
// post-processing and the fp32 (SIMT) mask head.  Entry points: include/se_b200.h.
// All of these are streaming / reduction kernels bounded by HBM bandwidth except the
// head GEMM, whose tensor-core (tcgen05) variant lives in head_tc.cu.
#include <algorithm>
#include <cmath>
#include "objective_math.cuh"
#include "se_common.cuh"

using secommon::fail;
using secommon::block_accumulate_to;

namespace sehead {
int launch_linear_head_tc(const float* x, long long ldx, const float* mean, const float* stdv, long long ld_stats, float cmvn_eps,
                          const float* W, long long ldw, const float* b, long long R, int n_frames, int Din, int Dout, int act,
                          const float* linears, float* offset_out, float* pred_out, long long ld_out, cudaStream_t st);
}

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float relu(float x) { return x > 0.0f ? x : 0.0f; }

// ------------------------------------------------------------------ finalize (gain + metrics)
// level_or_neg: 10^(target_dB/10) computed on the host, or < 0 to match the clean reference's own level.
// 10^(10 log10(x) / 10) == x, so the reference's dB round trip (utils.py:38-42) needs no pow/log here.
__global__ void finalize_metrics_kernel(const double* __restrict__ sums, const long long* __restrict__ lengths,
                                        int T, double level_or_neg, float* __restrict__ wav, long long wav_stride,
                                        int width, float* __restrict__ gain_out, float* __restrict__ sisdr_wave,
                                        float* __restrict__ loss_spec, double* __restrict__ metric_acc, int chunks,
                                        unsigned long long* trace_buf) {
    secommon::TraceScope trace(trace_buf, 4);
    asm volatile("griddepcontrol.wait;" ::: "memory");                   // sums and wav come from the upstream kernel
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    // the first batch of waveform loads does not depend on the gain: issue it before the (double precision) gain arithmetic
    float* row = wav ? wav + (long long)u * wav_stride : nullptr;
    const int per = (((width + chunks - 1) / chunks) + 3) & ~3;
    const int lo = chunk * per, hi = min(width, lo + per);
    const bool vec = wav && (reinterpret_cast<uintptr_t>(row) & 15) == 0;
    float4* r4 = reinterpret_cast<float4*>(row);
    const int n4 = (hi & ~3) / 4, bd = blockDim.x;
    const int i0 = lo / 4 + threadIdx.x;
    float4 v[8];
    if (vec) {
#pragma unroll
        for (int q = 0; q < 8; ++q) if (i0 + q * bd < n4) v[q] = r4[i0 + q * bd];
    }
    const double* s = sums + (long long)u * SE_NSUMS;
    // clamped to [0, T] as se_mask_istft clamps it for the sums: the means divide by the samples that were summed
    const double len = lengths ? (double)min((long long)T, max(0LL, lengths[u])) : (double)T;
    const double eps_mean = 1e-8;                                       // utils.py:26, utils.py:31
    const double mean_yy = s[SE_SUM_YY] / (len + eps_mean);
    const double level = level_or_neg < 0.0 ? s[SE_SUM_CC] / (len + eps_mean) : level_or_neg;
    const double gain = sqrt(level / (mean_yy + eps_mean));
    if (chunk == 0 && threadIdx.x == 0) {
        if (gain_out) gain_out[u] = (float)gain;
        const float sd = (float)sisdr_from_sums(gain * s[SE_SUM_YC], s[SE_SUM_CC], gain * gain * s[SE_SUM_YY], 1e-10);
        const float ls = (float)(-sisdr_from_sums(s[SE_SUM_SPEC_ST], s[SE_SUM_SPEC_TT], s[SE_SUM_SPEC_SS], 1e-10));
        if (sisdr_wave) sisdr_wave[u] = sd;
        if (loss_spec) loss_spec[u] = ls;
        if (metric_acc) {                                               // running sums of an evaluation pass (runner.py:602)
            if (loss_spec) atomicAdd(metric_acc, (double)ls);           // only the terms this call produces
            if (sisdr_wave) atomicAdd(metric_acc + 1, (double)sd);
            atomicAdd(metric_acc + 2, 1.0);
        }
    }
    if (!wav) { trace.finish(); return; }
    const float g = (float)gain;
    if (vec) {
        for (int i = i0; i < n4; i += 8 * bd) {                              // eight (predicated) loads in flight per thread
            if (i != i0) {
#pragma unroll
                for (int q = 0; q < 8; ++q) if (i + q * bd < n4) v[q] = r4[i + q * bd];
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (i + q * bd < n4) {
                    v[q].x *= g; v[q].y *= g; v[q].z *= g; v[q].w *= g;
                    r4[i + q * bd] = v[q];
                }
        }
        for (int k = (hi & ~3) + threadIdx.x; k < hi; k += blockDim.x) row[k] *= g;
    } else {
        for (int k = lo + threadIdx.x; k < hi; k += blockDim.x) row[k] *= g;
    }
    if (trace_buf) { __syncthreads(); trace.finish(); }
}

// ------------------------------------------------------------------ spectral SI-SDR objective
// one block: per-utterance losses and (loss_mean != null) their batch mean (objective.py:100) in one launch
__global__ void __launch_bounds__(256) sisdr_finish_mean_kernel(const double* __restrict__ sums3, int n_utt, float eps,
                                                                float* __restrict__ loss, float* __restrict__ loss_mean) {
    __shared__ double part[8];
    double acc = 0.0;
    for (int u = threadIdx.x; u < n_utt; u += blockDim.x) {
        const float l = (float)(-sisdr_from_sums(sums3[3 * u], sums3[3 * u + 1], sums3[3 * u + 2], (double)eps));
        if (loss) loss[u] = l;
        acc += (double)l;
    }
    acc = secommon::warp_sum(acc);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0 && loss_mean) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
        *loss_mean = (float)(t / (double)n_utt);
    }
}

// The sums and the backward run on predicted = offset * linear_inp (model.py:33) without materialising `predicted`, on row-strided
// tensors (rows ld floats apart; V = 4: 16-byte aligned rows read as float4, V = 1: any stride); offset = null: predicted =
// linear_inp (the dense entry points pass ld = K).  The backward writes d loss / d offset = d loss / d predicted * linear_inp
// directly (0 on padded frames and on the pad columns of a row).
template <int V> __device__ __forceinline__ void ldv(const float* p, float (&v)[V]) {
    if (V == 4) { const float4 q = *reinterpret_cast<const float4*>(p); v[0] = q.x; v[1 % V] = q.y; v[2 % V] = q.z; v[3 % V] = q.w; }
    else v[0] = *p;
}
template <int V> __device__ __forceinline__ void stv(float* p, const float (&v)[V]) {
    if (V == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1 % V], v[2 % V], v[3 % V]);
    else *p = v[0];
}

struct SisdrMaskArgs {
    const float* offset; const float* inp; const float* tar;     // offset may be null (predicted = inp)
    long long ld_off, ld_inp, ld_tar;
    const long long* stft_len;
    int n_utt, n_frames, K, chunks;
    double* sums3;
    float eps; const float* grad_out; float* grad_offset; long long ld_g;   // backward only
    int len_hop;             // > 0: stft_len holds SAMPLE lengths, frames = len / len_hop + 1 (runner.py:455)
    float grad_uniform;      // grad_out == nullptr: every utterance's upstream gradient (1 / B for the batch-mean loss)
};

__device__ __forceinline__ int mask_valid_frames(const SisdrMaskArgs& a, int u) {
    long long v = a.n_frames;
    if (a.stft_len) v = a.len_hop > 0 ? a.stft_len[u] / a.len_hop + 1 : a.stft_len[u];
    return (int)min((long long)a.n_frames, v);
}

template <int V>
__global__ void __launch_bounds__(256) sisdr_mask_sums_kernel(const SisdrMaskArgs a) {
    const int u = blockIdx.x / a.chunks, chunk = blockIdx.x - u * a.chunks;
    const int valid = mask_valid_frames(a, u);
    const int KV = (a.K + V - 1) / V;
    const int per = (valid + a.chunks - 1) / a.chunks;
    const int f_lo = chunk * per, f_hi = min(valid, f_lo + per);
    const long long row0 = (long long)u * a.n_frames;
    float acc[3] = {0.f, 0.f, 0.f};
    const int items = max(f_hi - f_lo, 0) * KV;
#pragma unroll 4
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int fr = i / KV, c = (i - fr * KV) * V;
        const long long r = row0 + f_lo + fr;
        float x[V], t[V], o[V];
        ldv<V>(a.inp + r * a.ld_inp + c, x);
        ldv<V>(a.tar + r * a.ld_tar + c, t);
        if (a.offset) ldv<V>(a.offset + r * a.ld_off + c, o);
#pragma unroll
        for (int e = 0; e < V; ++e)
            if (c + e < a.K) {
                const float rp = relu(a.offset ? o[e] * x[e] : x[e]), rt = relu(t[e]);
                acc[0] += sqrtf(rp) * sqrtf(rt);
                acc[1] += rt;
                acc[2] += rp;
            }
    }
    block_accumulate_to<3, float>(acc, a.sums3 + (long long)u * 3);
}

template <int V>
__global__ void __launch_bounds__(256) sisdr_mask_bwd_kernel(const SisdrMaskArgs a) {
    const int u = blockIdx.x / a.chunks, chunk = blockIdx.x - u * a.chunks;
    const int valid = mask_valid_frames(a, u);
    const int KV = (int)(a.ld_g / V) < (a.K + V - 1) / V ? (a.K + V - 1) / V : (int)(a.ld_g / V);   // whole rows of grad_offset
    const int per = (a.n_frames + a.chunks - 1) / a.chunks;
    const int f_lo = chunk * per, f_hi = min(a.n_frames, f_lo + per);
    const float2 coef = sisdr_coef(a.sums3 + 3 * u, (double)a.eps, a.grad_out ? (double)a.grad_out[u] : (double)a.grad_uniform);
    const long long row0 = (long long)u * a.n_frames;
    const int items = max(f_hi - f_lo, 0) * KV;
#pragma unroll 4
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int fr = i / KV, c = (i - fr * KV) * V;
        const int f = f_lo + fr;
        const long long r = row0 + f;
        float g[V];
#pragma unroll
        for (int e = 0; e < V; ++e) g[e] = 0.0f;
        if (f < valid && c < a.K) {
            float x[V], t[V], o[V];
            ldv<V>(a.inp + r * a.ld_inp + c, x);
            ldv<V>(a.tar + r * a.ld_tar + c, t);
            if (a.offset) ldv<V>(a.offset + r * a.ld_off + c, o);
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float pi = a.offset ? o[e] * x[e] : x[e];
                if (c + e < a.K && pi > 0.0f) {
                    const float sq = sqrtf(pi), ti = sqrtf(relu(t[e]));
                    g[e] = (coef.x * ti + coef.y * sq) * (0.5f / sq) * (a.offset ? x[e] : 1.0f);
                }
            }
        }
        if (c + V <= a.ld_g) stv<V>(a.grad_offset + r * a.ld_g + c, g);
    }
}

// ------------------------------------------------------------------ gradient clipping + Adam for the head's parameters
// runner.py:463-466 (clip_grad_norm_ -> optimizer.step) on a handful of small tensors: torch runs ~15 launches for it,
// here it is two -- the squared gradient norm, then clip + update.  All state (moments, step count, norm accumulator) lives
// on the device, so the pair replays from a CUDA graph.  32 tensors cover a bidirectional 3-layer LSTM body and its projection (26);
// AdamArgs (1976 bytes) travels by value, far inside the kernel-parameter limit.
constexpr int kAdamMaxTensors = 32;
struct AdamArgs {
    float* p[kAdamMaxTensors]; float* g[kAdamMaxTensors]; float* m[kAdamMaxTensors]; float* v[kAdamMaxTensors];
    long long n[kAdamMaxTensors];
    int count;
    float lr, beta1, beta2, eps, weight_decay, max_norm;   // max_norm <= 0: no clipping
    float* mir[kAdamMaxTensors]; int mir_cols[kAdamMaxTensors]; long long mir_ld[kAdamMaxTensors]; int mir_tf32;   // optional row-padded copies
    double* acc;       // [1] sum of squared gradients of this step (zeroed by the update kernel's last CTA)
    int* state;        // [0] steps taken, [1] CTAs of the update kernel that have finished, [2] steps skipped (NaN / inf norm)
};

__global__ void __launch_bounds__(256) adam_norm_kernel(const AdamArgs a) {
    float acc[1] = {0.0f};
    for (int t = 0; t < a.count; ++t)
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n[t]; i += (long long)gridDim.x * blockDim.x) {
            const float g = a.g[t][i];
            acc[0] += g * g;
        }
    block_accumulate_to<1, float>(acc, a.acc);
}

__global__ void __launch_bounds__(256) adam_update_kernel(const AdamArgs a) {
    const int step = a.state[0] + 1;                                        // torch.optim.Adam: bias corrections use the new count
    const double sumsq = *a.acc;
    // runner.py:467-470: a NaN / inf gradient norm skips optimizer.step() -- parameters, moments and the step count stay as
    // they are (the gradients too: the runner zeroes them next).  The norm is always accumulated so that the guard also holds
    // without clipping.
    const bool finite = sumsq == sumsq && sumsq <= 3.0e38;
    float clip = 1.0f;
    if (a.max_norm > 0.0f) {
        const float total = (float)sqrt(sumsq);
        clip = fminf(a.max_norm / (total + 1e-6f), 1.0f);                   // torch.nn.utils.clip_grad_norm_
    }
    const double bc1 = 1.0 - pow((double)a.beta1, (double)step), bc2 = 1.0 - pow((double)a.beta2, (double)step);
    const float step_size = (float)(a.lr / bc1), inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
    if (finite)
    for (int t = 0; t < a.count; ++t)
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n[t]; i += (long long)gridDim.x * blockDim.x) {
            float g = a.g[t][i] * clip;
            a.g[t][i] = g;                                                  // the clipped gradient stays visible, as in torch
            const float p = a.p[t][i];
            if (a.weight_decay != 0.0f) g += a.weight_decay * p;
            const float m = a.beta1 * a.m[t][i] + (1.0f - a.beta1) * g;
            const float v = a.beta2 * a.v[t][i] + (1.0f - a.beta2) * g * g;
            a.m[t][i] = m;
            a.v[t][i] = v;
            const float pn = p - step_size * m / (sqrtf(v) * inv_sqrt_bc2 + a.eps);
            a.p[t][i] = pn;
            if (a.mir[t]) {                                                 // the row-padded (TF32-rounded) copy the head kernels read
                const long long row = i / a.mir_cols[t];
                const int col = (int)(i - row * a.mir_cols[t]);
                float w = pn;
                if (a.mir_tf32) w = __int_as_float((__float_as_int(pn) + 0x1000) & ~0x1FFF);   // nearest, ties away (cvt.rna.tf32)
                a.mir[t][row * a.mir_ld[t] + col] = w;
            }
        }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(a.state + 1, 1) == (int)gridDim.x - 1) {              // every CTA has read acc and the step count
            *a.acc = 0.0;
            a.state[1] = 0;
            if (finite) a.state[0] = step;
            else a.state[2] += 1;                                           // skipped steps (ClipAdam.steps_skipped)
        }
    }
}

// ------------------------------------------------------------------ active-sampling match scores (sampler.py:113-116)
// scores[j] = < key_j / (|key_j| + eps),  mean_i query_i / (|query_i| + eps) >
__global__ void __launch_bounds__(256) row_sumsq_kernel(const float* __restrict__ x, long long P, int chunks, double* __restrict__ out) {
    const int row = blockIdx.x / chunks, chunk = blockIdx.x - row * chunks;
    const long long per = (P + chunks - 1) / chunks, lo = chunk * per, hi = min(P, lo + per);
    const float* r = x + (long long)row * P;
    float acc[1] = {0.0f};
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) acc[0] += r[i] * r[i];
    block_accumulate_to<1, float>(acc, out + row);
}
__global__ void __launch_bounds__(256) match_qbar_kernel(const float* __restrict__ q, int nq, long long P, float eps,
                                                         const double* __restrict__ q_sumsq, float* __restrict__ qbar) {
    // the row norms once per CTA (256 rows at a time) instead of a double-precision sqrt and a divide per element
    __shared__ float s_inv[256];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // grid covers P (se_match_scores)
    float s = 0.0f;
    for (int r0 = 0; r0 < nq; r0 += 256) {
        __syncthreads();
        if (r0 + (int)threadIdx.x < nq) s_inv[threadIdx.x] = 1.0f / ((float)sqrt(q_sumsq[r0 + threadIdx.x]) + eps);
        __syncthreads();
        const int n = min(256, nq - r0);
        if (i < P) {
#pragma unroll 8
            for (int r = 0; r < n; ++r) s = fmaf(q[(long long)(r0 + r) * P + i], s_inv[r], s);
        }
    }
    if (i < P) qbar[i] = s / (float)nq;
}
__global__ void __launch_bounds__(256) match_dot_kernel(const float* __restrict__ k, long long P, int chunks,
                                                        const float* __restrict__ qbar, double* __restrict__ dots) {
    const int row = blockIdx.x / chunks, chunk = blockIdx.x - row * chunks;
    const long long per = (P + chunks - 1) / chunks, lo = chunk * per, hi = min(P, lo + per);
    const float* r = k + (long long)row * P;
    float acc[1] = {0.0f};
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) acc[0] += r[i] * qbar[i];
    block_accumulate_to<1, float>(acc, dots + row);
}
__global__ void match_finish_kernel(const double* __restrict__ k_sumsq, const double* __restrict__ dots, int nk, float eps,
                                    float* __restrict__ scores) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nk) scores[j] = (float)(dots[j] / ((double)((float)sqrt(k_sumsq[j]) + eps)));
}

// ------------------------------------------------------------------ log-spectral L1 objective
__global__ void l1_logspec_fwd_kernel(const float* __restrict__ logp, const float* __restrict__ tar,
                                      const long long* __restrict__ stft_len, int n_frames, int K, float eps,
                                      double* __restrict__ acc2, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const long long valid = (long long)min((long long)n_frames, stft_len ? stft_len[u] : (long long)n_frames) * K;
    const long long per = (valid + chunks - 1) / chunks;
    const long long lo = chunk * per, hi = min(valid, lo + per);
    const float* p = logp + (long long)u * n_frames * K;
    const float* t = tar + (long long)u * n_frames * K;
    float acc[2] = {0.f, 0.f};
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) acc[0] += fabsf(p[i] - logf(t[i] + eps));
    if (threadIdx.x == 0 && hi > lo) acc[1] = (float)(hi - lo);         // exact for < 2^24 elements per chunk
    block_accumulate_to<2, float>(acc, acc2);
}

__global__ void l1_logspec_bwd_kernel(const float* __restrict__ logp, const float* __restrict__ tar,
                                      const long long* __restrict__ stft_len, int n_frames, int K, float eps,
                                      double count, const float* __restrict__ grad_out, float* __restrict__ grad, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const long long total = (long long)n_frames * K;
    const long long valid = (long long)min((long long)n_frames, stft_len ? stft_len[u] : (long long)n_frames) * K;
    const long long per = (total + chunks - 1) / chunks;
    const long long lo = chunk * per, hi = min(total, lo + per);
    const float scale = (float)((double)grad_out[0] / count);
    const float* p = logp + (long long)u * total;
    const float* t = tar + (long long)u * total;
    float* g = grad + (long long)u * total;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        float out = 0.0f;
        if (i < valid) {
            const float d = p[i] - logf(t[i] + eps);
            out = d > 0.0f ? scale : (d < 0.0f ? -scale : 0.0f);
        }
        g[i] = out;
    }
}

// ------------------------------------------------------------------ weighted speech distortion objective (objective.py:120-153)
// energy[u,f] = sum_k S[u,f,k] for EVERY frame (the reference takes energy.max() over the whole padded batch), and the
// batch maximum.  One warp per frame (rows ld floats apart).  The maximum stays a plain float in memory, so that an
// all-reduce(max) of the buffer across data-parallel ranks gives the global one: the caller fills it with 0xff bytes (a
// NaN that every value replaces), non-negative sums go through a signed atomicMax of the bit pattern (their order as
// ints), negative ones through an unsigned atomicMin (reversed order), and a non-negative value beats a negative one in both.
__global__ void wsd_energy_kernel(const float* __restrict__ tar, long long ld, long long n_rows, int K, float* __restrict__ energy,
                                  float* __restrict__ max_energy) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    float best = -INFINITY;
    for (long long r = warp; r < n_rows; r += nwarps) {
        const float* t = tar + r * ld;
        float s = 0.0f;
        for (int k = lane; k < K; k += 32) s += t[k];
        s = secommon::warp_sum(s);
        if (lane == 0) energy[r] = s;
        best = fmaxf(best, s);
    }
    if (lane == 0 && best > -INFINITY) {
        if (best >= 0.0f) atomicMax(reinterpret_cast<int*>(max_energy), __float_as_int(best));
        else atomicMin(reinterpret_cast<unsigned*>(max_energy), __float_as_uint(best));
    }
}
int launch_wsd_energy(const float* tar, long long ld, long long rows, int K, float* energy, float* max_energy, cudaStream_t st) {
    SE_CUDA_CHECK(cudaMemsetAsync(max_energy, 0xff, sizeof(float), st));
    const long long want = (rows + 7) / 8;
    wsd_energy_kernel<<<(unsigned)(want < 148 * 8 ? want : 148 * 8), 256, 0, st>>>(tar, ld, rows, K, energy, max_energy);
    return secommon::check_launch("wsd_energy_kernel");
}
// Per-utterance sums over valid frames, sums2[u] = { sum ((S - G S) voiced)^2, sum (G N)^2 } with N = max(X - S, 0), and the
// backward, on row-strided tensors (the training step's padded spectra; the dense entry points pass ld = K), lengths as in the
// SISDR mask kernels and the batch maximum read from a device buffer that may have been all-reduced across ranks in between
// (se_wsd_energy)
struct WsdMaskArgs : SisdrMaskArgs {           // sums3 holds the (n_utt, 2) sums here; grad_out: d L / d loss_mean (one float)
    float alpha, db_interval;
    const float* energy; const float* max_energy;
};

template <int V>
__global__ void __launch_bounds__(256) wsd_mask_sums_kernel(const WsdMaskArgs a) {
    const int u = blockIdx.x / a.chunks, chunk = blockIdx.x - u * a.chunks;
    const int valid = mask_valid_frames(a, u);
    const int KV = (a.K + V - 1) / V;
    const int per = (valid + a.chunks - 1) / a.chunks;
    const int f_lo = chunk * per, f_hi = min(valid, f_lo + per);
    const long long row0 = (long long)u * a.n_frames;
    const float thres = wsd_threshold(*a.max_energy, a.eps, a.db_interval);
    float acc[2] = {0.f, 0.f};
    const int items = max(f_hi - f_lo, 0) * KV;
#pragma unroll 4
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int fr = i / KV, c = (i - fr * KV) * V;
        const long long r = row0 + f_lo + fr;
        float x[V], t[V], o[V];
        ldv<V>(a.inp + r * a.ld_inp + c, x);
        ldv<V>(a.tar + r * a.ld_tar + c, t);
        ldv<V>(a.offset + r * a.ld_off + c, o);
        const bool voiced = wsd_voiced(a.energy[r], a.eps, thres);
#pragma unroll
        for (int e = 0; e < V; ++e)
            if (c + e < a.K) {
                const float d = voiced ? t[e] - o[e] * t[e] : 0.0f;
                const float n = o[e] * fmaxf(x[e] - t[e], 0.0f);
                acc[0] += d * d;
                acc[1] += n * n;
            }
    }
    block_accumulate_to<2, float>(acc, a.sums3 + (long long)u * 2);
}

// one block: loss_per_utt[u] = alpha sd_u + (1 - alpha) rn_u and the batch mean
__global__ void __launch_bounds__(256) wsd_finish_mean_kernel(const double* __restrict__ sums2, int n_utt, float alpha,
                                                              float* __restrict__ loss, float* __restrict__ loss_mean) {
    __shared__ double part[2][8];
    double sp = 0.0, no = 0.0;
    for (int u = threadIdx.x; u < n_utt; u += blockDim.x) {
        const double s = sums2[2 * u], n = sums2[2 * u + 1];
        if (loss) loss[u] = (float)((double)alpha * s + (1.0 - (double)alpha) * n);
        sp += s;
        no += n;
    }
    sp = secommon::warp_sum(sp);
    no = secommon::warp_sum(no);
    if ((threadIdx.x & 31) == 0) { part[0][threadIdx.x >> 5] = sp; part[1][threadIdx.x >> 5] = no; }
    __syncthreads();
    if (threadIdx.x == 0) {
        sp = no = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { sp += part[0][w]; no += part[1][w]; }
        *loss_mean = (float)(((double)alpha * sp + (1.0 - (double)alpha) * no) / n_utt);
    }
}

// the evaluation step's WSD terms (se_mask_istft_wsd) -> loss_per_utt; one CTA per utterance.  Every thread sums its own run of
// consecutive frames, then a fixed reduction order: the result does not change from run to run.  The last CTA to finish puts the
// maximum and the CTA counter back to 0 for the next step (a captured step then needs no fill node).
// the slow route of the evaluation step's L1: sum |lp - log(tar + eps)| over each utterance's valid frames of row-strided
// (n_utt, n_frames, ld) tensors -> sums[u, SE_SUM_SPEC_ST] and l1_acc[0]; the first chunk of each utterance adds its element count
// to l1_acc[1] (the same contract as se_mask_istft_l1's sums)
__global__ void __launch_bounds__(256) l1_eval_sums_kernel(const float* __restrict__ logp, long long ld_lp, const float* __restrict__ tar,
                                                           long long ld_tar, const long long* __restrict__ lengths, long long T, int hop,
                                                           int K, float eps, double* sums, double* l1_acc, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const long long F = T / hop + 1;
    const long long len = lengths ? min(T, max(0LL, lengths[u])) : T;
    const long long valid = min(F, len / hop + 1) * K;
    const long long per = (valid + chunks - 1) / chunks;
    const long long lo = chunk * per, hi = min(valid, lo + per);
    const float* p = logp + (long long)u * F * ld_lp;
    const float* t = tar + (long long)u * F * ld_tar;
    float acc[1] = {0.f};
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const long long f = i / K, k = i - f * K;
        acc[0] += fabsf(p[f * ld_lp + k] - logf(t[f * ld_tar + k] + eps));
    }
    block_accumulate_to<1, float>(acc, sums + (long long)u * SE_NSUMS + SE_SUM_SPEC_ST);
    block_accumulate_to<1, float>(acc, l1_acc);
    if (chunk == 0 && threadIdx.x == 0) atomicAdd(l1_acc + 1, (double)valid);
}

// the evaluation step's L1 (se_mask_istft_l1, or the slow route's se_l1_eval_sums) -> per-utterance and batch losses; one
// CTA.  Thread 0 reads the (all-reduced) [sum, count] pair before the barrier and clears it after: a captured step needs no fill.
__global__ void __launch_bounds__(256) l1_eval_finish_kernel(const double* __restrict__ sums, const long long* __restrict__ lengths,
                                                             int n_utt, long long T, int hop, long long K, double* l1_acc,
                                                             float* __restrict__ loss_per_utt, float* __restrict__ loss,
                                                             double* __restrict__ metric_acc) {
    __shared__ double s_acc[2];
    if (threadIdx.x == 0) { s_acc[0] = __ldcg(l1_acc); s_acc[1] = __ldcg(l1_acc + 1); }
    const long long F = T / hop + 1;
    for (int u = threadIdx.x; u < n_utt; u += blockDim.x) {
        const long long len = lengths ? min(T, max(0LL, lengths[u])) : T;
        const long long frames = min(F, len / hop + 1);
        loss_per_utt[u] = (float)(sums[(long long)u * SE_NSUMS + SE_SUM_SPEC_ST] / (double)(frames * K));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const float l = (float)(s_acc[0] / s_acc[1]);
        loss[0] = l;
        if (metric_acc) metric_acc[0] += (double)n_utt * (double)l;
        l1_acc[0] = 0.0;
        l1_acc[1] = 0.0;
    }
}

__global__ void __launch_bounds__(256) wsd_eval_finish_kernel(const float2* __restrict__ terms, const double* __restrict__ sums,
                                                              int n_frames, float alpha, float db_interval, float eps,
                                                              float* wsd_state, float* __restrict__ loss, double* __restrict__ metric_acc) {
    __shared__ double part[8];
    const int u = blockIdx.x;
    const float thres = wsd_threshold(__ldcg(wsd_state), eps, db_interval);          // after any all-reduce of wsd_state[0]
    const float2* row = terms + (long long)u * n_frames;
    const int per = (n_frames + blockDim.x - 1) / blockDim.x;
    const int lo = threadIdx.x * per, hi = min(n_frames, lo + per);
    double sd = 0.0;
    for (int f = lo; f < hi; ++f) {
        const float2 t = row[f];
        if (wsd_voiced(t.x, eps, thres)) sd += (double)t.y;
    }
    sd = secommon::warp_sum(sd);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sd;
    __syncthreads();
    if (threadIdx.x == 0) {
        sd = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sd += part[w];
        const double rn = sums[(long long)u * SE_NSUMS + SE_SUM_SPEC_ST];
        const float l = (float)((double)alpha * sd + (1.0 - (double)alpha) * rn);
        loss[u] = l;
        if (metric_acc) atomicAdd(metric_acc, (double)l);
        __threadfence();
        unsigned* done = reinterpret_cast<unsigned*>(wsd_state + 1);
        if (atomicAdd(done, 1u) == gridDim.x - 1) {                                  // every CTA has read the maximum
            wsd_state[0] = 0.0f;
            *done = 0u;
        }
    }
}

// d L / d offset for L = grad_out[0] * loss_mean (grad_out null: L = loss_mean), whole rows of grad_offset: 0 on padded frames and
// pad columns
template <int V>
__global__ void __launch_bounds__(256) wsd_mask_bwd_kernel(const WsdMaskArgs a) {
    const int u = blockIdx.x / a.chunks, chunk = blockIdx.x - u * a.chunks;
    const int valid = mask_valid_frames(a, u);
    const int KV = (int)(a.ld_g / V) < (a.K + V - 1) / V ? (a.K + V - 1) / V : (int)(a.ld_g / V);
    const int per = (a.n_frames + a.chunks - 1) / a.chunks;
    const int f_lo = chunk * per, f_hi = min(a.n_frames, f_lo + per);
    const float thres = wsd_threshold(*a.max_energy, a.eps, a.db_interval);
    const float scale = a.grad_out ? a.grad_out[0] / (float)a.n_utt : a.grad_uniform;
    const long long row0 = (long long)u * a.n_frames;
    const int items = max(f_hi - f_lo, 0) * KV;
#pragma unroll 4
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int fr = i / KV, c = (i - fr * KV) * V;
        const int f = f_lo + fr;
        const long long r = row0 + f;
        float g[V];
#pragma unroll
        for (int e = 0; e < V; ++e) g[e] = 0.0f;
        if (f < valid && c < a.K) {
            float x[V], t[V], o[V];
            ldv<V>(a.inp + r * a.ld_inp + c, x);
            ldv<V>(a.tar + r * a.ld_tar + c, t);
            ldv<V>(a.offset + r * a.ld_off + c, o);
            const bool voiced = wsd_voiced(a.energy[r], a.eps, thres);
#pragma unroll
            for (int e = 0; e < V; ++e)
                if (c + e < a.K) g[e] = wsd_grad(o[e], x[e], t[e], voiced, a.alpha, scale);
        }
        if (c + V <= a.ld_g) stv<V>(a.grad_offset + r * a.ld_g + c, g);
    }
}

// ------------------------------------------------------------------ log-spectral L1 objective on row-padded tensors (training step)
// objective.L1 of log_predicted against log(linear_tar + eps) over the valid frames: one CTA per (utterance, frame chunk) writes the
// double sum of its chunk to its own slot of `partials` (no atomics), the finish kernel adds the slots in a fixed order -- the loss
// is bitwise repeatable.  The same pass writes d loss / d log_predicted = sign(d) / count (the sign of se_l1_logspec_bwd: 0 for
// d == 0 and for NaN), 0 on padded frames and on the pad columns of a row.
struct L1MaskArgs {
    const float* lp; const float* tar;
    long long ld_lp, ld_tar;
    const long long* lengths;
    int len_hop;             // > 0: lengths holds SAMPLE lengths, frames = len / len_hop + 1 (runner.py:455)
    int n_utt, n_frames, K, chunks;
    float eps;
    double* partials;        // (n_utt, chunks)
    float* grad; long long ld_g;   // grad may be null
};

__device__ __forceinline__ int l1_valid_frames(const L1MaskArgs& a, int u) {
    long long v = a.n_frames;
    if (a.lengths) v = a.len_hop > 0 ? a.lengths[u] / a.len_hop + 1 : a.lengths[u];
    return (int)max(0LL, min((long long)a.n_frames, v));
}

template <int V>
__global__ void __launch_bounds__(256) l1_mask_step_kernel(const L1MaskArgs a) {
    __shared__ double part[8];
    __shared__ long long count[8];
    const int u = blockIdx.x / a.chunks, chunk = blockIdx.x - u * a.chunks;
    const int warp = threadIdx.x >> 5, nwarps = (int)(blockDim.x >> 5);
    const int valid = l1_valid_frames(a, u);
    float scale = 0.0f;
    if (a.grad) {            // 1 / (K * sum_u valid_u): every CTA counts the batch's frames itself (n_utt loads)
        long long c = 0;
        for (int v = threadIdx.x; v < a.n_utt; v += blockDim.x) c += l1_valid_frames(a, v);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if ((threadIdx.x & 31) == 0) count[warp] = c;
        __syncthreads();
        c = 0;
        for (int w = 0; w < nwarps; ++w) c += count[w];
        scale = c > 0 ? (float)(1.0 / (double)(c * a.K)) : 0.0f;
    }
    const int KV = a.grad ? max((int)(a.ld_g / V), (a.K + V - 1) / V) : (a.K + V - 1) / V;   // whole rows of grad
    const int per = (a.n_frames + a.chunks - 1) / a.chunks;
    const int f_lo = chunk * per, f_hi = min(a.grad ? a.n_frames : valid, f_lo + per);
    const long long row0 = (long long)u * a.n_frames;
    const int items = max(f_hi - f_lo, 0) * KV;
    float acc = 0.0f;
#pragma unroll 4
    for (int i = threadIdx.x; i < items; i += blockDim.x) {
        const int fr = i / KV, c = (i - fr * KV) * V;
        const int f = f_lo + fr;
        const long long r = row0 + f;
        float g[V];
#pragma unroll
        for (int e = 0; e < V; ++e) g[e] = 0.0f;
        if (f < valid && c < a.K) {
            float p[V], t[V];
            ldv<V>(a.lp + r * a.ld_lp + c, p);
            ldv<V>(a.tar + r * a.ld_tar + c, t);
#pragma unroll
            for (int e = 0; e < V; ++e)
                if (c + e < a.K) {
                    const float d = p[e] - logf(t[e] + a.eps);
                    acc += fabsf(d);
                    g[e] = d > 0.0f ? scale : (d < 0.0f ? -scale : 0.0f);
                }
        }
        if (a.grad && c + V <= a.ld_g) stv<V>(a.grad + r * a.ld_g + c, g);
    }
    const double s = secommon::warp_sum((double)acc);
    if ((threadIdx.x & 31) == 0) part[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < nwarps; ++w) t += part[w];
        a.partials[blockIdx.x] = t;
    }
}

// one CTA: loss_per_utt[u] = (sum of u's slots) / (valid_u K) (may be null) and loss_mean = the batch's sum / (K sum_u valid_u)
__global__ void __launch_bounds__(256) l1_mask_finish_kernel(const L1MaskArgs a, float* __restrict__ loss_per_utt,
                                                             float* __restrict__ loss_mean) {
    __shared__ double part[8];
    __shared__ long long count[8];
    double s = 0.0;
    long long n = 0;
    for (int u = threadIdx.x; u < a.n_utt; u += blockDim.x) {
        double su = 0.0;
        for (int c = 0; c < a.chunks; ++c) su += a.partials[(long long)u * a.chunks + c];
        const int v = l1_valid_frames(a, u);
        if (loss_per_utt) loss_per_utt[u] = (float)(su / ((double)v * a.K));
        s += su;
        n += v;
    }
    s = secommon::warp_sum(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0) { part[threadIdx.x >> 5] = s; count[threadIdx.x >> 5] = n; }
    __syncthreads();
    if (threadIdx.x == 0) {
        s = 0.0;
        n = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { s += part[w]; n += count[w]; }
        *loss_mean = (float)(s / ((double)n * a.K));
    }
}

// g <- g * act'(out) on row-strided tensors, out = the head's output AFTER the activation (Sigmoid: out (1 - out), ReLU: out > 0):
// d loss / d output becomes d loss / d pre-activation.  Columns [K, ld_g) of g are set to 0 (the pad columns of `out` are unspecified).
template <int V>
__global__ void __launch_bounds__(256) act_grad_kernel(float* __restrict__ g, long long ld_g, const float* __restrict__ out, long long ld_out,
                                                       long long n_rows, int K, int act) {
    const long long per_row = ld_g / V, n = n_rows * per_row;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / per_row;
        const int c = (int)(i - r * per_row) * V;
        float gv[V], o[V];
#pragma unroll
        for (int e = 0; e < V; ++e) o[e] = 0.0f;
        ldv<V>(g + r * ld_g + c, gv);
        if (c < K) ldv<V>(out + r * ld_out + c, o);
#pragma unroll
        for (int e = 0; e < V; ++e) {
            const float y = o[e];
            gv[e] = c + e >= K ? 0.0f : (act == SE_ACT_SIGMOID ? gv[e] * y * (1.0f - y) : gv[e] * (y > 0.0f ? 1.0f : 0.0f));
        }
        stv<V>(g + r * ld_g + c, gv);
    }
}

// ------------------------------------------------------------------ on-device batch synthesis (dataset.py:54-74, 106-111, 128-161, 169-179)
// sums4[u] = { sum s^2 over [0, Ls), sum n^2 over [0, Ln), sum n^2 over [0, Ls mod Ln) (0 if Ls < Ln: crop), unused }
__global__ void mix_sums_kernel(const float* __restrict__ speech, long long s_stride, const long long* __restrict__ s_len,
                                const float* __restrict__ noise, long long n_stride, const long long* __restrict__ n_len,
                                double* __restrict__ sums4, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const long long Ls = s_len[u], Ln = n_len[u];
    const long long rem = Ls >= Ln ? Ls % Ln : Ls;                      // tiled: the partial last copy; cropped: the kept prefix
    const long long span = Ls > Ln ? Ls : Ln;
    const long long per = (span + chunks - 1) / chunks;
    const long long lo = chunk * per, hi = min(span, lo + per);
    const float* s = speech + (long long)u * s_stride;
    const float* n = noise + (long long)u * n_stride;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        if (i < Ls) { const float v = s[i]; acc[0] += v * v; }
        if (i < Ln) { const float v = n[i]; acc[1] += v * v; if (i < rem) acc[2] += v * v; }
    }
    block_accumulate_to<4, float>(acc, sums4 + (long long)u * 4);
}
// out[u] = [noisy, speech_n, scaled_noise] (3, T_out), zero beyond Ls (collate_fn's padding)
__global__ void mix_write_kernel(const float* __restrict__ speech, long long s_stride, const long long* __restrict__ s_len,
                                 const float* __restrict__ noise, long long n_stride, const long long* __restrict__ n_len,
                                 const float* __restrict__ snr_db, const double* __restrict__ sums4, int T_out,
                                 float level, float eps, float* __restrict__ out, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const long long Ls = s_len[u], Ln = n_len[u];
    const double ss = sums4[4 * u], nn = sums4[4 * u + 1], nrem = sums4[4 * u + 2];
    // normalize_wav_decibel (dataset.py:106-111): x * 10^(level/20) / (rms + 1e-10)
    const float s_gain = level / ((float)sqrt(ss / (double)Ls) + 1e-10f);
    const float n_gain = level / ((float)sqrt(nn / (double)Ln) + 1e-10f);
    // add_noise (dataset.py:54-74) on the normalised signals: powers over the speech length, noise tiled or cropped
    const double reps = Ls >= Ln ? (double)(Ls / Ln) : 0.0;
    const float p_s = (float)(ss * (double)s_gain * (double)s_gain);
    const float p_n = (float)((reps * nn + nrem) * (double)n_gain * (double)n_gain);
    const float ratio = powf(10.0f, snr_db[u] / 10.0f);
    const float mix_gain = sqrtf(p_s / (ratio * p_n + eps)) * n_gain;     // applied to the raw noise samples
    const int per = (((T_out + chunks - 1) / chunks) + 3) & ~3;
    const int lo = chunk * per, hi = min(T_out, lo + per);
    const float* s = speech + (long long)u * s_stride;
    const float* n = noise + (long long)u * n_stride;
    float* o = out + (long long)u * 3 * T_out;
    for (int t = lo + threadIdx.x; t < hi; t += blockDim.x) {
        float sp = 0.0f, sc = 0.0f;
        if (t < Ls) {
            sp = s[t] * s_gain;
            sc = n[t % Ln] * mix_gain;
        }
        o[t] = sp + sc;
        o[T_out + t] = sp;
        o[2LL * T_out + t] = sc;
    }
}

// ------------------------------------------------------------------ waveform-level reductions
// sums3[u] += (<s,t>, <t,t>, <s,s>) over t < len[u]
__global__ void wave_sums_kernel(const float* __restrict__ src, long long src_stride, const float* __restrict__ tar,
                                 long long tar_stride, const long long* __restrict__ lengths, int T,
                                 double* __restrict__ sums3, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const int len = lengths ? (int)min((long long)T, lengths[u]) : T;
    const int per = (len + chunks - 1) / chunks;
    const int lo = chunk * per, hi = min(len, lo + per);
    const float* s = src + (long long)u * src_stride;
    const float* t = tar ? tar + (long long)u * tar_stride : nullptr;
    float acc[3] = {0.f, 0.f, 0.f};
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const float a = s[i];
        acc[2] += a * a;
        if (t) { const float b = t[i]; acc[0] += a * b; acc[1] += b * b; }
    }
    block_accumulate_to<3, float>(acc, sums3 + (long long)u * 3);
}

__global__ void sisdr_wave_finish_kernel(const double* __restrict__ sums3, int n_utt, float eps, float* __restrict__ out) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n_utt) out[u] = (float)sisdr_from_sums(sums3[3 * u], sums3[3 * u + 1], sums3[3 * u + 2], (double)eps);
}

// objective.WaveSISDR from [<y,c>, <c,c>, <y,y>] at sums + u * ld_sums (K3's SE_SUM_YC / CC / YY, or se_sisdr_wave's workspace):
// loss_per_utt[u] = -sisdr_eval, loss[0] = their batch mean, coef[u] = (alpha, beta) with d loss[0] / d y = alpha y + beta c,
// metric_acc += [sum loss, sum SI-SDR, n_utt].  One block: the mean is summed in a fixed order.
__global__ void __launch_bounds__(256) wave_sisdr_finish_kernel(const double* __restrict__ sums, int ld_sums, int n_utt, float eps,
                                                                float* __restrict__ loss_per_utt, float* __restrict__ loss,
                                                                float2* __restrict__ coef, double* __restrict__ metric_acc) {
    __shared__ double part[8];
    double acc = 0.0;
    for (int u = threadIdx.x; u < n_utt; u += blockDim.x) {
        const double* s = sums + (long long)u * ld_sums;
        const float l = (float)(-sisdr_from_sums(s[0], s[1], s[2], (double)eps));
        if (loss_per_utt) loss_per_utt[u] = l;
        if (coef) {
            const float2 c = sisdr_coef(s, (double)eps, 1.0 / (double)n_utt);      // (coefficient of c, coefficient of y)
            coef[u] = make_float2(c.y, c.x);
        }
        acc += (double)l;
    }
    acc = secommon::warp_sum(acc);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
        if (loss) *loss = (float)(t / (double)n_utt);
        if (metric_acc) {
            atomicAdd(metric_acc, t);
            atomicAdd(metric_acc + 1, -t);
            atomicAdd(metric_acc + 2, (double)n_utt);
        }
    }
}

// grad[u, t] = scale * grad_out[u] * (coef[u].x src[u, t] + coef[u].y tar[u, t]) for t < len[u], 0 for len[u] <= t < T
__global__ void wave_sisdr_bwd_kernel(const float* __restrict__ src, long long src_stride, const float* __restrict__ tar,
                                      long long tar_stride, const long long* __restrict__ lengths, int T, const float2* __restrict__ coef,
                                      const float* __restrict__ grad_out, float scale, float* __restrict__ grad, long long grad_stride,
                                      int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const int len = lengths ? (int)min((long long)T, max(0LL, lengths[u])) : T;
    const int per = (T + chunks - 1) / chunks;
    const int lo = chunk * per, hi = min(T, lo + per);
    const float w = scale * grad_out[u];
    const float2 c = coef[u];
    const float a = w * c.x, b = w * c.y;
    const float* s = src + (long long)u * src_stride;
    const float* t = tar + (long long)u * tar_stride;
    float* g = grad + (long long)u * grad_stride;
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) g[i] = i < len ? a * s[i] + b * t[i] : 0.0f;
}

// out = audio * sqrt(10^(target/10) / (mean(audio^2) + eps)); sums3[u] = (<a,r>, <r,r>, <a,a>) with r = ref.
// The masked means divide by len + 1e-8 whatever eps is (utils.py:26 masked_mean's own default); eps enters only the
// gain's denominator (utils.py:42).
__global__ void normalize_db_kernel(const float* __restrict__ audio, long long stride, const long long* __restrict__ lengths,
                                    int width, const float* __restrict__ target_db, int have_ref, float eps,
                                    const double* __restrict__ sums3, float* __restrict__ out, long long out_stride, int chunks) {
    const int u = blockIdx.x / chunks, chunk = blockIdx.x - u * chunks;
    const double len = lengths ? (double)min((long long)width, max(0LL, lengths[u])) : (double)width;
    const double eps_mean = 1e-8;
    const double mean_aa = sums3[3 * u + 2] / (len + eps_mean);
    double tdb;
    if (target_db) tdb = (double)target_db[u];
    else tdb = have_ref ? 10.0 * log10(sums3[3 * u + 1] / (len + eps_mean)) : -25.0;
    const float g = (float)sqrt(pow(10.0, tdb / 10.0) / (mean_aa + (double)eps));
    const int per = (width + chunks - 1) / chunks;
    const int lo = chunk * per, hi = min(width, lo + per);
    const float* a = audio + (long long)u * stride;
    float* o = out + (long long)u * out_stride;
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) o[i] = a[i] * g;
}

__global__ void length_masks_kernel(const long long* __restrict__ lengths, long long n_utt, long long width,
                                    long long* __restrict__ masks) {
    const long long total = n_utt * width;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long u = i / width, t = i - u * width;
        masks[i] = t < lengths[u] ? 1 : 0;
    }
}

// ------------------------------------------------------------------ CMVN statistics over time
// x (n_utt, F, D): mean / unbiased std per (u, d).  block = 32 features x 8 frame lanes.
// One pass: sums of (x - x0) and (x - x0)^2 with x0 = the utterance's first frame (a shift that removes the
// cancellation of the one-pass variance), eight independent loads in flight per thread, double accumulators.
__global__ void cmvn_stats_kernel(const float* __restrict__ x, long long ldx, int n_frames, int D, float* __restrict__ mean,
                                  float* __restrict__ stdv, long long ld_stats) {
    const int dchunks = (D + 31) / 32;
    const int u = blockIdx.x / dchunks, dc = blockIdx.x - u * dchunks;
    const int lane = threadIdx.x & 31, row = threadIdx.x >> 5, nrows = blockDim.x >> 5;
    const int d = dc * 32 + lane;
    const float* base = x + (long long)u * n_frames * ldx + d;
    __shared__ double red1[8][33], red2[8][33];
    double s = 0.0, q = 0.0;
    float x0 = 0.0f;
    if (d < D) {
        x0 = base[0];
        int f = row;
        for (; f + 7 * nrows < n_frames; f += 8 * nrows) {
            float a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = base[(long long)(f + i * nrows) * ldx];
            float ps = 0.0f, pq = 0.0f;                                   // eight terms: fp32 partials are exact enough
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float v = a[i] - x0; ps += v; pq += v * v; }
            s += (double)ps; q += (double)pq;
        }
        for (; f < n_frames; f += nrows) { const float v = base[(long long)f * ldx] - x0; s += (double)v; q += (double)v * v; }
    }
    red1[row][lane] = s;
    red2[row][lane] = q;
    __syncthreads();
    if (row == 0 && d < D) {
        double st = 0.0, qt = 0.0;
        for (int r = 0; r < nrows; ++r) { st += red1[r][lane]; qt += red2[r][lane]; }
        const double n = (double)n_frames;
        const double var = (qt - st * st / n) / (n - 1.0);                  // unbiased (model.py:30)
        mean[(long long)u * ld_stats + d] = (float)((double)x0 + st / n);
        stdv[(long long)u * ld_stats + d] = (float)sqrt(var > 0.0 ? var : 0.0);
    }
}

// sums[(u, d)] = [sum_f x, sum_f x^2] (double), the form the fused head consumes (head_fused.cu)
__global__ void feature_sums_kernel(const float* __restrict__ x, long long ldx, int n_frames, int D, double* __restrict__ sums,
                                    long long ld_stats) {
    const int dchunks = (D + 31) / 32;
    const int u = blockIdx.x / dchunks, dc = blockIdx.x - u * dchunks;
    const int lane = threadIdx.x & 31, row = threadIdx.x >> 5, nrows = blockDim.x >> 5;
    const int d = dc * 32 + lane;
    const float* base = x + (long long)u * n_frames * ldx + d;
    __shared__ double red1[8][33], red2[8][33];
    double s = 0.0, q = 0.0;
    if (d < D)
        for (int f = row; f < n_frames; f += nrows) { const double v = (double)base[(long long)f * ldx]; s += v; q += v * v; }
    red1[row][lane] = s;
    red2[row][lane] = q;
    __syncthreads();
    if (row == 0 && d < D) {
        double st = 0.0, qt = 0.0;
        for (int r = 0; r < nrows; ++r) { st += red1[r][lane]; qt += red2[r][lane]; }
        double* p = sums + ((long long)u * ld_stats + d) * 2;
        p[0] = st;
        p[1] = qt;
    }
}

__global__ void cmvn_apply_kernel(float* __restrict__ x, long long n_frames, int D, const float* __restrict__ mean,
                                  const float* __restrict__ stdv, float eps, long long total) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int d = (int)(i - row * D);
        const long long u = row / n_frames;
        x[i] = (x[i] - mean[u * D + d]) / (stdv[u * D + d] + eps);
    }
}

// ------------------------------------------------------------------ mel filterbank / deltas
// one warp per spectrogram row: out[row, m] = log?(sum_k power[row,k] fb[k,m] + eps)
__global__ void mel_kernel(const float* __restrict__ power, long long n_rows, int K, const float* __restrict__ fb,
                           int n_mels, int take_log, float eps, float* __restrict__ out, long long out_stride) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const float* p = power + row * K;
    for (int m0 = 0; m0 < n_mels; m0 += 64) {
        const int ma = m0 + lane, mb = m0 + 32 + lane;
        float acc_a = 0.f, acc_b = 0.f;
        for (int k0 = 0; k0 < K; k0 += 32) {
            const float pv = (k0 + lane < K) ? p[k0 + lane] : 0.f;
            const int kn = min(32, K - k0);
            for (int j = 0; j < kn; ++j) {
                const float pk = __shfl_sync(0xffffffffu, pv, j);
                const float* f = fb + (long long)(k0 + j) * n_mels;
                if (ma < n_mels) acc_a = fmaf(pk, f[ma], acc_a);
                if (mb < n_mels) acc_b = fmaf(pk, f[mb], acc_b);
            }
        }
        if (ma < n_mels) out[row * out_stride + ma] = take_log ? logf(acc_a + eps) : acc_a;
        if (mb < n_mels) out[row * out_stride + mb] = take_log ? logf(acc_b + eps) : acc_b;
    }
}

// columns [dst_col, dst_col+D) <- 5-tap regression delta over time of columns [src_col, src_col+D)
__global__ void delta_kernel(float* __restrict__ x, int n_frames, int D, int row_stride, int src_col, int dst_col, long long total) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int d = (int)(i - row * D);
        const long long u = row / n_frames;
        const int f = (int)(row - u * n_frames);
        const float* base = x + u * n_frames * (long long)row_stride + src_col + d;
        auto at = [&](int t) { t = t < 0 ? 0 : (t >= n_frames ? n_frames - 1 : t); return base[(long long)t * row_stride]; };
        const float v = (-2.0f * at(f - 2) - at(f - 1) + at(f + 1) + 2.0f * at(f + 2)) / 10.0f;
        x[row * row_stride + dst_col + d] = v;
    }
}

// ------------------------------------------------------------------ fp32 mask head (SIMT GEMM)
// offset = act( cmvn(x) W^T + b ),  predicted = linears * offset
// x (R, Din) with R = n_utt*n_frames, W (Dout, Din); 64x64 tile, 16-deep k-slab, 4x4 micro-tile.
constexpr int BM = 64, BN = 64, BK = 16;

__device__ __forceinline__ float activate(float z, int act) {
    if (act == SE_ACT_RELU) return z > 0.f ? z : 0.f;
    if (act == SE_ACT_SIGMOID) return 1.0f / (1.0f + expf(-z));
    return z;
}

__global__ void __launch_bounds__(256) linear_head_fwd_kernel(
    const float* __restrict__ x, const float* __restrict__ mean, const float* __restrict__ stdv, float cmvn_eps,
    const float* __restrict__ W, const float* __restrict__ bias, long long R, int n_frames, int Din, int Dout, int act,
    const float* __restrict__ linears, float* __restrict__ offset_out, float* __restrict__ pred_out,
    long long ldx, long long ld_stats, long long ldw, long long ld_out) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const long long r0 = (long long)blockIdx.y * BM;
    const int n0 = blockIdx.x * BN;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16 threads, 4x4 outputs each
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    // loader mapping: 256 threads fetch a 64 x 16 slab: thread -> (row = tid/4, 4 consecutive k)
    const int lrow = threadIdx.x >> 2, lk = (threadIdx.x & 3) * 4;
    for (int k0 = 0; k0 < Din; k0 += BK) {
        {
            const long long r = r0 + lrow;
            const long long u = r / n_frames;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = k0 + lk + j;
                float v = 0.f;
                if (r < R && k < Din) {
                    v = x[r * ldx + k];
                    if (mean) v = (v - mean[u * ld_stats + k]) / (stdv[u * ld_stats + k] + cmvn_eps);
                }
                As[lk + j][lrow] = v;
            }
            const int n = n0 + lrow;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = k0 + lk + j;
                Bs[lk + j][lrow] = (n < Dout && k < Din) ? W[(long long)n * ldw + k] : 0.f;
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long long r = r0 + ty * 4 + i;
        if (r >= R) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n >= Dout) continue;
            const float o = activate(acc[i][j] + (bias ? bias[n] : 0.f), act);
            if (offset_out) offset_out[r * ld_out + n] = o;
            if (pred_out) pred_out[r * ld_out + n] = linears[r * ld_out + n] * o;
        }
    }
}

// grad_W[n,k] += sum_r gz[r,n] * xn[r,k],  grad_b[n] += sum_r gz[r,n],  gz = grad_offset * act'(offset)
__global__ void __launch_bounds__(256) linear_head_bwd_kernel(
    const float* __restrict__ x, const float* __restrict__ mean, const float* __restrict__ stdv, float cmvn_eps,
    const float* __restrict__ offset, const float* __restrict__ grad_offset, long long R, int n_frames, int Din, int Dout,
    int act, float* __restrict__ grad_W, float* __restrict__ grad_b, long long rows_per_split) {
    __shared__ float Gs[BK][BM + 4];      // [r][n]
    __shared__ float Xs[BK][BN + 4];      // [r][k]
    const int n0 = blockIdx.y * BM, k0 = blockIdx.x * BN;
    const long long ra = (long long)blockIdx.z * rows_per_split, rb = min(R, ra + rows_per_split);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4];
    float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    // loader: thread -> (r = tid/16 in [0,16), 4 consecutive columns starting at (tid%16)*4)
    const int lr = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;
    for (long long rr = ra; rr < rb; rr += BK) {
        const long long r = rr + lr;
        const long long u = r / n_frames;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + lc + j;
            float g = 0.f;
            if (r < rb && n < Dout) {
                const float o = offset[r * Dout + n];
                g = grad_offset[r * Dout + n];
                if (act == SE_ACT_SIGMOID) g *= o * (1.0f - o);
                else if (act == SE_ACT_RELU) g = o > 0.f ? g : 0.f;
            }
            Gs[lr][lc + j] = g;
            const int k = k0 + lc + j;
            float v = 0.f;
            if (r < rb && k < Din) {
                v = x[r * Din + k];
                if (mean) v = (v - mean[u * Din + k]) / (stdv[u * Din + k] + cmvn_eps);
            }
            Xs[lr][lc + j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = Gs[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Xs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                bsum[i] += a[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= Dout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < Din) atomicAdd(grad_W + (long long)n * Din + k, acc[i][j]);
        }
        if (grad_b && blockIdx.x == 0 && tx == 0) atomicAdd(grad_b + n, bsum[i]);
    }
}

int pick_chunks(long long n_utt, long long work_per_utt, long long min_per_chunk) {
    // enough CTAs to fill 148 SMs a few times over without making chunks tiny
    long long want = (148LL * 8 + n_utt - 1) / n_utt;
    long long cap = work_per_utt / min_per_chunk;
    if (cap < 1) cap = 1;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return (int)want;
}

bool vec4_ok(const float* p, long long ld, long long K) {
    return p == nullptr || ((reinterpret_cast<uintptr_t>(p) & 15) == 0 && ld % 4 == 0 && ld >= (K + 3) / 4 * 4);
}

// The fields every launch of the strided objective kernels shares (the dense entry points pass ld = K, len_hop = 0), chunks of at
// least min_per_chunk elements.  Returns whether the float4 variant applies: the rows of every operand given, grad_offset
// included, are 16-byte aligned, a multiple of 4 floats apart and cover K rounded up to 4.
bool set_mask_args(SisdrMaskArgs& a, const float* offset, long long ld_off, const float* inp, long long ld_inp, const float* tar,
                   long long ld_tar, const int64_t* lengths, long long len_hop, long long n_utt, long long n_frames, long long K,
                   long long min_per_chunk, double* sums, float eps, float* grad_offset, long long ld_g) {
    a.offset = offset; a.inp = inp; a.tar = tar; a.ld_off = ld_off; a.ld_inp = ld_inp; a.ld_tar = ld_tar;
    a.stft_len = (const long long*)lengths; a.len_hop = (int)len_hop; a.n_utt = (int)n_utt; a.n_frames = (int)n_frames; a.K = (int)K;
    a.chunks = pick_chunks(n_utt, n_frames * K, min_per_chunk); a.sums3 = sums; a.eps = eps; a.grad_offset = grad_offset; a.ld_g = ld_g;
    return vec4_ok(offset, ld_off, K) && vec4_ok(inp, ld_inp, K) && vec4_ok(tar, ld_tar, K) && vec4_ok(grad_offset, ld_g, K);
}

}  // namespace

extern "C" {

int se_finalize_metrics(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T, float target_db_or_nan,
                        float* wav, int64_t wav_stride, int64_t width, float* gain, float* sisdr_wave, float* loss_spec,
                        void* stream) {
    return se_finalize_metrics_acc(sums, lengths, n_utt, T, target_db_or_nan, wav, wav_stride, width, gain, sisdr_wave, loss_spec,
                                   nullptr, stream);
}

int se_finalize_metrics_acc(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T, float target_db_or_nan,
                            float* wav, int64_t wav_stride, int64_t width, float* gain, float* sisdr_wave, float* loss_spec,
                            double* metric_acc, void* stream) {
    SE_REQUIRE(sums && n_utt > 0, "sums must not be null");
    // two CTAs per SM in one wave: the launch ramp of ~1000 small CTAs costs more than the scaling itself
    int chunks = 1;
    if (wav) {
        long long want = (2LL * 148 + n_utt - 1) / n_utt, cap = width / 4096;
        chunks = (int)(want < 1 ? 1 : (cap >= 1 && want > cap ? cap : want));
    }
    const double level = std::isnan(target_db_or_nan) ? -1.0 : std::pow(10.0, (double)target_db_or_nan / 10.0);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(n_utt * chunks));
    cfg.blockDim = dim3(kThreads);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;       // CTAs become resident while the upstream kernel drains
    attr[0].val.programmaticStreamSerializationAllowed = (secommon::pdl_mask() & 4) ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, finalize_metrics_kernel, sums, (const long long*)lengths, (int)T, level, wav,
                                     (long long)wav_stride, (int)width, gain, sisdr_wave, loss_spec, metric_acc, chunks,
                                     secommon::trace_ptr()));
    return secommon::check_launch("finalize_metrics_kernel");
}

int se_sisdr_spec_fwd(const float* predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double* sums3, float* loss_per_utt, void* stream) {
    SE_REQUIRE(predicted && linear_tar && sums3 && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(sums3, 0, sizeof(double) * 3 * n_utt, st));
    SisdrMaskArgs a{};
    const bool v4 = set_mask_args(a, nullptr, K, predicted, K, linear_tar, K, stft_len, 0, n_utt, n_frames, K, 8192, sums3, eps, nullptr, 0);
    if (v4) sisdr_mask_sums_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_sums_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    int rc = secommon::check_launch("sisdr_mask_sums_kernel");
    if (rc != SE_OK || !loss_per_utt) return rc;
    sisdr_finish_mean_kernel<<<1, 256, 0, st>>>(sums3, (int)n_utt, eps, loss_per_utt, nullptr);
    return secommon::check_launch("sisdr_finish_mean_kernel");
}

int se_sisdr_spec_bwd(const float* predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, const double* sums3, const float* grad_out,
                      float* grad_predicted, void* stream) {
    SE_REQUIRE(predicted && linear_tar && sums3 && grad_out && grad_predicted && n_utt > 0, "bad argument");
    SisdrMaskArgs a{};
    const bool v4 = set_mask_args(a, nullptr, K, predicted, K, linear_tar, K, stft_len, 0, n_utt, n_frames, K, 8192,
                                  const_cast<double*>(sums3), eps, grad_predicted, K);
    a.grad_out = grad_out;
    cudaStream_t st = (cudaStream_t)stream;
    if (v4) sisdr_mask_bwd_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_bwd_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    return secommon::check_launch("sisdr_mask_bwd_kernel");
}

int se_sisdr_mask_fwd(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                      int64_t ld_tar, const int64_t* stft_len, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                      double* sums3, float* loss_per_utt, void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && sums3 && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_inp >= K && ld_tar >= K && (!offset || ld_off >= K), "row stride smaller than K");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(sums3, 0, sizeof(double) * 3 * n_utt, st));
    SisdrMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, ld_off, linear_inp, ld_inp, linear_tar, ld_tar, stft_len, 0, n_utt, n_frames, K, 2048, sums3,
                                  eps, nullptr, 0);
    if (v4) sisdr_mask_sums_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_sums_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    int rc = secommon::check_launch("sisdr_mask_sums_kernel");
    if (rc != SE_OK || !loss_per_utt) return rc;
    sisdr_finish_mean_kernel<<<1, 256, 0, st>>>(sums3, (int)n_utt, eps, loss_per_utt, nullptr);
    return secommon::check_launch("sisdr_finish_mean_kernel");
}

int se_sisdr_mask_bwd(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                      int64_t ld_tar, const int64_t* stft_len, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                      const double* sums3, const float* grad_out, float* grad_offset, int64_t ld_g, void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && sums3 && grad_out && grad_offset && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_inp >= K && ld_tar >= K && ld_g >= K && (!offset || ld_off >= K), "row stride smaller than K");
    SisdrMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, ld_off, linear_inp, ld_inp, linear_tar, ld_tar, stft_len, 0, n_utt, n_frames, K, 2048,
                                  const_cast<double*>(sums3), eps, grad_offset, ld_g);
    a.grad_out = grad_out;
    cudaStream_t st = (cudaStream_t)stream;
    if (v4) sisdr_mask_bwd_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_bwd_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    return secommon::check_launch("sisdr_mask_bwd_kernel");
}

int se_sisdr_mask_step(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                       int64_t ld_tar, const int64_t* lengths, int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                       double* sums3, int sums_zeroed, float* loss_per_utt, float* loss_mean, float* grad_offset, int64_t ld_g,
                       void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && sums3 && loss_mean && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_inp >= K && ld_tar >= K && (!grad_offset || ld_g >= K) && (!offset || ld_off >= K), "row stride smaller than K");
    SE_REQUIRE(len_hop >= 0 && len_hop < (1LL << 30), "len_hop=%lld out of range", (long long)len_hop);
    cudaStream_t st = (cudaStream_t)stream;
    if (!sums_zeroed) SE_CUDA_CHECK(cudaMemsetAsync(sums3, 0, sizeof(double) * 3 * n_utt, st));
    SisdrMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, ld_off, linear_inp, ld_inp, linear_tar, ld_tar, lengths, len_hop, n_utt, n_frames, K, 2048,
                                  sums3, eps, grad_offset, ld_g);
    a.grad_uniform = 1.0f / (float)n_utt;
    if (v4) sisdr_mask_sums_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_sums_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    int rc = secommon::check_launch("sisdr_mask_sums_kernel");
    if (rc != SE_OK) return rc;
    sisdr_finish_mean_kernel<<<1, 256, 0, st>>>(sums3, (int)n_utt, eps, loss_per_utt, loss_mean);
    if ((rc = secommon::check_launch("sisdr_finish_mean_kernel")) != SE_OK || !grad_offset) return rc;
    if (v4) sisdr_mask_bwd_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else sisdr_mask_bwd_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    return secommon::check_launch("sisdr_mask_bwd_kernel");
}

int se_adam_clip_step(float* const* params, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                      const int64_t* numels, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                      float max_norm, double* ws_acc, int* ws_state, void* stream) {
    // this entry keeps its original limit of 8 tensors (callers may size their arrays by it); the mirror form takes 32
    SE_REQUIRE(n_tensors > 0 && n_tensors <= 8, "n_tensors=%d must be in [1, 8] (se_adam_clip_step_mirror takes up to %d)", n_tensors,
               kAdamMaxTensors);
    return se_adam_clip_step_mirror(params, grads, exp_avg, exp_avg_sq, numels, n_tensors, lr, beta1, beta2, eps, weight_decay, max_norm,
                                    nullptr, nullptr, nullptr, 0, ws_acc, ws_state, stream);
}

int se_adam_clip_step_mirror(float* const* params, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                             const int64_t* numels, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                             float max_norm, float* const* mirrors, const int64_t* mirror_cols, const int64_t* mirror_lds,
                             int mirror_tf32, double* ws_acc, int* ws_state, void* stream) {
    SE_REQUIRE(params && grads && exp_avg && exp_avg_sq && numels && ws_acc && ws_state, "null pointer");
    SE_REQUIRE(!mirrors || (mirror_cols && mirror_lds), "mirrors need their column counts and row strides");
    SE_REQUIRE(n_tensors > 0 && n_tensors <= kAdamMaxTensors, "n_tensors=%d must be in [1, %d]", n_tensors, kAdamMaxTensors);
    AdamArgs a{};
    long long total = 0;
    for (int t = 0; t < n_tensors; ++t) {
        SE_REQUIRE(params[t] && grads[t] && exp_avg[t] && exp_avg_sq[t] && numels[t] > 0, "tensor %d: null pointer or empty", t);
        a.p[t] = params[t]; a.g[t] = grads[t]; a.m[t] = exp_avg[t]; a.v[t] = exp_avg_sq[t]; a.n[t] = numels[t];
        total += numels[t];
        if (mirrors && mirrors[t]) {
            SE_REQUIRE(mirror_cols[t] > 0 && mirror_cols[t] < (1LL << 31) && numels[t] % mirror_cols[t] == 0 && mirror_lds[t] >= mirror_cols[t],
                       "tensor %d: mirror shape does not match", t);
            a.mir[t] = mirrors[t]; a.mir_cols[t] = (int)mirror_cols[t]; a.mir_ld[t] = mirror_lds[t];
        }
    }
    a.mir_tf32 = mirror_tf32;
    a.count = n_tensors; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay; a.max_norm = max_norm;
    a.acc = ws_acc; a.state = ws_state;
    cudaStream_t st = (cudaStream_t)stream;
    long long blocks = (total + 4 * 256 - 1) / (4 * 256);
    if (blocks > 592) blocks = 592;
    {   // the norm is needed for clipping AND for the NaN / inf guard of runner.py:467-470
        adam_norm_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
        int rc = secommon::check_launch("adam_norm_kernel");
        if (rc != SE_OK) return rc;
    }
    adam_update_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
    return secommon::check_launch("adam_update_kernel");
}

int se_match_scores(const float* query, int64_t n_query, const float* key, int64_t n_key, int64_t P, float eps, double* ws_d,
                    float* ws_qbar, float* scores, void* stream) {
    SE_REQUIRE(query && key && ws_d && ws_qbar && scores && n_query > 0 && n_key > 0 && P > 0, "bad argument");
    SE_REQUIRE(n_query < (1 << 20) && n_key < (1 << 20), "too many rows");
    cudaStream_t st = (cudaStream_t)stream;
    double* q_sumsq = ws_d;                       // [n_query] | k_sumsq [n_key] | dots [n_key]
    double* k_sumsq = ws_d + n_query;
    double* dots = k_sumsq + n_key;
    SE_CUDA_CHECK(cudaMemsetAsync(ws_d, 0, sizeof(double) * (size_t)(n_query + 2 * n_key), st));
    const int cq = pick_chunks(n_query, P, 4096), ck = pick_chunks(n_key, P, 4096);
    row_sumsq_kernel<<<(unsigned)(n_query * cq), 256, 0, st>>>(query, P, cq, q_sumsq);
    row_sumsq_kernel<<<(unsigned)(n_key * ck), 256, 0, st>>>(key, P, ck, k_sumsq);
    const long long blocks = (P + 255) / 256;
    SE_REQUIRE(blocks < 0x7fffffffLL, "P=%lld too large", (long long)P);
    match_qbar_kernel<<<(unsigned)blocks, 256, 0, st>>>(query, (int)n_query, P, eps, q_sumsq, ws_qbar);
    match_dot_kernel<<<(unsigned)(n_key * ck), 256, 0, st>>>(key, P, ck, ws_qbar, dots);
    match_finish_kernel<<<(unsigned)((n_key + 127) / 128), 128, 0, st>>>(k_sumsq, dots, (int)n_key, eps, scores);
    return secommon::check_launch("match_scores");
}

int se_mix_batch(const float* speech, int64_t speech_stride, const int64_t* speech_len, const float* noise, int64_t noise_stride,
                 const int64_t* noise_len, const float* snr_db, int64_t n_utt, int64_t T_out, float target_level_db, float eps,
                 double* ws_sums4, float* wavs_out, void* stream) {
    SE_REQUIRE(speech && speech_len && noise && noise_len && snr_db && ws_sums4 && wavs_out && n_utt > 0 && T_out > 0, "bad argument");
    SE_REQUIRE(T_out < (1LL << 30), "T_out=%lld too long", (long long)T_out);
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(ws_sums4, 0, sizeof(double) * 4 * n_utt, st));
    const int chunks = pick_chunks(n_utt, T_out, 8192);
    mix_sums_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(speech, speech_stride, (const long long*)speech_len, noise,
                                                                     noise_stride, (const long long*)noise_len, ws_sums4, chunks);
    int rc = secommon::check_launch("mix_sums_kernel");
    if (rc != SE_OK) return rc;
    mix_write_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(speech, speech_stride, (const long long*)speech_len, noise,
                                                                      noise_stride, (const long long*)noise_len, snr_db, ws_sums4,
                                                                      (int)T_out, powf(10.0f, target_level_db / 20.0f), eps,
                                                                      wavs_out, chunks);
    return secommon::check_launch("mix_write_kernel");
}

int se_wsd_fwd(const float* linear_inp, const float* offset, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
               int64_t n_frames, int64_t K, float alpha, float db_interval, float eps, float* ws_energy, float* ws_max,
               double* ws_sums2, float* loss, void* stream) {
    SE_REQUIRE(linear_inp && offset && linear_tar && ws_energy && ws_max && ws_sums2 && loss && n_utt > 0 && n_frames > 0 && K > 0,
               "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(ws_sums2, 0, sizeof(double) * 2 * n_utt, st));
    int rc = launch_wsd_energy(linear_tar, K, n_utt * n_frames, (int)K, ws_energy, ws_max, st);
    if (rc != SE_OK) return rc;
    WsdMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, K, linear_inp, K, linear_tar, K, stft_len, 0, n_utt, n_frames, K, 8192, ws_sums2, eps,
                                  nullptr, 0);
    a.alpha = alpha; a.db_interval = db_interval; a.energy = ws_energy; a.max_energy = ws_max;
    if (v4) wsd_mask_sums_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else wsd_mask_sums_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    if ((rc = secommon::check_launch("wsd_mask_sums_kernel")) != SE_OK) return rc;
    wsd_finish_mean_kernel<<<1, 256, 0, st>>>(ws_sums2, (int)n_utt, alpha, nullptr, loss);
    return secommon::check_launch("wsd_finish_mean_kernel");
}

int se_wsd_bwd(const float* linear_inp, const float* offset, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
               int64_t n_frames, int64_t K, float alpha, float db_interval, float eps, const float* ws_energy,
               const float* ws_max, const float* grad_loss, float* grad_offset, void* stream) {
    SE_REQUIRE(linear_inp && offset && linear_tar && ws_energy && ws_max && grad_loss && grad_offset && n_utt > 0, "bad argument");
    WsdMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, K, linear_inp, K, linear_tar, K, stft_len, 0, n_utt, n_frames, K, 8192, nullptr, eps,
                                  grad_offset, K);
    a.grad_out = grad_loss; a.alpha = alpha; a.db_interval = db_interval; a.energy = ws_energy; a.max_energy = ws_max;
    cudaStream_t st = (cudaStream_t)stream;
    if (v4) wsd_mask_bwd_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else wsd_mask_bwd_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    return secommon::check_launch("wsd_mask_bwd_kernel");
}

int se_wsd_energy(const float* linear_tar, int64_t ld_tar, int64_t n_utt, int64_t n_frames, int64_t K, float* energy, float* max_energy,
                  void* stream) {
    SE_REQUIRE(linear_tar && energy && max_energy && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_tar >= K, "row stride smaller than K");
    return launch_wsd_energy(linear_tar, ld_tar, n_utt * n_frames, (int)K, energy, max_energy, (cudaStream_t)stream);
}

int se_wsd_mask_step(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                     const int64_t* lengths, int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float alpha, float db_interval,
                     float eps, const float* energy, const float* max_energy, double* sums2, int sums_zeroed, float* loss_per_utt,
                     float* loss_mean, float* grad_offset, int64_t ld_g, void* stream) {
    SE_REQUIRE(offset && linear_inp && linear_tar && energy && max_energy && sums2 && loss_mean && n_utt > 0 && n_frames > 0 && K > 0,
               "bad argument");
    SE_REQUIRE(ld_off >= K && ld_inp >= K && ld_tar >= K && (!grad_offset || ld_g >= K), "row stride smaller than K");
    SE_REQUIRE(len_hop >= 0 && len_hop < (1LL << 30), "len_hop=%lld out of range", (long long)len_hop);
    cudaStream_t st = (cudaStream_t)stream;
    if (!sums_zeroed) SE_CUDA_CHECK(cudaMemsetAsync(sums2, 0, sizeof(double) * 2 * n_utt, st));
    WsdMaskArgs a{};
    const bool v4 = set_mask_args(a, offset, ld_off, linear_inp, ld_inp, linear_tar, ld_tar, lengths, len_hop, n_utt, n_frames, K, 2048,
                                  sums2, eps, grad_offset, ld_g);
    a.grad_uniform = 1.0f / (float)n_utt; a.alpha = alpha; a.db_interval = db_interval; a.energy = energy; a.max_energy = max_energy;
    if (v4) wsd_mask_sums_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else wsd_mask_sums_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    int rc = secommon::check_launch("wsd_mask_sums_kernel");
    if (rc != SE_OK) return rc;
    wsd_finish_mean_kernel<<<1, 256, 0, st>>>(sums2, (int)n_utt, alpha, loss_per_utt, loss_mean);
    if ((rc = secommon::check_launch("wsd_finish_mean_kernel")) != SE_OK || !grad_offset) return rc;
    if (v4) wsd_mask_bwd_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else wsd_mask_bwd_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    return secommon::check_launch("wsd_mask_bwd_kernel");
}

int se_wsd_eval_finish(const float* frame_terms, const double* sums, int64_t n_utt, int64_t n_frames, float alpha, float db_interval,
                       float eps, float* wsd_state, float* loss_per_utt, double* metric_acc, void* stream) {
    SE_REQUIRE(frame_terms && sums && wsd_state && loss_per_utt && n_utt > 0 && n_frames > 0, "bad argument");
    SE_REQUIRE(n_utt <= 0x7fffffffLL && n_frames <= 0x7fffffffLL, "too many utterances or frames");
    wsd_eval_finish_kernel<<<(unsigned)n_utt, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(frame_terms), sums,
                                                                              (int)n_frames, alpha, db_interval, eps, wsd_state,
                                                                              loss_per_utt, metric_acc);
    return secommon::check_launch("wsd_eval_finish_kernel");
}

int se_l1_eval_sums(const float* log_predicted, int64_t ld_lp, const float* linear_tar, int64_t ld_tar, const int64_t* lengths,
                    int64_t n_utt, int64_t T, int hop, int64_t K, float eps, double* sums, double* l1_acc, void* stream) {
    SE_REQUIRE(log_predicted && linear_tar && sums && l1_acc && n_utt > 0 && T > 0 && hop > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_lp >= K && ld_tar >= K && K <= 0x7fffffffLL, "ld_lp / ld_tar smaller than K");
    const int chunks = pick_chunks(n_utt, (T / hop + 1) * K, 8192);
    SE_REQUIRE(n_utt * chunks <= 0x7fffffffLL, "too many utterances");
    l1_eval_sums_kernel<<<(unsigned)(n_utt * chunks), 256, 0, (cudaStream_t)stream>>>(
        log_predicted, (long long)ld_lp, linear_tar, (long long)ld_tar, reinterpret_cast<const long long*>(lengths), (long long)T, hop,
        (int)K, eps, sums, l1_acc, chunks);
    return secommon::check_launch("l1_eval_sums_kernel");
}

int se_l1_eval_finish(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T, int hop, int64_t K, double* l1_acc,
                      float* loss_per_utt, float* loss, double* metric_acc, void* stream) {
    SE_REQUIRE(sums && l1_acc && loss_per_utt && loss && n_utt > 0 && T > 0 && hop > 0 && K > 0, "bad argument");
    SE_REQUIRE(n_utt <= 0x7fffffffLL, "too many utterances");
    l1_eval_finish_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(sums, reinterpret_cast<const long long*>(lengths), (int)n_utt,
                                                              (long long)T, hop, (long long)K, l1_acc, loss_per_utt, loss, metric_acc);
    return secommon::check_launch("l1_eval_finish_kernel");
}

int64_t se_l1_mask_step_workspace(int64_t n_utt, int64_t n_frames, int64_t K) {
    if (n_utt <= 0 || n_frames <= 0 || K <= 0) return 0;
    return n_utt * pick_chunks(n_utt, n_frames * K, 2048);
}

int se_l1_mask_step(const float* log_predicted, int64_t ld_lp, const float* linear_tar, int64_t ld_tar, const int64_t* lengths,
                    int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float eps, double* ws_partials, int64_t ws_doubles,
                    float* loss_per_utt, float* loss_mean, float* grad, int64_t ld_g, void* stream) {
    SE_REQUIRE(log_predicted && linear_tar && ws_partials && loss_mean && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(ld_lp >= K && ld_tar >= K && (!grad || ld_g >= K), "row stride smaller than K");
    SE_REQUIRE(len_hop >= 0 && len_hop < (1LL << 30), "len_hop=%lld out of range", (long long)len_hop);
    SE_REQUIRE(n_utt <= 0x7fffffffLL && n_frames <= 0x7fffffffLL && K <= 0x7fffffffLL, "shape too large");
    SE_REQUIRE(ws_doubles >= se_l1_mask_step_workspace(n_utt, n_frames, K), "ws_partials holds %lld doubles, %lld needed",
               (long long)ws_doubles, (long long)se_l1_mask_step_workspace(n_utt, n_frames, K));
    L1MaskArgs a{};
    a.lp = log_predicted; a.tar = linear_tar; a.ld_lp = ld_lp; a.ld_tar = ld_tar;
    a.lengths = reinterpret_cast<const long long*>(lengths); a.len_hop = (int)len_hop;
    a.n_utt = (int)n_utt; a.n_frames = (int)n_frames; a.K = (int)K; a.chunks = pick_chunks(n_utt, n_frames * K, 2048);
    a.eps = eps; a.partials = ws_partials; a.grad = grad; a.ld_g = ld_g;
    cudaStream_t st = (cudaStream_t)stream;
    const bool v4 = vec4_ok(log_predicted, ld_lp, K) && vec4_ok(linear_tar, ld_tar, K) && vec4_ok(grad, ld_g, K);
    if (v4) l1_mask_step_kernel<4><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    else l1_mask_step_kernel<1><<<(unsigned)(n_utt * a.chunks), 256, 0, st>>>(a);
    int rc = secommon::check_launch("l1_mask_step_kernel");
    if (rc != SE_OK) return rc;
    l1_mask_finish_kernel<<<1, 256, 0, st>>>(a, loss_per_utt, loss_mean);
    return secommon::check_launch("l1_mask_finish_kernel");
}

int se_act_grad_inplace(float* grad, int64_t ld_g, const float* out, int64_t ld_out, int64_t n_rows, int64_t K, int act, void* stream) {
    SE_REQUIRE(act >= SE_ACT_IDENTITY && act <= SE_ACT_SIGMOID, "unknown activation %d", act);
    if (act == SE_ACT_IDENTITY) return SE_OK;                           // act' = 1: nothing to do
    SE_REQUIRE(grad && out && n_rows > 0 && K > 0 && K <= 0x7fffffffLL, "bad argument");
    SE_REQUIRE(ld_g >= K && ld_out >= K, "row stride smaller than K");
    const bool v4 = vec4_ok(grad, ld_g, K) && vec4_ok(out, ld_out, K);
    const long long n = n_rows * (v4 ? ld_g / 4 : ld_g);
    const long long blocks = std::min((n + 255) / 256, 148LL * 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (v4) act_grad_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(grad, ld_g, out, ld_out, n_rows, (int)K, act);
    else act_grad_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(grad, ld_g, out, ld_out, n_rows, (int)K, act);
    return secommon::check_launch("act_grad_kernel");
}

int se_l1_logspec_fwd(const float* log_predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double* acc2, void* stream) {
    SE_REQUIRE(log_predicted && linear_tar && acc2 && n_utt > 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(acc2, 0, sizeof(double) * 2, st));
    int chunks = pick_chunks(n_utt, n_frames * K, 8192);
    const long long per = (n_frames * K + chunks - 1) / chunks;
    if (per > (1LL << 24)) chunks = (int)((n_frames * K + (1LL << 24) - 1) >> 24);
    l1_logspec_fwd_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(log_predicted, linear_tar, (const long long*)stft_len,
                                                                           (int)n_frames, (int)K, eps, acc2, chunks);
    return secommon::check_launch("l1_logspec_fwd_kernel");
}

int se_l1_logspec_bwd(const float* log_predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double count, const float* grad_out,
                      float* grad_log_predicted, void* stream) {
    SE_REQUIRE(log_predicted && linear_tar && grad_out && grad_log_predicted && n_utt > 0 && count > 0, "bad argument");
    const int chunks = pick_chunks(n_utt, n_frames * K, 8192);
    l1_logspec_bwd_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, (cudaStream_t)stream>>>(
        log_predicted, linear_tar, (const long long*)stft_len, (int)n_frames, (int)K, eps, count, grad_out, grad_log_predicted, chunks);
    return secommon::check_launch("l1_logspec_bwd_kernel");
}

int se_sisdr_wave(const float* src, int64_t src_stride, const float* tar, int64_t tar_stride, const int64_t* lengths,
                  int64_t n_utt, int64_t T, float eps, double* ws_sums3, float* sisdr, void* stream) {
    SE_REQUIRE(src && tar && ws_sums3 && sisdr && n_utt > 0 && T > 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(ws_sums3, 0, sizeof(double) * 3 * n_utt, st));
    const int chunks = pick_chunks(n_utt, T, 8192);
    wave_sums_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(src, src_stride, tar, tar_stride, (const long long*)lengths,
                                                                      (int)T, ws_sums3, chunks);
    int rc = secommon::check_launch("wave_sums_kernel");
    if (rc != SE_OK) return rc;
    sisdr_wave_finish_kernel<<<(unsigned)((n_utt + 127) / 128), 128, 0, st>>>(ws_sums3, (int)n_utt, eps, sisdr);
    return secommon::check_launch("sisdr_wave_finish_kernel");
}

int se_wave_sisdr_finish(const double* sums, int64_t ld_sums, int64_t n_utt, float eps, float* loss_per_utt, float* loss, float* coef,
                         double* metric_acc, void* stream) {
    SE_REQUIRE(sums && n_utt > 0 && ld_sums >= 3, "bad argument");
    SE_REQUIRE(!coef || (reinterpret_cast<uintptr_t>(coef) & 7) == 0, "coef must be 8-byte aligned");
    wave_sisdr_finish_kernel<<<1, kThreads, 0, (cudaStream_t)stream>>>(sums, (int)ld_sums, (int)n_utt, eps, loss_per_utt, loss,
                                                                      reinterpret_cast<float2*>(coef), metric_acc);
    return secommon::check_launch("wave_sisdr_finish_kernel");
}

int se_wave_sisdr_bwd(const float* src, int64_t src_stride, const float* tar, int64_t tar_stride, const int64_t* lengths, int64_t n_utt,
                      int64_t T, const float* coef, const float* grad_out, float scale, float* grad, int64_t grad_stride, void* stream) {
    SE_REQUIRE(src && tar && coef && grad_out && grad && n_utt > 0 && T > 0 && T < (1LL << 31), "bad argument");
    SE_REQUIRE((reinterpret_cast<uintptr_t>(coef) & 7) == 0, "coef must be 8-byte aligned");
    const int chunks = pick_chunks(n_utt, T, 8192);
    wave_sisdr_bwd_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, (cudaStream_t)stream>>>(
        src, src_stride, tar, tar_stride, (const long long*)lengths, (int)T, reinterpret_cast<const float2*>(coef), grad_out, scale, grad,
        grad_stride, chunks);
    return secommon::check_launch("wave_sisdr_bwd_kernel");
}

int se_masked_normalize_db(const float* audio, int64_t stride, const int64_t* lengths, int64_t n_utt, int64_t width,
                           const float* target_db, const float* ref, int64_t ref_stride, float eps, double* ws_sums3,
                           float* out, int64_t out_stride, void* stream) {
    SE_REQUIRE(audio && out && ws_sums3 && n_utt > 0 && width > 0, "bad argument");
    SE_REQUIRE(target_db || ref, "either target_db or ref must be given");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(ws_sums3, 0, sizeof(double) * 3 * n_utt, st));
    const int chunks = pick_chunks(n_utt, width, 8192);
    wave_sums_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(audio, stride, target_db ? nullptr : ref, ref_stride,
                                                                      (const long long*)lengths, (int)width, ws_sums3, chunks);
    int rc = secommon::check_launch("wave_sums_kernel");
    if (rc != SE_OK) return rc;
    normalize_db_kernel<<<(unsigned)(n_utt * chunks), kThreads, 0, st>>>(audio, stride, (const long long*)lengths, (int)width,
                                                                         target_db, ref ? 1 : 0, eps, ws_sums3, out, out_stride, chunks);
    return secommon::check_launch("normalize_db_kernel");
}

int se_length_masks(const int64_t* lengths, int64_t n_utt, int64_t width, int64_t* masks, void* stream) {
    SE_REQUIRE(lengths && masks && n_utt > 0 && width > 0, "bad argument");
    const long long total = n_utt * width;
    const unsigned blocks = (unsigned)std::min<long long>((total + kThreads - 1) / kThreads, 148LL * 16);
    length_masks_kernel<<<blocks, kThreads, 0, (cudaStream_t)stream>>>((const long long*)lengths, n_utt, width, (long long*)masks);
    return secommon::check_launch("length_masks_kernel");
}

int se_cmvn_stats(const float* x, int64_t n_utt, int64_t n_frames, int64_t D, float* mean, float* std, void* stream) {
    return se_cmvn_stats_strided(x, D, n_utt, n_frames, D, mean, std, D, stream);
}

int se_cmvn_stats_strided(const float* x, int64_t ldx, int64_t n_utt, int64_t n_frames, int64_t D, float* mean, float* std,
                          int64_t ld_stats, void* stream) {
    SE_REQUIRE(x && mean && std && n_utt > 0 && n_frames > 0 && D > 0 && ldx >= D && ld_stats >= D, "bad argument");
    const long long blocks = n_utt * ((D + 31) / 32);
    cmvn_stats_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, (int)n_frames, (int)D, mean, std, ld_stats);
    return secommon::check_launch("cmvn_stats_kernel");
}

int se_feature_sums(const float* x, int64_t ldx, int64_t n_utt, int64_t n_frames, int64_t D, double* sums, int64_t ld_stats,
                    void* stream) {
    SE_REQUIRE(x && sums && n_utt > 0 && n_frames > 0 && D > 0 && ldx >= D && ld_stats >= D, "bad argument");
    const long long blocks = n_utt * ((D + 31) / 32);
    feature_sums_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, (int)n_frames, (int)D, sums, ld_stats);
    return secommon::check_launch("feature_sums_kernel");
}

int se_cmvn_apply(float* x, int64_t n_utt, int64_t n_frames, int64_t D, const float* mean, const float* std, float eps,
                  void* stream) {
    SE_REQUIRE(x && mean && std && n_utt > 0, "bad argument");
    const long long total = n_utt * n_frames * D;
    const unsigned blocks = (unsigned)std::min<long long>((total + kThreads - 1) / kThreads, 148LL * 16);
    cmvn_apply_kernel<<<blocks, kThreads, 0, (cudaStream_t)stream>>>(x, n_frames, (int)D, mean, std, eps, total);
    return secommon::check_launch("cmvn_apply_kernel");
}

// ------------------------------------------------------------------ K1b fused: mel -> log -> deltas -> CMVN sums, final layout
// One CTA = kMfTile consecutive frames of one utterance.  The mel(-log) rows of the tile and of 2 * order halo frames on
// either side (frame indices clamped to the utterance: compute_deltas pads by replication) are computed once into shared
// memory, the recursive 5-tap regression deltas are taken there, and the finished (order + 1) * n_mels columns are written
// straight into the output row -- one launch instead of se_mel + order x se_delta (+ se_cmvn_stats).  With stat_sums the
// per-(utterance, column) sum and sum of squares accumulate in double for the CMVN that follows (se_cmvn_apply_sums).
constexpr int kMfTile = 32, kMfMaxOrder = 2, kMfMaxMels = 64;
__global__ void __launch_bounds__(256) mel_features_kernel(const float* __restrict__ power, long long ld_power, int n_frames, int K,
                                                           const float* __restrict__ fb, int n_mels, int take_log, float eps, int order,
                                                           float* __restrict__ out, long long ld_out, double* __restrict__ stat_sums,
                                                           const int* __restrict__ fb_ranges, int tiles) {
    __shared__ float s_m[kMfMaxOrder + 1][kMfTile + 4 * kMfMaxOrder][kMfMaxMels];
    __shared__ float s_red[2][8][kMfMaxMels];
    const int u = blockIdx.x / tiles, tile = blockIdx.x - u * tiles;
    const int f0 = tile * kMfTile;
    const int nf = min(kMfTile, n_frames - f0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* prow = power + (long long)u * n_frames * ld_power;
    // level 0: mel rows of frames f0 - 2 order .. f0 + nf + 2 order - 1 (clamped)
    const int w0 = nf + 4 * order;
    if (fb_ranges) {
        // triangular filters are sparse (a bin feeds at most two of them): thread = (frame, filter) sums only the bins
        // [lo, hi) where its filter is non-zero -- ~2 K multiply-adds per frame instead of 40 K
        for (int idx = threadIdx.x; idx < w0 * n_mels; idx += blockDim.x) {
            const int i = idx / n_mels, m = idx - i * n_mels;
            int f = f0 - 2 * order + i;
            f = f < 0 ? 0 : (f >= n_frames ? n_frames - 1 : f);
            const float* p = prow + (long long)f * ld_power;
            const int lo = fb_ranges[2 * m], hi = fb_ranges[2 * m + 1];
            float acc = 0.f;
            for (int kk = lo; kk < hi; ++kk) acc = fmaf(__ldg(p + kk), __ldg(fb + (long long)kk * n_mels + m), acc);
            s_m[0][i][m] = take_log ? logf(acc + eps) : acc;
        }
    } else {
        for (int i = warp; i < w0; i += 8) {
            int f = f0 - 2 * order + i;
            f = f < 0 ? 0 : (f >= n_frames ? n_frames - 1 : f);
            const float* p = prow + (long long)f * ld_power;
            const int ma = lane, mb = 32 + lane;
            float acc_a = 0.f, acc_b = 0.f;
            for (int k0 = 0; k0 < K; k0 += 32) {
                const float pv = (k0 + lane < K) ? p[k0 + lane] : 0.f;
                const int kn = min(32, K - k0);
                for (int j = 0; j < kn; ++j) {
                    const float pk = __shfl_sync(0xffffffffu, pv, j);
                    const float* frow = fb + (long long)(k0 + j) * n_mels;
                    if (ma < n_mels) acc_a = fmaf(pk, frow[ma], acc_a);
                    if (mb < n_mels) acc_b = fmaf(pk, frow[mb], acc_b);
                }
            }
            if (ma < n_mels) s_m[0][i][ma] = take_log ? logf(acc_a + eps) : acc_a;
            if (mb < n_mels) s_m[0][i][mb] = take_log ? logf(acc_b + eps) : acc_b;
        }
    }
    __syncthreads();
    // level o: deltas of level o - 1 on frames f0 - 2 (order - o) .. ; position i of level o is frame f0 - 2 (order - o) + i
    for (int o = 1; o <= order; ++o) {
        const int wo = nf + 4 * (order - o);
        for (int idx = threadIdx.x; idx < wo * n_mels; idx += blockDim.x) {
            const int i = idx / n_mels, m = idx - i * n_mels;
            int f = f0 - 2 * (order - o) + i;
            f = f < 0 ? 0 : (f >= n_frames ? n_frames - 1 : f);
            // frame f +- k (clamped) sits at position clamp(f + k) - (f0 - 2 (order - o + 1)) of level o - 1
            const int base = f0 - 2 * (order - o + 1);
            auto at = [&](int t) { t = t < 0 ? 0 : (t >= n_frames ? n_frames - 1 : t); return s_m[o - 1][t - base][m]; };
            s_m[o][i][m] = (-2.0f * at(f - 2) - at(f - 1) + at(f + 1) + 2.0f * at(f + 2)) / 10.0f;
        }
        __syncthreads();
    }
    // output rows + CMVN sums: thread = (frame lane r, column m); level o's own frames start at position 2 (order - o)
    const int cols = (order + 1) * n_mels;
    for (int c0 = 0; c0 < cols; c0 += kMfMaxMels) {
        const int m = threadIdx.x & (kMfMaxMels - 1), r0 = threadIdx.x / kMfMaxMels;          // 4 frame lanes x 64 columns
        const int c = c0 + m;
        float s1 = 0.f, s2 = 0.f;
        if (m < kMfMaxMels && c < cols) {
            const int o = c / n_mels, mm = c - o * n_mels;
            for (int r = r0; r < nf; r += 256 / kMfMaxMels) {
                const float v = s_m[o][2 * (order - o) + r][mm];
                out[((long long)u * n_frames + f0 + r) * ld_out + c] = v;
                s1 += v; s2 += v * v;
            }
        }
        if (stat_sums) {
            s_red[0][r0][m] = s1;
            s_red[1][r0][m] = s2;
            __syncthreads();
            if (threadIdx.x < kMfMaxMels && c0 + (int)threadIdx.x < cols) {
                double a = 0.0, b = 0.0;
                for (int r = 0; r < 256 / kMfMaxMels; ++r) { a += (double)s_red[0][r][threadIdx.x]; b += (double)s_red[1][r][threadIdx.x]; }
                double* dst = stat_sums + ((long long)u * cols + c0 + threadIdx.x) * 2;
                atomicAdd(dst, a);
                atomicAdd(dst + 1, b);
            }
            __syncthreads();
        }
    }
}

// x = (x - mean) / (std + eps) in place with mean / unbiased std from the (n_utt, D, 2) double sums [sum x, sum x^2]
__global__ void cmvn_apply_sums_kernel(float* __restrict__ x, long long n_frames, int D, const double* __restrict__ sums, float eps,
                                       long long total) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long row = i / D;
        const int d = (int)(i - row * D);
        const long long u = row / n_frames;
        const double s1 = sums[(u * D + d) * 2], s2 = sums[(u * D + d) * 2 + 1];
        const double n = (double)n_frames, mean = s1 / n;
        const double var = (s2 - s1 * mean) / (n - 1.0);
        x[i] = (x[i] - (float)mean) / ((float)sqrt(var > 0.0 ? var : 0.0) + eps);
    }
}

int se_mel_features(const float* power, int64_t ld_power, int64_t n_utt, int64_t n_frames, int64_t K, const float* fb,
                    const int32_t* fb_ranges, int64_t n_mels, int take_log, float eps, int order, float* out, int64_t ld_out,
                    double* stat_sums, void* stream) {
    SE_REQUIRE(power && fb && out && n_utt > 0 && n_frames > 0 && K > 0, "bad argument");
    SE_REQUIRE(n_mels > 0 && n_mels <= kMfMaxMels && order >= 0 && order <= kMfMaxOrder, "n_mels=%lld (<= %d) / order=%d (<= %d) out of range",
               (long long)n_mels, kMfMaxMels, order, kMfMaxOrder);
    SE_REQUIRE(ld_power >= K && ld_out >= (order + 1) * n_mels, "row stride smaller than the row");
    cudaStream_t st = (cudaStream_t)stream;
    if (stat_sums) SE_CUDA_CHECK(cudaMemsetAsync(stat_sums, 0, sizeof(double) * 2 * (order + 1) * n_mels * n_utt, st));
    const int tiles = (int)((n_frames + kMfTile - 1) / kMfTile);
    const long long blocks = n_utt * tiles;
    SE_REQUIRE(blocks <= 0x7fffffffLL, "grid too large");
    mel_features_kernel<<<(unsigned)blocks, 256, 0, st>>>(power, ld_power, (int)n_frames, (int)K, fb, (int)n_mels, take_log, eps, order, out,
                                                          ld_out, stat_sums, fb_ranges, tiles);
    return secommon::check_launch("mel_features_kernel");
}

int se_cmvn_apply_sums(float* x, int64_t n_utt, int64_t n_frames, int64_t D, const double* sums, float eps, void* stream) {
    SE_REQUIRE(x && sums && n_utt > 0 && n_frames > 1 && D > 0, "bad argument");
    const long long total = n_utt * n_frames * D;
    const unsigned blocks = (unsigned)std::min<long long>((total + kThreads - 1) / kThreads, 148LL * 16);
    cmvn_apply_sums_kernel<<<blocks, kThreads, 0, (cudaStream_t)stream>>>(x, n_frames, (int)D, sums, eps, total);
    return secommon::check_launch("cmvn_apply_sums_kernel");
}

int se_mel(const float* power, int64_t n_rows, int64_t K, const float* fb, int64_t n_mels, int take_log, float eps,
           float* out, int64_t out_row_stride, void* stream) {
    SE_REQUIRE(power && fb && out && n_rows > 0 && K > 0 && n_mels > 0 && out_row_stride >= n_mels, "bad argument");
    const int warps = 8;
    mel_kernel<<<(unsigned)((n_rows + warps - 1) / warps), warps * 32, 0, (cudaStream_t)stream>>>(
        power, n_rows, (int)K, fb, (int)n_mels, take_log, eps, out, out_row_stride);
    return secommon::check_launch("mel_kernel");
}

int se_delta(float* x, int64_t n_utt, int64_t n_frames, int64_t D, int order, void* stream) {
    SE_REQUIRE(x && n_utt > 0 && n_frames > 0 && D > 0 && order >= 0 && order <= 4, "bad argument");
    const long long total = n_utt * n_frames * D;
    const unsigned blocks = (unsigned)std::min<long long>((total + kThreads - 1) / kThreads, 148LL * 16);
    const int stride = (int)((order + 1) * D);
    for (int o = 1; o <= order; ++o) {
        delta_kernel<<<blocks, kThreads, 0, (cudaStream_t)stream>>>(x, (int)n_frames, (int)D, stride, (int)((o - 1) * D), (int)(o * D), total);
        int rc = secommon::check_launch("delta_kernel");
        if (rc != SE_OK) return rc;
    }
    return SE_OK;
}

int se_linear_head_fwd(const float* x, const float* mean, const float* std, float cmvn_eps, const float* W,
                       const float* b, int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act,
                       const float* linears, float* offset_out, float* predicted_out, int precision, void* stream) {
    return se_linear_head_fwd_strided(x, D_in, mean, std, D_in, cmvn_eps, W, D_in, b, n_utt, n_frames, D_in, D_out, act, linears,
                                      offset_out, predicted_out, D_out, precision, stream);
}

int se_linear_head_fwd_strided(const float* x, int64_t ldx, const float* mean, const float* std, int64_t ld_stats,
                               float cmvn_eps, const float* W, int64_t ldw, const float* b, int64_t n_utt,
                               int64_t n_frames, int64_t D_in, int64_t D_out, int act, const float* linears,
                               float* offset_out, float* predicted_out, int64_t ld_out, int precision, void* stream) {
    SE_REQUIRE(x && W && n_utt > 0 && n_frames > 0 && D_in > 0 && D_out > 0, "bad argument");
    SE_REQUIRE(ldx >= D_in && ldw >= D_in && ld_out >= D_out && (!mean || ld_stats >= D_in), "row stride smaller than the row");
    SE_REQUIRE((mean == nullptr) == (std == nullptr), "mean and std go together");
    SE_REQUIRE(offset_out || predicted_out, "no output requested");
    SE_REQUIRE(!predicted_out || linears, "predicted_out needs linears");
    SE_REQUIRE(act >= SE_ACT_IDENTITY && act <= SE_ACT_SIGMOID, "unknown activation %d", act);
    const long long R = n_utt * n_frames;
    if (precision == 1)
        return sehead::launch_linear_head_tc(x, ldx, mean, std, ld_stats, cmvn_eps, W, ldw, b, R, (int)n_frames, (int)D_in, (int)D_out,
                                             act, linears, offset_out, predicted_out, ld_out, (cudaStream_t)stream);
    if (precision != 0) return fail(SE_ERR_BAD_ARG, "precision=%d (0 = fp32 SIMT, 1 = TF32 tcgen05)", precision);
    dim3 grid((unsigned)((D_out + BN - 1) / BN), (unsigned)((R + BM - 1) / BM));
    linear_head_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, mean, std, cmvn_eps, W, b, R, (int)n_frames, (int)D_in,
                                                                   (int)D_out, act, linears, offset_out, predicted_out,
                                                                   ldx, ld_stats, ldw, ld_out);
    return secommon::check_launch("linear_head_fwd_kernel");
}

int se_linear_head_bwd(const float* x, const float* mean, const float* std, float cmvn_eps, const float* W,
                       const float* offset, const float* grad_offset, int64_t n_utt, int64_t n_frames, int64_t D_in,
                       int64_t D_out, int act, float* grad_W, float* grad_b, void* stream) {
    (void)W;
    SE_REQUIRE(x && offset && grad_offset && grad_W && n_utt > 0 && n_frames > 0, "bad argument");
    SE_REQUIRE((mean == nullptr) == (std == nullptr), "mean and std go together");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemsetAsync(grad_W, 0, sizeof(float) * D_in * D_out, st));
    if (grad_b) SE_CUDA_CHECK(cudaMemsetAsync(grad_b, 0, sizeof(float) * D_out, st));
    const long long R = n_utt * n_frames;
    const int tiles = (int)(((D_out + BM - 1) / BM) * ((D_in + BN - 1) / BN));
    long long splits = std::max<long long>(1, (148LL * 4) / tiles);
    long long rows_per_split = (R + splits - 1) / splits;
    rows_per_split = ((rows_per_split + BK - 1) / BK) * BK;
    splits = (R + rows_per_split - 1) / rows_per_split;
    dim3 grid((unsigned)((D_in + BN - 1) / BN), (unsigned)((D_out + BM - 1) / BM), (unsigned)splits);
    linear_head_bwd_kernel<<<grid, 256, 0, st>>>(x, mean, std, cmvn_eps, offset, grad_offset, R, (int)n_frames, (int)D_in,
                                                 (int)D_out, act, grad_W, grad_b, rows_per_split);
    return secommon::check_launch("linear_head_bwd_kernel");
}

}  // extern "C"
