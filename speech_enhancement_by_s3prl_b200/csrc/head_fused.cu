// libse_b200.so -- fused CMVN + mask head for the evaluation step (model.py:28-34):
//
//     offset = act( ((x - mean) / (std + eps)) W^T + b )
//
// with mean / std taken from the per-(utterance, feature) sums that the STFT kernel accumulates
// (se_stft_stats), so no separate statistics pass runs between the STFT and the head.
//
// One CTA owns ONE tile of up to 128 consecutive rows (frames) and ALL output columns:
//   * warp 9 (one lane)  TMA producer: SWIZZLE_128B tensor-map loads through a 4-stage ring; a stage is one
//                        32-float k-block of the A tile (16 KB K-major tile) plus the same k-block of all
//                        weight rows (34 KB)
//   * warps 0-7          normalise the A tile IN PLACE in shared memory (CMVN scale/shift from the
//                        sums, round to TF32), later run the epilogue
//   * warp 8 (one lane)  tcgen05.mma kind::tf32, fp32 accumulators in tensor memory: columns
//                        [0,256) by one N=256 instruction, the remaining <= 16 by a second one
//   * more than 272 output columns (n_fft 1024: 513 -> 528): blockIdx.x % n_split selects one of the column slabs of
//                        <= 256 (3 x 176); each CTA streams the same A tile (re-reads come from L2) and its
//                        own slab of weight rows, and stores its slab of every output row
//   * more tiles than SMs: two CTAs per SM (2-stage rings, 256 tensor-memory columns each, direct stores)
//   * epilogue           tcgen05.ld -> +bias -> activation -> row-major staging tile in shared
//                        memory (reusing the A tile) -> ONE bulk async store per 32-row quadrant:
//                        with ld_out == padded row length the CTA's output is contiguous in HBM
// The kernel is launched with programmatic stream serialisation: barrier init, TMEM allocation and
// the first weight loads overlap the tail of the upstream kernel (griddepcontrol.wait guards the
// first read of its outputs).
#include <cuda.h>
#include "se_common.cuh"

using secommon::fail;

namespace {

constexpr int BM = 128, BK = 32, kMaxKB = 17, kMaxStages = 4;
constexpr int kWorkWarps = 8, kWorkThreads = kWorkWarps * 32, kThreads = kWorkThreads + 64;   // + MMA warp + TMA warp
constexpr int kATileBytes = BM * BK * 4;                       // 16 KB: one 32-float k-block of the A tile
constexpr int kMaxWRows = 272;
constexpr int kWTileBytes = kMaxWRows * BK * 4;                // 34 816: the same k-block of all weight rows
constexpr int kMaxStageBytes = kATileBytes + kWTileBytes;      // 51 200 (multiple of 1024: SWIZZLE_128B atoms stay aligned)
constexpr int kStatLd = kMaxKB * BK;                           // 544: features per utterance (n_fft 1024: 513)
// shared memory: fixed part (CMVN scale / shift of two utterances, bias, mbarriers, TMEM slot) | ring of `stages` stages.
// Two launch shapes share the kernel: ONE CTA per SM with a 4-stage ring, 512 tensor-memory columns and bulk stores from a
// staging tile (a single wave of <= 272-column tiles: the headline), or TWO CTAs per SM with 2-stage rings, 256 columns
// each and direct stores -- when the tiles outnumber the SMs, the second CTA's loads fill the L2 pipe while the first one
// is in its prologue / epilogue (the kernel is bound by the chip-wide L2 throughput of the weight re-reads).
constexpr int kOffScale = 0;
constexpr int kOffShift = kOffScale + 2 * kStatLd * 4;
constexpr int kOffBias = kOffShift + 2 * kStatLd * 4;
constexpr int kOffExtra = kOffBias + kStatLd * 4;              // [BM] the "+1" output column of a 256 + 1 slab (SIMT dot products)
constexpr int kOffBar = kOffExtra + BM * 4;
constexpr int kNumBars = 3 * kMaxStages + 1;
constexpr int kOffTmem = kOffBar + kNumBars * 8;
constexpr int kOffRing = (kOffTmem + 16 + 1023) / 1024 * 1024;
constexpr int kSmemBytes = kOffRing + kMaxStages * kMaxStageBytes;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(kMaxStageBytes % 1024 == 0 && kATileBytes % 1024 == 0, "swizzle atom alignment");
constexpr unsigned kSpinLimit = 1u << 22;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (unsigned spin = 0; !done; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (spin > kSpinLimit) __trap();                          // never hang the GPU on a protocol bug
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// K-major SWIZZLE_128B shared-memory matrix descriptor: rows 128 B apart, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ uint32_t make_idesc(int n) {           // kind::tf32, fp32 accumulate, A/B K-major, M = 128
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

struct Head2Args {
    const double* sums;        // (n_utt, ld_stats, 2): sum x, sum x^2 over the utterance's frames; null = no CMVN
    long long ld_stats;
    float cmvn_eps;
    double inv_n, inv_nm1;     // 1 / n_frames, 1 / (n_frames - 1)
    const float* bias;
    long long R;               // n_utt * n_frames
    int n_utt, n_frames, Din, Dout, act;
    float* out;
    long long ld_out;
    int tile_rows;             // rows per CTA: multiple of 8, <= 128, <= n_frames (a tile touches <= 2 utterances)
    int kblocks;               // ceil(Din / 32) <= 17
    int w_rows;                // Dout rounded up to 16, <= 544
    int cta_cols;              // output columns (weight rows) per CTA slab: multiple of 16, <= 272; slab = blockIdx.x % n_split
    int n_split;               // column slabs per row tile
    int w_box_rows, w_boxes;   // weight tensor-map box rows and boxes per k-block
    int sld;                   // floats per row of the staging tile
    int bulk_out;              // staging rows == output rows and 16-byte aligned: one bulk store per quadrant
    int stages, stage_bytes;   // ring depth (2 or 4) and bytes per stage (A k-block + this launch's weight k-block, 1024-aligned)
    int tmem_cols;             // tensor-memory columns allocated per CTA (256: two CTAs per SM; 512: one)
    int direct_out;            // epilogue stores registers straight to global memory (no staging tile: 2-stage rings are too small)
    const float* w_extra;      // 256 m + 1 output columns (K = 257, 513) as m slabs of 256 tensor-core columns: the last column's
    long long ldw;             //   weight row (its dot products run in the CMVN warps while they normalise the A tile), or null
    unsigned long long* trace; // CTA timeline buffer (se_set_trace) or null
};

// DUAL = two CTAs per SM: 2-stage ring of `a.stage_bytes` stages, "+1" SIMT column, direct stores; else one CTA per SM with
// the 4-stage ring of full-size stages (compile-time constants: this is the headline's shape)
template <bool DUAL>
__global__ void __launch_bounds__(kThreads, DUAL ? 2 : 1)
linear_head_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const Head2Args a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    secommon::TraceScope trace(a.trace, 2);
    const uint32_t sbase = smem_u32(smem);
    float* s_scale = reinterpret_cast<float*>(smem + kOffScale);
    float* s_shift = reinterpret_cast<float*>(smem + kOffShift);
    float* s_bias = reinterpret_cast<float*>(smem + kOffBias);
    float* s_extra = reinterpret_cast<float*>(smem + kOffExtra);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffTmem);
    const uint32_t bar_full = sbase + kOffBar;                         // [stages] TMA landed the stage's A and W k-block
    const uint32_t bar_norm = bar_full + 8 * kMaxStages;               // [stages] A k-block normalised in place
    const uint32_t bar_empty = bar_norm + 8 * kMaxStages;              // [stages] the MMAs have read the stage
    const uint32_t bar_accum = bar_empty + 8 * kMaxStages;
    constexpr int kStages = DUAL ? 2 : kMaxStages;
    const int kStageBytes = DUAL ? a.stage_bytes : kMaxStageBytes;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // slab index fastest: the slabs of one row tile are dispatched together, so the second read of the A tile hits L2
    const int slab = (int)(blockIdx.x % (unsigned)a.n_split);
    const long long r0 = (long long)(blockIdx.x / (unsigned)a.n_split) * a.tile_rows;
    const int col0 = slab * a.cta_cols;                                  // this CTA's slab of output columns
    const int ncols = a.w_rows - col0 < a.cta_cols ? a.w_rows - col0 : a.cta_cols;
    const int n_main = ncols > 256 ? 256 : ncols, n_tail = ncols - n_main;   // MMA column split: [0, n_main) and [n_main, ncols)
    const uint32_t w_bytes = (uint32_t)(a.w_box_rows * a.w_boxes) * BK * 4;  // whole boxes land (rows past Dout read as zero)

    if (threadIdx.x == 0) {
        if (sbase & 1023) __trap();
        for (int s = 0; s < kMaxStages; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_norm + 8 * s, kWorkWarps);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kWorkWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)a.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    griddep_launch();                                   // the next kernel may start its own prologue
    if (threadIdx.x == 0) trace.mark(11);

    if (warp == kWorkWarps + 1) {
        // ===================== TMA producer =====================
        // ring of kStages stages, each holding one 32-float k-block of the A tile and of all weight rows
        if (lane == 0) {
            const uint32_t a_bytes = (uint32_t)a.tile_rows * BK * 4;
            auto load_w = [&](int kb, int s) {
                const uint32_t dst = sbase + kOffRing + s * kStageBytes + kATileBytes;
                for (int b = 0; b < a.w_boxes; ++b)
                    tma_load_2d(dst + b * a.w_box_rows * BK * 4, &tmW, kb * BK, col0 + b * a.w_box_rows, bar_full + 8 * s);
            };
            auto load_a = [&](int kb, int s) {
                tma_load_2d(sbase + kOffRing + s * kStageBytes, &tmA, kb * BK, (int)r0, bar_full + 8 * s);
            };
            const int first = a.kblocks < kStages ? a.kblocks : kStages;
            for (int s = 0; s < first; ++s) {                              // weights do not depend on the upstream kernel
                mbar_expect_tx(bar_full + 8 * s, a_bytes + w_bytes);
                load_w(s, s);
            }
            griddep_wait();
            for (int s = 0; s < first; ++s) load_a(s, s);
            for (int kb = kStages; kb < a.kblocks; ++kb) {
                const int s = kb % kStages;
                mbar_wait(bar_empty + 8 * s, ((kb / kStages) - 1) & 1);     // MMAs of k-block kb - kStages have read the stage
                mbar_expect_tx(bar_full + 8 * s, a_bytes + w_bytes);
                load_w(kb, s);
                load_a(kb, s);
            }
        }
    } else if (warp == kWorkWarps) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc_main = make_idesc(n_main), idesc_tail = make_idesc(n_tail > 0 ? n_tail : 16);
            for (int kb = 0; kb < a.kblocks; ++kb) {
                const int s = kb % kStages;
                mbar_wait(bar_norm + 8 * s, (kb / kStages) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_addr = sbase + kOffRing + s * kStageBytes;
                const uint32_t b_addr = a_addr + kATileBytes;
                const int kvalid = a.Din - kb * BK;
                const int ksteps = kvalid >= BK ? BK / 8 : (kvalid + 7) / 8;
                for (int kk = 0; kk < ksteps; ++kk) {
                    const uint64_t ad = make_desc(a_addr + kk * 32);
                    umma_tf32(tmem_base, ad, make_desc(b_addr + kk * 32), idesc_main, (kb | kk) ? 1u : 0u);
                    if (n_tail > 0)
                        umma_tf32(tmem_base + (uint32_t)n_main, ad, make_desc(b_addr + n_main * BK * 4 + kk * 32), idesc_tail,
                                  (kb | kk) ? 1u : 0u);
                }
                umma_commit(bar_empty + 8 * s);
            }
            umma_commit(bar_accum);
        }
    } else {
        // ===================== CMVN in place, then epilogue =====================
        const int t = threadIdx.x;
        griddep_wait();                                                   // the sums come from the upstream kernel
        const long long u0 = r0 / a.n_frames;
        const int split = (int)((u0 + 1) * a.n_frames - r0);              // first tile row of the next utterance
        // per-utterance CMVN scale / shift for the (at most two) utterances of the tile; loads first, then the arithmetic
        const float bscale = a.act == SE_ACT_SIGMOID ? -1.4426950408889634f : 1.0f;     // see the epilogue
        float bias_r[2];                                                  // 288 local columns over 256 threads; in flight with the sums
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int i = t + q * kWorkThreads;
            bias_r[q] = (i < 288 && a.bias && col0 + i < a.Dout) ? bscale * __ldg(a.bias + col0 + i) : 0.f;
        }
        {
            constexpr int kPer = (2 * kStatLd + kWorkThreads - 1) / kWorkThreads;
            double2 p[kPer];
#pragma unroll
            for (int q = 0; q < kPer; ++q) {
                const int i = t + q * kWorkThreads, ul = i / kStatLd, k = i - ul * kStatLd;
                const long long u = u0 + ul;
                p[q] = make_double2(0.0, 0.0);
                if (i < 2 * kStatLd && k < a.Din && a.sums && u < a.n_utt)
                    p[q] = *reinterpret_cast<const double2*>(a.sums + (u * a.ld_stats + k) * 2);
            }
#pragma unroll
            for (int q = 0; q < kPer; ++q) {
                const int i = t + q * kWorkThreads, ul = i / kStatLd, k = i - ul * kStatLd;
                if (i < 2 * kStatLd) {
                    float sc = 0.f, sh = 0.f;
                    if (k < a.Din) {
                        sc = 1.f;
                        if (a.sums && u0 + ul < a.n_utt) {
                            const double mean = p[q].x * a.inv_n;
                            const float var = (float)((p[q].y - p[q].x * mean) * a.inv_nm1);   // unbiased (model.py:30); cancellation in double
                            const float inv = __fdividef(1.0f, sqrtf(fmaxf(var, 0.0f)) + a.cmvn_eps);
                            sc = inv;
                            sh = -(float)mean * inv;
                        }
                    }
                    s_scale[i] = sc;
                    s_shift[i] = sh;
                }
            }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q)                                         // local column i = output column col0 + i
            if (t + q * kWorkThreads < 288) s_bias[t + q * kWorkThreads] = bias_r[q];
        asm volatile("bar.sync 1, %0;" ::"n"(kWorkThreads) : "memory");
        if (t == 0) trace.mark(12);

        // the "+1" column (last slab only): every thread owns one 4-float chunk of four rows per k-block
        const bool has_extra = DUAL && a.w_extra != nullptr && slab == a.n_split - 1;
        const int cx = (t & 7) ^ ((t >> 3) & 7);                          // logical chunk of this thread's four rows
        float dot[4] = {0.f, 0.f, 0.f, 0.f};
        for (int kb = 0; kb < a.kblocks; ++kb) {
            const int s = kb % kStages;
            float4 wx = make_float4(0.f, 0.f, 0.f, 0.f);
            const int kx = kb * BK + 4 * cx;
            if (has_extra && kx + 4 <= (int)a.ldw) wx = __ldg(reinterpret_cast<const float4*>(a.w_extra + kx));
            if (kx + 4 > a.Din) {                                         // the weight row's padding past D_in may hold NaN (NaN * 0 = NaN)
                wx.x = kx < a.Din ? wx.x : 0.f;
                wx.y = kx + 1 < a.Din ? wx.y : 0.f;
                wx.z = kx + 2 < a.Din ? wx.z : 0.f;
                wx.w = 0.f;
            }
            mbar_wait(bar_full + 8 * s, (kb / kStages) & 1);
            if (t == 0 && kb == 0) trace.mark(13);
            float4* tile = reinterpret_cast<float4*>(smem + kOffRing + s * kStageBytes);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int idx = t + kWorkThreads * i;                     // physical 16-byte chunk: conflict-free LDS/STS.128
                const int row = idx >> 3;
                if (row < a.tile_rows) {
                    const int c = (idx & 7) ^ (row & 7);                  // logical chunk (SWIZZLE_128B)
                    const int so = (row >= split ? kStatLd : 0) + kb * BK + 4 * c;
                    const float4 sc = *reinterpret_cast<const float4*>(s_scale + so);
                    const float4 sh = *reinterpret_cast<const float4*>(s_shift + so);
                    float4 v = tile[idx];
                    v.x = to_tf32(fmaf(v.x, sc.x, sh.x));
                    v.y = to_tf32(fmaf(v.y, sc.y, sh.y));
                    v.z = to_tf32(fmaf(v.z, sc.z, sh.z));
                    v.w = to_tf32(fmaf(v.w, sc.w, sh.w));
                    tile[idx] = v;
                    if (has_extra) dot[i] = fmaf(v.x, wx.x, fmaf(v.y, wx.y, fmaf(v.z, wx.z, fmaf(v.w, wx.w, dot[i]))));
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the MMA (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_norm + 8 * s);
        }
        if (has_extra) {                                                   // the 8 lanes that share a row add up their chunks
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float d = dot[i];
                d += __shfl_xor_sync(0xffffffffu, d, 1);
                d += __shfl_xor_sync(0xffffffffu, d, 2);
                d += __shfl_xor_sync(0xffffffffu, d, 4);
                if ((t & 7) == 0) s_extra[(t >> 3) + 32 * i] = d;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kWorkThreads) : "memory");
        }

        // ---- epilogue: warp w reads TMEM lanes 32 (w & 3) .. +31, column half (w >> 2)
        if (t == 0) trace.mark(14);
        mbar_wait(bar_accum, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (t == 0) trace.mark(15);
        float* stage = reinterpret_cast<float*>(smem + kOffRing);           // every stage has been consumed: reuse the ring
        const int quad = warp & 3, half = warp >> 2;
        const int row = quad * 32 + lane;
        const int ncol16 = ncols / 16;
        const int c_lo = 16 * (half == 0 ? 0 : ncol16 / 2), c_hi = 16 * (half == 0 ? ncol16 / 2 : ncol16);
        float* srow = stage + (long long)row * a.sld;
        // direct mode: registers -> global memory (row = this lane's frame; 64 contiguous bytes per 16-column chunk)
        const bool row_ok = row < a.tile_rows && r0 + row < a.R;
        float* grow = a.out + (r0 + row) * a.ld_out + col0;
        // two 16-column chunks in flight: the tensor-memory load of chunk c+1 overlaps the activation of chunk c
        const uint32_t tbase = tmem_base + ((uint32_t)(quad * 32) << 16);
        // The activation of a chunk is written stage by stage over all 16 values (all exponentials, then all adds, then
        // all reciprocals): a warp issues in order, so element-by-element code would expose the SFU latency 16 times.
        // Sigmoid: s_bias holds -log2(e) * bias and z is scaled by -log2(e) in the same FFMA: 1 / (1 + 2^t).
        const int act = a.act;
        const float zscale = act == SE_ACT_SIGMOID ? -1.4426950408889634f : 1.0f;
        // direct mode, aligned rows: each warp turns its 32 rows x 32 columns around in a private 4 KB scratch of the (consumed)
        // ring -- lanes own rows on the tensor-memory side, 8 lanes share a row on the store side, so one store instruction writes
        // four whole 128-byte lines instead of 16 bytes of 32 different rows.  Chunk j of row r sits at r * 8 + (j ^ (r & 7)).
        float4* sw = reinterpret_cast<float4*>(stage) + warp * 256;
        auto emit = [&](const uint32_t (&acc)[16], int c0, int cb) {
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
                const float4 bz = *reinterpret_cast<const float4*>(s_bias + c0 + j);
                v[j] = fmaf(__uint_as_float(acc[j]), zscale, bz.x);
                v[j + 1] = fmaf(__uint_as_float(acc[j + 1]), zscale, bz.y);
                v[j + 2] = fmaf(__uint_as_float(acc[j + 2]), zscale, bz.z);
                v[j + 3] = fmaf(__uint_as_float(acc[j + 3]), zscale, bz.w);
            }
            if (act == SE_ACT_SIGMOID) {
#pragma unroll
                for (int j = 0; j < 16; ++j) asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(v[j]) : "f"(v[j]));
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] += 1.0f;
#pragma unroll
                for (int j = 0; j < 16; ++j) asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(v[j]) : "f"(v[j]));
            } else if (act == SE_ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
            }
            if (a.direct_out == 2) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    sw[lane * 8 + ((cb + j) ^ (lane & 7))] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                return;
            }
            if (a.direct_out) {
                if (row_ok) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const int c = col0 + c0 + j;
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (c + e < a.Dout) grow[c0 + j + e] = v[j + e];
                    }
                }
                return;
            }
#pragma unroll
            for (int j = 0; j < 16; j += 4)
                if (c0 + j < a.sld) *reinterpret_cast<float4*>(srow + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        };
        auto flush = [&](int c0, int ncol) {                                 // scratch columns [0, ncol) -> output columns col0 + c0 ...
            __syncwarp();
            const int c = lane & 7;
            if (4 * c < ncol) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + (lane >> 3), trow = quad * 32 + r;
                    if (trow < a.tile_rows && r0 + trow < a.R) {
                        const float4 x = sw[r * 8 + (c ^ (r & 7))];
                        float* g = a.out + (r0 + trow) * a.ld_out + col0 + c0 + 4 * c;
                        const int gc = col0 + c0 + 4 * c;
                        if (gc + 4 <= (int)a.ld_out) *reinterpret_cast<float4*>(g) = x;
                        else {
                            if (gc < a.Dout) g[0] = x.x;
                            if (gc + 1 < a.Dout) g[1] = x.y;
                            if (gc + 2 < a.Dout) g[2] = x.z;
                            if (gc + 3 < a.Dout) g[3] = x.w;
                        }
                    }
                }
            }
            __syncwarp();
        };
        uint32_t acc0[16], acc1[16];
        tmem_ld16(tbase + (uint32_t)c_lo, acc0);
        tmem_ld_wait();
        for (int c0 = c_lo; c0 < c_hi; c0 += 32) {
            if (c0 + 16 < c_hi) tmem_ld16(tbase + (uint32_t)(c0 + 16), acc1);
            emit(acc0, c0, 0);
            tmem_ld_wait();
            if (c0 + 16 < c_hi) {
                if (c0 + 32 < c_hi) tmem_ld16(tbase + (uint32_t)(c0 + 32), acc0);
                emit(acc1, c0 + 16, 4);
                tmem_ld_wait();
            }
            if (a.direct_out == 2) flush(c0, c_hi - c0 < 32 ? c_hi - c0 : 32);
        }
        if (has_extra && half == 0 && row_ok) {                             // column Dout - 1 of this row
            float z = fmaf(s_extra[row], zscale, (a.bias ? zscale * __ldg(a.bias + a.Dout - 1) : 0.f));
            if (act == SE_ACT_SIGMOID) {
                asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(z) : "f"(z));
                z += 1.0f;
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(z) : "f"(z));
            } else if (act == SE_ACT_RELU) z = fmaxf(z, 0.0f);
            a.out[(r0 + row) * a.ld_out + a.Dout - 1] = z;
        }
        if (!a.direct_out) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync %0, 64;" ::"r"(2 + quad) : "memory");        // both warps of the quadrant have staged their columns
        }
        if (t == 0) trace.mark(16);
        long long rows_left = a.R - r0;
        if (rows_left > a.tile_rows) rows_left = a.tile_rows;
        int rows_valid = (int)rows_left - quad * 32;
        rows_valid = rows_valid > 32 ? 32 : rows_valid;
        if (rows_valid > 0 && !a.direct_out) {
            float* gdst = a.out + (r0 + quad * 32) * a.ld_out + col0;
            const float* ssrc = stage + (long long)quad * 32 * a.sld;
            if (a.bulk_out) {
                if (half == 0 && lane == 0) {
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                 ::"l"(gdst), "r"(smem_u32(ssrc)), "r"((uint32_t)(rows_valid * a.sld * 4)) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the staging tile has been read; the writes land on their own
                }
            } else {
                for (int r = half; r < rows_valid; r += 2)
                    for (int c = lane; c < ncols && col0 + c < a.Dout; c += 32) gdst[(long long)r * a.ld_out + c] = ssrc[(long long)r * a.sld + c];
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    trace.finish();
    if (warp == kWorkWarps) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)a.tmem_cols) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D fp32 tensor map: `cols` x `rows` elements, `ld` floats between rows, box = 32 floats x box_rows, SWIZZLE_128B,
// out-of-bounds elements read as zero
int make_map(CUtensorMap* map, const float* base, long long cols, long long rows, long long ld, int box_rows) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) return fail(SE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return SE_OK;
}

int num_sms() { return secommon::device_sms(); }

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

extern "C" {

int se_linear_head_fused_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ldw,
                                   int64_t ld_out) {
    if (n_utt <= 0 || n_frames < 8 || D_in <= 0 || D_out <= 0) return 0;
    if (D_in > kMaxKB * BK || D_out > kMaxKB * BK) return 0;
    if (ldx % 4 || ldw % 4 || ldx < D_in || ldw < D_in || ld_out < D_out) return 0;
    const int64_t dout4 = (D_out + 3) / 4 * 4;
    if (D_out > kMaxWRows) return 1;                                                            // column slabs, direct stores
    if ((ld_out == dout4 ? ld_out : dout4 + 4) * 4 * BM > kMaxStages * kMaxStageBytes) return 0;  // staging tile must fit in the ring
    return 1;
}

int se_linear_head_fused(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps,
                         const float* W, int64_t ldw, const float* b, int64_t n_utt, int64_t n_frames, int64_t D_in,
                         int64_t D_out, int act, float* offset_out, int64_t ld_out, void* stream) {
    SE_REQUIRE(x && W && offset_out, "null pointer");
    SE_REQUIRE(act >= SE_ACT_IDENTITY && act <= SE_ACT_SIGMOID, "unknown activation %d", act);
    SE_REQUIRE(!stat_sums || ld_stats >= D_in, "ld_stats smaller than D_in");
    if (!se_linear_head_fused_supported(n_utt, n_frames, D_in, D_out, ldx, ldw, ld_out) || !aligned16(x) || !aligned16(W))
        return fail(SE_ERR_UNSUPPORTED, "fused head: shape / alignment outside the fast path (D_in=%lld, D_out=%lld, n_frames=%lld)",
                    (long long)D_in, (long long)D_out, (long long)n_frames);
    Head2Args a{};
    a.sums = stat_sums; a.ld_stats = ld_stats; a.cmvn_eps = cmvn_eps; a.bias = b;
    a.R = n_utt * n_frames; a.n_utt = (int)n_utt; a.n_frames = (int)n_frames; a.Din = (int)D_in; a.Dout = (int)D_out; a.act = act;
    a.out = offset_out; a.ld_out = ld_out;
    a.trace = secommon::trace_ptr();
    a.inv_n = 1.0 / (double)n_frames;
    a.inv_nm1 = 1.0 / (double)(n_frames - 1);
    a.kblocks = (int)((D_in + BK - 1) / BK);
    a.w_rows = (int)((D_out + 15) / 16 * 16);
    const int sms = num_sms();
    const long long tiles128 = (a.R + BM - 1) / BM;
    // Launch shape (see the shared-memory comment at the top): ONE CTA per SM with the deep ring (bulk stores from a staging
    // tile for a single slab, direct stores for the two <= 272-column slabs of K = 513), or TWO CTAs per SM when the slab
    // fits 256 tensor-memory columns and the tiles outnumber the SMs.
    // Two CTAs per SM need slabs of <= 256 tensor-memory columns.  K = 2^k + 1 (257, 513: every power-of-two n_fft) is cut into
    // slabs of 256 tensor-core columns plus ONE column of SIMT dot products in the CMVN warps, so it gets there without an extra
    // slab (cutting 272 into 2 x 136 or 528 into 3 x 176 re-reads every A tile once more and loses: measured 17.5 -> 20.0 us
    // and 45.3 -> 52.9 us, tools/time_head_fused.py).  Used when the tiles of the one-CTA shape outnumber the SMs.
    const bool plus_one = D_out > 256 && (D_out - 1) % 256 == 0;
    const int single_split = (a.w_rows + kMaxWRows - 1) / kMaxWRows;
    const bool fits256 = a.w_rows <= 256 || plus_one;
    const bool dual = fits256 && tiles128 * single_split > sms;
    int n_split = 1;
    long long slots = sms;
    a.w_extra = nullptr; a.ldw = ldw;
    if (dual) {
        if (plus_one) {
            n_split = (int)((D_out - 1) / 256);
            a.w_rows = 256 * n_split;                                       // tensor-core columns; column D_out - 1 is the SIMT one
            a.w_extra = W + (D_out - 1) * ldw;
        }
        slots = 2LL * sms;
        a.stages = 2; a.tmem_cols = 256;
        a.direct_out = (ld_out % 4 == 0 && aligned16(offset_out)) ? 2 : 1;
    } else {
        n_split = single_split;                                             // <= 2 slabs of <= 272 columns
        a.stages = kMaxStages; a.tmem_cols = 512;
        a.direct_out = n_split > 1 ? ((ld_out % 4 == 0 && aligned16(offset_out)) ? 2 : 1) : 0;
    }
    a.cta_cols = ((a.w_rows + n_split - 1) / n_split + 15) / 16 * 16;
    a.stage_bytes = dual ? kATileBytes + (a.cta_cols * BK * 4 + 1023) / 1024 * 1024 : kMaxStageBytes;
    // rows per tile: the fewest waves of (tiles x slabs) CTAs over the resident slots, then tiles as even as the waves allow
    const long long waves = (tiles128 * n_split + slots - 1) / slots;
    long long want_tiles = waves * slots / n_split;
    if (want_tiles < 1) want_tiles = 1;
    long long rows = (a.R + want_tiles - 1) / want_tiles;
    rows = (rows + 7) / 8 * 8;
    if (rows > BM) rows = BM;
    if (rows > n_frames) rows = n_frames / 8 * 8;                           // a tile may touch at most two utterances
    a.tile_rows = (int)rows;
    a.w_boxes = a.cta_cols > 256 ? 2 : 1;                              // cta_cols is a multiple of 16: both boxes are whole 8-row atoms
    a.w_box_rows = a.cta_cols / a.w_boxes;
    const int dout4 = (int)((D_out + 3) / 4 * 4);
    a.bulk_out = (!a.direct_out && ld_out == dout4 && aligned16(offset_out)) ? 1 : 0;
    a.sld = a.bulk_out ? (int)ld_out : dout4 + 4;
    const size_t smem_bytes = (size_t)kOffRing + (size_t)a.stages * a.stage_bytes;
    CUtensorMap tmA, tmW;
    int rc = make_map(&tmA, x, D_in, a.R, ldx, a.tile_rows);
    if (rc != SE_OK) return rc;
    if ((rc = make_map(&tmW, W, D_in, D_out, ldw, a.w_box_rows)) != SE_OK) return rc;
    static unsigned long long opted = 0;                       // per device: cudaFuncSetAttribute is not process-wide
    if (secommon::first_use_on_device(opted)) {
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kOffRing + 2 * (kATileBytes + 256 * BK * 4)));
    }
    cudaLaunchConfig_t cfg{};
    unsigned tiles = (unsigned)((a.R + a.tile_rows - 1) / a.tile_rows);
    a.n_split = n_split;
    cfg.gridDim = dim3(tiles * (unsigned)n_split);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (secommon::pdl_mask() & 1) ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (dual) SE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, linear_head_fused_kernel<true>, tmA, tmW, a));
    else SE_CUDA_CHECK(cudaLaunchKernelEx(&cfg, linear_head_fused_kernel<false>, tmA, tmW, a));
    return secommon::check_launch("linear_head_fused_kernel");
}

}  // extern "C"
