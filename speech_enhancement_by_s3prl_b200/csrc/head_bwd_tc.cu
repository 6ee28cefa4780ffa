// libse_b200.so -- tensor-core weight gradient of the mask head (autograd of model.py:14-17, 28-34):
//
//     grad_W[n, k] = sum_r dZ[r, n] * xhat[r, k]        grad_b[n] = sum_r dZ[r, n]
//     dZ = grad_offset * act'(offset)                   xhat = (x - mean) / (std + eps)   (the head's CMVN input)
//
// A split-K tcgen05 GEMM: CTA (split s, m-tile mt) owns rows [ra, rb) of the batch and output features
// [128 mt, 128 mt + 128), and accumulates D[128 n][272 k] in tensor memory over its row blocks of 32.  A second kernel sums the
// partials over the splits (deterministic), or packs one partial per utterance (per-sample gradients, sampler.py:95-108).
//
// TWO kernels share the plan, the epilogue and the reduction:
//   linear_head_bwd_tma_kernel<LOSS>  (further down; 16-byte aligned, row-padded operands -- the engine's tensors): TMA lands the
//       operands as they lie in HBM, MN-major tcgen05 operands, in-place rewrite; LOSS = kLossSisdr / kLossWsd also folds the
//       backward of that objective in
//   linear_head_bwd_tc_kernel         (below; any strides -- the autograd custom op on un-padded tensors): transposing producers
//
// linear_head_bwd_tc_kernel:
//   * warps 0-7  producers: both operands are row-major in r (the reduction index), so they are TRANSPOSED on the way
//                into shared memory: thread -> one n (or k), four consecutive rows per 16-byte chunk, coalesced 128-byte
//                loads across the warp, one conflict-free STS.128 into the K-major SWIZZLE_128B tile; dZ's activation
//                derivative and xhat's CMVN are applied here, operands rounded to TF32 (cvt.rna).  Column k = D_in of
//                the B tile is the constant 1, so grad_b falls out of the GEMM as column D_in of D.
//   * warp 0     also issues the tcgen05.mma kind::tf32 (M = 128, N = 256 + 16) of the previous block and commits stages back
//   * epilogue   tcgen05.ld -> staging tile -> coalesced stores of the CTA's partial into the workspace
// Output rows that do not fill a 128-row tile are few when D_out = 257 (one row): up to kMaxSimtRows such rows go through a
// fp32 dot products accumulated by the B-operand producers of the first tile's CTAs (they hold xhat in registers anyway)
// instead of a third tensor-core tile that would transpose the whole B operand again for one useful row.
#include <cuda.h>
#include "objective_math.cuh"
#include "se_common.cuh"

using secommon::fail;

namespace {

constexpr int BM = 128, BK = 32, kStages = 4;
constexpr int kProdWarps = 8, kProdThreads = kProdWarps * 32, kThreads = kProdThreads;   // 8 warps: 2 per scheduler, 255-register cap
constexpr int kATileBytes = BM * BK * 4;                       // 16 KB
constexpr int kMaxBRows = 272;
constexpr int kBTileBytes = kMaxBRows * BK * 4;                // 34 816
constexpr int kStageBytes = kATileBytes + kBTileBytes;         // 51 200
constexpr int kMaxUtt = 8;                                     // utterances one CTA's row range may touch
constexpr int kMaxSimtRows = 4;                                // leftover output rows handled without the tensor cores
constexpr int kOffRing = 0;
constexpr int kOffStats = kOffRing + kStages * kStageBytes;    // [kMaxUtt][272] (mean, 1/(std+eps))
constexpr int kOffDz = kOffStats + kMaxUtt * kMaxBRows * 8;    // [2][kMaxSimtRows][32] dZ of the leftover rows, double-buffered
constexpr int kOffTail = kOffDz + 2 * 4 * 32 * 4;              // [kMaxSimtRows][16][8] partial sums of the shared-out columns
constexpr int kOffBar = kOffTail + 4 * 16 * 8 * 4;
constexpr int kNumBars = 2 * kStages + 1;
constexpr int kOffTmem = kOffBar + kNumBars * 8;
constexpr int kSmemBytes = kOffTmem + 16;
constexpr int kStageLd = 276;                                  // staging row stride (floats): conflict-free STS.128 by row
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(kMaxSimtRows == 4, "kOffDz / kOffTail are sized for 4 leftover rows");
static_assert(BM * kStageLd * 4 <= kStages * kStageBytes, "staging tile fits in the ring");
constexpr unsigned kSpinLimit = 1u << 22;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {   // K-major SWIZZLE_128B: rows 128 B apart, 8-row groups 1024 B
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
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct BwdArgs {
    const float* x; long long ldx;
    const float* mean; const float* stdv; long long ld_stats; float cmvn_eps;
    const double* sums; double inv_n, inv_nm1;   // alternative to mean / stdv: (n_utt, ld_stats, 2) [sum x, sum x^2] over the frames
    const float* offset; const float* grad_offset; long long ld_off;
    long long R; int n_frames, Din, Dout, act;
    long long rows_per_split;      // multiple of 32
    int sub;                       // per-utterance mode: splits per utterance (0: rows [split * rows_per_split, ...) of the whole batch)
    int b_rows;                    // round16(Din + 1) <= 272
    int n_main, n_tail;
    float* partials;               // (splits, m_rows, 272)
    int m_rows;                    // m_tiles * 128 + simt_rows
    // LOSS kernels: grad_offset is not read; d loss / d offset of objective.SISDR on predicted = offset * linear_inp (or of objective.WSD)
    // is rebuilt per element
    const float* inp; const float* tar; long long ld_inp, ld_tar;
    const double* sums3; const long long* lengths; int len_hop; float loss_eps; float grad_uniform; const float* grad_out;
    // kLossWsd: objective.WSD instead -- frame energies (n_utt * n_frames) and the batch maximum (1 float) of se_wsd_energy
    float alpha, db_interval; const float* energy; const float* max_energy;
    int m_tiles, simt_rows;        // tensor-core tiles; leftover rows [128 m_tiles, 128 m_tiles + simt_rows) done by SIMT CTAs
};

// dZ = grad_offset * act'(offset)
__device__ __forceinline__ float dact(float g, float o, int act) {
    if (act == SE_ACT_SIGMOID) return g * (o * (1.0f - o));
    if (act == SE_ACT_RELU) return o > 0.f ? g : 0.f;
    return g;
}

__global__ void __launch_bounds__(kThreads, 1) linear_head_bwd_tc_kernel(const BwdArgs a) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    float2* s_stats = reinterpret_cast<float2*>(smem + kOffStats);
    float* s_dz = reinterpret_cast<float*>(smem + kOffDz);
    float* s_tail = reinterpret_cast<float*>(smem + kOffTail);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffTmem);
    const uint32_t bar_full = sbase + kOffBar, bar_empty = bar_full + 8 * kStages, bar_accum = bar_empty + 8 * kStages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int split = blockIdx.x, n0 = blockIdx.y * BM;
    long long ra = (long long)split * a.rows_per_split;
    long long rb = ra + a.rows_per_split < a.R ? ra + a.rows_per_split : a.R;
    if (a.sub > 0) {                                                   // per-utterance mode: split = (utterance, part of its frames)
        const long long u = split / a.sub, ue = (u + 1) * a.n_frames;
        ra = u * a.n_frames + (long long)(split - u * a.sub) * a.rows_per_split;
        rb = ra + a.rows_per_split < ue ? ra + a.rows_per_split : ue;
        if (ra > ue) ra = ue;
    }
    const int nkb = rb > ra ? (int)((rb - ra + BK - 1) / BK) : 0;

    if (threadIdx.x == 0) {
        if (sbase & 1023) __trap();
        for (int s = 0; s < kStages; ++s) { mbar_init(bar_full + 8 * s, kProdWarps); mbar_init(bar_empty + 8 * s, 1); }
        mbar_init(bar_accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // CMVN constants of the (at most kMaxUtt) utterances this CTA's rows touch
    const long long u_first = ra / a.n_frames;
    for (int i = threadIdx.x; i < kMaxUtt * kMaxBRows; i += kThreads) {
        const int ul = i / kMaxBRows, k = i - ul * kMaxBRows;
        const long long u = u_first + ul;
        float2 st = make_float2(0.0f, 1.0f);
        if (a.mean && k < a.Din && u * a.n_frames < a.R) {
            st.x = __ldg(a.mean + u * a.ld_stats + k);
            st.y = 1.0f / (__ldg(a.stdv + u * a.ld_stats + k) + a.cmvn_eps);
        } else if (a.sums && k < a.Din && u * a.n_frames < a.R) {   // same arithmetic as the fused forward head (head_fused.cu)
            const double2 p = *reinterpret_cast<const double2*>(a.sums + (u * a.ld_stats + k) * 2);
            const double mean = p.x * a.inv_n;
            const float var = (float)((p.y - p.x * mean) * a.inv_nm1);
            st.x = (float)mean;
            st.y = __fdividef(1.0f, sqrtf(fmaxf(var, 0.0f)) + a.cmvn_eps);
        }
        s_stats[i] = st;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    {
        // ===================== producers: transpose both operands into K-major tiles =====================
        // Warp 0 doubles as the MMA issuer: before it starts on block kb it issues the MMAs of block kb - 1 (whose stage the
        // other warps have filled, or are about to -- they run in step), so the CTA is 8 warps = 2 per scheduler and the
        // two register sets of the software pipeline below fit without spills.
        const int t = threadIdx.x;
        const uint32_t idesc_main = make_idesc(a.n_main), idesc_tail = make_idesc(a.n_tail > 0 ? a.n_tail : 16);
        auto issue_mma = [&](int kb) {
            const int s = kb % kStages;
            mbar_wait(bar_full + 8 * s, (kb / kStages) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                const uint32_t a_addr = sbase + kOffRing + s * kStageBytes;
                const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
                for (int kk = 0; kk < BK / 8; ++kk) {
                    const uint64_t ad = make_desc(a_addr + kk * 32);
                    umma_tf32(tmem_base, ad, make_desc(b_addr + kk * 32), idesc_main, (kb | kk) ? 1u : 0u);
                    if (a.n_tail > 0)
                        umma_tf32(tmem_base + (uint32_t)a.n_main, ad, make_desc(b_addr + a.n_main * BK * 4 + kk * 32), idesc_tail,
                                  (kb | kk) ? 1u : 0u);
                }
                umma_commit(bar_empty + 8 * s);
            }
            __syncwarp();
        };
        // leftover output rows [128 m_tiles, +simt_rows): the thread that normalises column k of a block also accumulates
        // sum_r dZ[r, n_left] * xhat[r, k] in fp32 (dZ of the block's 32 rows is shared through s_dz); first-tile CTAs only
        const bool do_left = a.simt_rows > 0 && blockIdx.y == 0;
        const int n_left = a.m_tiles * BM;
        float acc_l[kMaxSimtRows], acc_t[kMaxSimtRows];
#pragma unroll
        for (int i = 0; i < kMaxSimtRows; ++i) { acc_l[i] = 0.0f; acc_t[i] = 0.0f; }
        // Software pipeline: the global loads of block kb + 1 are issued BEFORE block kb is transposed into shared memory, so the
        // load latency of one block hides under the arithmetic / stores of the previous one (two register sets, loop unrolled by 2).
        struct Regs { float ao[16], ag[16], bv[32], bx[4], dzg, dzo; };
        const int n = t & (BM - 1), ch = t >> 7;
        const bool nvalid = n0 + n < a.Dout;
        const bool kvalid = t < a.b_rows, isx = t < a.Din;
        const bool has_shared = a.b_rows > kProdThreads && t < 16 * 8 && kProdThreads + (t & 15) < a.b_rows;
        const int ks = kProdThreads + (t & 15), cs = t >> 4;               // shared-out column / chunk of this thread
        const bool dz_owner = do_left && t < 32 * a.simt_rows;
        // Loads are UNCONDITIONAL in a full block (the column index is clamped into the row, out-of-range lanes are zeroed by
        // selects when the values are consumed): a guarded `ok ? __ldg(p) : 0` per element compiles into a branch with its own
        // convergence barrier per load, which serialises the 70 loads of a block.
        const int ncl = nvalid ? n : 0, tcl = isx ? t : 0, kcl = (has_shared && ks < a.Din) ? ks : 0;
        auto issue = [&](int kb, Regs& R) {
            const long long r0 = ra + (long long)kb * BK;
            const float* po = a.offset + r0 * a.ld_off + n0 + ncl;
            const float* pg = a.grad_offset + r0 * a.ld_off + n0 + ncl;
            const float* px = a.x + r0 * a.ldx;
            R.dzg = 0.0f; R.dzo = 0.0f;
            if (r0 + BK <= rb) {                                           // all 32 rows of the block exist
#pragma unroll
                for (int e = 0; e < 16; ++e) {                             // A: chunks c = ch + 2 (e >> 2), rows 4 c + (e & 3)
                    const int rr = 4 * (ch + 2 * (e >> 2)) + (e & 3);
                    R.ao[e] = __ldg(po + (long long)rr * a.ld_off);
                    R.ag[e] = __ldg(pg + (long long)rr * a.ld_off);
                }
#pragma unroll
                for (int rr = 0; rr < 32; ++rr) R.bv[rr] = __ldg(px + (long long)rr * a.ldx + tcl);       // B: column t, rows 0..31
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) R.bx[jj] = __ldg(px + (long long)(4 * cs + jj) * a.ldx + kcl);   // B: columns 256 ..
                if (dz_owner) {                                            // dZ of the leftover rows (whole warps)
                    R.dzg = __ldg(a.grad_offset + (r0 + (t & 31)) * a.ld_off + n_left + (t >> 5));
                    R.dzo = __ldg(a.offset + (r0 + (t & 31)) * a.ld_off + n_left + (t >> 5));
                }
            } else {                                                       // last block of the split: row guards
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int rr = 4 * (ch + 2 * (e >> 2)) + (e & 3);
                    const bool ok = r0 + rr < rb;
                    R.ao[e] = ok ? __ldg(po + (long long)rr * a.ld_off) : 0.0f;
                    R.ag[e] = ok ? __ldg(pg + (long long)rr * a.ld_off) : 0.0f;
                }
#pragma unroll
                for (int rr = 0; rr < 32; ++rr) R.bv[rr] = r0 + rr < rb ? __ldg(px + (long long)rr * a.ldx + tcl) : 0.0f;
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) R.bx[jj] = r0 + 4 * cs + jj < rb ? __ldg(px + (long long)(4 * cs + jj) * a.ldx + kcl) : 0.0f;
                if (dz_owner && r0 + (t & 31) < rb) {
                    R.dzg = __ldg(a.grad_offset + (r0 + (t & 31)) * a.ld_off + n_left + (t >> 5));
                    R.dzo = __ldg(a.offset + (r0 + (t & 31)) * a.ld_off + n_left + (t >> 5));
                }
            }
        };
        auto process = [&](int kb, const Regs& R) {
            const int s = kb % kStages;
            unsigned char* At = smem + kOffRing + s * kStageBytes;
            unsigned char* Bt = At + kATileBytes;
            const long long r0 = ra + (long long)kb * BK;
            const bool full = r0 + BK <= rb;
            if (dz_owner) s_dz[((kb & 1) * kMaxSimtRows + (t >> 5)) * 32 + (t & 31)] = dact(R.dzg, R.dzo, a.act);   // dact(0, 0) = 0
            if (warp == 0 && kb > 0) issue_mma(kb - 1);
            if (kb >= kStages) mbar_wait(bar_empty + 8 * s, ((kb / kStages) - 1) & 1);   // the MMAs that read this stage are done
            // ---- A tile: dZ^T (rows of the tile past D_out: zero)
            const float nz = nvalid ? 1.0f : 0.0f;
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const int c = ch + 2 * h;
                *reinterpret_cast<float4*>(At + n * 128 + ((c ^ (n & 7)) << 4)) =
                    make_float4(to_tf32(nz * dact(R.ag[4 * h], R.ao[4 * h], a.act)), to_tf32(nz * dact(R.ag[4 * h + 1], R.ao[4 * h + 1], a.act)),
                                to_tf32(nz * dact(R.ag[4 * h + 2], R.ao[4 * h + 2], a.act)), to_tf32(nz * dact(R.ag[4 * h + 3], R.ao[4 * h + 3], a.act)));
            }
            // ---- B tile: xhat^T with the ones column at k = Din.  thread -> column k = t; the columns 256 .. b_rows - 1 are
            // shared out afterwards as (k = 256 + (t & 15), chunk t >> 4) over the first 128 threads
            const long long uq = r0 / a.n_frames;                          // utterance of the block's first row
            const int ul0 = (int)(uq - u_first);
            const int bnd = (int)((uq + 1) * a.n_frames - r0);             // rows of the block before the next utterance (n_frames >= 32)
            if (do_left) asm volatile("bar.sync 1, %0;" ::"n"(kProdThreads) : "memory");   // s_dz[kb & 1] is complete
            const float* dzb = s_dz + (kb & 1) * kMaxSimtRows * 32;
            if (kvalid) {
                const float2 st0 = s_stats[ul0 * kMaxBRows + t];
                const float2 st1 = bnd < BK ? s_stats[(ul0 + 1) * kMaxBRows + t] : st0;
                const float fill = t == a.Din ? 1.0f : 0.0f;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float w[4];
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int rr = 4 * c + jj;
                        const float2 st = rr >= bnd ? st1 : st0;
                        w[jj] = isx ? (R.bv[rr] - st.x) * st.y : fill;
                        if (!full && r0 + rr >= rb) w[jj] = 0.0f;
                    }
                    *reinterpret_cast<float4*>(Bt + t * 128 + ((c ^ (t & 7)) << 4)) =
                        make_float4(to_tf32(w[0]), to_tf32(w[1]), to_tf32(w[2]), to_tf32(w[3]));
                    if (do_left) {
#pragma unroll
                        for (int i = 0; i < kMaxSimtRows; ++i)
                            if (i < a.simt_rows) {
                                const float4 d = *reinterpret_cast<const float4*>(dzb + i * 32 + 4 * c);
                                acc_l[i] += w[0] * d.x + w[1] * d.y + w[2] * d.z + w[3] * d.w;
                            }
                    }
                }
            }
            if (has_shared) {
                const int k = ks, c = cs;
                const bool tx = k < a.Din;
                const float2 st0 = s_stats[ul0 * kMaxBRows + k];
                const float2 st1 = bnd < BK ? s_stats[(ul0 + 1) * kMaxBRows + k] : st0;
                const float fill = k == a.Din ? 1.0f : 0.0f;
                float w[4];
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) {
                    const int rr = 4 * c + jj;
                    const bool ok = full || r0 + rr < rb;
                    const float2 st = rr >= bnd ? st1 : st0;
                    w[jj] = !ok ? 0.0f : (tx ? (R.bx[jj] - st.x) * st.y : fill);
                }
                *reinterpret_cast<float4*>(Bt + k * 128 + ((c ^ (k & 7)) << 4)) =
                    make_float4(to_tf32(w[0]), to_tf32(w[1]), to_tf32(w[2]), to_tf32(w[3]));
                if (do_left) {
#pragma unroll
                    for (int i = 0; i < kMaxSimtRows; ++i)
                        if (i < a.simt_rows) {
                            const float4 d = *reinterpret_cast<const float4*>(dzb + i * 32 + 4 * c);
                            acc_t[i] += w[0] * d.x + w[1] * d.y + w[2] * d.z + w[3] * d.w;
                        }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the MMA
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_full + 8 * s);
        };
        Regs r_even, r_odd;
        if (nkb > 0) issue(0, r_even);
        for (int kb = 0; kb < nkb; kb += 2) {
            if (kb + 1 < nkb) issue(kb + 1, r_odd);
            process(kb, r_even);
            if (kb + 1 < nkb) {
                if (kb + 2 < nkb) issue(kb + 2, r_even);
                process(kb + 1, r_odd);
            }
        }
        if (warp == 0 && nkb > 0) {
            issue_mma(nkb - 1);
            if (lane == 0) umma_commit(bar_accum);
            __syncwarp();
        }
        if (do_left) {
            // partial rows n_left + i of this split: main columns straight from the registers, the shared-out columns
            // (256 ..) summed over their 8 chunk owners through shared memory
            float* dst = a.partials + ((long long)split * a.m_rows + n_left) * kMaxBRows;
            if (t < 16 * 8) {
#pragma unroll
                for (int i = 0; i < kMaxSimtRows; ++i) s_tail[(i * 16 + (t & 15)) * 8 + (t >> 4)] = acc_t[i];
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kProdThreads) : "memory");
#pragma unroll
            for (int i = 0; i < kMaxSimtRows; ++i)
                if (i < a.simt_rows) {
                    if (t < a.b_rows && t < kProdThreads) dst[(long long)i * kMaxBRows + t] = acc_l[i];
                    if (t < 16 && kProdThreads + t < a.b_rows) {
                        float sum = 0.0f;
#pragma unroll
                        for (int c = 0; c < 8; ++c) sum += s_tail[(i * 16 + t) * 8 + c];
                        dst[(long long)i * kMaxBRows + kProdThreads + t] = sum;
                    }
                }
        }
        // ===================== epilogue: the CTA's partial D -> workspace =====================
        if (nkb > 0) {
            mbar_wait(bar_accum, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        float* stage = reinterpret_cast<float*>(smem + kOffRing);
        const int quad = warp & 3, half = warp >> 2;
        const int row = quad * 32 + lane;
        const int ncol16 = a.b_rows / 16;
        const int c_lo = 16 * (half == 0 ? 0 : ncol16 / 2), c_hi = 16 * (half == 0 ? ncol16 / 2 : ncol16);
        for (int c0 = c_lo; c0 < c_hi; c0 += 16) {
            uint32_t acc[16];
            if (nkb > 0) tmem_ld16(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, acc);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4)
                *reinterpret_cast<float4*>(stage + row * kStageLd + c0 + jj) =
                    nkb > 0 ? make_float4(__uint_as_float(acc[jj]), __uint_as_float(acc[jj + 1]), __uint_as_float(acc[jj + 2]),
                                          __uint_as_float(acc[jj + 3]))
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kProdThreads) : "memory");
        float* dst = a.partials + ((long long)split * a.m_rows + n0) * kMaxBRows;
        for (int rr = warp; rr < BM; rr += kProdWarps)
            for (int c = lane; c < a.b_rows; c += 32) dst[(long long)rr * kMaxBRows + c] = stage[rr * kStageLd + c];
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------------------------
// TMA variant (aligned operands: row strides multiples of 4 floats, 16-byte aligned bases, at most one leftover output row).
// Both operands are row-major in r, the reduction index -- which is exactly the MN-MAJOR shared-memory layout of tcgen05
// (M / N contiguous, K strided): a TMA box of 32 rows x 32 floats with SWIZZLE_128B_ATOM_32B is one MN-major atom column (4-row K
// groups 512 B apart, 32-element M / N groups one box = 4096 B apart).  So nothing is transposed: TMA lands grad_offset,
// offset and x as they lie in HBM, the worker warps rewrite the tiles IN PLACE (dZ = grad * act'(offset), xhat = x * scale +
// shift with scale = 0 / shift = 1 in the ones column, TF32 rounding) with 128-bit shared-memory accesses, and the MMAs read
// them with the transpose bits of the instruction descriptor set.  Per 32-row block a CTA pulls 16 + 16 + <= 36 KB through
// TMA instead of ~70 scalar loads per thread (the LSU path could not keep enough bytes in flight: 4 us per block).
constexpr int kTStages = 3;
constexpr int kTBox = 32 * 32 * 4;                              // one TMA box: 32 rows x 128 B
constexpr int kTMaxXBoxes = 9;                                  // 288 columns >= 272
constexpr int kTOffG = 0, kTOffO = 4 * kTBox, kTOffX = 8 * kTBox;
constexpr int kTStageBytes = (8 + kTMaxXBoxes) * kTBox;         // 69 632
constexpr int kTStatLd = kTMaxXBoxes * 32;                      // 288
constexpr int kTOffScale = kTStages * kTStageBytes;             // [kMaxUtt][288]
constexpr int kTOffShift = kTOffScale + kMaxUtt * kTStatLd * 4;
constexpr int kTOffBar = kTOffShift + kMaxUtt * kTStatLd * 4;
constexpr int kTNumBars = 3 * kTStages + 1;                     // full, norm, empty per stage + accum
constexpr int kTOffTmem = kTOffBar + kTNumBars * 8;
constexpr int kTOffCoef = kTOffTmem + 16;                       // LOSS: [kMaxUtt] (c_t, c_s) + [kMaxUtt] valid frames + WSD threshold
constexpr int kTSmemBytes = kTOffCoef + kMaxUtt * 12 + 16;
// LOSS variants (an objective's backward folded in): stages of inp | offset | tar | x = 12 + 9 boxes, two of them
constexpr int kLStages = 2, kLOffT = 8 * kTBox, kLOffX = 12 * kTBox, kLStageBytes = (12 + kTMaxXBoxes) * kTBox;
static_assert(kLStages * kLStageBytes <= kTStages * kTStageBytes && BM * kStageLd * 4 <= kLStages * kLStageBytes, "LOSS ring inside the plain ring");
constexpr int kTWorkWarps = 16, kTWorkThreads = kTWorkWarps * 32, kTThreads = kTWorkThreads + 64;   // + MMA warp + TMA warp
// (16 worker warps: the in-place rewrite of a stage -- shared-memory round trips and MUFU latency -- is the critical path of a block, not TMA)
static_assert(kTSmemBytes <= 227 * 1024, "shared memory budget");
static_assert(BM * kStageLd * 4 <= kTStages * kTStageBytes && 32 * kTStatLd * 4 <= kTStages * kTStageBytes, "staging tiles fit in the ring");

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// MN-major TF32 operands have ONE legal shared-memory layout: the 128-byte swizzle with 32-byte atoms (layout type 1; TMA's
// CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): rows of 128 B = 32 consecutive M / N elements, the 32-byte unit index XORed with
// (row & 3), K groups of FOUR rows 512 B apart (stride offset), 32-element M / N groups one box = 4096 B apart (leading offset).
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)(kTBox >> 4) << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}
__device__ __forceinline__ uint32_t make_idesc_mn(int n) {        // as make_idesc, A and B MN-major (transpose bits 15, 16)
    return make_idesc(n) | (1u << 15) | (1u << 16);
}

// grad_offset of one element: predicted = o * x, target power t, c = sisdr_coef (objective_math.cuh)
__device__ __forceinline__ float sisdr_grad(float o, float x, float t, float2 c) {
    const float pi = o * x, tp = fmaxf(t, 0.0f);
    const float rs = rsqrtf(fmaxf(pi, 1e-37f));                              // one MUFU each instead of sqrt + divide
    const float ti = tp * rsqrtf(fmaxf(tp, 1e-37f));
    const float g = (c.x * ti + c.y * (pi * rs)) * (0.5f * rs) * x;
    return pi > 0.0f ? g : 0.0f;
}
constexpr int kLossNone = 0, kLossSisdr = 1, kLossWsd = 2;
// c: SISDR's per-utterance coefficients, or (1 if the row's frame is voiced else 0, unused) for WSD
template <int LOSS>
__device__ __forceinline__ float loss_grad(float o, float x, float t, float2 c, const BwdArgs& a) {
    return LOSS == kLossWsd ? wsd_grad(o, x, t, c.x != 0.0f, a.alpha, a.grad_uniform) : sisdr_grad(o, x, t, c);
}

template <int LOSS>
__global__ void __launch_bounds__(kTThreads, 1) linear_head_bwd_tma_kernel(const __grid_constant__ CUtensorMap tmG,
                                                                            const __grid_constant__ CUtensorMap tmO,
                                                                            const __grid_constant__ CUtensorMap tmX,
                                                                            const __grid_constant__ CUtensorMap tmT, const BwdArgs a) {
    constexpr int STAGES = LOSS ? kLStages : kTStages, STAGE_BYTES = LOSS ? kLStageBytes : kTStageBytes;
    constexpr int OFF_X = LOSS ? kLOffX : kTOffX;
    static_assert(LOSS == kLossNone || LOSS == kLossSisdr || LOSS == kLossWsd, "loss kind");
    extern __shared__ __align__(1024) unsigned char smem[];
    const uint32_t sbase = smem_u32(smem);
    float* s_scale = reinterpret_cast<float*>(smem + kTOffScale);
    float* s_shift = reinterpret_cast<float*>(smem + kTOffShift);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kTOffTmem);
    const uint32_t bar_full = sbase + kTOffBar, bar_norm = bar_full + 8 * kTStages, bar_empty = bar_norm + 8 * kTStages,
                   bar_accum = bar_empty + 8 * kTStages;
    float2* s_coef = reinterpret_cast<float2*>(smem + kTOffCoef);
    int* s_valid = reinterpret_cast<int*>(smem + kTOffCoef + kMaxUtt * 8);
    float* s_thres = reinterpret_cast<float*>(smem + kTOffCoef + kMaxUtt * 12);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int split = blockIdx.x, n0 = blockIdx.y * BM;
    long long ra = (long long)split * a.rows_per_split;
    long long rb = ra + a.rows_per_split < a.R ? ra + a.rows_per_split : a.R;
    if (a.sub > 0) {                                                   // per-utterance mode: split = (utterance, part of its frames)
        const long long u = split / a.sub, ue = (u + 1) * a.n_frames;
        ra = u * a.n_frames + (long long)(split - u * a.sub) * a.rows_per_split;
        rb = ra + a.rows_per_split < ue ? ra + a.rows_per_split : ue;
        if (ra > ue) ra = ue;
    }
    const int nkb = rb > ra ? (int)((rb - ra + BK - 1) / BK) : 0;
    const int nbx = (a.b_rows + 31) / 32;                              // x boxes per block

    if (threadIdx.x == 0) {
        if (sbase & 1023) __trap();
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_norm + 8 * s, kTWorkWarps);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kTWorkWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // xhat = x * scale + shift for the (at most kMaxUtt) utterances of this CTA's rows: scale = 1 / (std + eps), shift = -mean * scale;
    // column Din: scale 0, shift 1 (the ones column that makes grad_b column Din of D); columns past it: 0, 0
    const long long u_first = ra / a.n_frames;
    for (int i = threadIdx.x; i < kMaxUtt * kTStatLd; i += kTThreads) {
        const int ul = i / kTStatLd, k = i - ul * kTStatLd;
        const long long u = u_first + ul;
        float sc = k < a.Din ? 1.0f : 0.0f, sh = k == a.Din ? 1.0f : 0.0f;
        if (k < a.Din && u * a.n_frames < a.R) {
            if (a.mean) {
                sc = 1.0f / (__ldg(a.stdv + u * a.ld_stats + k) + a.cmvn_eps);
                sh = -__ldg(a.mean + u * a.ld_stats + k) * sc;
            } else if (a.sums) {                                       // same arithmetic as the fused forward head (head_fused.cu)
                const double2 p = *reinterpret_cast<const double2*>(a.sums + (u * a.ld_stats + k) * 2);
                const double mean = p.x * a.inv_n;
                const float var = (float)((p.y - p.x * mean) * a.inv_nm1);
                sc = __fdividef(1.0f, sqrtf(fmaxf(var, 0.0f)) + a.cmvn_eps);
                sh = -(float)mean * sc;
            }
        }
        s_scale[i] = sc;
        s_shift[i] = sh;
    }
    if (LOSS && threadIdx.x < kMaxUtt) {
        const long long u = u_first + threadIdx.x;
        float2 c = make_float2(0.f, 0.f);
        int valid = 0;
        if (u * a.n_frames < a.R) {
            if (LOSS == kLossSisdr)
                c = sisdr_coef(a.sums3 + 3 * u, (double)a.loss_eps, a.grad_out ? (double)a.grad_out[u] : (double)a.grad_uniform);
            long long v = a.n_frames;
            if (a.lengths) v = a.len_hop > 0 ? a.lengths[u] / a.len_hop + 1 : a.lengths[u];
            valid = (int)(v < a.n_frames ? v : a.n_frames);
        }
        s_coef[threadIdx.x] = c;
        s_valid[threadIdx.x] = valid;
        if (LOSS == kLossWsd && threadIdx.x == 0)                      // voicing threshold of the (all-reduced) batch maximum, once per CTA
            *s_thres = wsd_threshold(__ldg(a.max_energy), a.loss_eps, a.db_interval);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == kTWorkWarps + 1) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            const uint32_t tx = (uint32_t)((LOSS ? 12 : 8) + nbx) * kTBox;
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                if (kb >= STAGES) mbar_wait(bar_empty + 8 * s, ((kb / STAGES) - 1) & 1);
                const uint32_t st = sbase + s * STAGE_BYTES, bar = bar_full + 8 * s;
                const int r0 = (int)(ra + (long long)kb * BK);
                mbar_expect_tx(bar, tx);
                for (int m = 0; m < 4; ++m) {
                    tma_load_2d(st + kTOffG + m * kTBox, &tmG, n0 + 32 * m, r0, bar);       // grad_offset, or linear_inp (LOSS)
                    tma_load_2d(st + kTOffO + m * kTBox, &tmO, n0 + 32 * m, r0, bar);
                    if (LOSS) tma_load_2d(st + kLOffT + m * kTBox, &tmT, n0 + 32 * m, r0, bar);
                }
                for (int j = 0; j < nbx; ++j) tma_load_2d(st + OFF_X + j * kTBox, &tmX, 32 * j, r0, bar);
            }
        }
    } else if (warp == kTWorkWarps) {
        // ===================== MMA issuer =====================
        if (lane == 0 && nkb > 0) {
            const uint32_t idesc_main = make_idesc_mn(a.n_main), idesc_tail = make_idesc_mn(a.n_tail > 0 ? a.n_tail : 16);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                mbar_wait(bar_norm + 8 * s, (kb / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_addr = sbase + s * STAGE_BYTES + kTOffG, b_addr = sbase + s * STAGE_BYTES + OFF_X;
#pragma unroll
                for (int kk = 0; kk < BK / 8; ++kk) {                    // 8 rows of r per instruction = one 1024-byte K group
                    const uint64_t ad = make_desc_mn(a_addr + kk * 1024);
                    umma_tf32(tmem_base, ad, make_desc_mn(b_addr + kk * 1024), idesc_main, (kb | kk) ? 1u : 0u);
                    if (a.n_tail > 0)
                        umma_tf32(tmem_base + (uint32_t)a.n_main, ad, make_desc_mn(b_addr + (a.n_main / 32) * kTBox + kk * 1024),
                                  idesc_tail, (kb | kk) ? 1u : 0u);
                }
                umma_commit(bar_empty + 8 * s);
            }
            umma_commit(bar_accum);
        }
    } else {
        // ===================== workers: rewrite the landed tiles in place, then the epilogue =====================
        const int t = threadIdx.x, tl = t & 255, th = t >> 8;              // th: which half of the boxes this thread rewrites
        const int row = tl >> 3, pc = tl & 7, lc = pc ^ ((row & 3) << 1);  // this thread's row of every box, physical / logical 16-byte chunk
        const bool do_left = a.simt_rows > 0 && blockIdx.y == 0;           // leftover output row n_left (at most one here)
        const int n_left = a.m_tiles * BM;
        const float thres = LOSS == kLossWsd ? *s_thres : 0.0f;
        constexpr int kXPer = (kTMaxXBoxes + 1) / 2;                       // x boxes per thread: j = th, th + 2, ...
        float4 acc_l[kXPer];
#pragma unroll
        for (int j = 0; j < kXPer; ++j) acc_l[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            const long long r0 = ra + (long long)kb * BK;
            const long long uq = r0 / a.n_frames;
            const int bnd = (int)((uq + 1) * a.n_frames - r0);             // rows of the block before the next utterance (n_frames >= 32)
            const int ui = (int)(uq - u_first) + (row >= bnd ? 1 : 0);     // this row's utterance (index into the staged constants)
            const int so = ui * kTStatLd + 4 * lc;
            float live = r0 + row < rb ? 1.0f : 0.0f;                      // rows past the split (the next utterance's, per-utterance mode)
            float2 coef = make_float2(0.f, 0.f);
            if (LOSS) {                                                    // padded frames of the utterance carry no loss
                const int fr = (int)(r0 + row - (u_first + ui) * a.n_frames);
                if (fr >= s_valid[ui]) live = 0.0f;
                if (LOSS == kLossSisdr) {
                    coef = s_coef[ui];
                } else {                                                   // WSD: one voiced flag per row (frame)
                    const bool voiced = r0 + row < a.R && wsd_voiced(__ldg(a.energy + r0 + row), a.loss_eps, thres);
                    coef = make_float2(voiced ? 1.0f : 0.0f, 0.0f);
                }
            }
            float dzl = 0.0f;
            if (do_left && live != 0.0f) {                                 // in flight while the stage lands
                const float ol = __ldg(a.offset + (r0 + row) * a.ld_off + n_left);
                const float gl = LOSS ? loss_grad<LOSS>(ol, __ldg(a.inp + (r0 + row) * a.ld_inp + n_left), __ldg(a.tar + (r0 + row) * a.ld_tar + n_left), coef, a)
                                      : __ldg(a.grad_offset + (r0 + row) * a.ld_off + n_left);
                dzl = dact(gl, ol, a.act);
            }
            mbar_wait(bar_full + 8 * s, (kb / STAGES) & 1);
            float4* G = reinterpret_cast<float4*>(smem + s * STAGE_BYTES + kTOffG);
            const float4* O = reinterpret_cast<const float4*>(smem + s * STAGE_BYTES + kTOffO);
            const float4* Tt = reinterpret_cast<const float4*>(smem + s * STAGE_BYTES + kLOffT);
            float4* X = reinterpret_cast<float4*>(smem + s * STAGE_BYTES + OFF_X);
#pragma unroll
            for (int mi = 0; mi < 2; ++mi) {                               // dZ = grad * act'(offset); rows past R / columns past D_out landed as 0
                const int ci = tl + 256 * (th + 2 * mi);
                float4 g = G[ci];
                const float4 o = O[ci];
                if (LOSS) {                                                // G holds linear_inp: rebuild d loss / d offset first
                    const float4 tt = Tt[ci];
                    g = make_float4(loss_grad<LOSS>(o.x, g.x, tt.x, coef, a), loss_grad<LOSS>(o.y, g.y, tt.y, coef, a),
                                    loss_grad<LOSS>(o.z, g.z, tt.z, coef, a), loss_grad<LOSS>(o.w, g.w, tt.w, coef, a));
                }
                G[ci] = make_float4(to_tf32(live * dact(g.x, o.x, a.act)), to_tf32(live * dact(g.y, o.y, a.act)),
                                    to_tf32(live * dact(g.z, o.z, a.act)), to_tf32(live * dact(g.w, o.w, a.act)));
            }
#pragma unroll
            for (int ji = 0; ji < kXPer; ++ji) {
                const int j = th + 2 * ji;
                if (j < nbx) {
                    const float4 sc = *reinterpret_cast<const float4*>(s_scale + so + 32 * j);
                    const float4 sh = *reinterpret_cast<const float4*>(s_shift + so + 32 * j);
                    float4 v = X[tl + 256 * j];
                    v.x = to_tf32(fmaf(v.x, sc.x, sh.x));
                    v.y = to_tf32(fmaf(v.y, sc.y, sh.y));
                    v.z = to_tf32(fmaf(v.z, sc.z, sh.z));
                    v.w = to_tf32(fmaf(v.w, sc.w, sh.w));
                    if (r0 + row >= rb) v = make_float4(0.f, 0.f, 0.f, 0.f);   // (only the ones column matters: dZ of these rows is 0)
                    X[tl + 256 * j] = v;
                    if (do_left) {
                        acc_l[ji].x = fmaf(v.x, dzl, acc_l[ji].x);
                        acc_l[ji].y = fmaf(v.y, dzl, acc_l[ji].y);
                        acc_l[ji].z = fmaf(v.z, dzl, acc_l[ji].z);
                        acc_l[ji].w = fmaf(v.w, dzl, acc_l[ji].w);
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the MMA (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_norm + 8 * s);
        }
        if (nkb > 0) {
            mbar_wait(bar_accum, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        float* stage = reinterpret_cast<float*>(smem);                       // every stage has been consumed: reuse the ring
        if (do_left) {
            // partial row n_left of this split: column sums over the 32 rows of the per-thread accumulators
#pragma unroll
            for (int ji = 0; ji < kXPer; ++ji)
                if (th + 2 * ji < nbx) *reinterpret_cast<float4*>(stage + row * kTStatLd + 32 * (th + 2 * ji) + 4 * lc) = acc_l[ji];
            asm volatile("bar.sync 1, %0;" ::"n"(kTWorkThreads) : "memory");
            float* dst = a.partials + ((long long)split * a.m_rows + n_left) * kMaxBRows;
            for (int k = t; k < a.b_rows; k += kTWorkThreads) {
                float sum = 0.0f;
#pragma unroll 8
                for (int r = 0; r < 32; ++r) sum += stage[r * kTStatLd + k];
                dst[k] = sum;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(kTWorkThreads) : "memory");
        }
        // ---- epilogue: the CTA's partial D -> workspace
        const int quad = warp & 3, part = warp >> 2;                        // TMEM lane quadrant, quarter of the columns
        const int trow = quad * 32 + lane;
        const int ncol16 = a.b_rows / 16;
        const int c_lo = 16 * (ncol16 * part / (kTWorkWarps / 4)), c_hi = 16 * (ncol16 * (part + 1) / (kTWorkWarps / 4));
        for (int c0 = c_lo; c0 < c_hi; c0 += 16) {
            uint32_t acc[16];
            if (nkb > 0) tmem_ld16(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, acc);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4)
                *reinterpret_cast<float4*>(stage + trow * kStageLd + c0 + jj) =
                    nkb > 0 ? make_float4(__uint_as_float(acc[jj]), __uint_as_float(acc[jj + 1]), __uint_as_float(acc[jj + 2]),
                                          __uint_as_float(acc[jj + 3]))
                            : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTWorkThreads) : "memory");
        float* dst = a.partials + ((long long)split * a.m_rows + n0) * kMaxBRows;
        for (int rr = warp; rr < BM; rr += kTWorkWarps)
            for (int c = lane; c < a.b_rows; c += 32) dst[(long long)rr * kMaxBRows + c] = stage[rr * kStageLd + c];
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == kTWorkWarps) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
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

// 2-D fp32 tensor map: `cols` x `rows` elements, `ld` floats between rows, box = 32 floats x 32 rows, SWIZZLE_128B_ATOM_32B; elements
// outside [0, cols) x [0, rows) read as zero
bool make_map32(CUtensorMap* map, const float* base, long long cols, long long rows, long long ld) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    const cuuint32_t box[2] = {32, 32};
    const cuuint32_t estr[2] = {1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// grad_W[n, k] = sum_s partials[s, n, k], grad_b[n] = sum_s partials[s, n, Din]
__global__ void head_bwd_reduce_kernel(const float* __restrict__ partials, int splits, int m_rows, int Din, int Dout,
                                       float* __restrict__ grad_W, float* __restrict__ grad_b) {
    const int cols = Din + 1;
    const long long total = (long long)Dout * cols;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i / cols), k = (int)(i - (long long)n * cols);
        const float* p = partials + (long long)n * kMaxBRows + k;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int s = 0;
        const long long stride = (long long)m_rows * kMaxBRows;
        for (; s + 3 < splits; s += 4) {
            s0 += p[(long long)s * stride]; s1 += p[(long long)(s + 1) * stride];
            s2 += p[(long long)(s + 2) * stride]; s3 += p[(long long)(s + 3) * stride];
        }
        for (; s < splits; ++s) s0 += p[(long long)s * stride];
        const float v = (s0 + s1) + (s2 + s3);
        if (k < Din) grad_W[(long long)n * Din + k] = v;
        else if (grad_b) grad_b[n] = v;
    }
}

// per-utterance partials (n_utt, m_rows, 272) -> embeddings (n_utt, Dout * Din + Dout) = [grad_W.view(-1), grad_b] (sampler.py:95-108)
__global__ void head_grad_pack_kernel(const float* __restrict__ partials, int m_rows, int Din, int Dout, int sub, float* __restrict__ out) {
    const long long P = (long long)Dout * Din + Dout;
    const long long stride = (long long)m_rows * kMaxBRows;
    const float* src = partials + (long long)blockIdx.y * sub * stride;      // `sub` partials per utterance, summed in a fixed order
    float* dst = out + (long long)blockIdx.y * P;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
        const long long wn = (long long)Dout * Din;
        const int n = i < wn ? (int)(i / Din) : (int)(i - wn);
        const int k = i < wn ? (int)(i - (long long)n * Din) : Din;
        float v = src[(long long)n * kMaxBRows + k];
        for (int q = 1; q < sub; ++q) v += src[q * stride + (long long)n * kMaxBRows + k];
        dst[i] = v;
    }
}

int num_sms() { return secommon::device_sms(); }

struct Geometry { int m_tiles, simt_rows, m_rows, splits, sub; long long rows_per_split; };

// per_utt: one split per utterance (its partial IS that utterance's gradient: per-sample gradients for sampler.py:59-110)
bool plan(long long R, long long n_frames, long long Din, long long Dout, Geometry* g, bool per_utt = false) {
    if (R <= 0 || n_frames < BK || Din <= 0 || Dout <= 0 || Din + 1 > kMaxBRows) return false;
    const int rem = (int)(Dout % BM);
    g->simt_rows = (Dout > BM && rem > 0 && rem <= kMaxSimtRows) ? rem : 0;
    g->m_tiles = (int)((Dout - g->simt_rows + BM - 1) / BM);
    g->m_rows = g->m_tiles * BM + g->simt_rows;
    g->sub = 0;
    if (per_utt) {
        // one split per utterance, or up to 4 per utterance while the grid stays below one wave (few long utterances)
        const long long n_utt = R / n_frames;
        if (n_utt > 0x3fffffffLL) return false;
        long long sub = num_sms() / (n_utt * g->m_tiles);
        sub = sub < 1 ? 1 : (sub > 4 ? 4 : sub);
        long long rows = ((n_frames + sub - 1) / sub + BK - 1) / BK * BK;
        sub = (n_frames + rows - 1) / rows;
        g->sub = (int)sub;
        g->rows_per_split = rows;
        g->splits = (int)(n_utt * sub);
        return true;
    }
    long long splits = num_sms() / g->m_tiles;
    if (splits < 1) splits = 1;
    long long rows = (R + splits - 1) / splits;
    rows = (rows + BK - 1) / BK * BK;
    // a split may touch at most kMaxUtt utterances (their CMVN constants are staged in shared memory): large batches of short
    // utterances get more splits than one wave of CTAs instead of longer row ranges
    const long long max_rows = (kMaxUtt - 2) * n_frames / BK * BK;
    if (rows > max_rows) rows = max_rows;
    g->rows_per_split = rows;
    const long long n_splits = (R + rows - 1) / rows;
    if (n_splits > 65535) return false;
    g->splits = (int)n_splits;
    return (rows + n_frames - 1) / n_frames + 1 <= kMaxUtt;
}

}  // namespace

extern "C" {

int64_t se_linear_head_bwd_tc_workspace(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out) {
    Geometry g;
    if (!plan(n_utt * n_frames, n_frames, D_in, D_out, &g)) return 0;
    return (int64_t)g.splits * g.m_rows * kMaxBRows;
}

struct LossArgs {          // an objective's backward folded into the weight gradient (TMA kernel only)
    const float* inp; int64_t ld_inp; const float* tar; int64_t ld_tar; const double* sums3; const int64_t* lengths; int64_t len_hop;
    float eps, grad_uniform; const float* grad_out;
    int kind = kLossSisdr;                                     // kLossWsd: energy / max_energy / alpha / db_interval instead of sums3
    float alpha = 0.0f, db_interval = 0.0f; const float* energy = nullptr; const float* max_energy = nullptr;
};
static int head_bwd_impl(const float* x, int64_t ldx, const float* mean, const float* std, const double* stat_sums, int64_t ld_stats,
                         float cmvn_eps, const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt,
                         int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats,
                         float* grad_W, float* grad_b, void* stream, float* per_utt_out = nullptr, const LossArgs* loss = nullptr);

int se_linear_head_bwd_tc(const float* x, int64_t ldx, const float* mean, const float* std, int64_t ld_stats, float cmvn_eps,
                          const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt, int64_t n_frames,
                          int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W,
                          float* grad_b, void* stream) {
    SE_REQUIRE((mean == nullptr) == (std == nullptr), "mean and std go together");
    return head_bwd_impl(x, ldx, mean, std, nullptr, ld_stats, cmvn_eps, offset, grad_offset, ld_off, n_utt, n_frames, D_in, D_out,
                         act, ws_partials, ws_floats, grad_W, grad_b, stream);
}

int se_linear_head_bwd_fused(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps,
                             const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt, int64_t n_frames,
                             int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W,
                             float* grad_b, void* stream) {
    SE_REQUIRE(!stat_sums || n_frames >= 2, "CMVN statistics need at least two frames");
    return head_bwd_impl(x, ldx, nullptr, nullptr, stat_sums, ld_stats, cmvn_eps, offset, grad_offset, ld_off, n_utt, n_frames, D_in,
                         D_out, act, ws_partials, ws_floats, grad_W, grad_b, stream);
}

int64_t se_head_grad_embeddings_workspace(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out) {
    Geometry g;
    if (!plan(n_utt * n_frames, n_frames, D_in, D_out, &g, true)) return 0;
    return (int64_t)g.splits * g.m_rows * kMaxBRows;
}

int se_head_grad_embeddings(const float* x, int64_t ldx, const float* mean, const float* std, const double* stat_sums,
                            int64_t ld_stats, float cmvn_eps, const float* offset, const float* grad_offset, int64_t ld_off,
                            int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws, int64_t ws_floats,
                            float* grads_out, void* stream) {
    SE_REQUIRE(grads_out, "null pointer");
    SE_REQUIRE((mean == nullptr) == (std == nullptr) && !(mean && stat_sums), "CMVN: give mean and std, or stat_sums, or neither");
    return head_bwd_impl(x, ldx, mean, std, stat_sums, ld_stats, cmvn_eps, offset, grad_offset, ld_off, n_utt, n_frames, D_in, D_out,
                         act, ws, ws_floats, nullptr, nullptr, stream, grads_out);
}

int se_linear_head_bwd_sisdr_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                       int64_t ld_inp, int64_t ld_tar) {
    Geometry g;
    if (!plan(n_utt * n_frames, n_frames, D_in, D_out, &g)) return 0;
    return (g.simt_rows <= 1 && ldx % 4 == 0 && ld_off % 4 == 0 && ld_inp % 4 == 0 && ld_tar % 4 == 0 && n_utt * n_frames < 0x7fffffffLL) ? 1 : 0;
}

int se_linear_head_bwd_sisdr(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                             int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                             const int64_t* lengths, int64_t len_hop, const double* sums3, float loss_eps, int64_t n_utt, int64_t n_frames,
                             int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W, float* grad_b,
                             void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && sums3 && grad_W, "null pointer");
    SE_REQUIRE(ld_inp >= D_out && ld_tar >= D_out && len_hop >= 0 && len_hop < (1LL << 30), "bad stride / hop");
    SE_REQUIRE(!stat_sums || n_frames >= 2, "CMVN statistics need at least two frames");
    LossArgs l{linear_inp, ld_inp, linear_tar, ld_tar, sums3, lengths, len_hop, loss_eps, 1.0f / (float)n_utt, nullptr};
    return head_bwd_impl(x, ldx, nullptr, nullptr, stat_sums, ld_stats, cmvn_eps, offset, nullptr, ld_off, n_utt, n_frames, D_in, D_out, act,
                         ws_partials, ws_floats, grad_W, grad_b, stream, nullptr, &l);
}

int se_linear_head_bwd_wsd_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                     int64_t ld_inp, int64_t ld_tar) {
    return se_linear_head_bwd_sisdr_supported(n_utt, n_frames, D_in, D_out, ldx, ld_off, ld_inp, ld_tar);   // same kernel, same operands
}

int se_linear_head_bwd_wsd(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                           int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                           const int64_t* lengths, int64_t len_hop, const float* energy, const float* max_energy, float alpha,
                           float db_interval, float loss_eps, int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act,
                           float* ws_partials, int64_t ws_floats, float* grad_W, float* grad_b, void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && energy && max_energy && grad_W, "null pointer");
    SE_REQUIRE(ld_inp >= D_out && ld_tar >= D_out && len_hop >= 0 && len_hop < (1LL << 30), "bad stride / hop");
    SE_REQUIRE(!stat_sums || n_frames >= 2, "CMVN statistics need at least two frames");
    LossArgs l{linear_inp, ld_inp, linear_tar, ld_tar, nullptr, lengths, len_hop, loss_eps, 1.0f / (float)n_utt, nullptr,
               kLossWsd, alpha, db_interval, energy, max_energy};
    return head_bwd_impl(x, ldx, nullptr, nullptr, stat_sums, ld_stats, cmvn_eps, offset, nullptr, ld_off, n_utt, n_frames, D_in, D_out, act,
                         ws_partials, ws_floats, grad_W, grad_b, stream, nullptr, &l);
}

int se_head_grad_embeddings_sisdr_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                            int64_t ld_inp, int64_t ld_tar) {
    Geometry g;
    if (!plan(n_utt * n_frames, n_frames, D_in, D_out, &g, true)) return 0;
    return (g.simt_rows <= 1 && ldx % 4 == 0 && ld_off % 4 == 0 && ld_inp % 4 == 0 && ld_tar % 4 == 0 && n_utt * n_frames < 0x7fffffffLL) ? 1 : 0;
}

int se_head_grad_embeddings_sisdr(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                                  int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                                  const int64_t* lengths, int64_t len_hop, const double* sums3, float loss_eps, int64_t n_utt,
                                  int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws, int64_t ws_floats, float* grads_out,
                                  void* stream) {
    SE_REQUIRE(linear_inp && linear_tar && sums3 && grads_out, "null pointer");
    SE_REQUIRE(ld_inp >= D_out && ld_tar >= D_out && len_hop >= 0 && len_hop < (1LL << 30), "bad stride / hop");
    SE_REQUIRE(!stat_sums || n_frames >= 2, "CMVN statistics need at least two frames");
    LossArgs l{linear_inp, ld_inp, linear_tar, ld_tar, sums3, lengths, len_hop, loss_eps, 1.0f, nullptr};   // row u: gradient of loss_u alone
    return head_bwd_impl(x, ldx, nullptr, nullptr, stat_sums, ld_stats, cmvn_eps, offset, nullptr, ld_off, n_utt, n_frames, D_in, D_out, act,
                         ws, ws_floats, nullptr, nullptr, stream, grads_out, &l);
}

static int head_bwd_impl(const float* x, int64_t ldx, const float* mean, const float* std, const double* stat_sums, int64_t ld_stats,
                         float cmvn_eps, const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt,
                         int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats,
                         float* grad_W, float* grad_b, void* stream, float* per_utt_out, const LossArgs* loss) {
    SE_REQUIRE(x && offset && (grad_offset || loss) && ws_partials && (grad_W || per_utt_out) && n_utt > 0 && n_frames > 0, "bad argument");
    SE_REQUIRE(ldx >= D_in && ld_off >= D_out && ((!mean && !stat_sums) || ld_stats >= D_in), "row stride smaller than the row");
    SE_REQUIRE(act >= SE_ACT_IDENTITY && act <= SE_ACT_SIGMOID, "unknown activation %d", act);
    Geometry g;
    if (!plan(n_utt * n_frames, n_frames, D_in, D_out, &g, per_utt_out != nullptr))
        return fail(SE_ERR_UNSUPPORTED, "tensor-core head backward: shape outside its range (D_in=%lld, n_frames=%lld)",
                    (long long)D_in, (long long)n_frames);
    SE_REQUIRE(ws_floats >= (int64_t)g.splits * g.m_rows * kMaxBRows, "workspace too small");
    BwdArgs a{};
    a.x = x; a.ldx = ldx; a.mean = mean; a.stdv = std; a.ld_stats = ld_stats; a.cmvn_eps = cmvn_eps;
    a.sums = stat_sums; a.inv_n = 1.0 / (double)n_frames; a.inv_nm1 = n_frames > 1 ? 1.0 / (double)(n_frames - 1) : 0.0;
    a.offset = offset; a.grad_offset = grad_offset; a.ld_off = ld_off;
    a.R = n_utt * n_frames; a.n_frames = (int)n_frames; a.Din = (int)D_in; a.Dout = (int)D_out; a.act = act;
    a.rows_per_split = g.rows_per_split; a.sub = g.sub;
    a.b_rows = (int)((D_in + 1 + 15) / 16 * 16);
    a.n_main = a.b_rows > 256 ? 256 : a.b_rows;
    a.n_tail = a.b_rows - a.n_main;
    a.partials = ws_partials;
    a.m_rows = g.m_rows; a.m_tiles = g.m_tiles; a.simt_rows = g.simt_rows;
    static unsigned long long opted = 0;                       // per device: cudaFuncSetAttribute is not process-wide
    if (secommon::first_use_on_device(opted)) {
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    }
    cudaStream_t st = (cudaStream_t)stream;
    // aligned operands (the engine's padded tensors): the TMA / MN-major kernel; anything else: the transposing producers
    const float* gsrc = loss ? loss->inp : grad_offset;
    const int64_t ld_g = loss ? loss->ld_inp : ld_off;
    bool aligned = ldx % 4 == 0 && ld_off % 4 == 0 && ld_g % 4 == 0 &&
                   ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(offset) | reinterpret_cast<uintptr_t>(gsrc)) & 15) == 0;
    if (loss) aligned = aligned && loss->ld_tar % 4 == 0 && (reinterpret_cast<uintptr_t>(loss->tar) & 15) == 0;
    CUtensorMap tmG, tmO, tmX, tmT;
    int rc;
    const bool tma_ok = aligned && g.simt_rows <= 1 && a.R < 0x7fffffffLL && make_map32(&tmG, gsrc, D_out, a.R, ld_g) &&
                        make_map32(&tmO, offset, D_out, a.R, ld_off) && make_map32(&tmX, x, D_in, a.R, ldx) &&
                        (!loss || make_map32(&tmT, loss->tar, D_out, a.R, loss->ld_tar));
    if (loss) {
        if (!tma_ok) return fail(SE_ERR_UNSUPPORTED, "head backward with the objective folded in: operands must be 16-byte aligned with row "
                                                     "strides that are multiples of 4 floats");
        a.inp = loss->inp; a.ld_inp = loss->ld_inp; a.tar = loss->tar; a.ld_tar = loss->ld_tar; a.sums3 = loss->sums3;
        a.lengths = (const long long*)loss->lengths; a.len_hop = (int)loss->len_hop; a.loss_eps = loss->eps;
        a.grad_uniform = loss->grad_uniform; a.grad_out = loss->grad_out;
        a.alpha = loss->alpha; a.db_interval = loss->db_interval; a.energy = loss->energy; a.max_energy = loss->max_energy;
    }
    static unsigned long long opted_t = 0;
    if (tma_ok && secommon::first_use_on_device(opted_t)) {
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_bwd_tma_kernel<kLossNone>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTSmemBytes));
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_bwd_tma_kernel<kLossSisdr>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTSmemBytes));
        SE_CUDA_CHECK(cudaFuncSetAttribute(linear_head_bwd_tma_kernel<kLossWsd>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTSmemBytes));
    }
    if (loss && loss->kind == kLossWsd) {
        linear_head_bwd_tma_kernel<kLossWsd><<<dim3((unsigned)g.splits, (unsigned)g.m_tiles), kTThreads, kTSmemBytes, st>>>(tmG, tmO, tmX, tmT, a);
        rc = secommon::check_launch("linear_head_bwd_tma_kernel<wsd>");
    } else if (loss) {
        linear_head_bwd_tma_kernel<kLossSisdr><<<dim3((unsigned)g.splits, (unsigned)g.m_tiles), kTThreads, kTSmemBytes, st>>>(tmG, tmO, tmX, tmT, a);
        rc = secommon::check_launch("linear_head_bwd_tma_kernel<loss>");
    } else if (tma_ok) {
        linear_head_bwd_tma_kernel<kLossNone><<<dim3((unsigned)g.splits, (unsigned)g.m_tiles), kTThreads, kTSmemBytes, st>>>(tmG, tmO, tmX, tmX, a);
        rc = secommon::check_launch("linear_head_bwd_tma_kernel");
    } else {
        linear_head_bwd_tc_kernel<<<dim3((unsigned)g.splits, (unsigned)g.m_tiles), kThreads, kSmemBytes, st>>>(a);
        rc = secommon::check_launch("linear_head_bwd_tc_kernel");
    }
    if (rc != SE_OK) return rc;
    const long long total = D_out * (D_in + 1);
    if (per_utt_out) {
        head_grad_pack_kernel<<<dim3((unsigned)((total + 1023) / 1024), (unsigned)n_utt), 256, 0, st>>>(ws_partials, a.m_rows, (int)D_in,
                                                                                                      (int)D_out, g.sub, per_utt_out);
        return secommon::check_launch("head_grad_pack_kernel");
    }
    head_bwd_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ws_partials, g.splits, a.m_rows, (int)D_in, (int)D_out,
                                                                          grad_W, grad_b);
    return secommon::check_launch("head_bwd_reduce_kernel");
}

}  // extern "C"
