// Register-resident 256-point complex FFT executed by 16 lanes x 16 values, the building block of the n_fft 512 and
// n_fft 1024 cores of fastgeo.cu (Core<Geo512>: one transform per group of 16 lanes, two groups per warp; Core<Geo1024>:
// two transforms per warp plus a radix-2 exchange).
//
//   256 = 16 x 16:  radix-16 in registers -> one transpose through shared memory -> twiddle ->
//   radix-16 in registers.  Lane j holds z[j + 16 r] (r = 0..15) on entry and Z[j + 16 q] on exit.
//
// The transpose buffer is 16 rows x 128 B per transform.  Lane j writes its row with 8 STS.128 whose
// 16-byte chunk index is XOR-swizzled with (j & 7); lane j' then reads column j' of every row with 16
// LDS.64.  Both patterns touch all 32 banks exactly once per 128 B wavefront (no bank conflicts).  Every
// lane of the warp runs a transform in lock-step, so the barriers and shuffles use the full warp mask.
//
// The real-input split needs Z[M-k] next to Z[k]: with k = j + 16 q that value lives in lane
// (16 - j) mod 16 of the same group, register 15 - q (lane 0: register (16 - q) mod 16), so it is fetched
// with one shuffle per value and no shared memory.
#pragma once
#include "fft_core.cuh"

namespace fft256w {
using namespace sefft;

constexpr unsigned kFull = 0xffffffffu;

// per-lane constants: tw[r-1] = exp(-2*pi*i*r*j/256) (r = 1..15), twn[q] = exp(-2*pi*i*(j+16q)/512) (q < 8)
__device__ __forceinline__ void load_lane_constants(int j, const float2* __restrict__ twM, const float2* __restrict__ twN,
                                                    float2 (&tw)[15], float2 (&twn)[8]) {
#pragma unroll
    for (int r = 1; r < 16; ++r) tw[r - 1] = twM[r * j];
#pragma unroll
    for (int q = 0; q < 8; ++q) twn[q] = twN[j + 16 * q];
}

template <int DIR>
__device__ __forceinline__ void fft256(float2 (&v)[16], float2* __restrict__ xbuf, int j, const float2 (&tw)[15]) {
    bfly16<DIR>(v);
    float4* row = reinterpret_cast<float4*>(xbuf) + j * 8;
#pragma unroll
    for (int c = 0; c < 8; ++c) row[c ^ (j & 7)] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = xbuf[r * 16 + ((((j >> 1) ^ (r & 7)) << 1) | (j & 1))];
    __syncwarp();
#pragma unroll
    for (int r = 1; r < 16; ++r) {
        float2 w = tw[r - 1];
        if (DIR > 0) w.y = -w.y;
        v[r] = cmul(v[r], w);
    }
    bfly16<DIR>(v);
}

// zm[q] = Z[256 - (j + 16 q)] for q < 8, given v[q] = Z[j + 16 q] in every lane of the 16-lane group
__device__ __forceinline__ void fetch_mirror(const float2 (&v)[16], int lane, float2 (&zm)[8]) {
    const int j = lane & 15;
    const int src = (lane & 16) | ((16 - j) & 15);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const float2 offer = (j == 0) ? v[(16 - q) & 15] : v[15 - q];
        zm[q].x = __shfl_sync(kFull, offer.x, src);
        zm[q].y = __shfl_sync(kFull, offer.y, src);
    }
}

// Inverse of the above for values: every lane computed b[q] = W[256 - (j + 16 q)] (q < 8) next to its own
// a[q] = W[j + 16 q]; afterwards v[0..15] = W[j + 16 q] for all q.  w128 = W[128] (used by lane 0 only).
__device__ __forceinline__ void scatter_mirror(const float2 (&a)[8], const float2 (&b)[8], float2 w128, int lane, float2 (&v)[16]) {
    const int j = lane & 15;
    const int src = (lane & 16) | ((16 - j) & 15);
    float2 rcv[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        rcv[q].x = __shfl_sync(kFull, b[q].x, src);          // = W[j + 16 (15 - q)]   (lane 0: W[16 (16 - q)])
        rcv[q].y = __shfl_sync(kFull, b[q].y, src);
        v[q] = a[q];
    }
#pragma unroll
    for (int q = 0; q < 7; ++q) v[15 - q] = (j == 0) ? rcv[q + 1] : rcv[q];
    v[8] = (j == 0) ? w128 : rcv[7];
}

}  // namespace fft256w
