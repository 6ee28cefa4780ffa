// The 256-point 16-lane FFT of the fast paths in isolation (no global memory in the loop): time per transform against the
// number of resident warps.  nvcc -arch=sm_100a -O3 -std=c++17 -I../../speech_enhancement_by_s3prl_b200/csrc -I../../include -o fft_loop fft_loop.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "fft256_warp.cuh"
using namespace fft256w;
constexpr int ITERS = 512;
template <int MODE> __global__ void __launch_bounds__(128) k(const float2* twM, const float2* twN, float2* out, float seed) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, j = lane & 15, hw = threadIdx.x >> 4;
    float2* xbuf = reinterpret_cast<float2*>(smem) + hw * 256;
    float2 tw[15], twn[8];
    load_lane_constants(j, twM, twN, tw, twn);
    float2 v[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = make_float2(seed * (j + 16 * r), seed);
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it) {
        if (MODE == 0) fft256<-1>(v, xbuf, j, tw);
        if (MODE == 1) { bfly16<-1>(v); bfly16<-1>(v); }                       // butterflies only (no transpose, no twiddles)
        if (MODE == 2) {                                                        // twiddles only
#pragma unroll
            for (int r = 1; r < 16; ++r) v[r] = cmul(v[r], tw[r - 1]);
        }
        if (MODE == 3) {                                                        // transpose only
            float4* row = reinterpret_cast<float4*>(xbuf) + j * 8;
#pragma unroll
            for (int c = 0; c < 8; ++c) row[c ^ (j & 7)] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
            __syncwarp();
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = xbuf[r * 16 + ((((j >> 1) ^ (r & 7)) << 1) | (j & 1))];
            __syncwarp();
        }
    }
    float2 s = make_float2(0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 16; ++r) s = cadd(s, v[r]);
    if (s.x == 123.456f) out[threadIdx.x] = s;
}
template <int MODE> void run(const char* name, const float2* twM, const float2* twN, int ctas_per_sm) {
    int sms; cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
    int clk; cudaDeviceGetAttribute(&clk, cudaDevAttrClockRate, 0);
    float2* out; cudaMalloc(&out, 1024);
    const size_t smem = 8 * 256 * 8 + (ctas_per_sm == 1 ? 120 : ctas_per_sm == 2 ? 90 : ctas_per_sm == 3 ? 52 : 30) * 1024;  // caps residency
    cudaFuncSetAttribute(k<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    k<MODE><<<sms * ctas_per_sm, 128, smem>>>(twM, twN, out, 1e-3f); cudaDeviceSynchronize();
    cudaEventRecord(e0);
    for (int r = 0; r < 5; ++r) k<MODE><<<sms * ctas_per_sm, 128, smem>>>(twM, twN, out, 1e-3f);
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= 5;
    const double cycles = ms * 1e-3 * clk * 1e3;
    // per SM: ctas_per_sm * 8 half-warps * ITERS transforms
    printf("%-32s %d CTA/SM (%2d warps): %7.3f ms  %7.1f SM-cycles per transform  (%6.0f cycles per warp-iteration)\n", name, ctas_per_sm,
           4 * ctas_per_sm, ms, cycles / (ctas_per_sm * 8.0 * ITERS), cycles / ITERS);
}
int main() {
    float2 h[512];
    for (int i = 0; i < 512; ++i) h[i] = make_float2(cosf(-6.2831853f * i / 256), sinf(-6.2831853f * i / 256));
    float2 *twM, *twN; cudaMalloc(&twM, sizeof(h)); cudaMalloc(&twN, sizeof(h));
    cudaMemcpy(twM, h, sizeof(h), cudaMemcpyHostToDevice); cudaMemcpy(twN, h, sizeof(h), cudaMemcpyHostToDevice);
    for (int c : {1, 2, 3, 4}) {
        run<0>("fft256", twM, twN, c);
        run<1>("2 x bfly16", twM, twN, c);
        run<2>("15 twiddle cmul", twM, twN, c);
        run<3>("transpose (8 STS.128+16 LDS.64)", twM, twN, c);
    }
    return 0;
}
