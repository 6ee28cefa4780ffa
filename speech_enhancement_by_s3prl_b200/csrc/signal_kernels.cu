// libse_b200.so -- STFT / iSTFT / fused mask->iSTFT entry points (generic tile path).
// The per-CTA bodies live in tile_kernels.cuh (shared with the CPU test harness); this file
// supplies the CTA executor, the __global__ wrappers, the per-device twiddle tables and the
// extern "C" functions declared in include/se_b200.h.
#include <map>
#include <mutex>
#include <vector>
#include "se_common.cuh"
#include "tile_kernels.cuh"
#include "host_plan.h"

using namespace sekern;
using secommon::fail;

namespace sefast {
// fastgeo.cu: n_fft 512 / hop 256, n_fft 1024 / hop 256 and n_fft 400 / hop 160
bool geo_supported(int n_fft, int hop);
int prepare_geo_kernels(int n_fft);
int launch_stft_run(const StftArgs& a, int n_fft, cudaStream_t st);
int launch_mask_istft_run(const MaskIstftArgs& a, int n_fft, cudaStream_t st);
}

namespace {

struct BlockExec {
    template <class F> __device__ __forceinline__ void foreach(int n, F f) {
        for (int w = threadIdx.x; w < n; w += blockDim.x) f(w);
    }
    __device__ __forceinline__ void sync() { __syncthreads(); }
    template <int NS> __device__ __forceinline__ void block_accumulate(const float* acc, double* dst) {
        secommon::block_accumulate_to<NS, float>(acc, dst);
    }
};

template <int N> __global__ void __launch_bounds__(Cfg<N>::THREADS) stft_kernel(StftArgs a, int tiles) {
    extern __shared__ __align__(16) unsigned char smem[];
    BlockExec ex;
    const int utt = blockIdx.x / tiles, tile = blockIdx.x - utt * tiles;
    stft_tile<N>(ex, a, utt, tile, smem);
}
template <int N> __global__ void __launch_bounds__(Cfg<N>::THREADS) istft_kernel(IstftArgs a, int tiles) {
    extern __shared__ __align__(16) unsigned char smem[];
    BlockExec ex;
    const int utt = blockIdx.x / tiles, tile = blockIdx.x - utt * tiles;
    istft_tile<N>(ex, a, utt, tile, smem);
}
template <int N> __global__ void __launch_bounds__(Cfg<N>::THREADS) mask_istft_kernel(MaskIstftArgs a, int tiles) {
    extern __shared__ __align__(16) unsigned char smem[];
    BlockExec ex;
    const int utt = blockIdx.x / tiles, tile = blockIdx.x - utt * tiles;
    mask_istft_tile<N>(ex, a, utt, tile, smem);
}

// ------------------------------------------------------------------ per-device tables
struct DeviceTables { float2* twM = nullptr; float2* twN = nullptr; };
std::mutex g_mu;
std::map<std::pair<int, int>, DeviceTables> g_tables;      // (device, n_fft)
constexpr size_t kMaxSmem = 200 * 1024;

template <int N> int opt_in_smem() {
    SE_CUDA_CHECK(cudaFuncSetAttribute(stft_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    SE_CUDA_CHECK(cudaFuncSetAttribute(istft_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    SE_CUDA_CHECK(cudaFuncSetAttribute(mask_istft_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem));
    return SE_OK;
}

int get_tables(int n_fft, DeviceTables* out) {
    if (!seplan::supported_nfft(n_fft)) return fail(SE_ERR_UNSUPPORTED, "n_fft=%d has no kernel (supported: 256, 400, 512, 1024, 2048)", n_fft);
    int dev = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(SE_ERR_NO_DEVICE, "no CUDA device: %s (libse_b200 has no CPU fallback)", cudaGetErrorString(e));
    std::lock_guard<std::mutex> lock(g_mu);
    auto key = std::make_pair(dev, n_fft);
    auto it = g_tables.find(key);
    if (it == g_tables.end()) {
        std::vector<float> twM, twN;
        seplan::make_twiddles(n_fft, twM, twN);
        DeviceTables t;
        SE_CUDA_CHECK(cudaMalloc(&t.twM, twM.size() * sizeof(float)));
        SE_CUDA_CHECK(cudaMalloc(&t.twN, twN.size() * sizeof(float)));
        SE_CUDA_CHECK(cudaMemcpy(t.twM, twM.data(), twM.size() * sizeof(float), cudaMemcpyHostToDevice));
        SE_CUDA_CHECK(cudaMemcpy(t.twN, twN.data(), twN.size() * sizeof(float), cudaMemcpyHostToDevice));
        int rc = SE_OK;
        switch (n_fft) {
            case 256: rc = opt_in_smem<256>(); break;
            case 400: rc = opt_in_smem<400>(); if (rc == SE_OK) rc = sefast::prepare_geo_kernels(400); break;
            case 512: rc = opt_in_smem<512>(); if (rc == SE_OK) rc = sefast::prepare_geo_kernels(512); break;
            case 1024: rc = opt_in_smem<1024>(); if (rc == SE_OK) rc = sefast::prepare_geo_kernels(1024); break;
            case 2048: rc = opt_in_smem<2048>(); break;
        }
        if (rc != SE_OK) return rc;
        it = g_tables.emplace(key, t).first;
    }
    *out = it->second;
    return SE_OK;
}

template <int N> int launch_stft(StftArgs a, cudaStream_t st) {
    constexpr int G = Cfg<N>::G;
    const int tiles = (a.n_frames + G - 1) / G;
    const size_t smem = Smem<N>::bytes((G - 1) * a.hop + N, 0);
    if (smem > kMaxSmem) return fail(SE_ERR_UNSUPPORTED, "hop=%d needs %zu B of shared memory", a.hop, smem);
    const long long blocks = (long long)a.n_utt * tiles;
    if (blocks > 0x7fffffffLL) return fail(SE_ERR_BAD_ARG, "grid too large");
    stft_kernel<N><<<(unsigned)blocks, Cfg<N>::THREADS, smem, st>>>(a, tiles);
    return secommon::check_launch("stft_kernel");
}
template <int N> int launch_istft(IstftArgs a, cudaStream_t st) {
    constexpr int G = Cfg<N>::G;
    a.tile_len = seplan::inverse_tile_len(N, a.hop, G);
    if (a.tile_len <= 0) return fail(SE_ERR_UNSUPPORTED, "hop=%d too small for n_fft=%d", a.hop, N);
    const int tiles = seplan::inverse_num_tiles(a.out_len, a.pad_to, a.tile_len);
    const size_t smem = Smem<N>::bytes(0, 0);
    const long long blocks = (long long)a.n_utt * tiles;
    if (blocks > 0x7fffffffLL) return fail(SE_ERR_BAD_ARG, "grid too large");
    istft_kernel<N><<<(unsigned)blocks, Cfg<N>::THREADS, smem, st>>>(a, tiles);
    return secommon::check_launch("istft_kernel");
}
template <int N> int launch_mask_istft(MaskIstftArgs a, cudaStream_t st) {
    constexpr int G = Cfg<N>::G;
    a.tile_len = seplan::inverse_tile_len(N, a.hop, G);
    if (a.tile_len <= 0) return fail(SE_ERR_UNSUPPORTED, "hop=%d too small for n_fft=%d", a.hop, N);
    const int tiles = seplan::inverse_num_tiles(a.out_len, a.pad_to, a.tile_len);
    const size_t smem = Smem<N>::bytes((G - 1) * a.hop + N, a.want_spec ? G * (N / 2 + 1) : 0);
    if (smem > kMaxSmem) return fail(SE_ERR_UNSUPPORTED, "hop=%d needs %zu B of shared memory", a.hop, smem);
    const long long blocks = (long long)a.n_utt * tiles;
    if (blocks > 0x7fffffffLL) return fail(SE_ERR_BAD_ARG, "grid too large");
    mask_istft_kernel<N><<<(unsigned)blocks, Cfg<N>::THREADS, smem, st>>>(a, tiles);
    return secommon::check_launch("mask_istft_kernel");
}

#define SE_DISPATCH_NFFT(n_fft, FN, ...)                 \
    switch (n_fft) {                                     \
        case 256: return FN<256>(__VA_ARGS__);           \
        case 400: return FN<400>(__VA_ARGS__);           \
        case 512: return FN<512>(__VA_ARGS__);           \
        case 1024: return FN<1024>(__VA_ARGS__);         \
        case 2048: return FN<2048>(__VA_ARGS__);         \
        default: return fail(SE_ERR_UNSUPPORTED, "n_fft=%d has no kernel", n_fft); \
    }

int check_geometry(int64_t n_utt, int64_t T, int n_fft, int hop) {
    SE_REQUIRE(n_utt > 0 && T > 0, "n_utt=%lld and T=%lld must be positive", (long long)n_utt, (long long)T);
    SE_REQUIRE(hop > 0 && hop <= n_fft, "hop=%d must be in [1, n_fft=%d]", hop, n_fft);
    SE_REQUIRE(T > n_fft / 2, "T=%lld must exceed n_fft/2=%d (reflect padding, as torch.stft requires)", (long long)T, n_fft / 2);
    SE_REQUIRE(T < (1LL << 30), "T=%lld too long", (long long)T);
    return SE_OK;
}

}  // namespace

static int g_force_generic = 0;

extern "C" {

int se_version(void) { return 100; }

int se_set_option(int key, int value) {
    if (key == SE_OPT_FORCE_GENERIC) { g_force_generic = value; return SE_OK; }
    return fail(SE_ERR_BAD_ARG, "unknown option %d", key);
}

int se_set_trace(unsigned long long* d_buf) {
    secommon::trace_ptr() = d_buf;
    return SE_OK;
}

int se_last_error(char* h_buf, int n) {
    if (!h_buf || n <= 0) return SE_ERR_BAD_ARG;
    strncpy(h_buf, secommon::last_error_buf(), (size_t)n);
    h_buf[n - 1] = 0;
    return SE_OK;
}

int se_prepare(int n_fft) {
    DeviceTables t;
    return get_tables(n_fft, &t);
}

int se_stft(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
            float log_eps, float* power, float* phase, float* logpower, void* stream) {
    return se_stft_strided(wav, n_utt, utt_stride, T, n_fft, hop, window, log_eps, power, phase, logpower, n_fft / 2 + 1, stream);
}

int se_stft_strided(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                    float log_eps, float* power, float* phase, float* logpower, int64_t spec_stride, void* stream) {
    SE_REQUIRE(wav && window, "wav and window must not be null");
    SE_REQUIRE(spec_stride >= n_fft / 2 + 1, "spec_stride=%lld smaller than K", (long long)spec_stride);
    int rc = check_geometry(n_utt, T, n_fft, hop);
    if (rc != SE_OK) return rc;
    DeviceTables t;
    if ((rc = get_tables(n_fft, &t)) != SE_OK) return rc;
    StftArgs a{};
    a.wav = wav; a.utt_stride = utt_stride; a.n_utt = (int)n_utt; a.T = (int)T; a.hop = hop;
    a.n_frames = (int)(T / hop) + 1;
    a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
    a.power = power; a.phase = phase; a.logp = logpower; a.log_eps = log_eps; a.spec_stride = spec_stride;
    cudaStream_t st = (cudaStream_t)stream;
    if (sefast::geo_supported(n_fft, hop) && !g_force_generic) return sefast::launch_stft_run(a, n_fft, st);
    SE_DISPATCH_NFFT(n_fft, launch_stft, a, st)
}

static int stft_features_impl(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                              float log_eps, int take_log, float* feat, int64_t feat_stride, double* stat_sums, int64_t ld_stats,
                              int flags, void* stream);

int se_stft_features(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                     float log_eps, int take_log, float* feat, int64_t feat_stride, double* stat_sums, int64_t ld_stats,
                     int flags, void* stream) {
    return stft_features_impl(wav, n_utt, utt_stride, T, n_fft, hop, window, log_eps, take_log, feat, feat_stride, stat_sums,
                              ld_stats, flags, stream);
}

static int stft_features_impl(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                              float log_eps, int take_log, float* feat, int64_t feat_stride, double* stat_sums, int64_t ld_stats,
                              int flags, void* stream) {
    SE_REQUIRE(wav && window && feat && stat_sums, "null pointer");
    SE_REQUIRE(feat_stride >= n_fft / 2 + 1 && ld_stats >= n_fft / 2 + 1, "feat_stride / ld_stats smaller than K");
    int rc = check_geometry(n_utt, T, n_fft, hop);
    if (rc != SE_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!(flags & SE_FLAG_SUMS_ZEROED)) SE_CUDA_CHECK(cudaMemsetAsync(stat_sums, 0, sizeof(double) * 2 * ld_stats * n_utt, st));
    if (sefast::geo_supported(n_fft, hop) && !g_force_generic) {
        DeviceTables t;
        if ((rc = get_tables(n_fft, &t)) != SE_OK) return rc;
        StftArgs a{};
        a.wav = wav; a.utt_stride = utt_stride; a.n_utt = (int)n_utt; a.T = (int)T; a.hop = hop;
        a.n_frames = (int)(T / hop) + 1;
        a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
        a.power = take_log ? nullptr : feat; a.logp = take_log ? feat : nullptr; a.log_eps = log_eps; a.spec_stride = feat_stride;
        a.stat_sums = stat_sums; a.ld_stats = ld_stats;
        a.trace = secommon::trace_ptr();
        if (flags & SE_FLAG_WS_SELF_CLEAN) { a.zero_ptr = stat_sums + 2 * ld_stats * n_utt; a.zero_count = (long long)SE_NSUMS * n_utt; }
        return sefast::launch_stft_run(a, n_fft, st);
    }
    if (flags & SE_FLAG_WS_SELF_CLEAN)                      // no fast path for this geometry: the same contract by a memset
        SE_CUDA_CHECK(cudaMemsetAsync(stat_sums + 2 * ld_stats * n_utt, 0, sizeof(double) * SE_NSUMS * n_utt, st));
    // other n_fft: generic STFT, then one pass over the features for the sums
    rc = se_stft_strided(wav, n_utt, utt_stride, T, n_fft, hop, window, log_eps, take_log ? nullptr : feat, nullptr,
                         take_log ? feat : nullptr, feat_stride, stream);
    if (rc != SE_OK) return rc;
    return se_feature_sums(feat, feat_stride, n_utt, T / hop + 1, n_fft / 2 + 1, stat_sums, ld_stats, stream);
}

int se_stft_features2(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                      float log_eps, float* power, float* logpower, int64_t spec_stride, double* stat_sums, int64_t ld_stats,
                      int flags, void* stream) {
    SE_REQUIRE(wav && window && (power || logpower) && stat_sums, "null pointer");
    SE_REQUIRE(spec_stride >= n_fft / 2 + 1 && ld_stats >= n_fft / 2 + 1, "spec_stride / ld_stats smaller than K");
    int rc = check_geometry(n_utt, T, n_fft, hop);
    if (rc != SE_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!(flags & SE_FLAG_SUMS_ZEROED)) SE_CUDA_CHECK(cudaMemsetAsync(stat_sums, 0, sizeof(double) * 2 * ld_stats * n_utt, st));
    if (sefast::geo_supported(n_fft, hop) && !g_force_generic) {
        DeviceTables t;
        if ((rc = get_tables(n_fft, &t)) != SE_OK) return rc;
        StftArgs a{};
        a.wav = wav; a.utt_stride = utt_stride; a.n_utt = (int)n_utt; a.T = (int)T; a.hop = hop;
        a.n_frames = (int)(T / hop) + 1;
        a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
        a.power = power; a.logp = logpower; a.log_eps = log_eps; a.spec_stride = spec_stride;
        a.stat_sums = stat_sums; a.ld_stats = ld_stats;
        a.trace = secommon::trace_ptr();
        return sefast::launch_stft_run(a, n_fft, st);
    }
    rc = se_stft_strided(wav, n_utt, utt_stride, T, n_fft, hop, window, log_eps, power, nullptr, logpower, spec_stride, stream);
    if (rc != SE_OK) return rc;
    return se_feature_sums(logpower ? logpower : power, spec_stride, n_utt, T / hop + 1, n_fft / 2 + 1, stat_sums, ld_stats, stream);
}

int se_stft_features_pair_supported(int n_fft, int hop) { return (sefast::geo_supported(n_fft, hop) && !g_force_generic) ? 1 : 0; }

int se_stft_features_pair(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t chan_step, int64_t T, int n_fft, int hop,
                          const float* window, float log_eps, float* power2, float* logpower, int64_t spec_stride, double* stat_sums,
                          int64_t ld_stats, int flags, void* stream) {
    SE_REQUIRE(wav && window && power2 && stat_sums, "null pointer");
    SE_REQUIRE(spec_stride >= n_fft / 2 + 1 && ld_stats >= n_fft / 2 + 1, "spec_stride / ld_stats smaller than K");
    int rc = check_geometry(2 * n_utt, T, n_fft, hop);
    if (rc != SE_OK) return rc;
    if (!se_stft_features_pair_supported(n_fft, hop))
        return fail(SE_ERR_UNSUPPORTED, "se_stft_features_pair: n_fft=%d hop=%d has no register-resident kernel (use two se_stft_features2 calls)", n_fft, hop);
    cudaStream_t st = (cudaStream_t)stream;
    if (!(flags & SE_FLAG_SUMS_ZEROED)) SE_CUDA_CHECK(cudaMemsetAsync(stat_sums, 0, sizeof(double) * 2 * ld_stats * n_utt, st));
    DeviceTables t;
    if ((rc = get_tables(n_fft, &t)) != SE_OK) return rc;
    StftArgs a{};
    a.wav = wav; a.utt_stride = utt_stride; a.n_utt = (int)(2 * n_utt); a.n_real = (int)n_utt; a.chan_step = chan_step;
    a.T = (int)T; a.hop = hop; a.n_frames = (int)(T / hop) + 1;
    a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
    a.power = power2; a.logp = logpower; a.log_eps = log_eps; a.spec_stride = spec_stride;
    a.stat_sums = stat_sums; a.ld_stats = ld_stats;
    a.trace = secommon::trace_ptr();
    return sefast::launch_stft_run(a, n_fft, st);
}

int se_istft(const float* power, const float* phase, int64_t n_utt, int64_t n_frames, int n_fft, int hop,
             const float* window, float* wav_out, int64_t out_stride, int64_t pad_to, void* stream) {
    SE_REQUIRE(power && phase && window && wav_out, "null pointer");
    SE_REQUIRE(n_utt > 0 && n_frames > 1, "n_utt=%lld, n_frames=%lld", (long long)n_utt, (long long)n_frames);
    SE_REQUIRE(hop > 0 && hop <= n_fft, "hop=%d must be in [1, n_fft=%d]", hop, n_fft);
    DeviceTables t;
    int rc = get_tables(n_fft, &t);
    if (rc != SE_OK) return rc;
    IstftArgs a{};
    a.power = power; a.phase = phase; a.n_utt = (int)n_utt; a.n_frames = (int)n_frames; a.hop = hop;
    a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
    a.wav_out = wav_out; a.out_stride = out_stride; a.out_len = hop * ((int)n_frames - 1); a.pad_to = (int)pad_to;
    SE_REQUIRE(out_stride >= a.out_len && out_stride >= pad_to, "out_stride=%lld too small", (long long)out_stride);
    cudaStream_t st = (cudaStream_t)stream;
    SE_DISPATCH_NFFT(n_fft, launch_istft, a, st)
}

int se_mask_istft(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, const int64_t* lengths,
                  int64_t n_utt, int64_t T, int n_fft, int hop, const float* window, float* wav_out, int64_t out_stride,
                  int64_t pad_to, double* sums, int want_spec, void* stream) {
    return se_mask_istft_strided(noisy, clean, utt_stride, mask, n_fft / 2 + 1, lengths, n_utt, T, n_fft, hop, window, wav_out,
                                 out_stride, pad_to, sums, want_spec, stream);
}

int se_mask_istft_strided(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, int64_t mask_stride,
                          const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                          float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, int want_spec, void* stream) {
    return se_mask_istft_ex(noisy, clean, utt_stride, mask, mask_stride, lengths, n_utt, T, n_fft, hop, window, wav_out, out_stride,
                            pad_to, sums, want_spec ? SE_FLAG_WANT_SPEC : 0, stream);
}

int se_mask_istft_ex(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, int64_t mask_stride,
                     const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                     float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, int flags, void* stream) {
    const int want_spec = (flags & SE_FLAG_WANT_SPEC) ? 1 : 0;
    SE_REQUIRE(noisy && mask && window && wav_out, "null pointer");
    SE_REQUIRE(mask_stride >= n_fft / 2 + 1, "mask_stride=%lld smaller than K", (long long)mask_stride);
    int rc = check_geometry(n_utt, T, n_fft, hop);
    if (rc != SE_OK) return rc;
    DeviceTables t;
    if ((rc = get_tables(n_fft, &t)) != SE_OK) return rc;
    MaskIstftArgs a{};
    a.noisy = noisy; a.clean = clean; a.utt_stride = utt_stride; a.mask = mask;
    a.lengths = reinterpret_cast<const long long*>(lengths);
    a.n_utt = (int)n_utt; a.T = (int)T; a.hop = hop; a.n_frames = (int)(T / hop) + 1;
    a.tab.window = window; a.tab.twM = t.twM; a.tab.twN = t.twN;
    a.wav_out = wav_out; a.out_stride = out_stride; a.out_len = hop * (a.n_frames - 1); a.pad_to = (int)pad_to;
    a.sums = sums; a.want_spec = (want_spec && clean && sums) ? 1 : 0; a.mask_stride = mask_stride;
    a.mask_is_power = (flags & SE_FLAG_MASK_IS_POWER) ? 1 : 0;
    a.trace = secommon::trace_ptr();
    SE_REQUIRE(out_stride >= a.out_len && out_stride >= pad_to, "out_stride=%lld too small", (long long)out_stride);
    cudaStream_t st = (cudaStream_t)stream;
    if (sums && !(flags & SE_FLAG_SUMS_ZEROED)) SE_CUDA_CHECK(cudaMemsetAsync(sums, 0, sizeof(double) * SE_NSUMS * n_utt, st));
    const long long stat_doubles = 2LL * ((n_fft / 2 + 1 + 3) / 4 * 4) * n_utt;         // (n_utt, round4(K), 2) right before `sums`
    const bool self_clean = (flags & SE_FLAG_WS_SELF_CLEAN) && sums;
    if (self_clean) { a.zero_ptr = sums - stat_doubles; a.zero_count = stat_doubles; }
    if (sefast::geo_supported(n_fft, hop) && a.n_frames >= 6 && !g_force_generic) return sefast::launch_mask_istft_run(a, n_fft, st);
    if (self_clean) SE_CUDA_CHECK(cudaMemsetAsync(sums - stat_doubles, 0, sizeof(double) * stat_doubles, st));   // generic path: by a memset
    SE_DISPATCH_NFFT(n_fft, launch_mask_istft, a, st)
}

__global__ void __launch_bounds__(256) pcm16_to_float_kernel(const short4* __restrict__ src, float4* __restrict__ dst, long long n4,
                                                             const short* __restrict__ src1, float* __restrict__ dst1, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const float s = 1.0f / 32768.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const short4 v = src[i];
        dst[i] = make_float4(s * (float)v.x, s * (float)v.y, s * (float)v.z, s * (float)v.w);
    }
    for (long long i = 4 * n4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst1[i] = s * (float)src1[i];
}

int se_h2d_channels_pcm16(const int16_t* h_pcm, int64_t B, int64_t C, int64_t T, int64_t n_ch, int16_t* d_pcm, float* d_wavs,
                          void* stream) {
    SE_REQUIRE(h_pcm && d_pcm && d_wavs && B > 0 && T > 0 && n_ch > 0 && n_ch <= C, "bad argument");
    SE_REQUIRE((reinterpret_cast<uintptr_t>(d_pcm) & 7) == 0 && (reinterpret_cast<uintptr_t>(d_wavs) & 15) == 0, "unaligned device buffer");
    cudaStream_t st = (cudaStream_t)stream;
    SE_CUDA_CHECK(cudaMemcpy2DAsync(d_pcm, (size_t)(n_ch * T) * sizeof(int16_t), h_pcm, (size_t)(C * T) * sizeof(int16_t),
                                    (size_t)(n_ch * T) * sizeof(int16_t), (size_t)B, cudaMemcpyHostToDevice, st));
    const long long n = (long long)B * n_ch * T, n4 = n / 4;
    long long blocks = (n4 + 256 * 8 - 1) / (256 * 8);
    const long long cap = 4LL * secommon::device_sms();
    blocks = blocks < 1 ? 1 : (blocks > cap ? cap : blocks);
    pcm16_to_float_kernel<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const short4*>(d_pcm), reinterpret_cast<float4*>(d_wavs), n4,
                                                            d_pcm, d_wavs, n);
    return secommon::check_launch("pcm16_to_float_kernel");
}

int se_h2d_channels(const float* h_wavs, int64_t B, int64_t C, int64_t T, int64_t n_ch, float* d_wavs, void* stream) {
    SE_REQUIRE(h_wavs && d_wavs && B > 0 && T > 0 && n_ch > 0 && n_ch <= C, "bad argument");
    SE_CUDA_CHECK(cudaMemcpy2DAsync(d_wavs, (size_t)(n_ch * T) * sizeof(float), h_wavs, (size_t)(C * T) * sizeof(float),
                                    (size_t)(n_ch * T) * sizeof(float), (size_t)B, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return SE_OK;
}

}  // extern "C"
