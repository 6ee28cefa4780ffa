// g++ harness for the adjoint of the iSTFT: runs istft_bwd_tile (csrc/tile_kernels.cuh) serially on the CPU (HostExec)
// so tests/test_wave_sisdr.py can compare se_istft_bwd's and se_mask_istft_bwd's tile bodies with the float64 oracle.
#include <vector>
#include "../speech_enhancement_by_s3prl_b200/csrc/tile_kernels.cuh"
#include "../speech_enhancement_by_s3prl_b200/csrc/host_plan.h"

using namespace sekern;

namespace {

struct HostExec {
    template <class F> void foreach(int n, F f) { for (int w = 0; w < n; ++w) f(w); }
    void sync() {}
};

template <int N, bool MASK> int run_istft_bwd(IstftBwdArgs a) {
    std::vector<float> twM, twN;
    seplan::make_twiddles(N, twM, twN);
    a.tab.twM = reinterpret_cast<const float2*>(twM.data());
    a.tab.twN = reinterpret_cast<const float2*>(twN.data());
    std::vector<unsigned char> smem(Smem<N>::bytes(istft_bwd_seg<N>(a.hop, MASK), 0));
    HostExec ex;
    const int frames = istft_bwd_frames<N>(MASK);
    const int tiles = (a.n_frames + frames - 1) / frames;
    for (int u = 0; u < a.n_utt; ++u)
        for (int t = 0; t < tiles; ++t) istft_bwd_tile<N, MASK>(ex, a, u, t, smem.data());
    return 0;
}

}  // namespace

#define DISPATCH(n_fft, CALL)              \
    switch (n_fft) {                       \
        case 256: return CALL(256);        \
        case 400: return CALL(400);        \
        case 512: return CALL(512);        \
        case 1024: return CALL(1024);      \
        case 2048: return CALL(2048);      \
        default: return -2;                \
    }

extern "C" {

int h_istft_bwd(int n_fft, const float* grad_wav, long long grad_stride, const float* power, const float* phase, int n_utt,
                int n_frames, int hop, const float* window, float* grad_power, float* grad_phase) {
    IstftBwdArgs a{};
    a.n_utt = n_utt; a.hop = hop; a.n_frames = n_frames; a.T = a.out_len = hop * (n_frames - 1); a.tab.window = window;
    a.grad_wav = grad_wav; a.grad_stride = grad_stride; a.power = power; a.phase = phase;
    a.grad_power = grad_power; a.grad_phase = grad_phase;
#define CALL(NN) run_istft_bwd<NN, false>(a)
    DISPATCH(n_fft, CALL)
#undef CALL
}

int h_mask_istft_bwd(int n_fft, const float* noisy, const float* clean, long long utt_stride, const float* y, long long y_stride,
                     const float* coef, const long long* lengths, const float* mask, long long ld, int n_utt, int T, int hop,
                     const float* window, float* grad_mask, int log_power) {
    IstftBwdArgs a{};
    a.n_utt = n_utt; a.T = T; a.hop = hop; a.n_frames = T / hop + 1; a.out_len = hop * (a.n_frames - 1); a.tab.window = window;
    a.noisy = noisy; a.clean = clean; a.utt_stride = utt_stride; a.y = y; a.y_stride = y_stride;
    a.coef = reinterpret_cast<const float2*>(coef); a.lengths = lengths;
    a.mask = mask; a.grad_mask = grad_mask; a.ld = ld; a.mask_is_power = log_power ? 2 : 0;
#define CALL(NN) run_istft_bwd<NN, true>(a)
    DISPATCH(n_fft, CALL)
#undef CALL
}

}  // extern "C"
