// The arithmetic of objective.SISDR and objective.WSD that the streaming objective kernels (ops_kernels.cu) and the weight-gradient
// kernel with the objective's backward folded in (head_bwd_tc.cu) share: both routes must round the same values the same way.
#pragma once
#include <cuda_runtime.h>

// SI-SDR in dB from the three sums st = <s,t>, tt = <t,t>, ss = <s,s>  (evaluation.py:5-10,
// objective.py:94-97): a = st/(tt+eps); 10 log10(|a t|^2 / (|a t - s|^2 + eps) + eps)
__device__ __forceinline__ double sisdr_from_sums(double st, double tt, double ss, double eps) {
    const double a = st / (tt + eps);
    const double num = a * a * tt;
    double den = a * a * tt - 2.0 * a * st + ss;
    if (den < 0.0) den = 0.0;                      // rounding when s is (numerically) a multiple of t
    return 10.0 * log10(num / (den + eps) + eps);
}

// d loss_u / d s_i = c_t t_i + c_s s_i for loss_u = -sisdr_from_sums(sums3) (s, t: the magnitudes sqrt(relu(.))), scaled by the
// upstream gradient go: loss_u = -10 log10(R + eps), R = A / D, d loss_u / d s_i = kappa * ((ca*D - A*cd) t_i - 2 A s_i)
__device__ __forceinline__ float2 sisdr_coef(const double* sums3, double eps, double go) {
    const double st = sums3[0], tt = sums3[1], ss = sums3[2];
    const double al = st / (tt + eps);
    const double A = al * al * tt;
    const double D = al * al * tt - 2.0 * al * st + ss + eps;
    const double R = A / D;
    const double kappa = -10.0 / (log(10.0) * (R + eps) * D * D);
    const double ca = 2.0 * al * tt / (tt + eps);
    const double cd = 2.0 * (al * tt - st) / (tt + eps) - 2.0 * al;
    return make_float2((float)(go * kappa * (ca * D - A * cd)), (float)(go * kappa * (-2.0 * A)));
}

// objective.WSD's voicing rule: a frame of energy E (sum of its target power) is voiced when 10 log10(E + eps) lies above the
// threshold 10 log10(max + eps) - db_interval, max being the batch maximum of the frame energies
__device__ __forceinline__ float wsd_threshold(float max_energy, float eps, float db_interval) {
    return 10.0f * log10f(max_energy + eps) - db_interval;
}
__device__ __forceinline__ bool wsd_voiced(float energy, float eps, float thres) { return 10.0f * log10f(energy + eps) > thres; }

// d loss / d G of one element of objective.WSD: G = offset, X = linear_inp, S = linear_tar, scale = d L / d loss_u
__device__ __forceinline__ float wsd_grad(float G, float X, float S, bool voiced, float alpha, float scale) {
    const float n = fmaxf(X - S, 0.0f);
    return scale * ((voiced ? alpha * 2.0f * (S - G * S) * (-S) : 0.0f) + (1.0f - alpha) * 2.0f * G * n * n);
}
