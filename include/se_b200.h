/* se_b200.h -- C ABI of libse_b200.so: the B200 (sm_100a) enhancement signal path.
 *
 * Drop-in boundary for the hot path of leo19941227/Speech-Enhancement-by-S3PRL
 * (SURVEY.md section 8b).  The reference is pure Python: what it "binds" for this
 * path are PyTorch library calls made from the call sites cited on each entry
 * point below; a maintainer swaps those call sites for the ctypes stubs shown in
 * INTEGRATION.md (or simply imports the drop-in Python classes of
 * speech_enhancement_by_s3prl_b200, which wrap exactly these functions).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device unless the
 *     parameter name starts with h_ (host); all tensors are dense fp32 unless noted
 *   - the caller owns every buffer; the library allocates only its private
 *     twiddle tables (once per device and n_fft, see se_prepare) and keeps no
 *     reference to caller memory after return
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*)
 *   - return value: SE_OK or a negative SE_ERR_*; se_last_error() gives the text
 *     of the last failure on the calling thread.  No C++ exception crosses the ABI.
 *   - spectra are TIME-MAJOR (n_utt, n_frames, K), K = n_fft/2 + 1,
 *     n_frames = T / hop + 1  (runner.py:455: stft_lengths = lengths // hop + 1)
 *   - supported n_fft: 256, 400, 512, 1024, 2048; window length n_fft (a shorter
 *     analysis window is passed already centred and zero-padded, as torch.stft does)
 */
#ifndef SE_B200_H
#define SE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SE_OK 0
#define SE_ERR_BAD_ARG (-1)        /* null pointer, non-positive size, T <= n_fft/2 (reflect padding undefined) */
#define SE_ERR_UNSUPPORTED (-2)    /* n_fft / hop combination without a kernel */
#define SE_ERR_CUDA (-3)           /* a CUDA runtime call failed; text in se_last_error */
#define SE_ERR_NO_DEVICE (-4)      /* no sm_100 device: there is NO CPU fallback */

#define SE_NSUMS 6                 /* doubles per utterance written by se_mask_istft */
#define SE_SUM_YC 0                /* sum_t y*c  (t < length)   y = enhanced, c = clean */
#define SE_SUM_CC 1                /* sum_t c*c                                        */
#define SE_SUM_YY 2                /* sum_t y*y                                        */
#define SE_SUM_SPEC_ST 3           /* sum_{f,k} sqrt(relu(pred))*sqrt(tar)  (f < length/hop+1) */
#define SE_SUM_SPEC_TT 4           /* sum_{f,k} tar                                    */
#define SE_SUM_SPEC_SS 5           /* sum_{f,k} relu(pred)                             */

#define SE_ACT_IDENTITY 0
#define SE_ACT_RELU 1
#define SE_ACT_SIGMOID 2

#define SE_OPT_FORCE_GENERIC 0     /* 1: use the generic tile kernels even where a fast path exists (tests) */

int se_version(void);
int se_last_error(char* h_buf, int n);
int se_set_option(int key, int value);
/* Debugging aid: CTA timeline of the fused-step kernels.  d_buf = device buffer of 1 + 4*capacity uint64 (first word = record
 * count, zeroed by the caller) or NULL to switch tracing off; records are {kernel id << 32 | block, SM id, t_start, t_end}
 * (globaltimer ns; kernel ids 1 = STFT, 2 = head, 3 = mask->iSTFT, 4 = finalize).  Applies to launches (and graph captures)
 * made after the call. */
int se_set_trace(unsigned long long* d_buf);

/* Create the per-device twiddle tables for n_fft and opt the kernels into their
 * shared-memory size.  Idempotent.  Call once before capturing a CUDA graph. */
int se_prepare(int n_fft);

/* ---- K1: STFT + magphase (+log) ----------------------------------------------
 * Replaces OnlinePreprocessor.forward's torch.stft -> magphase(power=2) -> log ->
 * transpose chain (S3PRL utility/preprocessor.py; call sites runner.py:433,558,297,
 * sampler.py:60; the same primitives are used directly at sampler.py:226-229).
 * Row u of the input starts at wav + u*utt_stride (so one channel of a (B,3,T)
 * batch is wav + c*T with utt_stride 3*T).  center=True, reflect padding,
 * one-sided, not normalised.  Any of power / phase / logpower may be NULL.
 *   power    = re^2 + im^2            ("linear" feature)
 *   phase    = atan2(im, re)
 *   logpower = log(power + log_eps)   (feature config log: True) */
int se_stft(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop,
            const float* window, float log_eps, float* power, float* phase, float* logpower, void* stream);
/* same, with spec_stride floats between consecutive frames of every output (>= K).  A stride that is a
 * multiple of 4 floats makes the rows 16-byte aligned for the tensor-core head's vector loads. */
int se_stft_strided(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop,
                    const float* window, float log_eps, float* power, float* phase, float* logpower,
                    int64_t spec_stride, void* stream);

/* ---- iSTFT from (power, phase) --------------------------------------------------
 * Replaces OnlinePreprocessor.istft(linears, phases) (call site runner.py:267):
 * polar(power^(1/2), phase) -> irfft -> window -> overlap-add -> / sum w^2 -> trim.
 * Writes hop*(n_frames-1) samples per row and zero-fills up to pad_to (runner.py:268). */
int se_istft(const float* power, const float* phase, int64_t n_utt, int64_t n_frames, int n_fft, int hop,
             const float* window, float* wav_out, int64_t out_stride, int64_t pad_to, void* stream);

/* ---- adjoint of the iSTFT (training through the waveform) -----------------------
 * For y = iSTFT(Y) as se_istft computes it and a gradient waveform g = dL/dy (zero outside [0, hop*(n_frames-1))), the
 * gradient of every frame's spectrum G = dL/dRe Y + i dL/dIm Y is, with w the centred window and env[p] = sum_f w[p - f hop]^2,
 *   r_f[n] = w[n] g[f hop + n - n_fft/2] / env[f hop + n],
 *   G_f[k] = (c_k / n_fft) sum_n r_f[n] e^{-2 pi i k n / n_fft},  c_0 = c_{n_fft/2} = 1, else 2;  Im G_f[0] = Im G_f[n_fft/2] = 0
 * (the exact transpose of irfft + window + overlap-add + envelope division; one forward real FFT per frame).
 * se_istft_bwd: the backward of se_istft in power and phase, Y = sqrt(P) e^{i phase}: grad_wav row u at grad_wav + u*grad_stride
 *   (only its first hop*(n_frames-1) samples are read: the pad_to zero fill carries no gradient); power / phase / grad_power /
 *   grad_phase dense (n_utt, n_frames, K):
 *     grad_power = Re(G e^{-i phase}) / (2 sqrt(P)), 0 where P = 0;   grad_phase = sqrt(P) Im(G e^{-i phase}).
 * se_mask_istft_bwd: the backward of se_mask_istft_ex in its mask, for a loss whose gradient in K3's output y (wav_out, rows
 *   y_stride apart) is g[t] = coef[u].x y[t] + coef[u].y clean[t] for t < min(lengths[u], hop*(T/hop)) (0 elsewhere; coef (n_utt)
 *   float pairs, e.g. from se_wave_sisdr_finish): the noisy spectrum X is recomputed from `noisy` with K3's framing, and
 *     flags 0 (Y = sqrt(m) X):                             grad_mask = Re(G conj X) / (2 sqrt(m)), 0 where m <= 0;
 *     SE_FLAG_MASK_IS_LOG_POWER (Y = e^{m/2} X / |X|):     grad_mask = Re(G conj Y) / 2.
 *   mask and grad_mask are (n_utt, T/hop + 1, ld >= K) with rows ld floats apart; grad_mask's columns [K, ld) are written 0.
 *   Every n_fft and hop of se_mask_istft_ex, on the generic tile kernel. */
int se_istft_bwd(const float* grad_wav, int64_t grad_stride, const float* power, const float* phase, int64_t n_utt,
                 int64_t n_frames, int n_fft, int hop, const float* window, float* grad_power, float* grad_phase, void* stream);
int se_mask_istft_bwd(const float* noisy, const float* clean, int64_t utt_stride, const float* y, int64_t y_stride, const float* coef,
                      const int64_t* lengths, const float* mask, int64_t ld, int64_t n_utt, int64_t T, int n_fft, int hop,
                      const float* window, float* grad_mask, int flags, void* stream);

/* ---- K3: fused mask multiply + iSTFT + overlap-add (+ metric sums) ---------------
 * wav_out = istft(linear_inp * mask, phase_inp) computed as iSTFT(sqrt(mask) * STFT(noisy))
 * without materialising the spectrum, `predicted` or the phase
 * (model.py:33 `predicted = linears * offset`; runner.py:569-570 `_decode_wav`).
 * If sums != NULL (n_utt x SE_NSUMS doubles, overwritten) it accumulates the
 * reductions that masked_normalize_decibel (utils.py:31-46), sisdr_eval
 * (evaluation.py:5-10) and, with want_spec, objective.SISDR (objective.py:86-100)
 * need; `clean` may be NULL (only SE_SUM_YY is produced then).  lengths may be NULL (= T). */
int se_mask_istft(const float* noisy, const float* clean, int64_t utt_stride, const float* mask,
                  const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                  float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, int want_spec, void* stream);
int se_mask_istft_strided(const float* noisy, const float* clean, int64_t utt_stride, const float* mask,
                          int64_t mask_stride, const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop,
                          const float* window, float* wav_out, int64_t out_stride, int64_t pad_to, double* sums,
                          int want_spec, void* stream);

/* flags of the _ex / fused entry points */
#define SE_FLAG_WANT_SPEC 1        /* se_mask_istft_ex: also accumulate the spectral SI-SDR sums (= want_spec) */
#define SE_FLAG_SUMS_ZEROED 2      /* the caller has zeroed the sums buffer on this stream: skip the library's memset, so
                                      that consecutive kernels of the fused step keep their programmatic (PDL) edges */
#define SE_FLAG_MASK_IS_POWER 4    /* se_mask_istft_ex: `mask` holds a TARGET power spectrum P (e.g. the upstream SpecHead's
                                      output, runner.py:272-281): wav_out = istft(P, phase(STFT(noisy))) = iSTFT(sqrt(P) X / |X|),
                                      sqrt(P) where X = 0 -- _decode_wav on a predicted spectrum without materialising the phase */
#define SE_FLAG_WS_SELF_CLEAN 8     /* the fused step's workspace is ONE caller-owned block of doubles, zeroed once:
                                      [ stat_sums (n_utt, round4(K), 2) | sums (n_utt, SE_NSUMS) ].  With this flag (and
                                      SE_FLAG_SUMS_ZEROED) the step's kernels leave it zeroed for the next replay instead of the
                                      caller filling it every step: se_stft_features zeroes the `sums` part (consumed by the
                                      previous step's se_finalize_metrics), se_mask_istft_ex zeroes the stat_sums part (consumed
                                      by this step's head) -- a captured step then has no fill node at its start.  The STFT
                                      entry points require ld_stats == round4(K) with it (SE_ERR_BAD_ARG otherwise): both ends
                                      find the boundary from that layout */
#define SE_FLAG_MASK_IS_LOG_POWER 16 /* se_mask_istft_ex: `mask` holds the LOG of a target power spectrum (model.LSTM's
                                      log_predicted, model.py:37-60): wav_out = iSTFT(exp(lp / 2) X / |X|), exp(lp / 2) where
                                      X = 0 -- _decode_wav(exp(lp), phase_inp) without the phase or an exp pass; with
                                      SE_FLAG_WANT_SPEC the spectral SI-SDR sums take s = exp(lp / 2) as the estimate's
                                      magnitude.  Mutually exclusive with SE_FLAG_MASK_IS_POWER */
int se_mask_istft_ex(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, int64_t mask_stride,
                     const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                     float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, int flags, void* stream);

/* ---- K3 epilogue: level normalisation + metrics from the sums --------------------
 * Per utterance: gain so that the masked mean-square of wav matches the clean
 * reference's (target_db_or_nan = NaN; runner.py:570 + utils.py:38-40) or a fixed level
 * in dB (runner.py:266 default -25); wav *= gain in place over [0, width);
 * sisdr_wave[u] = evaluation.sisdr_eval(gain*y[:len], c[:len]);
 * loss_spec[u]  = per-utterance term of objective.SISDR (its batch mean is the loss); meaningful only if the sums
 *                came from se_mask_istft with want_spec (otherwise the spectral sums are 0 and the term is 100 dB).
 * lengths[u] is clamped to [0, T] as se_mask_istft clamps it, so the means divide by the samples that were summed;
 * lengths NULL = T.  Any of gain / sisdr_wave / loss_spec may be NULL; wav may be NULL (no scaling). */
int se_finalize_metrics(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T,
                        float target_db_or_nan, float* wav, int64_t wav_stride, int64_t width,
                        float* gain, float* sisdr_wave, float* loss_spec, void* stream);
/* Same, and metric_acc[0..2] (doubles, caller-owned, never zeroed here) += [sum_u loss_spec, sum_u sisdr_wave, n_utt]:
 * the running sums an evaluation pass averages at its end (runner.py:602; objective.py:100) stay on the device, so
 * a pass over many batches -- and the one all-reduce of a data-parallel pass -- needs no host read per batch.
 * A term is added only if it is produced: metric_acc[0] only when loss_spec != NULL, metric_acc[1] only when
 * sisdr_wave != NULL (pass loss_spec = NULL when the sums were made without want_spec); metric_acc[2] always counts. */
int se_finalize_metrics_acc(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T,
                            float target_db_or_nan, float* wav, int64_t wav_stride, int64_t width,
                            float* gain, float* sisdr_wave, float* loss_spec, double* metric_acc, void* stream);

/* ---- K4a: spectral SI-SDR objective (objective.py:86-100) -------------------------
 * fwd: per-utterance sums (n_utt x 3 doubles: st, tt, ss; overwritten) over frames
 *      f < stft_len[u] of src = sqrt(relu(predicted)), tar = sqrt(relu(linear_tar));
 *      loss_per_utt[u] = -10 log10(|a t|^2 / (|a t - s|^2 + eps) + eps), a = st/(tt+eps).
 * bwd: grad_predicted[u] = grad_out[u] * d loss_u / d predicted[u] (grad_out: (n_utt,), 1/B each
 *      for loss.mean(); 0 where predicted <= 0 or the frame is masked), from the saved sums.
 * Both are se_sisdr_mask_fwd / _bwd (below) on dense tensors: offset NULL and every row stride = K. */
int se_sisdr_spec_fwd(const float* predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double* sums3, float* loss_per_utt, void* stream);
int se_sisdr_spec_bwd(const float* predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, const double* sums3, const float* grad_out,
                      float* grad_predicted, void* stream);

/* ---- K4b: log-spectral L1 objective (objective.py:109-117) ------------------------
 * fwd: acc2[0] = sum |log_predicted - log(linear_tar + eps)| over valid frames,
 *      acc2[1] = number of valid elements (2 doubles, overwritten); loss = acc2[0]/acc2[1]
 *      (the global element mean: under data parallelism all-reduce both before dividing).
 * bwd: grad = sign(log_predicted - log(tar+eps)) * grad_out / count on valid frames, else 0. */
int se_l1_logspec_fwd(const float* log_predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double* acc2, void* stream);
int se_l1_logspec_bwd(const float* log_predicted, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
                      int64_t n_frames, int64_t K, float eps, double count, const float* grad_out,
                      float* grad_log_predicted, void* stream);

/* se_l1_mask_step: objective.L1's part of one training step (the counterpart of se_sisdr_mask_step) on row-strided tensors:
 * log_predicted (n_utt, n_frames, ld_lp) and the clean power linear_tar (n_utt, n_frames, ld_tar), rows ld_* floats apart (float4
 * loads when every ld is a multiple of 4 and the pointers are 16-byte aligned), columns >= K never read.  lengths / len_hop as in
 * se_sisdr_mask_step.  Over the valid frames f < frames_u and the K bins, d = log_predicted - log(linear_tar + eps):
 *   loss_mean (1 float) = sum |d| / count with count = K sum_u frames_u -- the element mean of the batch this rank holds, which is
 *     what objective.L1 returns on each rank under data parallelism;
 *   loss_per_utt[u] (may be NULL) = the utterance's own sum |d| / (K frames_u);
 *   grad (may be NULL; ld_g floats between rows) = d loss_mean / d log_predicted = sign(d) / count, with se_l1_logspec_bwd's sign
 *     (0 for d == 0 and for NaN), 0 on padded frames and on the pad columns [K, ld_g).
 * Two launches and no atomics: every CTA writes the double sum of its frame chunk to its own slot of ws_partials
 * (se_l1_mask_step_workspace doubles, caller-owned, no zeroing needed) and a one-CTA finish adds the slots in a fixed order, so the
 * loss is bitwise repeatable.  No host synchronisation: capturable. */
int64_t se_l1_mask_step_workspace(int64_t n_utt, int64_t n_frames, int64_t K);
int se_l1_mask_step(const float* log_predicted, int64_t ld_lp, const float* linear_tar, int64_t ld_tar, const int64_t* lengths,
                    int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float eps, double* ws_partials, int64_t ws_doubles,
                    float* loss_per_utt, float* loss_mean, float* grad, int64_t ld_g, void* stream);

/* se_act_grad_inplace: grad <- grad * act'(out) on n_rows rows (grad rows ld_g floats apart, out rows ld_out apart), where out is
 * the head's output AFTER its activation: Sigmoid out (1 - out), ReLU (out > 0); columns [K, ld_g) of grad are set to 0.  It turns
 * an objective's d loss / d output into d loss / d pre-activation (the operand of both weight- and input-gradient GEMMs).
 * act = SE_ACT_IDENTITY returns at once without a launch. */
int se_act_grad_inplace(float* grad, int64_t ld_g, const float* out, int64_t ld_out, int64_t n_rows, int64_t K, int act, void* stream);

/* ---- K4d: weighted speech distortion objective (objective.py:120-153) ------------------
 * loss = alpha * mean_u sum_{f<len,k} ((S - G S) voiced)^2 + (1 - alpha) * mean_u sum (G max(X - S, 0))^2 with
 * S = linear_tar, X = linear_inp, G = offset; voiced[u,f] = 10 log10(sum_k S + eps) > 10 log10(max_{u,f} sum_k S + eps)
 * - db_interval (the maximum runs over the whole padded batch, as in the reference).  Workspaces (caller-owned):
 * ws_energy (n_utt * n_frames) floats, ws_max 1 float, ws_sums2 (n_utt, 2) doubles; loss: 1 float.
 * bwd: grad_offset = grad_loss[0] * d loss / d offset (0 on padded frames), from the forward's workspaces (ws_max holds the
 * batch maximum as a plain float).
 * Both are the strided forms below on dense tensors (every row stride = K): fwd = se_wsd_energy, then the sums and batch mean of
 * se_wsd_mask_step; bwd = se_wsd_mask_step's backward scaled by grad_loss[0].
 * This form takes the maximum over the batch it is given.  Under data parallelism the maximum must be the GLOBAL batch's: use
 * the split form below (se_wsd_energy -> all-reduce(max) of its 1-float buffer -> se_wsd_mask_step), which se_wsd_bwd can
 * also differentiate (its ws_energy / ws_max are se_wsd_energy's outputs). */
int se_wsd_fwd(const float* linear_inp, const float* offset, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
               int64_t n_frames, int64_t K, float alpha, float db_interval, float eps, float* ws_energy, float* ws_max,
               double* ws_sums2, float* loss, void* stream);
int se_wsd_bwd(const float* linear_inp, const float* offset, const float* linear_tar, const int64_t* stft_len, int64_t n_utt,
               int64_t n_frames, int64_t K, float alpha, float db_interval, float eps, const float* ws_energy,
               const float* ws_max, const float* grad_loss, float* grad_offset, void* stream);

/* ---- the same objective split at the batch maximum (data-parallel form), on row-padded tensors --------------------------------
 * se_wsd_energy: energy[u * n_frames + f] = sum_{k<K} linear_tar[u, f, k] over EVERY frame of the padded batch (rows ld_tar floats
 *   apart, columns >= K never read; summation order of se_wsd_fwd) and max_energy[0] = their maximum, written as a plain float32 --
 *   so that torch.distributed.all_reduce(op=MAX) of that 1-element buffer gives the maximum of the global batch.  Sums of
 *   any sign are ordered as floats; NaN energies take no part (if every energy is NaN, max_energy is NaN).
 * se_wsd_mask_step: the objective's part of one training step (the counterpart of se_sisdr_mask_step), reading the maximum from
 *   max_energy AFTER any all-reduce: sums2 (n_utt, 2) doubles = {sum ((S - G S) voiced)^2, sum (G max(X - S, 0))^2} over the
 *   valid frames, loss_per_utt[u] = alpha sums2[u, 0] + (1 - alpha) sums2[u, 1] (may be NULL), loss_mean (1 float) = their batch
 *   mean, and grad_offset = d loss_mean / d offset (ld_g floats between rows; 0 on padded frames and pad columns), skipped when
 *   NULL (se_linear_head_bwd_wsd rebuilds it inside the weight-gradient kernel).  Rows of offset / linear_inp / linear_tar are
 *   ld_* floats apart (float4 loads when every ld is a multiple of 4 and the pointers are 16-byte aligned).  lengths / len_hop as
 *   in se_sisdr_mask_step; sums_zeroed != 0: sums2 is already zero. */
int se_wsd_energy(const float* linear_tar, int64_t ld_tar, int64_t n_utt, int64_t n_frames, int64_t K, float* energy, float* max_energy,
                  void* stream);
int se_wsd_mask_step(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                     const int64_t* lengths, int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float alpha, float db_interval,
                     float eps, const float* energy, const float* max_energy, double* sums2, int sums_zeroed, float* loss_per_utt,
                     float* loss_mean, float* grad_offset, int64_t ld_g, void* stream);

/* ---- the evaluation step with objective.WSD (objective.py:127-153; runner.py:575 `criterion(**locals())`) ---------------------
 * se_mask_istft_wsd: se_mask_istft_ex (same waveform output and SE_SUM_YC / SE_SUM_CC / SE_SUM_YY sums; clean and sums
 *   required) that computes, instead of the spectral SI-SDR sums, the WSD terms of mask G = `mask`, X = |STFT(noisy)|^2 and
 *   S = |STFT(clean)|^2 without materialising any spectrum:
 *     frame_terms (n_utt, n_frames) float2 = {E_f = sum_k S over EVERY frame of the padded batch,
 *                                             D_f = sum_k (S - G S)^2 on frames f < lengths[u] // hop + 1, else 0};
 *     sums[u * SE_NSUMS + SE_SUM_SPEC_ST] += sum over valid frames of (G max(X - S, 0))^2;
 *     wsd_state[0] (a float32 that rests at 0.0f) = max(itself, largest E_f), so that torch.distributed.all_reduce(op=MAX) of that
 *     1-element buffer gives the maximum of the global batch.  wsd_state is 2 x 32 bits, zeroed once by the caller;
 *     se_wsd_eval_finish puts it back to zero.
 *   flags: SE_FLAG_SUMS_ZEROED and SE_FLAG_WS_SELF_CLEAN as in se_mask_istft_ex.  Register-resident geometries only
 *   (se_mask_istft_wsd_supported, and T / hop + 1 >= 6 frames); otherwise SE_ERR_UNSUPPORTED: use se_wsd_energy and
 *   se_wsd_mask_step on the spectra.
 * se_wsd_eval_finish: after any all-reduce of wsd_state[0]: voiced[u, f] = 10 log10(E_f + eps) > 10 log10(wsd_state[0] + eps)
 *   - db_interval; loss_per_utt[u] = alpha sum_f voiced D_f (double, fixed order) + (1 - alpha) sums[u, SE_SUM_SPEC_ST]; the batch
 *   mean of loss_per_utt is objective.WSD's value.  metric_acc (or NULL) [0] += sum_u loss_per_utt; pair it with
 *   se_finalize_metrics_acc(loss_spec = NULL), which adds the SI-SDR sum and the count. */
int se_mask_istft_wsd_supported(int n_fft, int hop);
int se_mask_istft_wsd(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, int64_t mask_stride,
                      const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                      float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, float* frame_terms, float* wsd_state,
                      int flags, void* stream);
int se_wsd_eval_finish(const float* frame_terms, const double* sums, int64_t n_utt, int64_t n_frames, float alpha, float db_interval,
                       float eps, float* wsd_state, float* loss_per_utt, double* metric_acc, void* stream);

/* ---- the evaluation step with objective.L1 (objective.py:109-117) and model.LSTM (log_predicted) ------------------------
 * se_mask_istft_l1: se_mask_istft_ex with SE_FLAG_MASK_IS_LOG_POWER (same waveform output and SE_SUM_YC / SE_SUM_CC / SE_SUM_YY
 *   sums; clean and sums required) whose clean-frame pass computes, for lp = `mask` and C = STFT(clean), over the valid frames
 *   f < lengths[u] // hop + 1 and the K bins:
 *     sums[u * SE_NSUMS + SE_SUM_SPEC_ST] += sum |lp - log(|C|^2 + eps)|   (SE_SUM_SPEC_TT / _SS stay 0);
 *     l1_acc[0] += the same sums over the batch, l1_acc[1] += sum_u valid_frames_u * K
 *   (2 caller-owned doubles that rest at 0: the numerator and the element count of the global mean, which is what a data-parallel
 *   evaluation all-reduces before se_l1_eval_finish; one double atomic per run).
 *   flags: SE_FLAG_SUMS_ZEROED and SE_FLAG_WS_SELF_CLEAN as in se_mask_istft_ex.  Register-resident geometries only
 *   (se_mask_istft_l1_supported, and T / hop + 1 >= 6 frames); otherwise SE_ERR_UNSUPPORTED: use se_mask_istft_ex with
 *   SE_FLAG_MASK_IS_LOG_POWER and se_l1_eval_sums on the clean power spectrum.
 * se_l1_eval_sums: the same sums from materialised row-strided tensors (n_utt, T / hop + 1, ld): log_predicted and the clean
 *   power linear_tar; sums[u, SE_SUM_SPEC_ST] (zeroed by the caller) += the utterance's sum, l1_acc[0] += the batch's, l1_acc[1] +=
 *   sum_u valid_frames_u * K.
 * se_l1_eval_finish: after any all-reduce of l1_acc: loss_per_utt[u] = sums[u, SE_SUM_SPEC_ST] / (valid_frames_u * K) (the
 *   utterance's own L1, a batch of one), loss[0] = l1_acc[0] / l1_acc[1] (objective.L1 of the global batch), metric_acc (or NULL)
 *   [0] += n_utt * loss[0] (so that the pass mean of dp.means_from_acc stays the mean of the batch losses, weighted by their
 *   utterances), then l1_acc = {0, 0} for the next step.  Lengths are clamped to [0, T] as the mask-iSTFT kernels clamp them. */
int se_mask_istft_l1_supported(int n_fft, int hop);
int se_mask_istft_l1(const float* noisy, const float* clean, int64_t utt_stride, const float* mask, int64_t mask_stride,
                     const int64_t* lengths, int64_t n_utt, int64_t T, int n_fft, int hop, const float* window,
                     float* wav_out, int64_t out_stride, int64_t pad_to, double* sums, double* l1_acc, float eps, int flags,
                     void* stream);
int se_l1_eval_sums(const float* log_predicted, int64_t ld_lp, const float* linear_tar, int64_t ld_tar, const int64_t* lengths,
                    int64_t n_utt, int64_t T, int hop, int64_t K, float eps, double* sums, double* l1_acc, void* stream);
int se_l1_eval_finish(const double* sums, const int64_t* lengths, int64_t n_utt, int64_t T, int hop, int64_t K, double* l1_acc,
                      float* loss_per_utt, float* loss, double* metric_acc, void* stream);

/* ---- K4c: batched waveform SI-SDR (evaluation.py:5-10 over runner.py:587-602) -----
 * sisdr[u] = sisdr_eval(src[u, :len[u]], tar[u, :len[u]]).  ws_sums3: caller workspace of
 * n_utt x 3 doubles (overwritten: <s,t>, <t,t>, <s,s>). */
int se_sisdr_wave(const float* src, int64_t src_stride, const float* tar, int64_t tar_stride, const int64_t* lengths,
                  int64_t n_utt, int64_t T, float eps, double* ws_sums3, float* sisdr, void* stream);
/* ---- objective.WaveSISDR: the waveform SI-SDR as a training loss ------------------------------------------------
 * se_wave_sisdr_finish: from s = sums + u * ld_sums = [<y,c>, <c,c>, <y,y>] (K3's SE_SUM_YC / CC / YY with ld_sums = SE_NSUMS,
 *   or se_sisdr_wave's workspace with ld_sums = 3), in double with sisdr_eval's arithmetic (a = s0 / (s1 + eps)):
 *     loss_per_utt[u] = -10 log10(a^2 s1 / (a^2 s1 - 2 a s0 + s2 + eps) + eps),  loss[0] = their mean over the n_utt utterances;
 *     coef[u] = (alpha_u, beta_u), float pairs, such that d loss[0] / d y[t] = alpha_u y[t] + beta_u c[t] (the 1/n_utt included);
 *     metric_acc[0..2] += [sum loss_per_utt, sum SI-SDR, n_utt].
 *   Every output is optional.  A silent reference (s1 = 0) or a zero estimate gives finite values (coefficients 0).
 * se_wave_sisdr_bwd: grad[u, t] = scale * grad_out[u] * (coef[u].x src[u, t] + coef[u].y tar[u, t]) for t < lengths[u] (clamped
 *   to [0, T]; NULL = T), 0 for the rest of [0, T). */
int se_wave_sisdr_finish(const double* sums, int64_t ld_sums, int64_t n_utt, float eps, float* loss_per_utt, float* loss, float* coef,
                         double* metric_acc, void* stream);
int se_wave_sisdr_bwd(const float* src, int64_t src_stride, const float* tar, int64_t tar_stride, const int64_t* lengths, int64_t n_utt,
                      int64_t T, const float* coef, const float* grad_out, float scale, float* grad, int64_t grad_stride, void* stream);

/* ---- STOI / ESTOI (pystoi 0.3.x: stoi(clean, processed, fs), extended=False / True) -----------------------
 * stoi[u], estoi[u] of ref[u, :len[u]] (the clean reference, pystoi's x) and est[u, :len[u]] (the processed
 * signal); lengths NULL = T, otherwise clamped to [0, T].  Resampled to 10 kHz unless fs == 10000; fewer than
 * 30 STFT frames after silent-frame removal (also no frame at all) gives 1e-5.  Supported rates: 10000 / fs
 * reduced to p / q with p, q <= 48 (8, 16, 32, 48 kHz; 10 kHz without resampling); others SE_ERR_UNSUPPORTED.
 * se_stoi_workspace: bytes of `ws` (<= 0: unsupported fs or shape).  stoi, estoi, n_kept (frames kept by the
 * silent-frame removal) are each optional, but stoi or estoi must be given.  acc (optional, 3 doubles, never
 * zeroed here) += [sum stoi, sum estoi, n_utt], each sum only when that output is given.  No host
 * synchronisation, no allocation: capturable.  Per-utterance results are bitwise reproducible. */
int64_t se_stoi_workspace(int64_t n_utt, int64_t T, int fs);
int se_stoi(const float* est, int64_t est_stride, const float* ref, int64_t ref_stride, const int64_t* lengths,
            int64_t n_utt, int64_t T, int fs, void* ws, int64_t ws_bytes,
            float* stoi, float* estoi, int32_t* n_kept, double* acc, void* stream);

/* ---- a11: masked_normalize_decibel (utils.py:31-46) -------------------------------
 * out = audio * sqrt(10^(target/10) / (masked_mean(audio^2) + eps)); target per row is
 * target_db[u] if target_db != NULL, else the masked level of ref[u] (utils.py:38-40).  masked_mean divides by
 * min(lengths[u], width) + 1e-8 whatever eps is (utils.py:26: the reference's masked_mean keeps its own default).
 * ws_sums3: caller workspace of n_utt x 3 doubles.  out may alias audio. */
int se_masked_normalize_db(const float* audio, int64_t stride, const int64_t* lengths, int64_t n_utt, int64_t width,
                           const float* target_db, const float* ref, int64_t ref_stride, float eps,
                           double* ws_sums3, float* out, int64_t out_stride, void* stream);

/* ---- a4: length masks (runner.py:216-220) ------------------------------------------
 * masks[u, i] = i < lengths[u] ? 1 : 0, int64, shape (n_utt, width). */
int se_length_masks(const int64_t* lengths, int64_t n_utt, int64_t width, int64_t* masks, void* stream);

/* ---- K2: mask head (model.py:14-17 Linear, model.py:28-34 LinearResidual) ---------
 * se_cmvn_stats: per (utterance, feature) mean and unbiased std over ALL n_frames
 *   (padding included, as model.py:30 does).  mean/std: (n_utt, D).
 * se_linear_head_fwd: act((x - mean)/(std + cmvn_eps)) W^T + b) [* linears]
 *   x (n_utt*n_frames, D_in), W (D_out, D_in) row-major (nn.Linear layout), b (D_out) or NULL;
 *   mean/std NULL = no CMVN; offset_out and/or predicted_out (= linears * offset) may be NULL.
 *   precision: 0 = fp32 SIMT (bit-comparable with torch fp32), 1 = TF32 tcgen05 tensor cores.
 * se_linear_head_bwd: given grad_offset (dL/d offset after activation) computes grad_W, grad_b
 *   (overwritten).  grad_x is not produced: the head's input features come from the
 *   preprocessor and never require a gradient in the reference (runner.py:433-453). */
int se_cmvn_stats(const float* x, int64_t n_utt, int64_t n_frames, int64_t D, float* mean, float* std, void* stream);
int se_linear_head_fwd(const float* x, const float* mean, const float* std, float cmvn_eps, const float* W,
                       const float* b, int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act,
                       const float* linears, float* offset_out, float* predicted_out, int precision, void* stream);
/* strided forms used by the fused evaluation step: ldx = floats between rows of x, ld_stats between rows of
 * mean / std, ldw between rows of W, ld_out between rows of linears / offset_out / predicted_out.  With
 * precision 1 and every stride a multiple of 4 floats (16-byte aligned rows) the producers use 128-bit loads. */
int se_cmvn_stats_strided(const float* x, int64_t ldx, int64_t n_utt, int64_t n_frames, int64_t D, float* mean,
                          float* std, int64_t ld_stats, void* stream);
int se_linear_head_fwd_strided(const float* x, int64_t ldx, const float* mean, const float* std, int64_t ld_stats,
                               float cmvn_eps, const float* W, int64_t ldw, const float* b, int64_t n_utt,
                               int64_t n_frames, int64_t D_in, int64_t D_out, int act, const float* linears,
                               float* offset_out, float* predicted_out, int64_t ld_out, int precision, void* stream);
int se_linear_head_bwd(const float* x, const float* mean, const float* std, float cmvn_eps, const float* W,
                       const float* offset, const float* grad_offset, int64_t n_utt, int64_t n_frames,
                       int64_t D_in, int64_t D_out, int act, float* grad_W, float* grad_b, void* stream);

/* se_linear_head_bwd_fused: se_linear_head_bwd_tc with the CMVN statistics given as the sums se_stft_features wrote (the
 * counterpart of se_linear_head_fused: same mean / unbiased std arithmetic); stat_sums NULL = no CMVN. */
int se_linear_head_bwd_fused(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps,
                             const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt, int64_t n_frames,
                             int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W,
                             float* grad_b, void* stream);

/* se_linear_head_bwd_sisdr: se_linear_head_bwd_fused with the backward of objective.SISDR on predicted = offset * linear_inp
 * (objective.py:86-100 after model.py:33) folded in: d loss / d offset is rebuilt per element from offset, linear_inp, linear_tar and
 * the per-utterance sums3 of se_sisdr_mask_fwd / _step (same arithmetic as se_sisdr_mask_bwd with grad_out = 1 / n_utt), so grad_offset
 * is never written or read.  lengths / len_hop as in se_sisdr_mask_step.  Operands must be 16-byte aligned with row strides that are
 * multiples of 4 floats (se_linear_head_bwd_sisdr_supported; otherwise SE_ERR_UNSUPPORTED: use se_sisdr_mask_bwd + _bwd_fused). */
int se_linear_head_bwd_sisdr_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                       int64_t ld_inp, int64_t ld_tar);
int se_linear_head_bwd_sisdr(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                             int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                             const int64_t* lengths, int64_t len_hop, const double* sums3, float loss_eps, int64_t n_utt, int64_t n_frames,
                             int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W, float* grad_b,
                             void* stream);

/* se_linear_head_bwd_wsd: se_linear_head_bwd_fused with the backward of objective.WSD folded in: d loss / d offset =
 * (1 / n_utt) (alpha 2 (S - G S)(-S) voiced + (1 - alpha) 2 G max(X - S, 0)^2) is rebuilt per element from offset (G), linear_inp (X)
 * and linear_tar (S), with one voiced flag per frame from energy and the threshold from max_energy (se_wsd_energy, after any
 * all-reduce), so grad_offset is never written or read.  Padded frames carry no gradient.  lengths / len_hop as in se_wsd_mask_step.
 * Same operands and alignment rules as se_linear_head_bwd_sisdr (_supported; otherwise SE_ERR_UNSUPPORTED: use se_wsd_mask_step's
 * grad_offset + se_linear_head_bwd_fused). */
int se_linear_head_bwd_wsd_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                     int64_t ld_inp, int64_t ld_tar);
int se_linear_head_bwd_wsd(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                           int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                           const int64_t* lengths, int64_t len_hop, const float* energy, const float* max_energy, float alpha,
                           float db_interval, float loss_eps, int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act,
                           float* ws_partials, int64_t ws_floats, float* grad_W, float* grad_b, void* stream);

/* ---- spectral SI-SDR objective on predicted = offset * linear_inp (objective.py:86-100 after model.py:33) ----------------
 * Same sums / loss as se_sisdr_spec_fwd without materialising `predicted`; rows of the three tensors are ld_* floats apart
 * (float4 loads when every ld is a multiple of 4 and the pointers are 16-byte aligned).  offset NULL: predicted = linear_inp.
 * bwd: grad_offset = grad_out[u] * d loss_u / d predicted * linear_inp (0 on padded frames and on columns >= K of a row). */
int se_sisdr_mask_fwd(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                      int64_t ld_tar, const int64_t* stft_len, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                      double* sums3, float* loss_per_utt, void* stream);
int se_sisdr_mask_bwd(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                      int64_t ld_tar, const int64_t* stft_len, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                      const double* sums3, const float* grad_out, float* grad_offset, int64_t ld_g, void* stream);
/* se_sisdr_mask_step: the objective's part of one training step (runner.py:455-460) in three launches: the sums, the
 * per-utterance losses + their batch mean (objective.py:100; loss_mean: 1 float, loss_per_utt may be NULL) and
 * grad_offset = d loss_mean / d offset.  lengths: frame counts (len_hop = 0) or SAMPLE lengths with len_hop = hop, in which
 * case frames = length / hop + 1 is taken in the kernels (runner.py:455).  sums_zeroed != 0: sums3 is already zero.  grad_offset NULL:
 * the backward launch is skipped (se_linear_head_bwd_sisdr rebuilds the gradient inside the weight-gradient kernel). */
int se_sisdr_mask_step(const float* offset, int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar,
                       int64_t ld_tar, const int64_t* lengths, int64_t len_hop, int64_t n_utt, int64_t n_frames, int64_t K, float eps,
                       double* sums3, int sums_zeroed, float* loss_per_utt, float* loss_mean, float* grad_offset, int64_t ld_g,
                       void* stream);

/* ---- active sampling (sampler.py:59-120, driven by runner.py:383-411) ----------------------------------------------------
 * se_head_grad_embeddings: per-UTTERANCE gradients of the head -- row u of grads_out (n_utt, D_out*D_in + D_out) is
 *   [d loss_u / d W (row-major), d loss_u / d b], the vector sampler.scoring builds with one backward call per utterance.
 *   grad_offset holds d loss_u / d offset for every utterance at once (utterances do not interact, e.g. se_sisdr_mask_bwd
 *   with grad_out = 1).  The split-K weight-gradient kernel runs with one split per utterance, so its partials are the answer.
 *   CMVN of x: mean and std, or stat_sums, or neither.  ws: se_head_grad_embeddings_workspace(...) floats (0 = unsupported).
 * se_match_scores: sampler.matching -- scores[j] = <key_j / (|key_j| + eps), mean_i query_i / (|query_i| + eps)>;
 *   ws_d: n_query + 2 n_key doubles, ws_qbar: P floats. */
int64_t se_head_grad_embeddings_workspace(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out);
int se_head_grad_embeddings(const float* x, int64_t ldx, const float* mean, const float* std, const double* stat_sums,
                            int64_t ld_stats, float cmvn_eps, const float* offset, const float* grad_offset, int64_t ld_off,
                            int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws, int64_t ws_floats,
                            float* grads_out, void* stream);
int se_match_scores(const float* query, int64_t n_query, const float* key, int64_t n_key, int64_t P, float eps, double* ws_d,
                    float* ws_qbar, float* scores, void* stream);

/* se_head_grad_embeddings_sisdr: se_head_grad_embeddings for objective.SISDR on predicted = offset * linear_inp with the objective's
 * backward folded in (as se_linear_head_bwd_sisdr, upstream gradient 1 per utterance): row u of grads_out is the gradient of the loss
 * of utterance u ALONE (sampler.py:95-108).  Workspace: se_head_grad_embeddings_workspace.  Aligned operands only (_supported). */
int se_head_grad_embeddings_sisdr_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ld_off,
                                            int64_t ld_inp, int64_t ld_tar);
int se_head_grad_embeddings_sisdr(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps, const float* offset,
                                  int64_t ld_off, const float* linear_inp, int64_t ld_inp, const float* linear_tar, int64_t ld_tar,
                                  const int64_t* lengths, int64_t len_hop, const double* sums3, float loss_eps, int64_t n_utt,
                                  int64_t n_frames, int64_t D_in, int64_t D_out, int act, float* ws, int64_t ws_floats, float* grads_out,
                                  void* stream);

/* ---- gradient clipping + Adam on the head's parameters (runner.py:463-466: clip_grad_norm_ then optimizer.step) -------
 * params / grads / exp_avg / exp_avg_sq: HOST arrays of n_tensors device pointers (se_adam_clip_step: <= 8, its original limit;
 * se_adam_clip_step_mirror: <= 32, e.g. a bidirectional 3-layer LSTM body and its projection, 26 tensors), numels their sizes.
 * Semantics of
 * torch.nn.utils.clip_grad_norm_(max_norm) (skipped if max_norm <= 0; the scaled gradient is written back) followed by
 * torch.optim.Adam.step (L2 weight_decay, no amsgrad).  A NaN / inf gradient norm skips the update (runner.py:467-470):
 * parameters, moments and the step count keep their values and the skipped-step counter advances.  ws_acc: 1 double,
 * ws_state: 3 ints (steps taken, internal, steps skipped), all zero before the first call and owned by the caller; the
 * counts advance on the device (CUDA-graph replayable). */
int se_adam_clip_step(float* const* params, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                      const int64_t* numels, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                      float max_norm, double* ws_acc, int* ws_state, void* stream);
/* se_adam_clip_step_mirror: the same step; additionally tensor t (viewed as rows of mirror_cols[t] elements) is written to
 * mirrors[t] with mirror_lds[t] floats between rows (mirrors NULL or mirrors[t] NULL: none) -- the 16-byte-row copy of the
 * head weight that the TMA / tensor-core head reads, rounded to TF32 (nearest, ties away) if mirror_tf32 != 0 -- so the copy
 * follows the parameters inside the same launch (skipped steps leave both untouched). */
int se_adam_clip_step_mirror(float* const* params, float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
                             const int64_t* numels, int n_tensors, float lr, float beta1, float beta2, float eps, float weight_decay,
                             float max_norm, float* const* mirrors, const int64_t* mirror_cols, const int64_t* mirror_lds,
                             int mirror_tf32, double* ws_acc, int* ws_state, void* stream);

/* ---- K1 + K2 of the fused evaluation step ------------------------------------------
 * se_stft_features: STFT of one channel -> ONE feature tensor feat (n_utt, n_frames, feat_stride): power (take_log = 0)
 *   or log(power + log_eps) (take_log = 1), AND stat_sums (n_utt, ld_stats, 2) doubles += [sum_f x, sum_f x^2] per
 *   (utterance, bin) over all n_frames -- the CMVN statistics of model.py:30 in one-pass form.  stat_sums is zeroed
 *   first unless flags has SE_FLAG_SUMS_ZEROED.  (runner.py:433,558 preprocessor call + model.py:30.)
 * se_feature_sums: the same sums from an existing feature tensor x (rows ldx floats apart); overwrites sums.
 * se_linear_head_fused: offset = act(((x - mean)/(std + cmvn_eps)) W^T + b) with mean / unbiased std derived from
 *   stat_sums (NULL = no CMVN); tcgen05 TF32 (W is read as TF32: pass it pre-rounded for round-to-nearest).
 *   One CTA per <=128-row tile, TMA tensor-map loads, accumulators in tensor memory, bulk-store epilogue.
 *   Returns SE_ERR_UNSUPPORTED outside its shape range (se_linear_head_fused_supported(...) == 0):
 *   D_in <= 544, D_out <= 544 (more than 272 output columns run as column slabs), n_frames >= 8, ldx and ldw multiples of 4,
 *   16-byte aligned x and W, and for D_out <= 272 a 128-row staging tile of ld_out (ld_out == round4(D_out)) or round4(D_out) + 4
 *   floats per row that fits the 200 KB ring. */
int se_stft_features(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                     float log_eps, int take_log, float* feat, int64_t feat_stride, double* stat_sums, int64_t ld_stats,
                     int flags, void* stream);
int se_feature_sums(const float* x, int64_t ldx, int64_t n_utt, int64_t n_frames, int64_t D, double* sums, int64_t ld_stats,
                    void* stream);
int se_linear_head_fused_supported(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out, int64_t ldx, int64_t ldw,
                                   int64_t ld_out);
int se_linear_head_fused(const float* x, int64_t ldx, const double* stat_sums, int64_t ld_stats, float cmvn_eps,
                         const float* W, int64_t ldw, const float* b, int64_t n_utt, int64_t n_frames, int64_t D_in,
                         int64_t D_out, int act, float* offset_out, int64_t ld_out, void* stream);

/* se_stft_features2: se_stft_features with BOTH spectral tensors of the channel -- power ("linear", what the objectives and
 * `predicted = linears * offset` consume) and log-power (the head's feature) -- from one transform; either may be NULL.
 * stat_sums holds the sums of logpower if it is given, else of power.  One launch for n_fft 512 / hop 256, 1024 / 256 and 400 / 160. */
int se_stft_features2(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t T, int n_fft, int hop, const float* window,
                      float log_eps, float* power, float* logpower, int64_t spec_stride, double* stat_sums, int64_t ld_stats,
                      int flags, void* stream);
/* se_stft_features_pair: se_stft_features2 of the input channel AND the power spectrum of a second channel (the clean target,
 * runner.py:433: linear_tar) in ONE launch of the register-resident kernels (n_fft 512 / hop 256, 1024 / 256 and 400 / 160;
 * se_stft_features_pair_supported, else SE_ERR_UNSUPPORTED: call se_stft_features2 twice).  wav points at the input channel of
 * utterance 0, the second channel lies chan_step floats further in every utterance.  power2: (2, n_utt, n_frames, spec_stride) --
 * [0] the input channel's power, [1] the second channel's; logpower / stat_sums: the input channel only. */
int se_stft_features_pair_supported(int n_fft, int hop);
int se_stft_features_pair(const float* wav, int64_t n_utt, int64_t utt_stride, int64_t chan_step, int64_t T, int n_fft, int hop,
                          const float* window, float log_eps, float* power2, float* logpower, int64_t spec_stride, double* stat_sums,
                          int64_t ld_stats, int flags, void* stream);

/* Tensor-core form of se_linear_head_bwd (tcgen05 TF32 split-K GEMM; grad_b from a ones column of the same GEMM).
 * ws_partials: caller workspace of se_linear_head_bwd_tc_workspace(...) floats (0 = shape unsupported: D_in <= 271 and
 * n_frames >= 32).  A split of the rows touches at most 8 utterances: large batches of short utterances get shorter splits, and
 * then more of them than one wave of CTAs.  ldx / ld_off = floats between rows of x / of offset and grad_offset. */
int64_t se_linear_head_bwd_tc_workspace(int64_t n_utt, int64_t n_frames, int64_t D_in, int64_t D_out);
int se_linear_head_bwd_tc(const float* x, int64_t ldx, const float* mean, const float* std, int64_t ld_stats, float cmvn_eps,
                          const float* offset, const float* grad_offset, int64_t ld_off, int64_t n_utt, int64_t n_frames,
                          int64_t D_in, int64_t D_out, int act, float* ws_partials, int64_t ws_floats, float* grad_W,
                          float* grad_b, void* stream);

/* ---- K1b: feature post-processing (S3PRL OnlinePreprocessor feature configs:
 * config/pretrain_sample.yaml:54-65, config/pseudo_noise.yaml:10-15) ------------------
 * se_mel: out[u,f,m] = log?(sum_k power[u,f,k] * fb[k,m] (+eps)), fb (K, n_mels) row-major
 * se_delta: 5-tap regression deltas with replicate padding along time, order-times
 *           recursive, reading columns [0, D) of x and writing columns [D, (order+1)*D)
 *           of the same (n_utt, n_frames, (order+1)*D) buffer
 * se_cmvn_apply: x = (x - mean) / (std + eps) per (utterance, feature) in place */
int se_mel(const float* power, int64_t n_rows, int64_t K, const float* fb, int64_t n_mels, int take_log, float eps,
           float* out, int64_t out_row_stride, void* stream);
int se_delta(float* x, int64_t n_utt, int64_t n_frames, int64_t D, int order, void* stream);
/* The mel feature configs in ONE launch (pretrain_sample.yaml:54-59 "mel, log, delta 1, cmvn"; pseudo_noise.yaml:10-15
 * "mel, log, delta 2"): out (n_utt, n_frames, ld_out) columns [0, (order+1) n_mels) = [mel | delta | delta-delta] of
 * log?(power fb (+eps)), deltas as se_delta (order <= 2, n_mels <= 64).  stat_sums (n_utt, (order+1) n_mels, 2) doubles or
 * NULL: zeroed here, then [sum_f x, sum_f x^2] per column -- what se_cmvn_apply_sums turns into the CMVN
 * x = (x - mean) / (unbiased std + eps) in place.  fb_ranges (n_mels, 2) int32 device array or NULL: [first bin, last bin + 1)
 * where filter m is non-zero -- the triangular filters are sparse, so the projection costs ~2 K instead of 40 K
 * multiply-adds per frame (NULL: dense). */
int se_mel_features(const float* power, int64_t ld_power, int64_t n_utt, int64_t n_frames, int64_t K, const float* fb,
                    const int32_t* fb_ranges, int64_t n_mels, int take_log, float eps, int order, float* out, int64_t ld_out,
                    double* stat_sums, void* stream);
int se_cmvn_apply_sums(float* x, int64_t n_utt, int64_t n_frames, int64_t D, const double* sums, float eps, void* stream);
int se_cmvn_apply(float* x, int64_t n_utt, int64_t n_frames, int64_t D, const float* mean, const float* std,
                  float eps, void* stream);

/* ---- a13 + a1 on the device: batch synthesis (dataset.py:106-111 normalize_wav_decibel, 54-74 add_noise, 128-161
 * __getitem__, 169-179 collate_fn; SURVEY 8f rank 3) ------------------------------------
 * Per utterance u: speech[u, :speech_len[u]] and noise[u, :noise_len[u]] are RMS-normalised to target_level_db, the noise is
 * tiled (or cropped) to the speech length and scaled to snr_db[u] (add_noise's formula with eps), and
 * wavs_out[u] = [noisy, speech, scaled_noise] (3, T_out), zero beyond speech_len[u] -- collate_fn's output for the batch.
 * The reference's sample lengths are the speech lengths; T_out >= max(speech_len).  ws_sums4: (n_utt, 4) doubles. */
int se_mix_batch(const float* speech, int64_t speech_stride, const int64_t* speech_len, const float* noise, int64_t noise_stride,
                 const int64_t* noise_len, const float* snr_db, int64_t n_utt, int64_t T_out, float target_level_db, float eps,
                 double* ws_sums4, float* wavs_out, void* stream);

/* ---- a1: host batch -> device (dataset.py:169-179 collate_fn output; runner.py:431, 556) ----
 * Copies channels [0, n_ch) of a pinned HOST batch h_wavs (B, C, T) into a compact device batch
 * d_wavs (B, n_ch, T) with one strided async copy (the path consumes the noisy and clean channels
 * only; the scaled-noise channel never crosses PCIe). */
int se_h2d_channels(const float* h_wavs, int64_t B, int64_t C, int64_t T, int64_t n_ch, float* d_wavs, void* stream);
/* The same for 16-bit PCM host batches (what the corpora's wav files hold: dataset.py:96-103 reads them into floats on the
 * host): channels [0, n_ch) of h_pcm (B, C, T) int16 cross PCIe as 2 bytes per sample into the staging buffer
 * d_pcm (B, n_ch, T) int16, and one kernel widens them to d_wavs (B, n_ch, T) fp32 = sample / 32768 (exact). */
int se_h2d_channels_pcm16(const int16_t* h_pcm, int64_t B, int64_t C, int64_t T, int64_t n_ch, int16_t* d_pcm, float* d_wavs,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SE_B200_H */
