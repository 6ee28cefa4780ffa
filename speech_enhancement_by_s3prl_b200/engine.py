"""Fused evaluation / training step of the enhancement path.

``EnhancementEngine.eval_step`` computes what the reference's evaluation step computes
(runner.py:556-602): features of the noisy channel -> mask head -> enhanced waveform
(``_decode_wav``: iSTFT with the noisy phase, zero-pad, level-match to the clean reference)
-> spectral SISDR criterion -> per-utterance waveform SI-SDR -- in four kernels:

  K1  se_stft            noisy wav -> (log-)power features               read 4H  write 4K  /frame
  K2  se_cmvn_stats + se_linear_head_fwd   features -> mask             read 4K  write 4K
  K3  se_mask_istft      noisy+clean wav, mask -> enhanced wav + sums    read 8H+4K write 4H
  K3' se_finalize_metrics  gain, SI-SDR, loss terms; wav *= gain (in place)

Nothing else is materialised: no noise-channel STFT, no phase, no `predicted`, no int64 masks.
"""
import ctypes
import os

import torch

from . import _lib, dp, ops


def _c64(lengths):
    """contiguous int64 lengths (what the kernels read)"""
    return lengths if lengths.dtype == torch.int64 and lengths.is_contiguous() else lengths.to(torch.int64).contiguous()


def _eval_loss(criterion, head=None):
    """The evaluation step's loss: "sisdr" for None / objective.SISDR (spectral SI-SDR), "wsd" for objective.WSD, "l1" for
    objective.L1, "wave" for objective.WaveSISDR (any head: it reads the waveform).  The pairs follow the reference's ``criterion(**locals(), **model_results)`` call (runner.py:575): WSD reads
    ``offset`` (LinearResidual, Residual), L1 reads ``log_predicted`` (LSTM); any other pair raises, as the reference raises
    TypeError."""
    from . import model, objective as obj
    kind = type(head).__name__ if head is not None else None
    if criterion is None or type(criterion) is obj.SISDR:
        return "sisdr"
    if type(criterion) is obj.WSD and (head is None or type(head) in (model.LinearResidual, model.Residual)):
        return "wsd"
    if type(criterion) is obj.L1 and (head is None or type(head) is model.LSTM):
        return "l1"
    if type(criterion) is obj.WaveSISDR:
        return "wave"
    raise RuntimeError(f"EnhancementEngine: no evaluation route for the criterion {type(criterion).__name__}"
                       f"{' with a ' + kind + ' head' if kind else ''} (supported: None, objective.SISDR, objective.WSD with "
                       "LinearResidual / Residual, objective.L1 with LSTM, objective.WaveSISDR)")


def _criterion_key(criterion):
    """What a captured evaluation step bakes in of its criterion."""
    loss = _eval_loss(criterion)
    if loss == "wsd":
        return ("WSD", float(criterion.alpha), float(criterion.db_interval), float(criterion.eps))
    if loss == "l1":
        return ("L1", float(criterion.eps))
    if loss == "wave":
        return ("WaveSISDR",)
    return None


def _recurrent(head):
    """True for the heads with a cuDNN LSTM body (model.LSTM, model.Residual)."""
    from . import model
    return type(head) in (model.LSTM, model.Residual)


class EnhancementEngine:
    def __init__(self, preprocessor, head, log_features=True, precision=0, feat_cfg=None):
        """preprocessor: se_b200 OnlinePreprocessor (gives n_fft / hop / window, channel_inp/tar);
        head: se_b200 LinearResidual on the (log-)power spectrum of the input channel.
        feat_cfg: a preprocessor feature config (``get_feat_config``) for the head's input instead of the (log-)power
        spectrum -- e.g. the baseline feature of config/pseudo_noise.yaml:10-15, mel + log + delta 2 (120-d); the training
        step then takes the autograd route through the custom ops (the fused routes are for spectrum-in / spectrum-out heads)."""
        self.pre = preprocessor
        self.head = head
        self.log_features = bool(log_features)
        self.precision = precision
        self.feat_cfg = feat_cfg
        self.n_fft = preprocessor._win_args["n_fft"]
        self.hop = preprocessor._win_args["hop_length"]
        self.ch_inp = int(getattr(preprocessor, "channel_inp", 0))
        self.ch_tar = int(getattr(preprocessor, "channel_tar", 1))
        self._graphs = {}
        self._side_streams = {}
        self.fused_training = os.environ.get("SE_B200_FUSED_TRAIN", "1") != "0"  # train_step without autograd (see fused_training_supported)
        self.launches_per_step = 5          # library kernels per eval_step (set by eval_step: 4 on the fused path)

    # ------------------------------------------------------------------ device-resident step
    def step_workspace(self, B, device, criterion=None):
        """Persistent, zeroed workspace of one captured evaluation step: [CMVN sums (B, round4(K), 2) | K3 sums (B, 6)] doubles,
        + one double (the WSD maximum and the finish kernel's CTA counter) with an objective.WSD criterion, or two (the L1 sum
        and element count) with objective.L1.
        The step's kernels leave it zeroed for the next replay (SE_FLAG_WS_SELF_CLEAN), so the graph has no fill node."""
        return torch.zeros(ops.step_workspace_doubles(B, self.n_fft, _eval_loss(criterion)), device=device, dtype=torch.float64)

    def eval_step(self, lengths, wavs, want_spec_loss=True, metric_acc=None, ws=None, want_stoi=False, stoi_acc=None,
                  criterion=None):
        """lengths (B,) int64, wavs (B, C, T) fp32, both on the GPU.
        Returns dict(loss_per_utt (B,), sisdr (B,), wav_predicted (B, T), gain (B,)); loss_per_utt is None when
        want_spec_loss is False (the loss terms are not computed then).
        criterion: the objective the validation loss is reported in (runner.py:575): None or an objective.SISDR (the spectral
        SI-SDR), or an objective.WSD (its alpha, db_interval and eps; the voicing threshold comes from the loudest frame of the
        global batch, so under data parallelism every rank must run the step for every batch).  On the register-resident
        geometries (n_fft / hop 512 / 256, 1024 / 256, 400 / 160) the WSD terms come out of K3 itself; on any other geometry
        from both channels' power spectra through ops.wsd_energy / ops.wsd_mask_step -- a slower route that materialises them.
        objective.L1 (model.LSTM heads only): loss_per_utt[u] is utterance u's own L1 and out["loss"] (1,) the batch's -- the
        element mean over every rank's valid frames (its [sum, count] pair is all-reduced), which is what the criterion returns;
        metric_acc[0] += B * loss.  Other geometries and steps under 6 frames take a slower route through the clean power spectrum.
        objective.WaveSISDR (any head): loss_per_utt = -sisdr, the step's own waveform SI-SDR (sisdr_eval's eps, 1e-10), from the
        same K3 sums; metric_acc[0] += their sum on the device.
        head: LinearResidual (fused K1 / K2), or a recurrent LSTM / Residual: the cuDNN body runs through torch between K1 and the
        library's projection; LSTM's output is log_predicted and K3 decodes exp(log_predicted) with the noisy phase.
        metric_acc: float64 (3,) device tensor += [sum loss, sum SI-SDR, utterances] (the running sums of an evaluation
        pass, runner.py:587-602; ``dp.means_from_acc`` turns them into the global means with one all-reduce).  Without
        want_spec_loss the loss sum is left as it is; SI-SDR and the count are still added.
        ws: a ``step_workspace`` (of the same criterion) that this call may use and must leave zeroed (captured steps); None = a
        fresh one per call.
        want_stoi: also return "stoi" and "estoi" (B,) of wav_predicted against the target channel, at the preprocessor's
        sample rate (``ops.stoi``); stoi_acc: float64 (3,) device tensor += [sum STOI, sum ESTOI, utterances]."""
        head = self.head
        crit = _eval_loss(criterion, head) if want_spec_loss else (_eval_loss(criterion, head) and "sisdr")
        wsd, l1, wave = crit == "wsd", crit == "l1", crit == "wave"
        want_spec_loss = want_spec_loss and crit == "sisdr"     # the spectral SI-SDR sums of K3
        log_power = type(head).__name__ == "LSTM"               # K3 decodes exp(log_predicted)
        B, C, T = wavs.shape
        dev = wavs.device
        window = self.pre._frame_window
        if window.device != dev:
            self.pre.to(dev)
            window = self.pre._frame_window
        K = self.n_fft // 2 + 1
        with torch.no_grad():
            # internal tensors use rows padded to 16 bytes (K = 257 -> 260 floats): TMA / 128-bit loads for the
            # tensor-core head; nothing outside this function sees the padding
            LD = ops.round4(K)
            F = T // self.hop + 1
            wpad = self._padded_weight()
            Dout = wpad.shape[0]
            D = self._mel_feature_dim() if self.feat_cfg is not None else K
            state = None                                         # the criterion's persistent state at the workspace's end
            if ws is not None:
                state = ops.step_workspace_views(ws, B, self.n_fft)[2]
            if _recurrent(head):
                mask = self._recurrent_front(wavs, D, wpad)
                k3 = {}
            elif self.feat_cfg is not None:
                # head input = a mel feature config (e.g. pseudo_noise.yaml:10-15) built by the fused K1b kernel from the
                # power spectrum; the mask still applies to the K bins of the noisy spectrum
                if D is None or D % 4 or Dout != K or not ops.linear_head_tma_supported(B, F, D, K, D, wpad.shape[1], LD):
                    raise RuntimeError("EnhancementEngine.eval_step: feat_cfg must be a mel config (log / delta <= 2, no CMVN of its "
                                       "own) feeding a LinearResidual(D, K) head with the tensor-core path (precision=1)")
                cfg = self.feat_cfg
                self.launches_per_step = 7      # K1, K1b, sums (+ its zero fill), K2, K3, K3'
                power = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=False)
                feats = ops.mel_features(power, self.pre._tables(dev)[1], bool(cfg.get("log", False)), self.pre.eps,
                                         order=int(cfg.get("delta", 0)), K=K)
                stat_sums = ops.feature_sums(feats, D) if head.cmvn else None
                mask = ops.linear_head_tma(feats, D, wpad, head.linear.bias, head.activation, stat_sums, head.eps)
                k3 = {}
            elif self.precision == 1 and ops.linear_head_tma_supported(B, F, K, Dout, LD, wpad.shape[1], ops.round4(Dout)):
                # K1 (+ CMVN sums) -> K2 (TMA + tcgen05 head) -> K3 -> K3': one zeroed workspace, no other memset, so
                # the four kernels are chained by programmatic dependent launches
                self.launches_per_step = 4      # K1, K2, K3, K3' (+ torch's fill of the workspace unless `ws` is given)
                if ws is None:                  # a fresh zeroed one, used once: the kernels need not clean it
                    stat_sums, sums, state = ops.step_workspace_views(self.step_workspace(B, dev, criterion), B, self.n_fft)
                    k1, k3 = dict(stat_sums=stat_sums), dict(sums=sums, sums_zeroed=True)
                else:
                    k1 = k3 = dict(ws=ws)
                feats, stat_sums = ops.stft_features(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=self.log_features,
                                                     log_eps=self.pre.eps, **k1)
                mask = ops.linear_head_tma(feats, K, wpad, head.linear.bias, head.activation,
                                             stat_sums if head.cmvn else None, head.eps)
            else:
                self.launches_per_step = 5      # K1, K2 (+ CMVN statistics), the sums' fill, K3, K3'
                feats = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=self.log_features, log_eps=self.pre.eps)
                mean = std = None
                if head.cmvn:
                    mean, std = ops.cmvn_stats_padded(feats, K)
                mask = ops.linear_head_padded(feats, K, wpad, head.linear.bias, head.activation, mean, std,
                                              head.eps, precision=self.precision)
                k3 = {}
            batch_loss = None
            # K3' without the loss terms, for the L1 / WSD routes (their finish kernels compute those after the all-reduce)
            finalize = lambda: ops.finalize_metrics(sums, lengths, T, wav=wav, target_db=None, want_loss=False, metric_acc=metric_acc)
            if l1:
                # K3 (log-power target) with the L1 sums, or the slow route -> all-reduce of [sum, count] on the side stream under
                # K3' -> the finish kernel
                l1_acc = state if state is not None and state.numel() == 2 else torch.zeros(2, device=dev, dtype=torch.float64)
                self.launches_per_step += 1                         # the finish kernel (K3-L1 replaces K3)
                if ops.mask_istft_register_resident(self.n_fft, self.hop, T):
                    wav, sums = ops.mask_istft_l1(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                                  pad_to=T, l1_acc=l1_acc, eps=criterion.eps, **k3)
                else:
                    wav, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                               pad_to=T, want_sums=True, want_spec=False, mask_padded=True, mask_is_log_power=True,
                                               **k3)
                    self._l1_terms_from_spectra(wavs, mask, lengths, criterion, sums, l1_acc)
                gain, sisdr, _ = self._all_reduce_beside(dp.reduce_sums, l1_acc, finalize)
                loss, batch_loss = ops.l1_eval_finish(sums, lengths, T, self.hop, K, l1_acc, metric_acc)
            elif wsd and ops.mask_istft_register_resident(self.n_fft, self.hop, T):
                # K3 with the WSD terms -> all-reduce(max) of its 4-byte maximum on the side stream under K3' -> the finish kernel
                self.launches_per_step += 1
                if state is not None and state.numel() == 1:
                    state = state.view(torch.float32)                  # the step leaves it zeroed
                else:
                    state = torch.zeros(2, device=dev, dtype=torch.float32)
                wav, sums, terms = ops.mask_istft_wsd(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                                      pad_to=T, wsd_state=state, **k3)
                gain, sisdr, _ = self._all_reduce_beside(dp.global_max, state[:1], finalize)
                loss = ops.wsd_eval_finish(terms, sums, state, criterion.alpha, criterion.db_interval, criterion.eps, metric_acc)
            else:
                wav, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                           pad_to=T, want_sums=True, want_spec=want_spec_loss, mask_padded=True,
                                           mask_is_log_power=log_power, **k3)
                gain, sisdr, loss = ops.finalize_metrics(sums, lengths, T, wav=wav, target_db=None, want_loss=want_spec_loss,
                                                         metric_acc=metric_acc)
                if wsd:
                    self.launches_per_step += 8     # 2 STFTs, energies (+ fill), sums (+ fill), finish, the accumulator's sum + add
                    loss = self._wsd_terms_from_spectra(wavs, mask, lengths, criterion, metric_acc)
                elif wave:
                    loss = sisdr.neg()              # objective.WaveSISDR's terms are the step's own metric, bit for bit
                    self.launches_per_step += 1
                    if metric_acc is not None:
                        metric_acc[:1].sub_(sisdr.sum(dtype=torch.float64))
                        self.launches_per_step += 2
            out = {"loss_per_utt": loss, "sisdr": sisdr, "wav_predicted": wav, "gain": gain, "mask": mask[..., :K]}
            if batch_loss is not None:
                out["loss"] = batch_loss
            if want_stoi:
                # after K3' (both metrics are invariant to the gain of the estimate); the clean channel is read in place
                out["stoi"], out["estoi"] = ops.stoi(wav, wavs[:, self.ch_tar], lengths, fs=self.pre._sample_rate, acc=stoi_acc)
        return out

    def _recurrent_front(self, wavs, D, wpad):
        """K1 -> cuDNN LSTM body (torch, no_grad) -> [Residual's CMVN over the hidden states, torch] -> the library's projection
        (TMA head when the hidden width is a multiple of 4 and precision=1, else the padded head) -> mask (B, F, round4(K)):
        model.LSTM's log_predicted or model.Residual's offset.  launches_per_step counts everything but the body."""
        feats = self._recurrent_k1(wavs, D)[0]
        hidden = self._recurrent_body(self._recurrent_input(feats, D, "eval_step"))
        mask = self._recurrent_project(hidden, wpad)
        self.launches_per_step = (2 if self.feat_cfg is not None else 1) + int(D != feats.shape[2])   # K1 (+ K1b), the copy
        self.launches_per_step += 5 if self._recurrent_cmvn() else 0
        self.launches_per_step += 1 + 3                                  # projection, K3's sums fill, K3, K3'
        return mask

    def _recurrent_k1(self, wavs, D, spectra=False):
        """K1 of the recurrent routes: the head's input (B, F, LD) -- the (log-)power spectrum of the input channel, or the mel feature
        of ``feat_cfg`` -- and with ``spectra`` also both channels' power spectra linear_inp and linear_tar (B, F, round4(K)) that the
        training step's objectives read (one launch for all three where the register-resident pair kernel exists).  Returns
        (feats, linear_inp | None, linear_tar | None)."""
        dev, window = wavs.device, self.pre._frame_window
        K = self.n_fft // 2 + 1
        linear_inp = linear_tar = None
        if self.feat_cfg is not None:
            if D is None:
                raise RuntimeError(f"EnhancementEngine.{'train_step' if spectra else 'eval_step'}: feat_cfg must be a mel config "
                                   "(log / delta <= 2, no CMVN of its own)")
            cfg = self.feat_cfg
            linear_inp = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=False)
            feats = ops.mel_features(linear_inp, self.pre._tables(dev)[1], bool(cfg.get("log", False)), self.pre.eps,
                                     order=int(cfg.get("delta", 0)), K=K)
        elif not spectra:
            feats = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=self.log_features, log_eps=self.pre.eps)
        elif self.log_features:
            linear_inp, feats, linear_tar, _ = ops.stft_features_pair(wavs, self.ch_inp, self.ch_tar, self.n_fft, self.hop, window,
                                                                      log_eps=self.pre.eps)
        else:
            feats = linear_inp = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=False)
        if spectra and linear_tar is None:
            linear_tar = ops.stft_padded(wavs, self.ch_tar, self.n_fft, self.hop, window, logpower=False)
        return feats, linear_inp, linear_tar

    def _recurrent_input(self, feats, D, caller):
        """The recurrent head's input (B, F, D), copied out of K1's 16-byte padded rows where they are wider than D."""
        head = self.head
        if head.lstm.input_size != D:
            raise RuntimeError(f"EnhancementEngine.{caller}: the {type(head).__name__} head takes {head.lstm.input_size} features, "
                               f"the engine's feature has {D}")
        x = feats[..., :D]
        return x if x.is_contiguous() else x.contiguous()

    def _recurrent_cmvn(self):
        return type(self.head).__name__ == "Residual" and self.head.cmvn

    def _recurrent_body(self, x):
        """The cuDNN LSTM body (DESIGN section 7) [+ Residual's CMVN over every frame of the padded batch, model.py:88] in torch:
        recorded for autograd when grad mode is on.  Returns the projection's input (B, F, hidden * directions), contiguous."""
        head = self.head
        hidden, _ = head.lstm(x)
        if self._recurrent_cmvn():
            hidden = (hidden - hidden.mean(dim=1, keepdim=True)) / (hidden.std(dim=1, keepdim=True) + head.eps)
        return hidden.contiguous()

    def _recurrent_project(self, hidden, wpad):
        """The library's projection of the hidden states -> (B, F, round4(K)): the TMA head when the hidden width is a multiple of 4
        at precision 1, else the padded head."""
        B, F, H = hidden.shape
        K = self.n_fft // 2 + 1
        if self.precision == 1 and H % 4 == 0 and ops.linear_head_tma_supported(B, F, H, K, H, wpad.shape[1], ops.round4(K)):
            return ops.linear_head_tma(hidden, H, wpad, self._proj().bias, self.head.activation, None, 0.0)
        return ops.linear_head_padded(hidden, H, wpad, self._proj().bias, self.head.activation, None, None, 0.0,
                                      precision=self.precision)

    def _l1_terms_from_spectra(self, wavs, mask, lengths, criterion, sums, l1_acc):
        """objective.L1's sums where K3 has no L1 variant (other geometries, or fewer than 6 frames): the clean power spectrum is
        materialised (one more STFT) and one reduction (se_l1_eval_sums) adds each utterance's sum to its SE_SUM_SPEC_ST column of
        `sums` and the batch's [sum, count] to l1_acc -- what K3-L1 adds on the fused route."""
        T = wavs.shape[2]
        tar = ops.stft_padded(wavs, self.ch_tar, self.n_fft, self.hop, self.pre._frame_window, logpower=False)
        ops.l1_eval_sums(mask, tar, lengths, T, self.hop, self.n_fft // 2 + 1, sums, l1_acc, criterion.eps)
        self.launches_per_step += 2

    def _proj(self):
        """The head's output layer: LinearResidual.linear, or LSTM / Residual.scaling_layer[0]."""
        return self.head.scaling_layer[0] if _recurrent(self.head) else self.head.linear

    def _wsd_terms_from_spectra(self, wavs, mask, lengths, criterion, metric_acc):
        """objective.WSD's per-utterance terms where K3 has no WSD variant (other geometries, or fewer than 6 frames): both
        channels' power spectra are materialised (B, F, LD) and go through the training step's split kernels -- energies and
        their maximum (all-reduced across ranks), then the sums.  The slow route: two more STFTs and three passes over spectra."""
        K = self.n_fft // 2 + 1
        window = self.pre._frame_window
        linear_inp = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=False)
        linear_tar = ops.stft_padded(wavs, self.ch_tar, self.n_fft, self.hop, window, logpower=False)
        energy, emax = ops.wsd_energy(linear_tar, K)
        dp.global_max(emax)
        _, loss, _, _ = ops.wsd_mask_step(mask, linear_inp, linear_tar, lengths, self.hop, K, energy, emax, criterion.alpha,
                                          criterion.db_interval, criterion.eps, want_grad=False)
        if metric_acc is not None:
            metric_acc[:1] += loss.sum(dtype=torch.float64)
        return loss

    def _padded_weight(self, force=False):
        """16-byte-row (and, for the tensor cores, TF32-rounded) copy of the head weight.

        ONE persistent buffer per (shape, device): captured graphs bake its address in, so it is refreshed IN PLACE --
        eagerly here when the parameter's version changed (optimizer.step / load_state_dict), and by kernels inside the
        captured training step after every update (``force``; graph replays never bump ``_version``)."""
        w = self._proj().weight
        Dout, Din = w.shape
        buf = getattr(self, "_wpad", None)
        if buf is None or buf.device != w.device or buf.shape != (Dout, ops.round4(Din)):
            buf = self._wpad = torch.zeros(Dout, ops.round4(Din), device=w.device, dtype=torch.float32)
            self._wpad_key = None
            self._graphs = {}                    # graphs captured against another buffer are void
        key = (w.data_ptr(), w._version)
        if force or self._wpad_key != key:
            with torch.no_grad():
                buf[:, :Din].copy_(w.detach())
                if self.precision == 1:          # the tensor cores read TF32: round to nearest once (cvt.rna)
                    bits = buf.view(torch.int32)
                    bits.add_(0x1000).bitwise_and_(~0x1FFF)
            self._wpad_key = key
            self._refresh_weight_t()
        return buf

    def _padded_weight_t(self):
        """The transposed copy of ``_padded_weight``, (Din, round4(Dout)) with zero pad columns: the weight operand of the recurrent
        training step's input gradient dH = dZ W (the TMA head run on W^T).  A second persistent buffer under the same version key,
        refreshed in place whenever the first one is (also by the captured step after every update), so graphs always read the
        trained weights.  TF32 values copied from the rounded buffer stay TF32."""
        buf = self._padded_weight()
        Din = self._proj().weight.shape[1]
        if self._weight_t() is None:
            self._wtpad = torch.zeros(Din, ops.round4(buf.shape[0]), device=buf.device, dtype=torch.float32)
            self._refresh_weight_t()
        return self._wtpad

    def _weight_t(self):
        """The W^T buffer if it exists and matches the current padded weight, else None (and the stale one is dropped)."""
        wt, buf = getattr(self, "_wtpad", None), getattr(self, "_wpad", None)
        if wt is not None and (buf is None or wt.device != buf.device or
                               wt.shape != (self._proj().weight.shape[1], ops.round4(buf.shape[0]))):
            wt = self._wtpad = None
        return wt

    def _refresh_weight_t(self):
        wt = self._weight_t()
        if wt is not None:
            with torch.no_grad():
                wt[:, :self._wpad.shape[0]].copy_(self._wpad[:, :wt.shape[0]].t())

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def capture_bound(self, lengths, wavs, metric_acc=None, want_stoi=False, stoi_acc=None, criterion=None):
        """Capture eval_step into a CUDA graph that reads the GIVEN device tensors in place
        (no staging copy).  Returns dict(graph=, lengths=, wavs=, loss_per_utt=, sisdr=, wav_predicted=, ...).
        metric_acc, want_stoi, stoi_acc, criterion: see eval_step (every replay adds the batch's sums to the accumulators;
        the criterion's constants are baked into the graph)."""
        device = wavs.device
        ops.prepare(self.n_fft)
        if self.pre._frame_window.device != device:
            self.pre.to(device)
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        ws = self.step_workspace(wavs.shape[0], device, criterion)   # zeroed once here; every replay leaves it zeroed
        with torch.cuda.stream(side):
            for _ in range(2):                                   # warm up allocator + lazy init outside capture
                self.eval_step(lengths, wavs, ws=ws, want_stoi=want_stoi, criterion=criterion)   # (no accumulators: warm-up
                                                                                                   # batches are not part of a pass)
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        try:
            with torch.cuda.graph(graph):
                out = self.eval_step(lengths, wavs, metric_acc=metric_acc, ws=ws, want_stoi=want_stoi, stoi_acc=stoi_acc,
                                     criterion=criterion)
        except RuntimeError as exc:
            if not _recurrent(self.head):
                raise
            raise RuntimeError(f"EnhancementEngine.capture_bound: the evaluation step of the {type(self.head).__name__} head could "
                               f"not be captured into a CUDA graph (eager eval_step still runs it): {exc}") from exc
        static = {"lengths": lengths, "wavs": wavs, "graph": graph, "ws": ws}
        static.update(out)
        return static

    def capture(self, B, C, T, device, criterion=None):
        """Graph with its own static input buffers for a fixed (B, C, T) and criterion; cached."""
        key = (B, C, T, str(device), _criterion_key(criterion))
        if key not in self._graphs:
            lengths = torch.full((B,), T, dtype=torch.int64, device=device)
            wavs = torch.zeros(B, C, T, device=device).normal_(0, 0.05)
            self._graphs[key] = self.capture_bound(lengths, wavs, criterion=criterion)
        return self._graphs[key]

    def eval_step_graph(self, lengths, wavs, criterion=None):
        """Same result as eval_step through the cached graph (inputs are copied into its static buffers)."""
        B, C, T = wavs.shape
        st = self.capture(B, C, T, wavs.device, criterion)
        self._padded_weight()                                       # in-place refresh if the parameters changed since capture
        st["lengths"].copy_(lengths, non_blocking=True)
        st["wavs"].copy_(wavs, non_blocking=True)
        st["graph"].replay()
        return st

    # ------------------------------------------------------------------ host-facing step (e2e)
    def eval_step_host(self, lengths_cpu, wavs_cpu, criterion=None):
        """The call a user makes with collate_fn's output (CPU tensors): H2D of the batch, the fused
        step, D2H of the per-utterance loss terms and SI-SDR.  Returns (mean_loss, mean_sisdr, wav_predicted on device).
        mean_loss is the criterion's value of the batch: the mean of the per-utterance terms, and for objective.L1 (an element
        mean) their mean weighted by each utterance's valid frames."""
        pipe = self.host_pipeline(*wavs_cpu.shape, depth=1, criterion=criterion)
        pipe.submit(lengths_cpu, wavs_cpu)
        loss, sisdr = pipe.drain()[0]
        if _eval_loss(criterion) == "l1":
            T = wavs_cpu.shape[2]
            frames = (lengths_cpu.to(torch.int64).clamp(0, T) // self.hop + 1).clamp(max=T // self.hop + 1).double()
            mean_loss = float((loss.double() * frames).sum() / frames.sum())
        else:
            mean_loss = float(loss.mean())
        return mean_loss, float(sisdr.mean()), pipe.slots[0]["wav_predicted"]

    def host_pipeline(self, B, C, T, depth=2, device=None, pcm16=False, want_wav=False, copy_wav=True, criterion=None):
        """Host-facing evaluation loop for (B, C, T) batches; see HostPipeline.  pcm16: the host batches are int16 PCM
        (half the PCIe bytes; widened on the device); want_wav: the enhanced waveforms come back to pinned host memory
        (copy_wav=False: as views of the slot's pinned buffer, valid until that slot is submitted to again);
        criterion: the loss the per-utterance terms are in (see eval_step); with objective.L1 they are each utterance's own L1,
        whose batch value is their mean weighted by valid frames, not their plain mean (eval_step_host returns the weighted one)."""
        key = ("pipe", B, C, T, depth, bool(pcm16), bool(want_wav), bool(copy_wav), _criterion_key(criterion))
        if key not in self._graphs:
            device = device or torch.device("cuda", torch.cuda.current_device())
            self._graphs[key] = HostPipeline(self, B, C, T, depth, device, pcm16=pcm16, want_wav=want_wav, copy_wav=copy_wav,
                                             criterion=criterion)
        return self._graphs[key]

    # ------------------------------------------------------------------ training step (head fwd + bwd)
    def _mel_feature_dim(self):
        """Width of the head input if ``feat_cfg`` is a mel feature the fused training route can build in one launch
        (mel [+ log] [+ delta <= 2] of the input channel, no CMVN of its own: the head normalises), else None."""
        cfg = self.feat_cfg
        if cfg is None or cfg.get("feat_type") != "mel" or cfg.get("cmvn") or int(cfg.get("delta", 0)) > 2:
            return None
        if int(cfg.get("channel", 0)) != self.ch_inp or self.pre._n_mels > 64:
            return None
        return (int(cfg.get("delta", 0)) + 1) * self.pre._n_mels

    def fused_training_supported(self, objective, B, T):
        """True if train_step can take the fused route: LinearResidual with the SISDR, WSD or WaveSISDR objective and the tensor-core
        head, on the (log-)power spectrum or on a mel feature config (pseudo_noise.yaml:10-15), shapes inside the TMA head's / the
        split-K backward's range.  Recurrent heads: model.LSTM with objective.L1 / WaveSISDR and model.Residual with objective.SISDR / WSD /
        WaveSISDR (with
        or without its CMVN), a hidden width (x directions) that is a multiple of 4, and both projections -- hidden -> K forward and
        K -> hidden for the input gradient -- on the TMA head (see _fused_recurrent_forward_backward).  Every other pair (e.g. LSTM
        with SISDR, or Linear) takes the autograd route."""
        from . import model, objective as obj
        if not self.fused_training or self.precision != 1:
            return False
        if _recurrent(self.head):
            return self._fused_recurrent_supported(objective, B, T)
        if type(objective) not in (obj.SISDR, obj.WSD, obj.WaveSISDR) or type(self.head) is not model.LinearResidual:
            return False
        F, K = T // self.hop + 1, self.n_fft // 2 + 1
        LD = ops.round4(K)
        D = K if self.feat_cfg is None else self._mel_feature_dim()
        if D is None or D % 4 and self.feat_cfg is not None:
            return False
        if self.head.linear.weight.shape != (K, D):
            return False
        return (ops.linear_head_tma_supported(B, F, D, K, ops.round4(D), ops.round4(D), LD) and ops.linear_head_bwd_fused_supported(B, F, D, K))

    def _fused_recurrent_supported(self, objective, B, T):
        from . import model, objective as obj
        head = self.head
        if not ((type(head) is model.LSTM and type(objective) in (obj.L1, obj.WaveSISDR)) or
                (type(head) is model.Residual and type(objective) in (obj.SISDR, obj.WSD, obj.WaveSISDR))):
            return False
        F, K = T // self.hop + 1, self.n_fft // 2 + 1
        LD = ops.round4(K)
        D = K if self.feat_cfg is None else self._mel_feature_dim()
        H = head.lstm.hidden_size * (2 if head.lstm.bidirectional else 1)
        if D is None or head.lstm.input_size != D or getattr(head.lstm, "proj_size", 0) or H % 4 or self._proj().weight.shape != (K, H):
            return False
        return (ops.linear_head_tma_supported(B, F, H, K, H, H, LD) and ops.linear_head_tma_supported(B, F, K, H, LD, LD, H) and
                ops.linear_head_bwd_fused_supported(B, F, H, K))

    def _fused_recurrent_forward_backward(self, lengths, wavs, objective):
        """runner.py:431-460 for model.LSTM + objective.L1 and model.Residual + objective.SISDR / WSD: the cuDNN body and Residual's
        CMVN stay in torch autograd (DESIGN section 7); everything around them runs on the library's padded kernels.
          K1 (both channels) -> copy out of the padded rows -> body (+ CMVN), recorded for autograd
          -> projection forward on the TMA head (detached hidden states) -> the objective's step: loss and d loss / d output
             (objective.WSD: its batch maximum all-reduced on the side stream under the projection; objective.WaveSISDR: K3 ->
             se_wave_sisdr_finish -> se_mask_istft_bwd, LSTM's output decoded as a log target power)
          -> act'(output) in place: dZ, read by both GEMMs -> weight / bias gradient (split-K TMA kernel)
          -> dH = dZ W (TMA head on the persistent TF32 W^T copy) -> torch.autograd.backward(hidden, dH): cuDNN BPTT [+ CMVN's].
        Leaves the gradients in ``.grad`` and returns the loss (objective.L1: the element mean of this rank's batch)."""
        from . import objective as obj
        head, dev = self.head, wavs.device
        if self.pre._frame_window.device != dev:
            self.pre.to(dev)
        K = self.n_fft // 2 + 1
        D = K if self.feat_cfg is None else self._mel_feature_dim()
        kind = type(objective)
        wave = kind is obj.WaveSISDR
        with torch.no_grad():
            feats, linear_inp, linear_tar = self._recurrent_k1(wavs, D, spectra=not wave)
            x = self._recurrent_input(feats, D, "train_step")
        with torch.enable_grad():
            hidden = self._recurrent_body(x)
        proj = self._proj()
        with torch.no_grad():
            wpad, wt = self._padded_weight(), self._padded_weight_t()
            h = hidden.detach()
            H = h.shape[2]
            head_fwd = lambda: ops.linear_head_tma(h, H, wpad, proj.bias, head.activation, None, 0.0)
            lens = _c64(lengths)
            if kind is obj.WSD:
                energy, emax = ops.wsd_energy(linear_tar, K)
                out = self._all_reduce_beside(dp.global_max, emax, head_fwd)
                loss, _, dz, _ = ops.wsd_mask_step(out, linear_inp, linear_tar, lens, self.hop, K, energy, emax, objective.alpha,
                                                   objective.db_interval, objective.eps)
            elif kind is obj.SISDR:
                out = head_fwd()
                loss, _, dz, _ = ops.sisdr_mask_step(out, linear_inp, linear_tar, lens, self.hop, K, objective.eps)
            elif wave:
                out = head_fwd()
                loss, dz = self._wave_sisdr_step(wavs, lens, out, objective, log_power=type(head).__name__ == "LSTM")
            else:
                out = head_fwd()
                loss, _, dz = ops.l1_mask_step(out, linear_tar, lens, self.hop, K, objective.eps)
            ops.act_grad_(dz, out, K, head.activation)                  # dZ = d loss / d pre-activation; pad columns 0
            gw, gb = ops.linear_head_bwd_fused(h, H, None, 0.0, out, dz, K, "Identity")
            dh = ops.linear_head_tma(dz, K, wt, None, "Identity", None, 0.0)
            for p, g in ((proj.weight, gw), (proj.bias, gb)):
                if p.grad is None:
                    p.grad = g
                else:
                    p.grad.add_(g)
        if hidden.requires_grad:                                         # (a frozen body: nothing below the projection trains)
            torch.autograd.backward(hidden, dh)
        return loss

    def _fused_forward_backward(self, lengths, wavs, objective):
        """runner.py:431-460 in seven kernels, no autograd graph: K1 (noisy: power + log-power + CMVN sums), K1 (clean:
        power), TMA head, SISDR sums + finish on offset * linear_inp, its backward straight to grad_offset, split-K
        tensor-core weight gradient + reduction.  With a mel ``feat_cfg`` the head input comes from the fused K1b kernel
        (mel -> log -> deltas) and one sums pass instead.  objective.WSD: the frame energies of linear_tar and their maximum
        first (all-reduced across data-parallel ranks on a side stream while the head runs), then the WSD sums + finish and
        its backward in the weight-gradient kernel.  Leaves the gradients in ``.grad`` and returns the loss."""
        from . import objective as obj
        wsd = type(objective) is obj.WSD
        wave = type(objective) is obj.WaveSISDR
        B, C, T = wavs.shape
        dev = wavs.device
        head = self.head
        window = self.pre._frame_window
        if window.device != dev:
            self.pre.to(dev)
            window = self.pre._frame_window
        K = self.n_fft // 2 + 1
        LD = ops.round4(K)
        with torch.no_grad():
            if self.feat_cfg is None:
                ws = torch.zeros(B * (2 * LD + 3), device=dev, dtype=torch.float64)
                stat_sums = ws[:B * 2 * LD].view(B, LD, 2)
                sums3 = ws[B * 2 * LD:].view(B, 3)
                linear_tar = None
                if wave:                     # the loss reads the clean waveform: K1 on the noisy channel only
                    linear_inp, logp, _ = ops.stft_features2(wavs, self.ch_inp, self.n_fft, self.hop, window,
                                                             want_power=not self.log_features, want_logpower=self.log_features,
                                                             log_eps=self.pre.eps, stat_sums=stat_sums)
                elif self.log_features:      # one K1 launch for both channels where the register-resident kernel exists
                    linear_inp, logp, linear_tar, _ = ops.stft_features_pair(wavs, self.ch_inp, self.ch_tar, self.n_fft, self.hop, window,
                                                                             log_eps=self.pre.eps, stat_sums=stat_sums)
                else:
                    linear_inp, logp, _ = ops.stft_features2(wavs, self.ch_inp, self.n_fft, self.hop, window, want_power=True,
                                                             want_logpower=False, log_eps=self.pre.eps, stat_sums=stat_sums)
                feats, D = (logp if self.log_features else linear_inp), K
            else:
                cfg = self.feat_cfg
                sums3 = torch.zeros(B, 3, device=dev, dtype=torch.float64)
                linear_inp = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=False)
                feats = ops.mel_features(linear_inp, self.pre._tables(dev)[1], bool(cfg.get("log", False)), self.pre.eps,
                                         order=int(cfg.get("delta", 0)), K=K)
                D = feats.shape[2]
                stat_sums = ops.feature_sums(feats, D) if head.cmvn else None
            if not wave and (self.feat_cfg is not None or linear_tar is None):
                linear_tar = ops.stft_padded(wavs, self.ch_tar, self.n_fft, self.hop, window, logpower=False)
            wpad = self._padded_weight()            # current: refreshed in place after every update (_clip_and_step)
            stats = stat_sums if head.cmvn else None
            head_fwd = lambda: ops.linear_head_tma(feats, D, wpad, head.linear.bias, head.activation, stats, head.eps)
            if wsd:
                # the voicing threshold needs the loudest frame of the GLOBAL batch: its 4-byte all-reduce runs on a side stream
                # under the head's forward
                energy, emax = ops.wsd_energy(linear_tar, K)
                offset = self._all_reduce_beside(dp.global_max, emax, head_fwd)
            else:
                offset = head_fwd()
            lens = _c64(lengths)
            if wave:
                loss, grad_offset = self._wave_sisdr_step(wavs, lens, offset, objective)
                gw, gb = ops.linear_head_bwd_fused(feats, D, stats, head.eps, offset, grad_offset, K, head.activation)
                for p, g in ((head.linear.weight, gw), (head.linear.bias, gb)):
                    p.grad = g if p.grad is None else p.grad.add_(g)
                return loss
            # frames = lengths // hop + 1, the batch-mean loss and d loss / d offset inside three launches
            fold = (ops.linear_head_bwd_wsd_supported if wsd else ops.linear_head_bwd_sisdr_supported)(
                B, feats.shape[1], D, K, feats.shape[2], offset.shape[2], linear_inp.shape[2], linear_tar.shape[2])
            if wsd:
                sums2 = sums3.view(-1)[:2 * B].view(B, 2)          # the zeroed workspace's sums part, as (B, 2)
                loss, _, grad_offset, _ = ops.wsd_mask_step(offset, linear_inp, linear_tar, lens, self.hop, K, energy, emax,
                                                            objective.alpha, objective.db_interval, objective.eps, sums2=sums2,
                                                            sums_zeroed=True, want_grad=not fold)
            else:
                loss, _, grad_offset, _ = ops.sisdr_mask_step(offset, linear_inp, linear_tar, lens, self.hop, K, objective.eps,
                                                               sums3=sums3, sums_zeroed=True, want_grad=not fold)
            if fold and wsd:    # the objective's backward runs inside the weight-gradient kernel: no grad_offset tensor
                gw, gb = ops.linear_head_bwd_wsd(feats, D, stats, head.eps, offset, linear_inp, linear_tar, lens, self.hop, energy, emax, K,
                                                 head.activation, objective.alpha, objective.db_interval, objective.eps)
            elif fold:
                gw, gb = ops.linear_head_bwd_sisdr(feats, D, stats, head.eps, offset, linear_inp, linear_tar, lens, self.hop, sums3, K,
                                                   head.activation, objective.eps)
            else:
                gw, gb = ops.linear_head_bwd_fused(feats, D, stats, head.eps, offset, grad_offset, K, head.activation)
            for p, g in ((head.linear.weight, gw), (head.linear.bias, gb)):
                if p.grad is None:
                    p.grad = g
                else:
                    p.grad.add_(g)
        return loss

    def _wave_sisdr_step(self, wavs, lengths, mask, objective, log_power=False):
        """objective.WaveSISDR's step on a mask (B, F, round4(K)) of the head: K3 (the enhanced waveform y and its sums, no gain
        pass) -> se_wave_sisdr_finish (the batch-mean loss and d loss / d y = alpha y + beta clean) -> se_mask_istft_bwd.
        Returns (loss (1,), d loss / d mask (B, F, round4(K)), pad columns 0)."""
        window, T = self.pre._frame_window, wavs.shape[2]
        y, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window, pad_to=T,
                                 want_sums=True, want_spec=False, mask_padded=True, mask_is_log_power=log_power)
        _, loss, coef = ops.wave_sisdr_finish(sums, objective.eps)
        grad = ops.mask_istft_bwd(wavs, self.ch_inp, self.ch_tar, y, coef, lengths, mask, self.n_fft, self.hop, window,
                                  mask_is_log_power=log_power)
        return loss, grad

    def _all_reduce_beside(self, all_reduce, buf, work):
        """all_reduce(buf) (dp.global_max / dp.reduce_sums) on the device's side stream while the current stream runs work();
        returns work()'s result with the current stream joined to the side stream.  At world size 1 there is nothing to reduce:
        only work() runs.  The side stream is one per device and kept, so that a captured step records it as a fork / join."""
        if dp.world()[1] == 1:
            return work()
        key = str(buf.device)
        if key not in self._side_streams:
            self._side_streams[key] = torch.cuda.Stream(device=buf.device)
        main, side = torch.cuda.current_stream(buf.device), self._side_streams[key]
        side.wait_stream(main)
        with torch.cuda.stream(side):
            all_reduce(buf)
        result = work()
        main.wait_stream(side)
        return result

    def _clip_and_step(self, optimizer, grad_clip):
        """runner.py:463-470; two launches with se_b200.ClipAdam (NaN / inf norms skipped on the device), torch's kernels
        with any other optimizer (the guard is then the runner's host-side check, which cannot run under graph capture)."""
        from .optim import ClipAdam
        if isinstance(optimizer, ClipAdam):
            # the update kernel also writes the padded / TF32 copy the head kernels read (one persistent buffer, see _padded_weight);
            # the recurrent step's transposed copy follows it
            w = self._proj().weight
            buf = self._padded_weight()
            optimizer.clip_and_step(grad_clip, mirrors={w: buf}, mirror_tf32=self.precision == 1)
            self._wpad_key = (w.data_ptr(), w._version)
            self._refresh_weight_t()
            return
        else:
            params = list(self.head.parameters())
            if grad_clip is not None:
                grad_norm = torch.nn.utils.clip_grad_norm_(params, grad_clip)
            else:
                grad_norm = torch.linalg.vector_norm(torch.stack([p.grad.norm() for p in params if p.grad is not None]))
            if torch.cuda.is_current_stream_capturing() or bool(torch.isfinite(grad_norm)):
                optimizer.step()
        # the padded / TF32 copy the kernels read follows the parameters inside the same (possibly captured) step
        self._padded_weight(force=True)

    def train_step(self, lengths, wavs, objective, optimizer=None, grad_clip=None):
        """runner.py:431-471 on the kernels: preprocessor tensors -> head -> criterion -> backward
        (+ gradient all-reduce under DP) -> optimizer step.  Returns the loss tensor."""
        if optimizer is None:
            return self._autograd_loss(lengths, wavs, objective)
        optimizer.zero_grad(set_to_none=True)
        return self._train_body(lengths, wavs, objective, optimizer, grad_clip)

    def _autograd_loss(self, lengths, wavs, objective):
        """The reference's forward through the custom ops (preprocessor -> head -> objective), recorded for autograd."""
        from . import objective as obj
        c = self.pre.get_feat_config
        feat_cfg = self.feat_cfg or c("linear", self.ch_inp, log=self.log_features)
        if type(objective) is obj.WaveSISDR:
            # wav_predicted = istft(predicted, phase_inp) zero-padded to T (runner.py:266-268, before the level normalisation,
            # which the scale-invariant loss does not need), through the differentiable ops.istft
            feats, linear_inp, phase_inp = self.pre(wavs, [feat_cfg, c("linear", self.ch_inp), c("phase", self.ch_inp)])
            predicted, _ = self.head(features=feats, linears=linear_inp)
            wav_predicted = ops.istft(predicted, phase_inp, self.n_fft, self.hop, self.pre._frame_window, pad_to=wavs.shape[2])
            loss, _ = objective(wav_predicted=wav_predicted, wav_tar=wavs[:, self.ch_tar], lengths=lengths)
            return loss
        feats, linear_inp, linear_tar = self.pre(wavs, [feat_cfg, c("linear", self.ch_inp), c("linear", self.ch_tar)])
        predicted, extra = self.head(features=feats, linears=linear_inp)
        frames = lengths // self.hop + 1
        loss, _ = objective(predicted=predicted, linear_tar=linear_tar, linear_inp=linear_inp, stft_lengths=frames, **extra)
        return loss

    def capture_train(self, lengths, wavs, objective, optimizer, grad_clip=None):
        """Capture the training step of one batch shape -- forward, backward, gradient all-reduce (NCCL under DP), clipping
        and the optimizer update -- into a CUDA graph with its own static input buffers; cached per (shape, objective,
        optimizer).  Returns dict(graph=, lengths=, wavs=, loss=): fill the inputs, ``graph.replay()``, read ``loss``."""
        B, C, T = wavs.shape
        key = ("train", B, C, T, id(objective), id(optimizer), grad_clip)
        st = self._graphs.get(key)
        if st is None:
            dev = wavs.device
            ops.prepare(self.n_fft)
            st = {"lengths": lengths.clone(), "wavs": wavs.clone()}
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):                                   # warm-up: lazy state of autograd, NCCL and the optimizer
                    self.train_step(st["lengths"], st["wavs"], objective, optimizer, grad_clip)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            optimizer.zero_grad(set_to_none=True)
            graph = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(graph):
                    st["loss"] = self._train_body(st["lengths"], st["wavs"], objective, optimizer, grad_clip)
            except RuntimeError as exc:
                if not _recurrent(self.head):
                    raise
                raise RuntimeError(f"EnhancementEngine.capture_train: the training step of the {type(self.head).__name__} head could "
                                   f"not be captured into a CUDA graph (eager train_step still runs it): {exc}") from exc
            st["graph"] = graph
            self._graphs[key] = st
        return st

    def train_step_graph(self, lengths, wavs, objective, optimizer, grad_clip=None):
        """``train_step`` replayed from a CUDA graph (the eager step is launch-bound: ~40 small launches).  The optimizer
        must be capturable (``se_b200.ClipAdam``, or e.g. ``torch.optim.Adam(..., capturable=True)``).  Returns the loss
        tensor of the static step (valid until the next call)."""
        st = self.capture_train(lengths, wavs, objective, optimizer, grad_clip)
        st["lengths"].copy_(lengths, non_blocking=True)
        st["wavs"].copy_(wavs, non_blocking=True)
        st["graph"].replay()
        return st["loss"]

    def _train_body(self, lengths, wavs, objective, optimizer, grad_clip):
        """forward + backward + update without ``zero_grad`` (inside a graph the gradients live in the graph's pool)."""
        if self.fused_training_supported(objective, wavs.shape[0], wavs.shape[2]):
            fused = self._fused_recurrent_forward_backward if _recurrent(self.head) else self._fused_forward_backward
            loss = fused(lengths, wavs, objective)
        else:
            loss = self._autograd_loss(lengths, wavs, objective)
            loss.backward()
        dp.allreduce_gradients(self.head.parameters())
        self._clip_and_step(optimizer, grad_clip)
        return loss


class HostPipeline:
    """Host-facing evaluation loop: pinned host batches in, per-utterance (loss term, SI-SDR) out.

    ``depth`` slots, each with its own device input buffers, captured graph and pinned result buffer.
    ``submit`` enqueues, on a copy stream, the H2D of the noisy and clean channels (one strided
    cudaMemcpy2DAsync; the scaled-noise channel is never used by the path and never crosses PCIe)
    and of the lengths; the compute stream then replays the slot's graph and copies the 2*B result
    floats back.  With depth 2 the copy of batch i+1 overlaps the kernels of batch i.

    ``pcm16``: the host batches are int16 PCM (the sample format of the corpora's wav files): 2 bytes per sample
    cross PCIe and one kernel widens them to the fp32 the path computes in (sample / 32768, exact).
    ``want_wav``: every step also copies the level-matched enhanced waveforms (B, T) fp32 back to pinned host memory
    (``drain`` then returns (loss_per_utt, sisdr, wav) triples) -- what an "enhance these files" caller needs;
    ``Runner.evaluate()`` itself only needs the metrics."""

    N_CH = 2

    def __init__(self, engine, B, C, T, depth, device, pcm16=False, want_wav=False, copy_wav=True, criterion=None):
        assert engine.ch_inp in (0, 1) and engine.ch_tar in (0, 1), "pipeline ships channels 0 and 1 only"
        self.engine, self.shape, self.device = engine, (B, C, T), device
        self.pcm16, self.want_wav, self.copy_wav = bool(pcm16), bool(want_wav), bool(copy_wav)
        self.copy_stream = torch.cuda.Stream(device=device)
        self.compute_stream = torch.cuda.Stream(device=device)
        self.slots = []
        self.pending = []
        self.h2d_bytes = B * self.N_CH * T * (2 if pcm16 else 4) + B * 8
        self.d2h_bytes = 2 * B * 4 + (B * T * 4 if want_wav else 0)
        self.launches_per_step = 5 + (1 if pcm16 else 0) + (0 if _eval_loss(criterion) == "sisdr" else 1)   # (+ a finish kernel)
        with torch.cuda.stream(self.compute_stream):
            for _ in range(depth):
                lengths = torch.full((B,), T, dtype=torch.int64, device=device)
                wavs = torch.zeros(B, self.N_CH, T, device=device).normal_(0, 0.05)
                st = engine.capture_bound(lengths, wavs, criterion=criterion)
                st["result_host"] = torch.empty(2, B).pin_memory()
                if self.pcm16:
                    st["pcm"] = torch.empty(B, self.N_CH, T, device=device, dtype=torch.int16)
                if self.want_wav:
                    st["wav_host"] = torch.empty(B, T).pin_memory()
                st["copied"] = torch.cuda.Event()
                st["done"] = torch.cuda.Event()
                st["busy"] = False
                self.slots.append(st)
        torch.cuda.synchronize(device)
        if _recurrent(engine.head):              # (the library's launches around the cuDNN body, see eval_step)
            self.launches_per_step = engine.launches_per_step + (1 if pcm16 else 0)
        self._next = 0

    def submit(self, lengths_cpu, wavs_cpu):
        if self._results is None:
            self._results = []
        B, C, T = self.shape
        want_dtype = torch.int16 if self.pcm16 else torch.float32
        if tuple(wavs_cpu.shape) != (B, C, T) or wavs_cpu.dtype != want_dtype or not wavs_cpu.is_contiguous():
            raise RuntimeError(f"HostPipeline.submit: expected a contiguous {want_dtype} batch of shape {(B, C, T)}, "
                               f"got {wavs_cpu.dtype} {tuple(wavs_cpu.shape)}")
        st = self.slots[self._next]
        self._next = (self._next + 1) % len(self.slots)
        if st["busy"]:
            self._collect(st)
        self.engine._padded_weight()                                # in-place refresh if the parameters changed since capture
        lib = _lib.load()
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(st["done"])              # previous use of this slot's inputs has finished
            if self.pcm16:
                rc = lib.se_h2d_channels_pcm16(wavs_cpu.data_ptr(), B, C, T, self.N_CH, st["pcm"].data_ptr(), st["wavs"].data_ptr(),
                                               self.copy_stream.cuda_stream)
                _lib.check(rc, "se_h2d_channels_pcm16")
            else:
                rc = lib.se_h2d_channels(wavs_cpu.data_ptr(), B, C, T, self.N_CH, st["wavs"].data_ptr(), self.copy_stream.cuda_stream)
                _lib.check(rc, "se_h2d_channels")
            st["lengths"].copy_(lengths_cpu, non_blocking=True)
            st["copied"].record(self.copy_stream)
        with torch.cuda.stream(self.compute_stream):
            self.compute_stream.wait_event(st["copied"])
            st["graph"].replay()
            st["result_host"][0].copy_(st["loss_per_utt"], non_blocking=True)
            st["result_host"][1].copy_(st["sisdr"], non_blocking=True)
            if self.want_wav:
                st["wav_host"].copy_(st["wav_predicted"][:, :T], non_blocking=True)
            st["done"].record(self.compute_stream)
        st["busy"] = True
        self.pending.append(st)

    def _collect(self, st):
        st["done"].synchronize()
        st["busy"] = False
        res = st["result_host"].clone()
        if self.want_wav:                           # (a 16 MB host copy per step unless the caller consumes the slot's buffer in place)
            self._results.append((res[0], res[1], st["wav_host"].clone() if self.copy_wav else st["wav_host"]))
        else:
            self._results.append((res[0], res[1]))
        self.pending.remove(st)

    _results = None

    def drain(self):
        """Wait for everything submitted; returns [(loss_per_utt, sisdr[, wav]), ...] in submission order."""
        if self._results is None:
            self._results = []
        for st in list(self.pending):
            self._collect(st)
        out, self._results = self._results, []
        return out
