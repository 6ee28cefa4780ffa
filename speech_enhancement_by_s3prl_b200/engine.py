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
    def step_workspace(self, B, device):
        """Persistent, zeroed workspace of one captured evaluation step: [CMVN sums (B, round4(K), 2) | K3 sums (B, 6)] doubles.
        The step's kernels leave it zeroed for the next replay (SE_FLAG_WS_SELF_CLEAN), so the graph has no fill node."""
        LD = ops.round4(self.n_fft // 2 + 1)
        return torch.zeros(B * (2 * LD + ops.NSUMS), device=device, dtype=torch.float64)

    def eval_step(self, lengths, wavs, want_spec_loss=True, metric_acc=None, ws=None, want_stoi=False, stoi_acc=None):
        """lengths (B,) int64, wavs (B, C, T) fp32, both on the GPU.
        Returns dict(loss_per_utt (B,), sisdr (B,), wav_predicted (B, T), gain (B,)); loss_per_utt is None when
        want_spec_loss is False (the spectral SI-SDR sums are not computed then).
        metric_acc: float64 (3,) device tensor += [sum loss, sum SI-SDR, utterances] (the running sums of an evaluation
        pass, runner.py:587-602; ``dp.means_from_acc`` turns them into the global means with one all-reduce).  Without
        want_spec_loss the loss sum is left as it is; SI-SDR and the count are still added.
        ws: a ``step_workspace`` that this call may use and must leave zeroed (captured steps); None = a fresh one per call.
        want_stoi: also return "stoi" and "estoi" (B,) of wav_predicted against the target channel, at the preprocessor's
        sample rate (``ops.stoi``); stoi_acc: float64 (3,) device tensor += [sum STOI, sum ESTOI, utterances]."""
        B, C, T = wavs.shape
        dev = wavs.device
        window = self.pre._frame_window
        if window.device != dev:
            self.pre.to(dev)
            window = self.pre._frame_window
        head = self.head
        K = self.n_fft // 2 + 1
        with torch.no_grad():
            # internal tensors use rows padded to 16 bytes (K = 257 -> 260 floats): TMA / 128-bit loads for the
            # tensor-core head; nothing outside this function sees the padding
            LD = ops.round4(K)
            F = T // self.hop + 1
            wpad = self._padded_weight()
            Dout = wpad.shape[0]
            D = self._mel_feature_dim() if self.feat_cfg is not None else K
            if self.feat_cfg is not None:
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
                wav, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                           pad_to=T, want_sums=True, want_spec=want_spec_loss, mask_padded=True)
            elif self.precision == 1 and ops.linear_head_tma_supported(B, F, K, Dout, LD, wpad.shape[1], ops.round4(Dout)):
                # K1 (+ CMVN sums) -> K2 (TMA + tcgen05 head) -> K3 -> K3': one zeroed workspace, no other memset, so
                # the four kernels are chained by programmatic dependent launches
                self.launches_per_step = 4      # K1, K2, K3, K3' (+ torch's fill of the workspace unless `ws` is given)
                self_clean = ws is not None
                if ws is None:
                    ws = torch.zeros(B * (2 * LD + ops.NSUMS), device=dev, dtype=torch.float64)
                stat_sums = ws[:B * 2 * LD].view(B, LD, 2)
                sums = ws[B * 2 * LD:].view(B, ops.NSUMS)
                feats, _ = ops.stft_features(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=self.log_features,
                                             log_eps=self.pre.eps, stat_sums=stat_sums, self_clean=self_clean)
                mask = ops.linear_head_tma(feats, K, wpad, head.linear.bias, head.activation,
                                             stat_sums if head.cmvn else None, head.eps)
                wav, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                           pad_to=T, want_sums=True, want_spec=want_spec_loss, mask_padded=True, sums=sums,
                                           sums_zeroed=True, self_clean=self_clean)
            else:
                feats = ops.stft_padded(wavs, self.ch_inp, self.n_fft, self.hop, window, logpower=self.log_features, log_eps=self.pre.eps)
                mean = std = None
                if head.cmvn:
                    mean, std = ops.cmvn_stats_padded(feats, K)
                mask = ops.linear_head_padded(feats, K, wpad, head.linear.bias, head.activation, mean, std,
                                              head.eps, precision=self.precision)
                wav, sums = ops.mask_istft(wavs, self.ch_inp, self.ch_tar, mask, lengths, self.n_fft, self.hop, window,
                                           pad_to=T, want_sums=True, want_spec=want_spec_loss, mask_padded=True)
            gain, sisdr, loss = ops.finalize_metrics(sums, lengths, T, wav=wav, target_db=None, want_loss=want_spec_loss,
                                                     metric_acc=metric_acc)
            out = {"loss_per_utt": loss, "sisdr": sisdr, "wav_predicted": wav, "gain": gain, "mask": mask[..., :K]}
            if want_stoi:
                # after K3' (both metrics are invariant to the gain of the estimate); the clean channel is read in place
                out["stoi"], out["estoi"] = ops.stoi(wav, wavs[:, self.ch_tar], lengths, fs=self.pre._sample_rate, acc=stoi_acc)
        return out

    def _padded_weight(self, force=False):
        """16-byte-row (and, for the tensor cores, TF32-rounded) copy of the head weight.

        ONE persistent buffer per (shape, device): captured graphs bake its address in, so it is refreshed IN PLACE --
        eagerly here when the parameter's version changed (optimizer.step / load_state_dict), and by kernels inside the
        captured training step after every update (``force``; graph replays never bump ``_version``)."""
        w = self.head.linear.weight
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
        return buf

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def capture_bound(self, lengths, wavs, metric_acc=None, want_stoi=False, stoi_acc=None):
        """Capture eval_step into a CUDA graph that reads the GIVEN device tensors in place
        (no staging copy).  Returns dict(graph=, lengths=, wavs=, loss_per_utt=, sisdr=, wav_predicted=, ...).
        metric_acc, want_stoi, stoi_acc: see eval_step (every replay adds the batch's sums to the accumulators)."""
        device = wavs.device
        ops.prepare(self.n_fft)
        if self.pre._frame_window.device != device:
            self.pre.to(device)
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        ws = self.step_workspace(wavs.shape[0], device)          # zeroed once here; every replay leaves it zeroed
        with torch.cuda.stream(side):
            for _ in range(2):                                   # warm up allocator + lazy init outside capture
                self.eval_step(lengths, wavs, ws=ws, want_stoi=want_stoi)   # (no accumulators: warm-up batches are not part of a pass)
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = self.eval_step(lengths, wavs, metric_acc=metric_acc, ws=ws, want_stoi=want_stoi, stoi_acc=stoi_acc)
        static = {"lengths": lengths, "wavs": wavs, "graph": graph, "ws": ws}
        static.update(out)
        return static

    def capture(self, B, C, T, device):
        """Graph with its own static input buffers for a fixed (B, C, T); cached."""
        key = (B, C, T, str(device))
        if key not in self._graphs:
            lengths = torch.full((B,), T, dtype=torch.int64, device=device)
            wavs = torch.zeros(B, C, T, device=device).normal_(0, 0.05)
            self._graphs[key] = self.capture_bound(lengths, wavs)
        return self._graphs[key]

    def eval_step_graph(self, lengths, wavs):
        """Same result as eval_step through the cached graph (inputs are copied into its static buffers)."""
        B, C, T = wavs.shape
        st = self.capture(B, C, T, wavs.device)
        self._padded_weight()                                       # in-place refresh if the parameters changed since capture
        st["lengths"].copy_(lengths, non_blocking=True)
        st["wavs"].copy_(wavs, non_blocking=True)
        st["graph"].replay()
        return st

    # ------------------------------------------------------------------ host-facing step (e2e)
    def eval_step_host(self, lengths_cpu, wavs_cpu):
        """The call a user makes with collate_fn's output (CPU tensors): H2D of the batch, the fused
        step, D2H of the per-utterance loss terms and SI-SDR.  Returns (mean_loss, mean_sisdr, wav_predicted on device)."""
        pipe = self.host_pipeline(*wavs_cpu.shape, depth=1)
        pipe.submit(lengths_cpu, wavs_cpu)
        loss, sisdr = pipe.drain()[0]
        return float(loss.mean()), float(sisdr.mean()), pipe.slots[0]["wav_predicted"]

    def host_pipeline(self, B, C, T, depth=2, device=None, pcm16=False, want_wav=False, copy_wav=True):
        """Host-facing evaluation loop for (B, C, T) batches; see HostPipeline.  pcm16: the host batches are int16 PCM
        (half the PCIe bytes; widened on the device); want_wav: the enhanced waveforms come back to pinned host memory
        (copy_wav=False: as views of the slot's pinned buffer, valid until that slot is submitted to again)."""
        key = ("pipe", B, C, T, depth, bool(pcm16), bool(want_wav), bool(copy_wav))
        if key not in self._graphs:
            device = device or torch.device("cuda", torch.cuda.current_device())
            self._graphs[key] = HostPipeline(self, B, C, T, depth, device, pcm16=pcm16, want_wav=want_wav, copy_wav=copy_wav)
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
        """True if train_step can take the fused route: LinearResidual with the SISDR or the WSD objective and the tensor-core
        head, on the (log-)power spectrum or on a mel feature config (pseudo_noise.yaml:10-15), shapes inside the TMA head's / the
        split-K backward's range."""
        from . import model, objective as obj
        if not self.fused_training or self.precision != 1 or type(objective) not in (obj.SISDR, obj.WSD):
            return False
        if type(self.head) is not model.LinearResidual:
            return False
        F, K = T // self.hop + 1, self.n_fft // 2 + 1
        LD = ops.round4(K)
        D = K if self.feat_cfg is None else self._mel_feature_dim()
        if D is None or D % 4 and self.feat_cfg is not None:
            return False
        if self.head.linear.weight.shape != (K, D):
            return False
        return (ops.linear_head_tma_supported(B, F, D, K, ops.round4(D), ops.round4(D), LD) and ops.linear_head_bwd_fused_supported(B, F, D, K))

    def _fused_forward_backward(self, lengths, wavs, objective):
        """runner.py:431-460 in seven kernels, no autograd graph: K1 (noisy: power + log-power + CMVN sums), K1 (clean:
        power), TMA head, SISDR sums + finish on offset * linear_inp, its backward straight to grad_offset, split-K
        tensor-core weight gradient + reduction.  With a mel ``feat_cfg`` the head input comes from the fused K1b kernel
        (mel -> log -> deltas) and one sums pass instead.  objective.WSD: the frame energies of linear_tar and their maximum
        first (all-reduced across data-parallel ranks on a side stream while the head runs), then the WSD sums + finish and
        its backward in the weight-gradient kernel.  Leaves the gradients in ``.grad`` and returns the loss."""
        from . import objective as obj
        wsd = type(objective) is obj.WSD
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
                if self.log_features:        # one K1 launch for both channels where the register-resident kernel exists
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
            if self.feat_cfg is not None or linear_tar is None:
                linear_tar = ops.stft_padded(wavs, self.ch_tar, self.n_fft, self.hop, window, logpower=False)
            wpad = self._padded_weight()            # current: refreshed in place after every update (_clip_and_step)
            stats = stat_sums if head.cmvn else None
            if wsd:
                # the voicing threshold needs the loudest frame of the GLOBAL batch: its 4-byte all-reduce runs on a side stream
                # under the head's forward (nothing to fork at world size 1)
                energy, emax = ops.wsd_energy(linear_tar, K)
                main = torch.cuda.current_stream(dev)
                side = self._side_stream(dev) if dp.world()[1] > 1 else None
                if side is not None:
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        dp.global_max(emax)
            offset = ops.linear_head_tma(feats, D, wpad, head.linear.bias, head.activation, stats, head.eps)
            # frames = lengths // hop + 1, the batch-mean loss and d loss / d offset inside three launches
            lens = _c64(lengths)
            fold = (ops.linear_head_bwd_wsd_supported if wsd else ops.linear_head_bwd_sisdr_supported)(
                B, feats.shape[1], D, K, feats.shape[2], offset.shape[2], linear_inp.shape[2], linear_tar.shape[2])
            if wsd:
                if side is not None:
                    main.wait_stream(side)
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

    def _side_stream(self, device):
        """One side stream per device for the WSD maximum's all-reduce (kept: a captured step records it as a fork / join)."""
        key = str(device)
        if key not in self._side_streams:
            self._side_streams[key] = torch.cuda.Stream(device=device)
        return self._side_streams[key]

    def _clip_and_step(self, optimizer, grad_clip):
        """runner.py:463-470; two launches with se_b200.ClipAdam (NaN / inf norms skipped on the device), torch's kernels
        with any other optimizer (the guard is then the runner's host-side check, which cannot run under graph capture)."""
        from .optim import ClipAdam
        if isinstance(optimizer, ClipAdam):
            # the update kernel also writes the padded / TF32 copy the head kernels read (one persistent buffer, see _padded_weight)
            w = self.head.linear.weight
            buf = self._padded_weight()
            optimizer.clip_and_step(grad_clip, mirrors={w: buf}, mirror_tf32=self.precision == 1)
            self._wpad_key = (w.data_ptr(), w._version)
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
        if optimizer is not None and self.fused_training_supported(objective, wavs.shape[0], wavs.shape[2]):
            optimizer.zero_grad(set_to_none=True)
            loss = self._fused_forward_backward(lengths, wavs, objective)
            dp.allreduce_gradients(self.head.parameters())
            self._clip_and_step(optimizer, grad_clip)
            return loss
        c = self.pre.get_feat_config
        feat_cfg = self.feat_cfg or c("linear", self.ch_inp, log=self.log_features)
        feats, linear_inp, linear_tar = self.pre(wavs, [feat_cfg, c("linear", self.ch_inp), c("linear", self.ch_tar)])
        predicted, extra = self.head(features=feats, linears=linear_inp)
        frames = lengths // self.hop + 1
        loss, _ = objective(predicted=predicted, linear_tar=linear_tar, linear_inp=linear_inp, stft_lengths=frames, **extra)
        if optimizer is not None:
            optimizer.zero_grad(set_to_none=True)
            loss.backward()
            dp.allreduce_gradients(self.head.parameters())
            self._clip_and_step(optimizer, grad_clip)
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
            with torch.cuda.graph(graph):
                st["loss"] = self._train_body(st["lengths"], st["wavs"], objective, optimizer, grad_clip)
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
            loss = self._fused_forward_backward(lengths, wavs, objective)
            dp.allreduce_gradients(self.head.parameters())
            self._clip_and_step(optimizer, grad_clip)
            return loss
        c = self.pre.get_feat_config
        feat_cfg = self.feat_cfg or c("linear", self.ch_inp, log=self.log_features)
        feats, linear_inp, linear_tar = self.pre(wavs, [feat_cfg, c("linear", self.ch_inp), c("linear", self.ch_tar)])
        predicted, extra = self.head(features=feats, linears=linear_inp)
        frames = lengths // self.hop + 1
        loss, _ = objective(predicted=predicted, linear_tar=linear_tar, linear_inp=linear_inp, stft_lengths=frames, **extra)
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

    def __init__(self, engine, B, C, T, depth, device, pcm16=False, want_wav=False, copy_wav=True):
        assert engine.ch_inp in (0, 1) and engine.ch_tar in (0, 1), "pipeline ships channels 0 and 1 only"
        self.engine, self.shape, self.device = engine, (B, C, T), device
        self.pcm16, self.want_wav, self.copy_wav = bool(pcm16), bool(want_wav), bool(copy_wav)
        self.copy_stream = torch.cuda.Stream(device=device)
        self.compute_stream = torch.cuda.Stream(device=device)
        self.slots = []
        self.pending = []
        self.h2d_bytes = B * self.N_CH * T * (2 if pcm16 else 4) + B * 8
        self.d2h_bytes = 2 * B * 4 + (B * T * 4 if want_wav else 0)
        self.launches_per_step = 5 + (1 if pcm16 else 0)
        with torch.cuda.stream(self.compute_stream):
            for _ in range(depth):
                lengths = torch.full((B,), T, dtype=torch.int64, device=device)
                wavs = torch.zeros(B, self.N_CH, T, device=device).normal_(0, 0.05)
                st = engine.capture_bound(lengths, wavs)
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
