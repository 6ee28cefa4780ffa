#!/usr/bin/env python
"""bench.py -- enhanced audio-seconds per second through the fused STFT -> mask -> iSTFT + loss path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1]): VoiceBank-DEMAND-shaped synthetic batch, 16 kHz, 64 x 4 s
utterances per GPU, n_fft=512 hop=256, LinearResidual mask head on the log-power spectrum, the
reference's evaluation step (runner.py:556-602): enhanced waveform level-matched to the clean
reference, spectral SISDR criterion, per-utterance waveform SI-SDR.  One step = one batch.

Own arm: `value` = device-timed graph replays with the batches already in HBM (inputs rotate over
a ring of distinct batches larger than L2); `e2e` = the same through EnhancementEngine's host
pipeline with pinned HOST batches, H2D and D2H inside the timed region.  `roofline` is for the
dominant kernel (fused mask -> iSTFT), timed with CUDA events around its launches.  `cpu_baseline`
(rank 0, N=1) times the CPU oracle -- the reference's un-fused sequence on torch CPU ops -- on the
host cores.  `--impl reference` runs that oracle alone as the reference arm (the reference is pure
Python whose STFT lives in an un-vendored dependency; see DESIGN.md).

The same JSON line carries a `configs` object with the other BASELINE.json configurations, each timed the same way
(device-resident, CUDA events, max over ranks) with its own algorithmic-bytes roofline fraction:
  configs[3] long-form: 1024 utterances of 60 s in total (STRONG scaling: 1024 / N per GPU), n_fft 1024 / hop 256;
  configs[2] training: the fused training step (forward, backward, NCCL gradient all-reduce inside the captured graph,
             clipping + Adam) at the reference's default n_fft 400 / hop 160;
  configs[4] scoring: per-utterance gradient embeddings of 12 + 32 utterances and their cosine matching.

Timed regions: the ranks are aligned by a collective ON THE STREAM right before the first event, the metric sums of the
pass accumulate on the device (se_finalize_metrics_acc) and are all-reduced once before the second event; nothing between
the events reads back to the host.  Every timed loop runs exactly --steps steps.

--dump-outputs DIR (rank 0): after the timed pass, the arrays its last step returned (EnhancementEngine.eval_step's
loss_per_utt, sisdr, gain, wav_predicted, mask) and the pass's device sums [sum loss, sum SI-SDR, utterances] are written
as DIR/<name>.npy, float32 (pass_sums: float64), about 33 MB in all.  The inputs are seeded, so two builds run with the
same arguments can be compared array for array.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "enhanced audio-sec/sec (STFT->mask->iSTFT+loss)"
UNIT = "audio-s/s"
SR = 16000
N_UTT, SECONDS, N_FFT, HOP = 64, 4.0, 512, 256
PRE_KW = dict(sample_rate=SR, win_ms=32, hop_ms=16, n_freq=257, n_mels=40, n_mfcc=13)
WORKLOAD = "configs[1]: VoiceBank-DEMAND-shaped synthetic, 16 kHz, 64x4s per GPU, n_fft=512 hop=256, LinearResidual(257) on log-power, eval step + SISDR + waveform SI-SDR"
GEOMETRY = {512: dict(win_ms=32, hop_ms=16, n_freq=257, hop=256), 1024: dict(win_ms=64, hop_ms=16, n_freq=513, hop=256),
            400: dict(win_ms=25, hop_ms=10, n_freq=201, hop=160)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons sampled by NVML in a background thread while the GPU is busy."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        self.index = index
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": "nvmlClocksEventReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksEventReasonHwThermalSlowdown",
                 "sw_thermal_slowdown": "nvmlClocksEventReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksEventReasonSwPowerCap"}
        bits = {k: getattr(nv, v, None) for k, v in names.items()}
        legacy = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
                  "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap"}
        for k, v in legacy.items():
            if bits[k] is None:
                bits[k] = getattr(nv, v, None)
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, b in bits.items():
                    if b is not None and mask & b:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self.thread.start()

    def stop(self):
        self._stop.set()
        if self.nv is not None and self.thread.is_alive():
            self.thread.join(timeout=1.0)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def oracle_objects():
    from oracle import signal_path as sp
    from oracle.preprocessor import OnlinePreprocessor as OraclePre
    ora = OraclePre(**PRE_KW)
    ora.channel_inp, ora.channel_tar = 0, 1
    c = ora.get_feat_config
    # the six tensors of run_downstream.py:150-157 with the log-power spectrum as up/downstream feature
    ora.feat_list = [c("linear", 0, log=True), c("linear", 0, log=True), c("linear", 0), c("phase", 0), c("linear", 1), c("phase", 1)]
    return sp, ora


def time_cpu_oracle(lengths, wavs, weight, bias, budget_s, min_reps=2, max_reps=50):
    """Best-of wall-clock of the un-fused reference sequence on the host cores (torch CPU, fp32, no_grad)."""
    sp, ora = oracle_objects()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    head = dict(weight=weight, bias=bias)
    times = []
    t_start = time.perf_counter()
    with torch.no_grad():
        sp.eval_step(ora, head, lengths, wavs)                     # warm-up (thread pools, FFT plans)
        while len(times) < max_reps and (len(times) < min_reps or time.perf_counter() - t_start < budget_s):
            t0 = time.perf_counter()
            sp.eval_step(ora, head, lengths, wavs)
            times.append(time.perf_counter() - t0)
    return min(times), cores, len(times)


def run_reference_arm(args, rank):
    """--impl reference: the CPU oracle port of the reference path on all host threads."""
    if rank != 0:
        return
    from speech_enhancement_by_s3prl_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sp, ora = oracle_objects()
    torch.manual_seed(1337)
    lin = torch.nn.Linear(257, 257)
    head = dict(weight=lin.weight.detach(), bias=lin.bias.detach())
    n_utt = N_UTT
    lengths, wavs = synth.batch(n_utt, SECONDS)
    with torch.no_grad():
        t0 = time.perf_counter()
        sp.eval_step(ora, head, lengths, wavs)
        first = time.perf_counter() - t0
        while first * (args.steps + args.warmup) > 150.0 and n_utt > 4:   # keep the whole run within a few minutes
            n_utt //= 2
            first /= 2
        lengths, wavs = lengths[:n_utt], wavs[:n_utt].contiguous()
        for _ in range(args.warmup):
            sp.eval_step(ora, head, lengths, wavs)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            sp.eval_step(ora, head, lengths, wavs)
        total = time.perf_counter() - t0
    audio_s = n_utt * SECONDS
    value = audio_s * args.steps / total
    sample = f"{n_utt}x{SECONDS:g}s per step ({'full batch' if n_utt == N_UTT else 'sub-sampled batch'}), {args.steps} steps"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "where": "host CPU, torch ops (torch.stft/istft) restating the reference's un-fused sequence"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- shared helpers
class Ctx:
    """Per-process state: rank, device, the process group, a scratch tensor for stream-side rank alignment."""

    def __init__(self, args):
        import torch.distributed as dist
        self.dist = dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        # one process per GPU: keep the process and its pinned host batches on the GPU's NUMA node (the e2e feed of 8 ranks)
        from speech_enhancement_by_s3prl_b200 import dp
        self.numa_node = dp.bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.align = torch.zeros(1, device=self.dev)
        self.peak, self.peak_src = peaks()

    def timed(self, run, warm_collective=True):
        """Device time of run() in ms, max over ranks.  A collective ON THE STREAM right before the first event aligns the
        ranks' device timelines (a host barrier leaves the CPUs, not the GPUs, aligned); run() ends with its own
        collective when the workload has one, so every rank's second event waits for the slowest rank."""
        dist = self.dist
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if self.world > 1:
            dist.barrier()
            dist.all_reduce(self.align)                            # stream-ordered: e0 is recorded after it completes everywhere
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()


DUMP_KEYS = ("loss_per_utt", "sisdr", "gain", "wav_predicted", "mask")


def dump_outputs(path, step_out, acc):
    """--dump-outputs: one step's eval_step arrays as float32 and the pass's float64 sums, as <path>/<name>.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: step_out[k].float() for k in DUMP_KEYS}
    arrays["pass_sums"] = acc.double()
    for name, t in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), t.detach().cpu().numpy())


def make_engine(se, ctx, n_fft, precision=1):
    g = GEOMETRY[n_fft]
    pre = se.OnlinePreprocessor(sample_rate=SR, win_ms=g["win_ms"], hop_ms=g["hop_ms"], n_freq=g["n_freq"], n_mels=40, n_mfcc=13).to(ctx.dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=g["n_freq"], output_size=g["n_freq"], precision=precision).to(ctx.dev)
    return pre, head, se.EnhancementEngine(pre, head, log_features=True, precision=precision)


def eval_step_bytes(audio_s, n_fft, hop):
    """SURVEY 8(d): 16 H + 16 K bytes per frame = 16 sr (1 + K / H) per audio-second."""
    K = n_fft // 2 + 1
    return audio_s * 16 * SR * (1 + K / hop)


def time_eval_kernels(ctx, se, engine, pre, head, slots_in, n_fft, hop, reps, graph=True):
    """Every kernel of the fused evaluation step timed ALONE with CUDA events: captured in a CUDA graph that launches it
    once per slot (distinct, HBM-cold inputs; no CPU launch gaps) when graph=True, else launched eagerly (kernels of
    many ms).  Returns (kernel_ms per launch, algorithmic bytes per launch)."""
    from speech_enhancement_by_s3prl_b200 import ops
    window = pre._frame_window
    wpad = engine._padded_weight()
    K = n_fft // 2 + 1
    LD = ops.round4(K)
    B, _, T = slots_in[0][1].shape
    F = T // hop + 1
    if not (engine.precision == 1 and ops.linear_head_tma_supported(B, F, K, K, LD, wpad.shape[1], LD)):
        return None, None
    slots = []
    with torch.no_grad():
        for lengths, wavs in slots_in:
            sl = dict(lengths=lengths, wavs=wavs)
            sl["stat_sums"] = torch.zeros(B, LD, 2, device=ctx.dev, dtype=torch.float64)
            sl["feats"], _ = ops.stft_features(wavs, 0, n_fft, hop, window, logpower=True, stat_sums=sl["stat_sums"])
            sl["mask"] = ops.linear_head_tma(sl["feats"], K, wpad, head.linear.bias, head.activation, sl["stat_sums"], head.eps)
            sl["wav"], sl["sums"] = ops.mask_istft(wavs, 0, 1, sl["mask"], lengths, n_fft, hop, window, pad_to=T, mask_padded=True)
            slots.append(sl)
    torch.cuda.synchronize()
    # (the sums buffers keep accumulating across timing launches: the values are not used here)
    launchers = {
        "stft": lambda s: ops.stft_features(s["wavs"], 0, n_fft, hop, window, logpower=True, stat_sums=s["stat_sums"]),
        "head": lambda s: ops.linear_head_tma(s["feats"], K, wpad, head.linear.bias, head.activation, s["stat_sums"], head.eps),
        "mask_istft": lambda s: ops.mask_istft(s["wavs"], 0, 1, s["mask"], s["lengths"], n_fft, hop, window, pad_to=T,
                                               mask_padded=True, out=s["wav"], sums=s["sums"]),
        "finalize": lambda s: ops.finalize_metrics(s["sums"], s["lengths"], T, wav=s["wav"]),
    }
    kernel_ms = {}
    for name, fn in launchers.items():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for sl in slots[:2]:
                fn(sl)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if graph:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g), torch.no_grad():
                for sl in slots:
                    fn(sl)
            run = g.replay
        else:
            def run():
                with torch.no_grad():
                    for sl in slots:
                        fn(sl)
        run()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(reps):
            run()
        a1.record()
        torch.cuda.synchronize()
        kernel_ms[name] = a0.elapsed_time(a1) / (reps * len(slots))
    # algorithmic bytes per launch (DESIGN.md "kernels"): K3 reads noisy + clean (2 x 4T), the mask (4FK), writes 4T per utterance
    alg_bytes = {"stft": B * (4 * T + 4 * F * K), "head": B * 8 * F * K, "mask_istft": B * (12 * T + 4 * F * K), "finalize": B * 8 * T}
    return kernel_ms, alg_bytes


def roofline_of(ctx, kernel_ms, alg_bytes, step_bytes, step_ms, traffic=None):
    dominant = max(kernel_ms, key=kernel_ms.get)
    achieved = alg_bytes[dominant] / (kernel_ms[dominant] * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
            "traffic": traffic, "peak_source": ctx.peak_src, "algorithmic_bytes_per_launch": alg_bytes[dominant],
            "kernel_ms": {k: round(v, 5) for k, v in kernel_ms.items()},
            "kernel_frac_of_hbm_peak": {k: round(alg_bytes[k] / (v * 1e-3) / 1e9 / ctx.peak, 4) for k, v in kernel_ms.items()},
            "step_algorithmic_bytes": int(step_bytes),
            "step_frac_of_hbm_peak": step_bytes / (step_ms * 1e-3) / 1e9 / ctx.peak}


# ------------------------------------------------------------------------------------------------- configs[3]: long-form
def bench_longform(ctx, se, args):
    """1024 utterances of 60 s in total, n_fft 1024 / hop 256, evaluation step; STRONG scaling (1024 / N per GPU)."""
    from speech_enhancement_by_s3prl_b200 import dp, synth
    total_utt, secs, n_fft = args.long_utts, 60.0, 1024
    hop = GEOMETRY[n_fft]["hop"]
    B = total_utt // ctx.world
    T = int(secs * SR)
    pre, head, engine = make_engine(se, ctx, n_fft)
    # ONE global data set whatever N is (strong scaling: the pass means in `check` do not depend on N): utterance g of the 1024
    # is host-generated utterance 4 (g // 128) + g % 4 under a level-preserving circular shift (distinct bytes in every row;
    # generating 17 audio-hours on the host would take minutes); rank r owns utterances [r B, (r + 1) B)
    chunk, g0 = 128, ctx.rank * B
    bases = {}
    for c in range(g0 // chunk, (g0 + B - 1) // chunk + 1):
        bases[c] = synth.batch(4, secs, first_index=500000 + 4 * c)[1].to(ctx.dev)
    wavs = torch.empty(B, 3, T, device=ctx.dev)
    for b in range(B):
        g_utt = g0 + b
        wavs[b] = torch.roll(bases[g_utt // chunk][g_utt % 4], shifts=7919 * ((g_utt % chunk) // 4), dims=-1)
    del bases
    lengths = torch.full((B,), T, dtype=torch.int64, device=ctx.dev)
    acc = torch.zeros(3, device=ctx.dev, dtype=torch.float64)
    g = engine.capture_bound(lengths, wavs, metric_acc=acc)
    steps = args.steps
    for _ in range(2):
        g["graph"].replay()
    acc.zero_()

    def run():
        for _ in range(steps):
            g["graph"].replay()
        dp.reduce_sums(acc)                                         # the one collective of an evaluation pass
    ms = ctx.timed(run) / steps
    audio_s = total_utt * secs
    value = audio_s / (ms * 1e-3)
    loss, sisdr, n = acc[0] / acc[2], acc[1] / acc[2], acc[2]
    kernel_ms, alg_bytes = time_eval_kernels(ctx, se, engine, pre, head, [(lengths, wavs)], n_fft, hop, reps=3, graph=False)
    out = {"workload": f"configs[3]: long-form, {total_utt} utterances x {secs:g} s in total ({B} per GPU), n_fft={n_fft} hop={hop}, "
                       f"LinearResidual({n_fft // 2 + 1}) on log-power, eval step + SISDR + waveform SI-SDR",
           "metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": ms, "steps": steps, "scaling": "strong",
           "utterances_per_gpu": B, "seconds": secs, "l2": f"one pass reads {B * 2 * T * 4 / 1e9:.1f} GB of waveforms per GPU (>> 126 MB L2)",
           "check": {"mean_sisdr_db": float(sisdr), "mean_loss": float(loss), "utterances_counted": int(n.item()) // steps}}
    if kernel_ms:
        out["roofline"] = roofline_of(ctx, kernel_ms, alg_bytes, eval_step_bytes(B * secs, n_fft, hop), ms)
    del g, wavs
    engine._graphs.clear()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------- configs[2]: training
def bench_training(ctx, se, args):
    """The fused training step (runner.py:431-471) at the reference's default n_fft 400 / hop 160: STFT of both channels,
    CMVN sums, tcgen05 head, SISDR forward / backward, split-K head backward, NCCL all-reduce of the head gradients inside
    the captured graph, clipping + Adam.  48 utterances of 3-10 s per GPU (pseudo_noise.yaml batch_size 6, x 8)."""
    from speech_enhancement_by_s3prl_b200 import synth
    n_fft, B, secs = 400, 48, 10.0
    hop = GEOMETRY[n_fft]["hop"]
    K = n_fft // 2 + 1
    pre, head, engine = make_engine(se, ctx, n_fft)
    crit = se.SISDR()
    opt = se.ClipAdam(head.parameters(), lr=1e-4)
    lengths, wavs = synth.batch(B, secs, first_index=700000 + B * ctx.rank, min_seconds=3.0)
    audio_s = float(lengths.sum()) / SR
    lengths, wavs = lengths.to(ctx.dev), wavs.to(ctx.dev)
    fused = engine.fused_training_supported(crit, B, wavs.shape[2])
    st = engine.capture_train(lengths, wavs, crit, opt, 1.0)
    steps = args.steps
    for _ in range(3):
        st["graph"].replay()

    def run():
        for _ in range(steps):
            st["graph"].replay()
        if ctx.world > 1:
            ctx.dist.all_reduce(ctx.align)
    ms = ctx.timed(run) / steps
    t = torch.tensor([audio_s], device=ctx.dev, dtype=torch.float64)
    if ctx.world > 1:
        ctx.dist.all_reduce(t)
    frames = float((lengths // hop + 1).sum())
    # SURVEY 8(d) training path, recompute variant: custom kernels 4 (5 H + D + 3 K) per frame + head forward / backward I/O
    # (forward reads D writes K; backward reads D, offset K, grad K), D = K here
    step_bytes = frames * (4 * (5 * hop + K + 3 * K) + 4 * (K + K) + 4 * 3 * K)
    out = {"workload": f"configs[2]: training step at n_fft={n_fft} hop={hop}, LinearResidual({K}) on log-power + SISDR, fwd + bwd + "
                       f"gradient all-reduce + clip + Adam in one CUDA graph, {B} utterances of 3-10 s per GPU",
           "metric": "trained audio-sec/sec (fwd+bwd+update)", "value": t.item() / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
           "steps": steps, "scaling": "weak", "fused_route": bool(fused), "audio_s_per_gpu_step": audio_s,
           "grad_allreduce": "NCCL all-reduce of the flat head gradient (162 KB) captured inside the step's graph" if ctx.world > 1 else "world size 1",
           "step_algorithmic_bytes": int(step_bytes), "step_frac_of_hbm_peak": step_bytes / (ms * 1e-3) / 1e9 / ctx.peak,
           "check": {"loss": float(st["loss"]), "steps_taken": opt.steps_taken()[0], "steps_skipped": opt.steps_skipped()[0]}}
    # the same step with the baseline feature of config/pseudo_noise.yaml:10-15 -- mel + log + delta 2 (120-d, fused K1b kernel)
    # -- into LinearResidual(120 -> K): the fused route with the K1b kernel in front of the head, also captured with its all-reduce
    torch.manual_seed(1337)
    head2 = se.LinearResidual(input_size=120, output_size=K, precision=1).to(ctx.dev)
    eng2 = se.EnhancementEngine(pre, head2, precision=1, feat_cfg=pre.get_feat_config("mel", 0, log=True, delta=2))
    opt2 = se.ClipAdam(head2.parameters(), lr=1e-4)
    st2 = eng2.capture_train(lengths, wavs, crit, opt2, 1.0)
    for _ in range(3):
        st2["graph"].replay()

    def run2():
        for _ in range(steps):
            st2["graph"].replay()
        if ctx.world > 1:
            ctx.dist.all_reduce(ctx.align)
    ms2 = ctx.timed(run2) / steps
    out["mel_log_delta2"] = {"workload": f"mel(40) + log + delta 2 (120-d, fused K1b kernel) -> LinearResidual(120, {K}) + SISDR, "
                                         f"{'fused route (no autograd graph)' if eng2.fused_training_supported(crit, B, wavs.shape[2]) else 'autograd route'}, one CUDA graph",
                             "value": t.item() / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2, "loss": float(st2["loss"].detach())}
    return out


# ------------------------------------------------------------------------------------------------- configs[4]: scoring
def bench_scoring(ctx, se, args):
    """Active-sampling scoring (sampler.py:59-120): gradient embeddings of 12 training + 32 query utterances of up to 10 s
    and the cosine matching, n_fft 400 / hop 160.  Every rank scores its own 44 utterances (weak scaling, replicas)."""
    from speech_enhancement_by_s3prl_b200 import sampler_ops, synth
    n_fft = 400
    pre, head, engine = make_engine(se, ctx, n_fft)
    crit = se.SISDR()
    lengths, wavs = synth.batch(44, 10.0, first_index=900000 + 44 * ctx.rank, min_seconds=3.0)
    audio_s = float(lengths.sum()) / SR
    lengths, wavs = lengths.to(ctx.dev), wavs.to(ctx.dev)

    def one():
        grads = sampler_ops.scoring(pre, head, crit, lengths, wavs)
        return grads, sampler_ops.matching(grads[12:], grads[:12])
    for _ in range(3):
        grads, scores = one()
    steps = args.steps

    def run():
        for _ in range(steps):
            one()
        if ctx.world > 1:
            ctx.dist.all_reduce(ctx.align)
    ms = ctx.timed(run) / steps
    t = torch.tensor([audio_s], device=ctx.dev, dtype=torch.float64)
    if ctx.world > 1:
        ctx.dist.all_reduce(t)
    # run_active.sh's own combination: --downstream LSTM with the L1-trained checkpoint; the library part is the projection layer
    torch.manual_seed(1337)
    lstm = se.LSTM(input_size=201, output_size=201, hidden_size=201, num_layers=3, precision=1).to(ctx.dev)
    l1 = se.L1()

    def one_l1():
        g = sampler_ops.scoring(pre, lstm, l1, lengths, wavs, projection_only=True)
        return g, sampler_ops.matching(g[12:], g[:12])
    for _ in range(3):
        g_l1, s_l1 = one_l1()

    def run_l1():
        for _ in range(steps):
            one_l1()
        if ctx.world > 1:
            ctx.dist.all_reduce(ctx.align)
    ms_l1 = ctx.timed(run_l1) / steps
    l1_out = {"workload": "LSTM(3 x 201) head + L1 objective, gradient embeddings of the projection layer (cuDNN LSTM forward included)",
              "value": t.item() / (ms_l1 * 1e-3), "unit": UNIT, "ms_per_step": ms_l1, "parameters": int(g_l1.shape[1]),
              "finite": bool(torch.isfinite(g_l1).all())}
    return {"l1_lstm_projection": l1_out,
            "workload": "configs[4]: active-sampling scoring, 12 + 32 utterances of 3-10 s per GPU, n_fft=400 hop=160, per-utterance "
                        "gradient embeddings of LinearResidual(201) under the spectral SISDR objective + cosine matching",
            "metric": "scored audio-sec/sec", "value": t.item() / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
            "scaling": "weak", "parameters": int(grads.shape[1]), "launch": "eager (10 library launches per scoring call)",
            "check": {"selected": int((scores > 0).sum()), "finite": bool(torch.isfinite(grads).all())}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ring", type=int, default=8, help="distinct batches the device-resident run rotates over")
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU oracle timing for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--streams", type=int, default=3, help="independent steps in flight (CUDA streams) in the device-resident run")
    ap.add_argument("--head-precision", type=int, default=1, help="0 = fp32 SIMT head, 1 = TF32 tcgen05 head")
    ap.add_argument("--long-utts", type=int, default=1024, help="utterances (60 s each) of the long-form configuration, in total")
    ap.add_argument("--skip-configs", action="store_true", help="headline only (no `configs` object)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args, int(os.environ.get("RANK", "0")))
        return

    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp, ops, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    ctx = Ctx(args)
    rank, world, dev, dist = ctx.rank, ctx.world, ctx.dev, ctx.dist
    sampler = ClockSampler(ctx.local_rank)
    sampler.start()                                     # (started early: no thread start between the alignment and the first event)

    # ---------------------------------------------------------------- model + data
    pre = se.OnlinePreprocessor(**PRE_KW).to(dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=257, output_size=257).to(dev)
    engine = se.EnhancementEngine(pre, head, log_features=True, precision=args.head_precision)
    T = int(SECONDS * SR)
    ring_host = [synth.batch(N_UTT, SECONDS, first_index=(rank * args.ring + r) * N_UTT) for r in range(min(args.ring, 4))]
    # device ring: the first few slots come from the host batches, the rest are level-preserving
    # circular shifts of them (distinct bytes; generation on the host is the slow part)
    ring = []
    for r in range(args.ring):
        lengths, wavs = ring_host[r % len(ring_host)]
        d = wavs.to(dev)
        if r >= len(ring_host):
            d = torch.roll(d, shifts=1777 * r, dims=-1).contiguous()
        ring.append((lengths.to(dev), d))
    audio_s_per_step = N_UTT * SECONDS
    K = N_FFT // 2 + 1

    # ---------------------------------------------------------------- device-resident timed run
    acc = torch.zeros(3, device=dev, dtype=torch.float64)     # [sum loss, sum SI-SDR, utterances] of the pass, kept on the device
    if args.eager:
        outputs = [{} for _ in ring]                   # what each ring slot's latest step returned
        steps = [lambda l=l, w=w, o=o: o.update(engine.eval_step(l, w, metric_acc=acc)) for (l, w), o in zip(ring, outputs)]
    else:
        graphs = outputs = [engine.capture_bound(l, w, metric_acc=acc) for l, w in ring]
        steps = [g["graph"].replay for g in graphs]
    # Consecutive steps work on independent batches: with --streams S > 1, step i is enqueued on stream i % S, so the
    # ramp-up and tail of one step's kernels overlap the neighbouring step's kernels (every ring slot owns its buffers).
    main_stream = torch.cuda.current_stream()
    lanes = [torch.cuda.Stream(device=dev) for _ in range(args.streams)] if args.streams > 1 else [main_stream]

    def run_steps(n):
        if len(lanes) > 1:
            fork = torch.cuda.Event()
            fork.record(main_stream)
            for st in lanes:
                st.wait_event(fork)
        for i in range(n):
            with torch.cuda.stream(lanes[i % len(lanes)]):
                steps[i % len(steps)]()
        if len(lanes) > 1:
            for st in lanes:
                main_stream.wait_stream(st)

    run_steps(max(args.warmup, len(steps)))            # at least W steps, and every ring slot's graph has run once
    for _ in range(3):                                 # communicator setup and the first collectives stay out of the timed region
        dp.reduce_sums(acc)
    torch.cuda.synchronize()
    acc.zero_()

    def timed_pass():
        run_steps(args.steps)
        dp.reduce_sums(acc)                            # the one collective of an evaluation pass: [sum loss, sum SI-SDR, n] (no host read)
    ms_total = ctx.timed(timed_pass)
    value = world * audio_s_per_step * args.steps / (ms_total * 1e-3)
    pass_loss, pass_sisdr, pass_n = float(acc[0] / acc[2]), float(acc[1] / acc[2]), float(acc[2])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs[(args.steps - 1) % len(outputs)], acc)

    # ---------------------------------------------------------------- per-kernel timing, roofline of the dominant kernel
    kernel_ms, alg_bytes = time_eval_kernels(ctx, se, engine, pre, head, ring, N_FFT, HOP, reps=10)
    if kernel_ms is None:                              # fp32 SIMT head (--head-precision 0): no per-kernel breakdown
        kernel_ms, alg_bytes = {"step": ms_total / args.steps}, {"step": eval_step_bytes(audio_s_per_step, N_FFT, HOP)}
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    dominant = max(kernel_ms, key=kernel_ms.get)
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(dominant, {}).get("dram_bytes_per_launch")
    roofline = roofline_of(ctx, kernel_ms, alg_bytes, eval_step_bytes(audio_s_per_step, N_FFT, HOP), ms_total / args.steps, traffic)
    roofline["note"] = ("K1/K3 are bound by the fp32 pipe + shared-memory wavefronts, not HBM (DESIGN.md 4.1); "
                        "kernel times are per launch, each kernel timed alone over HBM-cold inputs")

    # ---------------------------------------------------------------- end-to-end through the host pipeline
    # e2e: fp32 host batches in, metrics out (the like-for-like headline, as in round 1).  Two more modes of the same
    # public call: int16 PCM host batches (half the PCIe bytes, widened on the device) and fp32 in + enhanced waveforms out.
    def run_e2e(pcm16, want_wav):
        pipe = engine.host_pipeline(N_UTT, 3, T, depth=2, device=dev, pcm16=pcm16, want_wav=want_wav, copy_wav=False)
        if pcm16:
            pinned = [(l.clone().pin_memory(), (w * 32768.0).round().clamp_(-32768, 32767).to(torch.int16).pin_memory()) for l, w in ring_host]
        else:
            pinned = [(l.clone().pin_memory(), w.clone().pin_memory()) for l, w in ring_host]
        for i in range(max(3, min(args.warmup, 10))):
            pipe.submit(*pinned[i % len(pinned)])
        pipe.drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            pipe.submit(*pinned[i % len(pinned)])
        results = pipe.drain()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out = {"value": world * audio_s_per_step * args.steps / t.item(), "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes,
               "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": 1e3 * t.item() / args.steps, "pipeline_depth": 2}
        return out, results

    e2e, results = run_e2e(False, False)
    mean_sisdr = float(torch.stack([r[1] for r in results]).mean())
    mean_loss = float(torch.stack([r[0] for r in results]).mean())
    e2e_pcm16, res16 = run_e2e(True, False)
    e2e_pcm16["input"] = "int16 PCM host batches (the corpora's sample format), sample / 32768 on the device"
    e2e_pcm16["mean_sisdr_db"] = float(torch.stack([r[1] for r in res16]).mean())
    e2e_wav, _ = run_e2e(False, True)
    e2e_wav["output"] = "per-utterance metrics + the enhanced waveforms (B, T) fp32 to pinned host memory (handed out as views of the slot buffers)"
    del results, res16
    clocks = sampler.stop()

    # ---------------------------------------------------------------- the other BASELINE configurations
    configs = None
    if not args.skip_configs:
        engine._graphs.clear()
        if not args.eager:
            del graphs, steps
        torch.cuda.empty_cache()
        configs = {}
        for name, fn in (("configs[3]", bench_longform), ("configs[2]", bench_training), ("configs[4]", bench_scoring)):
            try:
                configs[name] = fn(ctx, se, args)
            except Exception as exc:                   # a failed side configuration must not take the headline with it
                if world > 1:
                    raise                              # (ranks must stay in lock-step: fail loudly under torchrun)
                configs[name] = {"error": f"{type(exc).__name__}: {exc}"}

    # ---------------------------------------------------------------- CPU baseline on the host cores (rank 0, N = 1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        lengths, wavs = ring_host[0]
        best, cores, reps = time_cpu_oracle(lengths, wavs, head.linear.weight.detach().cpu(), head.linear.bias.detach().cpu(), args.cpu_budget)
        cpu = {"value": audio_s_per_step / best, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"full batch {N_UTT}x{SECONDS:g}s, best of {reps} runs of the un-fused oracle sequence (torch CPU fp32)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "head": "tf32 tcgen05 (fp32 accumulate)" if args.head_precision == 1 else "fp32 SIMT", "utterances_per_gpu": N_UTT, "seconds": SECONDS, "n_fft": N_FFT, "hop": HOP,
                           "launch": ("eager" if args.eager else "cuda-graph replay") + f", {args.streams} step(s) in flight (streams)",
                           "l2": f"inputs rotate over {args.ring} distinct device batches ({args.ring * N_UTT * 3 * T * 4 / 1e6:.0f} MB > 126 MB L2); no explicit flush",
                           "parallelism": f"dp{world} (utterance-sharded, no data-path collective; metric sums accumulate on the device, one all-reduce per pass)",
                           "timing": "ranks aligned by a collective on the stream before the first event; max over ranks",
                           "numa": f"rank 0 bound to NUMA node {ctx.numa_node}" if ctx.numa_node is not None else "no NUMA binding"},
                "e2e": e2e, "e2e_pcm16": e2e_pcm16, "e2e_wav_out": e2e_wav,
                "gpu_launches": engine.launches_per_step * args.steps, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
                "check": {"mean_sisdr_db": mean_sisdr, "mean_loss": mean_loss,
                          "device_pass": {"mean_sisdr_db": pass_sisdr, "mean_loss": pass_loss, "utterances": pass_n}},
                "configs": configs}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
