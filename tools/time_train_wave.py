"""Time the captured LinearResidual training step (train_step_graph, se_b200.ClipAdam, grad_clip 1.0) with objective.WaveSISDR
against objective.SISDR on the same engine and batches: configs[2]'s shape (48 x 10 s, n_fft / hop 400 / 160) and 64 x 4 s at
512 / 256.  The two objectives alternate within the run (--rounds times each).  Then, in a separate profiled pass of the WaveSISDR
step, the per-kernel times of K3 (mask_istft), the finish kernel and se_mask_istft_bwd from torch.profiler.
Prints the card, its power limit and max SM clock beside the numbers: python tools/time_train_wave.py [--steps N] [--rounds R]"""
import argparse, os, subprocess, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as exc:
    card = f"{torch.cuda.get_device_name(dev)}, power limit unknown ({exc})"
print(f"device: {card}", flush=True)
GEO = {(512, 256): (257, 32, 16), (400, 160): (201, 25, 10)}
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed(fn, n):
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


KERNELS = {"K3 (mask_istft)": "mask_istft_", "finish (wave_sisdr_finish)": "wave_sisdr_finish_kernel",
           "backward (mask_istft_bwd)": "mask_istft_bwd_kernel"}

for (n_fft, hop), B, secs in (((400, 160), 48, 10.0), ((512, 256), 64, 4.0)):
    n_freq, win_ms, hop_ms = GEO[(n_fft, hop)]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).to(dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    lengths, wavs = synth.batch(B, secs)
    lengths, wavs = lengths.to(dev), wavs.to(dev)
    T = wavs.shape[2]
    tag = f"{B} x {secs:g} s, {n_fft} / {hop}"
    torch.manual_seed(1337)
    head = se.LinearResidual(n_freq, n_freq, precision=1).to(dev)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crits = {"SISDR": se.SISDR(), "WaveSISDR": se.WaveSISDR()}
    opts = {}
    for name, crit in crits.items():
        assert eng.fused_training_supported(crit, B, T), name
        opts[name] = se.ClipAdam(head.parameters(), lr=1e-6)
        eng.train_step_graph(lengths, wavs, crit, opts[name], 1.0)
    times = {name: [] for name in crits}
    for _ in range(args.rounds):
        for name, crit in crits.items():
            times[name].append(timed(lambda: eng.train_step_graph(lengths, wavs, crit, opts[name], 1.0), args.steps))
    for name in crits:
        ts = ", ".join(f"{t:.3f}" for t in times[name])
        print(f"[{tag}] captured step, {name:9s}: best {min(times[name]):8.3f} ms  (rounds: {ts})", flush=True)

    from torch.profiler import ProfilerActivity, profile
    wave, opt = crits["WaveSISDR"], opts["WaveSISDR"]
    n_prof = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            eng.train_step(lengths, wavs, wave, opt, 1.0)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            for label, key in KERNELS.items():
                if key in e.name and (key != "mask_istft_" or "bwd" not in e.name):
                    per.setdefault(label, []).append(e.device_time_total / 1000.0)
    for label in KERNELS:
        ts = per.get(label, [])
        mean = sum(ts) / len(ts) if ts else float("nan")
        print(f"[{tag}] {label:28s} {mean * 1000:9.1f} us per call  ({len(ts)} calls in {n_prof} eager WaveSISDR steps, torch.profiler)",
              flush=True)
    del eng, head, opts
    torch.cuda.empty_cache()
