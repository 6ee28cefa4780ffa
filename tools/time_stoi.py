"""se_stoi (STOI + ESTOI) at 64 x 4 s and 128 x 60 s, 16 kHz: call time by CUDA events, time per kernel by torch.profiler,
the resampler's FMA rate against the fp32 FMA peak, and the float64 CPU oracle (oracle/stoi_f64.py, not pystoi) on the
64 x 4 s batch.  Synthetic amplitude-modulated noise with a silent gap; every row full length.

    python tools/time_stoi.py            (needs a GPU; prints the report)
"""
import os
import re
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from speech_enhancement_by_s3prl_b200 import ops  # noqa: E402
from oracle import stoi_f64  # noqa: E402

FS = 16000
assert torch.cuda.is_available(), "time_stoi.py measures on the GPU"
dev = torch.device("cuda", 0)
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                   capture_output=True, text=True).stdout.strip()
print(f"device: {q}")
max_clk_mhz = float(q.split(",")[2].split()[0])
sms = torch.cuda.get_device_properties(0).multi_processor_count
fma_peak = sms * 128 * max_clk_mhz * 1e6                     # fp32 FMA / s at the max SM clock


def batch(B, seconds, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    T = int(seconds * FS)
    t = torch.arange(T) / FS
    clean = torch.randn(B, T, generator=g) * (0.6 + 0.4 * torch.sin(2 * torch.pi * 3.1 * t))
    clean[:, int(0.4 * T):int(0.45 * T)] *= 1e-3
    est = 0.5 * clean + 0.2 * torch.randn(B, T, generator=g)
    return est.to(dev), clean.to(dev), torch.full((B,), T, dtype=torch.int64, device=dev)


def time_call(fn, min_s=0.2):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    n = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_s * 1e3:
            return ms / n
        n *= 2


def kernel_times(fn, reps=20):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            m = re.search(r"stoi_\w+_kernel", ev.key)
            name = m.group(0) if m else ev.key
            out[name] = out.get(name, 0.0) + ev.device_time_total / reps          # us per call
    return out


for B, sec in ((64, 4.0), (128, 60.0)):
    est, clean, L = batch(B, sec)
    T = est.shape[1]
    ws_bytes = ops._lib.load().se_stoi_workspace(B, T, FS)
    fn = lambda: ops.stoi(est, clean, L, fs=FS)              # noqa: E731
    ms = time_call(fn)
    ms2 = time_call(fn)
    kt = kernel_times(fn)
    p, qq = stoi_f64.rates(FS)
    _, Lh = stoi_f64.resample_filter(p, qq)
    K = 2 * Lh // p + 1
    n10 = -(-T * p // qq)
    fma = 2 * B * n10 * K
    rs_us = kt.get("stoi_resample_kernel", float("nan"))
    print(f"\n{B} x {sec:g} s @ {FS} Hz: se_stoi (STOI + ESTOI) {ms * 1e3:.1f} / {ms2 * 1e3:.1f} us per call (two CUDA-event windows of >= 200 ms), "
          f"workspace {ws_bytes / 2**20:.1f} MiB")
    for k, us in sorted(kt.items(), key=lambda kv: -kv[1]):
        print(f"  {k:<28s} {us:9.1f} us")
    print(f"  resampler: {fma / 1e9:.3f} G FMA ({K} taps per output, both channels) in {rs_us:.1f} us = "
          f"{fma / (rs_us * 1e-6) / 1e12:.2f} T FMA/s, {100 * fma / (rs_us * 1e-6) / fma_peak:.1f}% of the fp32 FMA peak "
          f"({sms} SMs x 128 x {max_clk_mhz:.0f} MHz = {fma_peak / 1e12:.1f} T FMA/s)")
    if B == 64:
        e, c = est.cpu().numpy(), clean.cpu().numpy()
        t0 = time.perf_counter()
        o = stoi_f64.batch(e, c, L.cpu().numpy(), FS)
        cpu_s = time.perf_counter() - t0
        s, es = fn()
        print(f"  CPU float64 oracle (NumPy, one process): {cpu_s * 1e3:.0f} ms for the batch, {cpu_s / B * 1e3:.1f} ms per utterance; "
              f"max |GPU - oracle| STOI {np.abs(s.cpu().double().numpy() - o['stoi']).max():.1e}, "
              f"ESTOI {np.abs(es.cpu().double().numpy() - o['estoi']).max():.1e}")
