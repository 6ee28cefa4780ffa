"""Long-form evaluation pass (BASELINE configs[3] at one GPU's share of 8: 128 utterances x 60 s, n_fft 1024 / hop 256):
ms per pass and per-kernel times.
python tools/time_longform.py [B] [seconds] [n_freq win_ms hop_ms]"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import ops, synth
B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
secs = float(sys.argv[2]) if len(sys.argv) > 2 else 60.0
nfreq, win, hop_ms = (int(v) for v in sys.argv[3:6]) if len(sys.argv) > 5 else (513, 64, 16)
dev = torch.device("cuda", 0)
pre = se.OnlinePreprocessor(sample_rate=16000, win_ms=win, hop_ms=hop_ms, n_freq=nfreq).to(dev)
pre.channel_inp, pre.channel_tar = 0, 1
torch.manual_seed(1337)
head = se.LinearResidual(input_size=nfreq, output_size=nfreq).to(dev)
eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
_, base = synth.batch(4, secs)
base = base.to(dev)
wavs = torch.stack([torch.roll(base[b % 4], shifts=7919 * (b // 4), dims=-1) for b in range(B)])
lengths = torch.full((B,), wavs.shape[2], dtype=torch.int64, device=dev)
n_fft, hop, K, T = pre._win_args["n_fft"], pre._win_args["hop_length"], nfreq, wavs.shape[2]


def timeit(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


with torch.no_grad():
    ms = timeit(lambda: eng.eval_step(lengths, wavs))
    LD = ops.round4(K)
    window, wpad = pre._frame_window, eng._padded_weight()
    sums = torch.zeros(B, LD, 2, device=dev, dtype=torch.float64)
    feats, _ = ops.stft_features(wavs, 0, n_fft, hop, window, logpower=True, stat_sums=sums)
    mask = ops.linear_head_tma(feats, K, wpad, head.linear.bias, head.activation, sums, head.eps)
    wav, s6 = ops.mask_istft(wavs, 0, 1, mask, lengths, n_fft, hop, window, pad_to=T, mask_padded=True)
    k1 = timeit(lambda: ops.stft_features(wavs, 0, n_fft, hop, window, logpower=True, stat_sums=sums))
    k2 = timeit(lambda: ops.linear_head_tma(feats, K, wpad, head.linear.bias, head.activation, sums, head.eps))
    k3 = timeit(lambda: ops.mask_istft(wavs, 0, 1, mask, lengths, n_fft, hop, window, pad_to=T, mask_padded=True, out=wav, sums=s6))
    k4 = timeit(lambda: ops.finalize_metrics(s6, lengths, T, wav=wav))
print(f"B {B} x {secs:g} s n_fft {n_fft}: {ms:.3f} ms/pass = {B * secs / ms * 1e3 / 1e6:.3f} M audio-s/s | "
      f"K1 {k1:.3f} K2 {k2:.3f} K3 {k3:.3f} K3' {k4:.3f} ms", flush=True)
