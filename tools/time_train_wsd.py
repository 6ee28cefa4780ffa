"""Time the captured training step at the configs[2] shape -- synth.batch(48, 10.0, min_seconds=3.0), n_fft 400 / hop 160,
LinearResidual(201) on log-power, TF32 head, ClipAdam, CUDA-graph replay -- for the fused SISDR step, the fused WSD step and
the WSD step through autograd (EnhancementEngine.fused_training = False).  Prints the card and its power limit beside the
numbers: python tools/time_train_wsd.py [--steps N]"""
import argparse, os, subprocess, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the three routes")
args = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as exc:                                  # (the name alone from torch then)
    card = f"{torch.cuda.get_device_name(dev)}, power limit unknown ({exc})"
print(f"device: {card}", flush=True)
pre = se.OnlinePreprocessor(sample_rate=16000, win_ms=25, hop_ms=10, n_freq=201).to(dev)
pre.channel_inp, pre.channel_tar = 0, 1
lengths, wavs = synth.batch(48, 10.0, min_seconds=3.0)
lengths, wavs = lengths.to(dev), wavs.to(dev)
audio_s = lengths.sum().item() / 16000.0
routes = {}
for name, crit, fused in (("fused SISDR", se.SISDR(), True), ("fused WSD", se.WSD(), True), ("autograd WSD", se.WSD(), False)):
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=201, output_size=201, precision=1).to(dev)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    eng.fused_training = fused
    assert eng.fused_training_supported(crit, 48, wavs.shape[2]) == fused
    opt = se.ClipAdam(head.parameters(), lr=1e-4)
    for _ in range(5):                                        # capture (3 eager warm-ups) + replays
        loss = eng.train_step_graph(lengths, wavs, crit, opt, 1.0)
    torch.cuda.synchronize()
    routes[name] = (eng, crit, opt)
times = {name: [] for name in routes}
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for _ in range(args.rounds):
    for name, (eng, crit, opt) in routes.items():
        st = eng.capture_train(lengths, wavs, crit, opt, 1.0)   # (cached: the inputs are already in its static buffers)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            st["graph"].replay()
        e1.record()
        torch.cuda.synchronize()
        times[name].append(e0.elapsed_time(e1) / args.steps)
for name, ts in times.items():
    loss = routes[name][0].capture_train(lengths, wavs, routes[name][1], routes[name][2], 1.0)["loss"].item()
    best = min(ts)
    print(f"configs[2] {name:13s}: {best:.3f} ms/step (rounds: {', '.join(f'{t:.3f}' for t in ts)})  "
          f"{audio_s / best * 1e3 / 1e6:.2f} M trained audio-s/s  loss {loss:.4f}", flush=True)
