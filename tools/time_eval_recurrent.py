"""Time the evaluation step of model.LSTM(hidden 256, 3 layers) with objective.L1 -- the pairing of the reference's
run_active.sh / run_uniform.sh -- at 64 x 4 s for n_fft / hop 512 / 256 and 400 / 160:
  step        the captured EnhancementEngine step (eager if the capture fails; the error is printed);
  body        an estimate of the cuDNN LSTM body's share of the step: CUDA events around a separately captured graph of
              head.lstm on a random input of the step's shape (cuDNN's time does not depend on the values; events inside the
              step's own graph cannot be read);
  library_ms  step - body: K1, the copy out of the padded rows, the projection, K3-L1, K3' and the finish kernel (an estimate,
              as the body time is);
  drop-in     the un-fused evaluation on the drop-in modules (STFT of every channel, the head module, exp, iSTFT, objective.L1,
              waveform SI-SDR).
Prints the card, its power limit and max SM clock beside the numbers: python tools/time_eval_recurrent.py [--steps N]"""
import argparse, os, subprocess, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import evaluation, ops, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=50)
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


def best(fn):
    fn()
    return min(timed(fn, args.steps) for _ in range(args.rounds))


def captured(fn):
    """fn replayed from a CUDA graph, or None if it cannot be captured."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    try:
        with torch.cuda.graph(g):
            fn()
    except RuntimeError as exc:
        print(f"  (capture failed: {exc})", flush=True)
        return None
    return g


for (n_fft, hop), B, secs in (((512, 256), 64, 4.0), ((400, 160), 64, 4.0)):
    n_freq, win_ms, hop_ms = GEO[(n_fft, hop)]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).to(dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LSTM(input_size=n_freq, output_size=n_freq, hidden_size=256, num_layers=3, precision=1).to(dev).eval()
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    lengths, wavs = synth.batch(B, secs)
    lengths, wavs = lengths.to(dev), wavs.to(dev)
    T = wavs.shape[2]
    tag = f"{B} x {secs:g} s, {n_fft} / {hop}"
    crit = se.L1()
    st = None
    try:
        st = eng.capture_bound(lengths, wavs, criterion=crit)
        step, mode = best(st["graph"].replay), "captured"
        loss = st["loss"].item()
    except RuntimeError as exc:
        print(f"[{tag}] capture failed: {exc}", flush=True)
        with torch.no_grad():
            step, mode = best(lambda: eng.eval_step(lengths, wavs, criterion=crit)), "eager"
        loss = eng.eval_step(lengths, wavs, criterion=crit)["loss"].item()
    x = torch.randn(B, T // hop + 1, n_freq, device=dev)

    def body():
        with torch.no_grad():
            head.lstm(x)

    g = captured(body) if mode == "captured" else None
    tb = best(g.replay if g is not None else body)
    print(f"[{tag}] step ({mode}, L1): {step * 1e3:9.1f} us  body (cuDNN LSTM): {tb * 1e3:9.1f} us  "
          f"library_ms: {(step - tb):.4f} ms ({eng.launches_per_step} library launches)  loss {loss:.4f}", flush=True)
    window = pre._frame_window
    c = pre.get_feat_config

    def dropin():
        with torch.no_grad():
            feats, phase_inp, linear_tar = pre(wavs, [c("linear", 0, log=True), c("phase", 0), c("linear", 1)])
            predicted, extra = head(features=feats)
            loss, _ = crit(linear_tar=linear_tar, stft_lengths=lengths // hop + 1, **extra)
            wav = ops.istft(predicted, phase_inp, n_fft, hop, window, pad_to=T)
            return loss, evaluation.sisdr_eval_batch(wav[:, :T], wavs[:, 1], lengths)

    td = best(dropin)
    print(f"[{tag}] drop-in L1 evaluation (eager): {td * 1e3:9.1f} us  -> fused step {td / step:.2f} x faster; "
          f"outside the body {(td - tb) / max(step - tb, 1e-9):.1f} x", flush=True)
    del eng, st
    torch.cuda.empty_cache()
