"""Time the training step of model.LSTM(hidden 256, 3 layers) with objective.L1 -- the pairing of the reference's run_active.sh /
run_uniform.sh -- at 64 x 4 s for n_fft / hop 512 / 256 and at 12 x 10 s for 400 / 160 (the train batch of active.yaml):
  autograd    train_step on the autograd route through the drop-in modules (SE_B200_FUSED_TRAIN=0) with torch.optim.Adam, eager;
  fused       train_step on the fused route with se_b200.ClipAdam, eager;
  captured    train_step_graph: the fused route with ClipAdam replayed from one CUDA graph (eager fused if the capture fails; the
              error is printed);
  body        an estimate of the cuDNN LSTM body's share of a step: CUDA events around a separately captured graph of head.lstm's
              forward + backward on a random input of the step's shape (cuDNN's time does not depend on the values);
  library_ms  step - body for each route: everything around the body (an estimate, as the body time is).
All steps run with grad_clip 1.0 and cuDNN without TF32 (the settings of tests/test_train_recurrent.py).
Prints the card, its power limit and max SM clock beside the numbers: python tools/time_train_recurrent.py [--steps N]"""
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
torch.backends.cudnn.allow_tf32 = False
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


def engine(pre, n_freq, fused):
    torch.manual_seed(1337)
    head = se.LSTM(input_size=n_freq, output_size=n_freq, hidden_size=256, num_layers=3, precision=1).to(dev)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    eng.fused_training = fused
    return eng, head


for (n_fft, hop), B, secs in (((512, 256), 64, 4.0), ((400, 160), 12, 10.0)):
    n_freq, win_ms, hop_ms = GEO[(n_fft, hop)]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).to(dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    lengths, wavs = synth.batch(B, secs)
    lengths, wavs = lengths.to(dev), wavs.to(dev)
    T = wavs.shape[2]
    tag = f"{B} x {secs:g} s, {n_fft} / {hop}"
    crit = se.L1()

    eng, head = engine(pre, n_freq, fused=False)
    assert not eng.fused_training_supported(crit, B, T)
    opt = torch.optim.Adam(head.parameters(), lr=1e-4)
    t_auto = best(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0))
    l_auto = eng.train_step(lengths, wavs, crit, opt, 1.0).item()

    eng, head = engine(pre, n_freq, fused=True)
    assert eng.fused_training_supported(crit, B, T)
    opt = se.ClipAdam(head.parameters(), lr=1e-4)
    t_fused = best(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0))
    l_fused = eng.train_step(lengths, wavs, crit, opt, 1.0).item()

    eng, head = engine(pre, n_freq, fused=True)
    opt = se.ClipAdam(head.parameters(), lr=1e-4)
    try:
        eng.train_step_graph(lengths, wavs, crit, opt, 1.0)
        t_graph, mode = best(lambda: eng.train_step_graph(lengths, wavs, crit, opt, 1.0)), "captured"
        l_graph = eng.train_step_graph(lengths, wavs, crit, opt, 1.0).item()
    except RuntimeError as exc:
        print(f"[{tag}] capture failed: {exc}", flush=True)
        t_graph, mode = best(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0)), "eager"
        l_graph = eng.train_step(lengths, wavs, crit, opt, 1.0).item()

    # the body alone: cuDNN forward + backward of head.lstm on the step's shape, captured
    x = torch.randn(B, T // hop + 1, n_freq, device=dev)
    gy = torch.randn(B, T // hop + 1, 256, device=dev)
    lstm = head.lstm

    def body():
        for p in lstm.parameters():                      # as in the step (zero_grad(set_to_none)): fresh gradients, no accumulation
            p.grad = None
        y, _ = lstm(x)
        torch.autograd.backward(y, gy)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            body()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    try:
        with torch.cuda.graph(g):
            body()
        t_body = best(g.replay)
    except RuntimeError as exc:
        print(f"[{tag}] body capture failed, eager body: {exc}", flush=True)
        t_body = best(body)
    print(f"[{tag}] autograd route + torch Adam (eager): {t_auto:8.3f} ms  outside the body {t_auto - t_body:7.3f} ms  loss {l_auto:.4f}",
          flush=True)
    print(f"[{tag}] fused route + ClipAdam (eager):      {t_fused:8.3f} ms  library_ms {t_fused - t_body:7.3f} ms  loss {l_fused:.4f}",
          flush=True)
    print(f"[{tag}] fused route + ClipAdam ({mode}):   {t_graph:8.3f} ms  library_ms {t_graph - t_body:7.3f} ms  loss {l_graph:.4f}",
          flush=True)
    print(f"[{tag}] body (cuDNN LSTM forward + backward, captured): {t_body:8.3f} ms  -> captured step {t_auto / t_graph:.2f} x the "
          f"autograd route; outside the body {(t_auto - t_body) / max(t_graph - t_body, 1e-9):.1f} x", flush=True)
    del eng, head, opt, g
    torch.cuda.empty_cache()
