"""Time the captured evaluation step (EnhancementEngine.capture, LinearResidual on log-power, TF32 head) with criterion SISDR
and WSD, alternated in one process, at 64 x 4 s for n_fft / hop 512 / 256, 400 / 160 and 1024 / 256 and at 128 x 60 s for
1024 / 256; K3 in both variants and the WSD finish kernel on their own (CUDA graphs of repeated launches); and the un-fused
drop-in WSD evaluation (STFT of every channel, the head module, objective.WSD, iSTFT, SI-SDR) on the same batch.
Prints the card, its power limit and max SM clock beside the numbers: python tools/time_eval_wsd.py [--steps N]"""
import argparse, os, subprocess, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import evaluation, ops, synth

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=100)
ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the criteria")
args = ap.parse_args()
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
try:
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as exc:                                  # (the name alone from torch then)
    card = f"{torch.cuda.get_device_name(dev)}, power limit unknown ({exc})"
print(f"device: {card}", flush=True)
GEO = {(512, 256): (257, 32, 16), (400, 160): (201, 25, 10), (1024, 256): (513, 64, 16)}
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def timed(fn, n):
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def graph_of(fn, reps):
    """CUDA graph of `reps` launches of fn (per-kernel times without host launch overhead)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    return g


for (n_fft, hop), B, secs in (((512, 256), 64, 4.0), ((400, 160), 64, 4.0), ((1024, 256), 64, 4.0), ((1024, 256), 128, 60.0)):
    n_freq, win_ms, hop_ms = GEO[(n_fft, hop)]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).to(dev)
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=n_freq, output_size=n_freq, precision=1).to(dev)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    lengths, wavs = synth.batch(B, secs)
    lengths, wavs = lengths.to(dev), wavs.to(dev)
    T = wavs.shape[2]
    tag = f"{B} x {secs:g} s, {n_fft} / {hop}"
    crits = {"SISDR": se.SISDR(), "WSD": se.WSD()}
    graphs = {}
    for name, crit in crits.items():
        st = eng.capture(B, 3, T, dev, crit)
        st["lengths"].copy_(lengths)
        st["wavs"].copy_(wavs)
        graphs[name] = st
    times = {name: [] for name in crits}
    for _ in range(args.rounds):
        for name, st in graphs.items():
            st["graph"].replay()                                   # (warm)
            times[name].append(timed(st["graph"].replay, args.steps))
    base = min(times["SISDR"])
    for name, ts in times.items():
        loss = graphs[name]["loss_per_utt"].mean().item()
        print(f"[{tag}] step {name:5s}: {min(ts) * 1e3:8.1f} us (rounds {', '.join(f'{t * 1e3:.1f}' for t in ts)})  "
              f"{min(ts) / base:.3f} x SISDR  mean loss {loss:.4f}", flush=True)
    # per kernel: K3 (SISDR sums), K3 (WSD terms), the finish kernel -- graphs of 20 launches on a random mask
    window = pre._frame_window
    mask = torch.rand(B, T // hop + 1, ops.round4(n_freq), device=dev)
    sums = torch.zeros(B, ops.NSUMS, device=dev, dtype=torch.float64)
    state = torch.zeros(2, device=dev)
    _, _, terms = ops.mask_istft_wsd(wavs, 0, 1, mask, lengths, n_fft, hop, window, T, state, sums=sums, sums_zeroed=True)
    k3 = lambda: ops.mask_istft(wavs, 0, 1, mask, lengths, n_fft, hop, window, T, want_spec=True, mask_padded=True, sums=sums,
                                sums_zeroed=True)
    k3w = lambda: ops.mask_istft_wsd(wavs, 0, 1, mask, lengths, n_fft, hop, window, T, state, sums=sums, sums_zeroed=True)
    fin = lambda: ops.wsd_eval_finish(terms, sums, state)
    reps = 20
    kt = {name: [] for name in ("K3 SISDR", "K3 WSD", "finish")}
    kg = {name: graph_of(fn, reps) for name, fn in (("K3 SISDR", k3), ("K3 WSD", k3w), ("finish", fin))}
    for _ in range(args.rounds):
        for name, g in kg.items():
            g.replay()
            kt[name].append(timed(g.replay, max(1, args.steps // 10)) / reps)
    print(f"[{tag}] kernels: " + "  ".join(f"{name} {min(ts) * 1e3:.1f} us" for name, ts in kt.items()) +
          f"  (K3 WSD / K3 SISDR {min(kt['K3 WSD']) / min(kt['K3 SISDR']):.3f})", flush=True)
    del kg
    # the un-fused drop-in evaluation with objective.WSD (runner.py:556-602 on the drop-in modules)
    if B * secs <= 64 * 4.0:
        c = pre.get_feat_config
        crit = crits["WSD"]

        def dropin():
            with torch.no_grad():
                feats, linear_inp, phase_inp, linear_tar = pre(wavs, [c("linear", 0, log=True), c("linear", 0), c("phase", 0),
                                                                      c("linear", 1)])
                predicted, extra = head(features=feats, linears=linear_inp)
                loss, _ = crit(predicted=predicted, linear_tar=linear_tar, linear_inp=linear_inp, stft_lengths=lengths // hop + 1,
                               **extra)
                wav = ops.istft(predicted, phase_inp, n_fft, hop, window, pad_to=T)
                return loss, evaluation.sisdr_eval_batch(wav[:, :T], wavs[:, 1], lengths)

        dropin()
        td = min(timed(dropin, max(1, args.steps // 10)) for _ in range(args.rounds))
        print(f"[{tag}] drop-in WSD evaluation (eager): {td * 1e3:8.1f} us  -> fused WSD step {td / min(times['WSD']):.1f} x faster",
              flush=True)
    del graphs, eng
    torch.cuda.empty_cache()
