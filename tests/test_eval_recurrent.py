"""The evaluation step with recurrent heads (EnhancementEngine.eval_step with model.LSTM / model.Residual) and objective.L1:
the log-power route of K3 (SE_FLAG_MASK_IS_LOG_POWER), the L1 variant of K3 on the register-resident geometries, the slow route
elsewhere, the finish kernel, captured replays and data parallelism (L1 is a global element mean: the numerator and the count
are all-reduced together, objective.py:113-116).

The reference state dict of tests/golden/recurrent_heads_ref.npz is not run through eval_step: its heads have 9 output bins
(n_fft 16), which no mask-iSTFT kernel supports.  oracle.signal_path.recurrent_head is pinned to that file
(test_oracle_golden.py), and the tests below compare the engine's heads against recurrent_head in float64."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import signal_path as sp
from oracle import stft_f64

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_parity import synth  # noqa: E402

gpu = pytest.mark.gpu
EPS = 1e-10
GEOS = {512: (257, 32), 400: (201, 25), 1024: (513, 64)}
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def _engine(se, n_fft, hop, kind="LSTM", hidden=32, layers=2, cmvn=False, activation=None, precision=1):
    n_freq, win_ms = GEOS[n_fft]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop // 16, n_freq=n_freq).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(7)
    if kind == "LSTM":
        head = se.LSTM(input_size=n_freq, output_size=n_freq, hidden_size=hidden, num_layers=layers,
                       activation=activation or "Identity", precision=precision)
    else:
        head = se.Residual(input_size=n_freq, output_size=n_freq, hidden_size=hidden, num_layers=layers, cmvn=cmvn,
                           activation=activation or "Sigmoid", precision=precision)
    return se.EnhancementEngine(pre, head.cuda().eval(), log_features=True, precision=precision)


def _ragged(B, T, seed, hop):
    lens = torch.LongTensor([T - (1777 * i) % (T // 2) - (hop // 3 if i else 0) for i in range(B)])
    return synth(B, T, seed=seed, lengths=lens)


def _oracle(eng, wavs, lengths, mask, kind="LSTM"):
    """float64 reference of the step from the engine's own head output `mask` (log_predicted for LSTM, offset for Residual):
    _decode_wav against the clean level, waveform SI-SDR, and the per-utterance / batch L1 of log_predicted."""
    n_fft, hop = eng.n_fft, eng.hop
    w = eng.pre._frame_window.double().cpu().numpy()
    x = wavs.double().numpy()
    X, C = stft_f64.stft(x[:, 0], n_fft, hop, w), stft_f64.stft(x[:, 1], n_fft, hop, w)
    m = mask.double().cpu().numpy()
    if kind == "LSTM":
        mag, ax = np.exp(m / 2), np.abs(X)
        Y = np.where(ax > 0, mag * X / np.where(ax > 0, ax, 1.0), mag)
    else:
        Y = np.sqrt(np.maximum(m, 0)) * X
    y = stft_f64.istft(Y, n_fft, hop, w)
    B, T = x.shape[0], x.shape[2]
    y = np.concatenate([y, np.zeros((B, T - y.shape[1]))], 1) if y.shape[1] < T else y[:, :T]
    y = sp.masked_normalize_decibel(torch.from_numpy(y), torch.from_numpy(x[:, 1]), sp.length_masks(lengths)).numpy()
    sisdr = np.array([sp.sisdr_eval(torch.from_numpy(y[b, :n]), torch.from_numpy(x[b, 1, :n])) for b, n in enumerate(lengths.tolist())])
    F = X.shape[1]
    frames = np.minimum(F, lengths.numpy() // hop + 1)
    valid = (np.arange(F)[None, :] < frames[:, None])[..., None]
    d = np.abs(m - np.log(np.abs(C) ** 2 + EPS)) * valid
    per_utt = d.sum((1, 2)) / (frames * X.shape[2])
    return y, sisdr, per_utt, d.sum() / (frames.sum() * X.shape[2]), X, C, valid


def _features64(eng, wavs):
    w = eng.pre._frame_window.double().cpu().numpy()
    X = stft_f64.stft(wavs[:, 0].double().numpy(), eng.n_fft, eng.hop, w)
    return torch.from_numpy(np.log(np.abs(X) ** 2 + eng.pre.eps))


def _head64(eng, feats64, linears=None, cmvn=False):
    """oracle.signal_path.recurrent_head in float64 from the engine's head's own state dict."""
    state = {k: v.detach().double().cpu() for k, v in eng.head.state_dict().items()}
    kind = type(eng.head).__name__
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.no_grad():
            _, extra = sp.recurrent_head(kind, state, feats64, linears, activation=eng.head.activation, cmvn=cmvn,
                                         eps=getattr(eng.head, "eps", 1e-6))
    finally:
        torch.set_default_dtype(prev)
    return extra["log_predicted" if kind == "LSTM" else "offset"]


def _check_step(out, ref, lengths, wav_rtol=2e-4):
    y, sisdr, per_utt, batch = ref[:4]
    for b, n in enumerate(lengths.tolist()):
        got = out["wav_predicted"][b, :n].double().cpu().numpy()
        assert np.abs(got - y[b, :n]).max() <= wav_rtol * np.abs(y[b, :n]).max(), f"utterance {b}: waveform"
    np.testing.assert_allclose(out["sisdr"].cpu().double().numpy(), sisdr, atol=0.01, rtol=0)     # 0.01 dB


# ------------------------------------------------------------------------------ 1. float64 oracle: LSTM + L1 on every route
# fp32 FFTs and lg2.approx put ~1e-6 relative error on each |lp - log(|C|^2 + eps)| term; per-run fp32 sums of <= 64 frames x K
# terms before the double atomics: 1e-4 relative leaves a wide margin.  The head itself (cuDNN LSTM, TF32 projection) is checked
# against its float64 restatement with a tolerance for TF32 operands.
@gpu
@pytest.mark.parametrize("n_fft,hop,T", [(512, 256, 20000), (400, 160, 20000), (1024, 256, 20000), (512, 128, 12000),
                                         (512, 256, 1200)])
def test_lstm_l1_step_matches_the_float64_oracle(se, n_fft, hop, T):
    from speech_enhancement_by_s3prl_b200 import ops
    B = 5 if T > 2000 else 3
    lengths, wavs = _ragged(B, T, seed=n_fft + hop, hop=hop) if T > 2000 else synth(B, T, 3, torch.LongTensor([T, 900, 700]))
    eng = _engine(se, n_fft, hop)
    eng.eval_step(lengths.cuda(), wavs.cuda())
    base = eng.launches_per_step                                                  # the SISDR step's launches
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    out = eng.eval_step(lengths.cuda(), wavs.cuda(), criterion=se.L1(), metric_acc=acc)
    torch.cuda.synchronize()
    fused = ops.mask_istft_l1_supported(n_fft, hop) and T // hop + 1 >= 6
    assert fused == ((n_fft, hop) in ((512, 256), (400, 160), (1024, 256)) and T > 2000)
    # the route taken: K3-L1 + finish (one launch more), or the slow route's STFT + sums + finish (three more)
    assert eng.launches_per_step == base + (1 if fused else 3)
    ref = _oracle(eng, wavs, lengths, out["mask"])
    _check_step(out, ref, lengths)
    np.testing.assert_allclose(out["loss_per_utt"].cpu().double().numpy(), ref[2], rtol=1e-4, atol=0)
    assert out["loss"].item() == pytest.approx(ref[3], rel=1e-4)
    assert acc[0].item() == pytest.approx(B * out["loss"].item(), rel=1e-6) and acc[2].item() == B
    lp64 = _head64(eng, _features64(eng, wavs)).numpy()
    lp = out["mask"].double().cpu().numpy()
    assert np.abs(lp - lp64).max() <= 1e-2 * max(1.0, np.abs(lp64).max())


@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (400, 160)])
def test_lstm_sisdr_mode_uses_exp_of_log_predicted(se, n_fft, hop):
    """criterion None: the spectral SI-SDR of predicted = exp(log_predicted) (objective.SISDR on the LSTM's output)."""
    B, T = 4, 16000
    lengths, wavs = _ragged(B, T, seed=5, hop=hop)
    eng = _engine(se, n_fft, hop)
    out = eng.eval_step(lengths.cuda(), wavs.cuda())
    torch.cuda.synchronize()
    assert "loss" not in out
    y, sisdr, _, _, X, C, valid = _oracle(eng, wavs, lengths, out["mask"])
    _check_step(out, (y, sisdr, None, None), lengths)
    lp = out["mask"].double().cpu().numpy()
    masks = torch.from_numpy(valid[..., 0].astype(np.int64))
    _, want = sp.sisdr_spectral(torch.from_numpy(np.exp(lp)), torch.from_numpy(np.abs(C) ** 2), masks)
    np.testing.assert_allclose(out["loss_per_utt"].cpu().double().numpy(), want.numpy(), atol=2e-3, rtol=0)


@gpu
@pytest.mark.parametrize("cmvn,crit", [(False, None), (True, "WSD")])
def test_residual_head_matches_the_float64_oracle(se, cmvn, crit):
    B, T, n_fft, hop = 4, 16000, 512, 256
    lengths, wavs = _ragged(B, T, seed=13, hop=hop)
    eng = _engine(se, n_fft, hop, kind="Residual", cmvn=cmvn)
    criterion = se.WSD() if crit == "WSD" else None
    out = eng.eval_step(lengths.cuda(), wavs.cuda(), criterion=criterion)
    torch.cuda.synchronize()
    ref = _oracle(eng, wavs, lengths, out["mask"], kind="Residual")
    _check_step(out, ref, lengths)
    X, C, valid = ref[4:]
    G = out["mask"].double().cpu().numpy()
    lin_x, lin_c = torch.from_numpy(np.abs(X) ** 2), torch.from_numpy(np.abs(C) ** 2)
    masks = torch.from_numpy(valid[..., 0].astype(np.int64))
    if crit == "WSD":
        want = sp.wsd(lin_x, torch.from_numpy(G), lin_c, masks)
        assert out["loss_per_utt"].double().mean().item() == pytest.approx(want.item(), rel=1e-4)
    else:
        _, want = sp.sisdr_spectral(lin_x * torch.from_numpy(G), lin_c, masks)
        np.testing.assert_allclose(out["loss_per_utt"].cpu().double().numpy(), want.numpy(), atol=2e-3, rtol=0)
    off64 = _head64(eng, _features64(eng, wavs), linears=lin_x, cmvn=cmvn).numpy()
    assert np.abs(G - off64).max() <= 1e-2


# ------------------------------------------------------------------------------ 2. the drop-ins
@gpu
def test_lstm_waveform_equals_the_drop_in_decode(se):
    from speech_enhancement_by_s3prl_b200 import runner_ops
    B, T, n_fft, hop = 4, 16000, 512, 256
    lengths, wavs = _ragged(B, T, seed=17, hop=hop)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    eng = _engine(se, n_fft, hop)
    crit = se.L1()
    out = eng.eval_step(lengths, wavs, criterion=crit)
    c = eng.pre.get_feat_config
    feats, phase, linear_tar = eng.pre(wavs, [c("linear", 0, log=True), c("phase", 0), c("linear", 1)])
    with torch.no_grad():
        _, extra = eng.head(features=feats, linears=None)
    want = runner_ops.decode_wav(eng.pre, out["mask"].exp().contiguous(), phase, lengths, wavs[:, 1])
    n = int(lengths.max())
    torch.testing.assert_close(out["wav_predicted"][:, :n], want[:, :n], rtol=1e-4, atol=2e-4 * want.abs().max().item())
    # the criterion of the drop-in modules on the drop-in head's output
    ref, _ = crit(log_predicted=extra["log_predicted"], linear_tar=linear_tar, stft_lengths=lengths // hop + 1)
    assert out["loss"].item() == pytest.approx(ref.item(), rel=2e-3)


# ------------------------------------------------------------------------------ 3. captured replays
@gpu
def test_captured_replays_equal_eager_steps_and_clear_the_l1_buffer(se):
    B, T = 4, 16000
    eng = _engine(se, 512, 256)
    crit = se.L1()
    batches = [_ragged(B, T, seed=s, hop=256) for s in (21, 22)]
    eager = []
    for l, w in batches:
        e = eng.eval_step(l.cuda(), w.cuda(), criterion=crit)
        eager.append({k: v.clone() for k, v in e.items() if v is not None})
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    l0, w0 = batches[0]
    st = eng.capture_bound(l0.cuda(), w0.cuda(), metric_acc=acc, criterion=crit)
    assert st["ws"][-2:].abs().sum().item() == 0.0
    for (l, w), e in zip(batches, eager):
        st["lengths"].copy_(l)
        st["wavs"].copy_(w)
        st["graph"].replay()
        torch.cuda.synchronize()
        assert st["ws"][-2:].abs().sum().item() == 0.0                          # [sum, count] back at zero
        torch.testing.assert_close(st["loss_per_utt"], e["loss_per_utt"], rtol=1e-5, atol=0)
        torch.testing.assert_close(st["loss"], e["loss"], rtol=1e-5, atol=0)
        torch.testing.assert_close(st["sisdr"], e["sisdr"], rtol=1e-5, atol=1e-5)
    want = sum(B * e["loss"].double().item() for e in eager)
    assert acc[0].item() == pytest.approx(want, rel=1e-5)
    assert acc[1].item() == pytest.approx(sum(e["sisdr"].double().sum().item() for e in eager), rel=1e-5, abs=1e-4)
    assert acc[2].item() == 2 * B
    # the cached graph of eval_step_graph gives the same
    g = eng.eval_step_graph(l0.cuda(), w0.cuda(), criterion=crit)
    torch.cuda.synchronize()
    torch.testing.assert_close(g["loss"], eager[0]["loss"], rtol=1e-5, atol=0)
    # the host path reports objective.L1 of the ragged batch (frame-weighted), not the plain mean of the per-utterance terms
    mean_loss, mean_sisdr, _ = eng.eval_step_host(l0, w0.contiguous(), criterion=crit)
    assert mean_loss == pytest.approx(eager[0]["loss"].item(), rel=1e-5)
    assert mean_sisdr == pytest.approx(eager[0]["sisdr"].double().mean().item(), rel=1e-5, abs=1e-5)
    assert abs(eager[0]["loss_per_utt"].double().mean().item() - mean_loss) > 1e-6 * mean_loss


# ------------------------------------------------------------------------------ 4. data parallelism
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_batch():
    lengths, wavs = _ragged(7, 16000, seed=31, hop=256)
    wavs[5] *= 10.0
    return lengths, wavs


def _gloo_worker(rank, world_size, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp
    lengths, wavs = dp.shard_batch(*_dp_batch(), rank, world_size)
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    out = _engine(se, 512, 256).eval_step(lengths.cuda(), wavs.cuda(), criterion=se.L1(), metric_acc=acc)
    mean_loss, mean_sisdr, n = dp.means_from_acc(acc)
    torch.cuda.synchronize()
    ret[rank] = (out["loss"].item(), out["loss_per_utt"].cpu(), mean_loss.item(), mean_sisdr.item(), n.item())
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_two_ranks_on_uneven_shards_report_the_whole_batch_l1(se):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_gloo_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    lengths, wavs = _dp_batch()
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    out = _engine(se, 512, 256).eval_step(lengths.cuda(), wavs.cuda(), criterion=se.L1(), metric_acc=acc)
    torch.cuda.synchronize()
    whole = out["loss"].item()
    for rank, (lo, hi) in enumerate([(0, 4), (4, 7)]):
        loss, per_utt, mean_loss, mean_sisdr, n = ret[rank]
        assert loss == pytest.approx(whole, rel=1e-5)                           # the global element mean on every rank
        np.testing.assert_allclose(per_utt.numpy(), out["loss_per_utt"][lo:hi].cpu().numpy(), rtol=1e-5)
        assert mean_loss == pytest.approx(acc[0].item() / 7, rel=1e-5)
        assert mean_sisdr == pytest.approx(acc[1].item() / 7, rel=1e-5, abs=1e-5)
        assert n == 7
    # each shard's own mean differs from the global one: the count is all-reduced with the sum
    assert abs(ret[0][1].mean().item() - whole) > 1e-4 * whole


# ------------------------------------------------------------------------------ 5. errors
@gpu
def test_unsupported_head_criterion_pairs_raise(se):
    lengths, wavs = _ragged(2, 8000, seed=1, hop=256)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    with pytest.raises(RuntimeError, match="L1 with a Residual head"):
        _engine(se, 512, 256, kind="Residual").eval_step(lengths, wavs, criterion=se.L1())
    with pytest.raises(RuntimeError, match="WSD with a LSTM head"):
        _engine(se, 512, 256).eval_step(lengths, wavs, criterion=se.WSD())


# ------------------------------------------------------------------------------ 6. CPU: the table, the exports, the flag
def test_head_criterion_table_is_host_logic():
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import engine
    lstm = se.LSTM(input_size=9, output_size=9, hidden_size=4, num_layers=1)
    res = se.Residual(input_size=9, output_size=9, hidden_size=4, num_layers=1)
    lin = se.Linear(input_size=9, output_size=9)
    linres = se.LinearResidual(input_size=9, output_size=9)
    assert engine._eval_loss(se.L1(), lstm) == "l1"
    for head in (lstm, res, lin, linres):
        assert engine._eval_loss(None, head) == engine._eval_loss(se.SISDR(), head) == "sisdr"
    assert engine._eval_loss(se.WSD(), res) == engine._eval_loss(se.WSD(), linres) == "wsd"
    for crit, head in ((se.L1(), res), (se.L1(), lin), (se.L1(), linres), (se.WSD(), lstm)):
        with pytest.raises(RuntimeError, match=f"{type(crit).__name__} with a {type(head).__name__} head"):
            engine._eval_loss(crit, head)
    assert engine._criterion_key(se.L1(eps=1e-8)) == ("L1", 1e-8)
    assert engine._recurrent(lstm) and engine._recurrent(res) and not engine._recurrent(linres)


def test_l1_eval_exports_flag_and_supported_geometries():
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    lib = _lib.load()
    for name in ("se_mask_istft_l1_supported", "se_mask_istft_l1", "se_l1_eval_sums", "se_l1_eval_finish"):
        assert name in _lib.EXPORTS and hasattr(lib, name)
    for n_fft, hop in ((512, 256), (1024, 256), (400, 160)):
        assert lib.se_mask_istft_l1_supported(n_fft, hop) == 1
    for n_fft, hop in ((512, 128), (256, 128), (400, 200)):
        assert lib.se_mask_istft_l1_supported(n_fft, hop) == 0
    assert ops.FLAG_MASK_IS_LOG_POWER == 16
    with open(os.path.join(ROOT, "include", "se_b200.h")) as f:
        header = f.read()
    assert re.search(r"#define SE_FLAG_MASK_IS_LOG_POWER 16\b", header)
    flags = [int(v) for v in re.findall(r"#define SE_FLAG_\w+ (\d+)", header)]
    assert len(flags) == len(set(flags)) and all(v & (v - 1) == 0 for v in flags)      # distinct single bits
