"""The evaluation step with objective.WSD (EnhancementEngine.eval_step(criterion=WSD)): the WSD variant of K3 on the
register-resident geometries, the split kernels on materialised spectra elsewhere, the finish kernel, captured replays and
data parallelism -- every rank thresholds voicing against the loudest frame of the GLOBAL padded batch (objective.py:127-153)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

from oracle import stft_f64

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_parity import synth  # noqa: E402

gpu = pytest.mark.gpu
EPS = 1e-10
# n_fft -> (n_freq, win_ms); hop_ms from the hop at 16 kHz
GEOS = {512: (257, 32), 400: (201, 25), 1024: (513, 64)}


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def _engine(se, n_fft, hop, route="log", activation="Sigmoid"):
    n_freq, win_ms = GEOS[n_fft]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop // 16, n_freq=n_freq).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(7)
    feat_cfg = pre.get_feat_config("mel", 0, log=True, delta=2) if route == "mel" else None
    precision = 0 if route == "p0" else 1
    head = se.LinearResidual(input_size=120 if feat_cfg else n_freq, output_size=n_freq, activation=activation,
                             precision=precision).cuda()
    return se.EnhancementEngine(pre, head, log_features=True, precision=precision, feat_cfg=feat_cfg)


def _power64(wavs, ch, n_fft, hop):
    return np.abs(stft_f64.stft(wavs[:, ch].double().numpy(), n_fft, hop)) ** 2


def _terms64(wavs, mask, lengths, n_fft, hop, alpha, db, emax=None, guard=True):
    """alpha sd_u + (1 - alpha) rn_u in float64 from float64 spectra of both channels and the engine's own mask as G.
    emax: the maximum to threshold against (default: over every frame of the padded batch).  guard: no valid frame's energy
    lies within 1e-3 dB of the threshold -- otherwise one voicing flip between fp32 and float64 would exceed the bound."""
    X, S = _power64(wavs, 0, n_fft, hop), _power64(wavs, 1, n_fft, hop)
    G = mask.double().cpu().numpy()
    F = S.shape[1]
    frames = np.minimum(F, lengths.numpy() // hop + 1)
    valid = (np.arange(F)[None, :] < frames[:, None])[..., None]
    energy = S.sum(-1)
    top = energy.max() if emax is None else emax
    thr = 10 * np.log10(top + EPS) - db
    level = 10 * np.log10(energy + EPS)
    if guard:
        assert np.abs(level - thr)[valid[..., 0]].min() > 1e-3, "a valid frame sits on the voicing threshold"
    voiced = (level > thr)[..., None]
    sd = (((S - G * S) * voiced * valid) ** 2).sum((1, 2))
    rn = ((G * np.maximum(X - S, 0.0) * valid) ** 2).sum((1, 2))
    return alpha * sd + (1 - alpha) * rn, energy, valid


def _ragged(B, T, seed, hop):
    lens = torch.LongTensor([T - (1777 * i) % (T // 2) - (hop // 3 if i else 0) for i in range(B)])
    return synth(B, T, seed=seed, lengths=lens)


# ------------------------------------------------------------------------------ 1. float64 oracle, every route
# fp32 FFTs (relative error ~1e-6 of a frame's energy per bin), fp32 per-frame sums of <= 513 terms and fp32 per-run sums of
# the residual noise before the float64 atomics: ~1e-5 relative per utterance at most, 1e-4 leaves a 10x margin.  A voicing
# flip would move a whole frame's D_f, hence the guard in _terms64.
@gpu
@pytest.mark.parametrize("n_fft,hop,route", [(512, 256, "log"), (512, 256, "mel"), (512, 256, "p0"),
                                             (400, 160, "log"), (400, 160, "mel"), (400, 160, "p0"),
                                             (1024, 256, "log"), (1024, 256, "mel"), (1024, 256, "p0"),
                                             (512, 128, "log")])
def test_wsd_loss_matches_the_float64_oracle(se, n_fft, hop, route):
    from speech_enhancement_by_s3prl_b200 import ops
    B, T = 5, 20000
    lengths, wavs = _ragged(B, T, seed=n_fft + hop, hop=hop)
    eng = _engine(se, n_fft, hop, route)
    alpha, db = 0.3, 30.0
    out = eng.eval_step(lengths.cuda(), wavs.cuda(), criterion=se.WSD(alpha=alpha, db_interval=db))
    torch.cuda.synchronize()
    assert ops.mask_istft_wsd_supported(n_fft, hop) == ((n_fft, hop) in ((512, 256), (400, 160), (1024, 256)))
    ref, _, _ = _terms64(wavs, out["mask"], lengths, n_fft, hop, alpha, db)
    assert np.all(ref > 0)
    np.testing.assert_allclose(out["loss_per_utt"].cpu().double().numpy(), ref, rtol=1e-4, atol=0)


@gpu
def test_wsd_loss_with_a_signed_mask(se):
    """Identity activation: masks of both signs (the residual-noise term is d^2 where G d > 0, d = G X - G S)."""
    B, T, n_fft, hop = 4, 16000, 512, 256
    lengths, wavs = _ragged(B, T, seed=3, hop=hop)
    eng = _engine(se, n_fft, hop, "log", activation="Identity")
    out = eng.eval_step(lengths.cuda(), wavs.cuda(), criterion=se.WSD())
    torch.cuda.synchronize()
    assert (out["mask"] < 0).any() and (out["mask"] > 0).any()
    ref, _, _ = _terms64(wavs, out["mask"], lengths, n_fft, hop, 0.5, 30.0)
    np.testing.assert_allclose(out["loss_per_utt"].cpu().double().numpy(), ref, rtol=1e-4, atol=0)


# ------------------------------------------------------------------------------ 2. the maximum runs over padded frames too
@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (400, 160)])
def test_loudest_frame_past_the_valid_length_sets_the_threshold(se, n_fft, hop):
    """Utterance 0 ends one sample before a hop boundary with a loud burst in its last n_fft / 8 samples: the frame just past its
    valid range is centred on the burst and is the loudest of the batch; the reference's threshold uses it."""
    B, T = 3, 16000
    L0 = (T // hop - 6) * hop + hop - 1
    lengths, wavs = synth(B, T, seed=11, lengths=torch.LongTensor([L0, T, T - 3000]))
    burst = torch.sin(torch.arange(n_fft // 8) * 0.7) * 2.0
    wavs[0, 0, L0 - n_fft // 8:L0] += burst
    wavs[0, 1, L0 - n_fft // 8:L0] += burst
    alpha, db = 0.5, 30.0
    out = _engine(se, n_fft, hop).eval_step(lengths.cuda(), wavs.cuda(), criterion=se.WSD(alpha=alpha, db_interval=db))
    torch.cuda.synchronize()
    ref, energy, valid = _terms64(wavs, out["mask"], lengths, n_fft, hop, alpha, db)
    valid_max = energy[valid[..., 0]].max()
    assert energy.max() > 2 * valid_max                                       # the loudest frame is past a valid range
    masked, _, _ = _terms64(wavs, out["mask"], lengths, n_fft, hop, alpha, db, emax=valid_max, guard=False)
    got = out["loss_per_utt"].cpu().double().numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=0)
    assert np.abs(masked - ref).max() > 10 * 1e-4 * np.abs(ref).max()        # the masked maximum gives another loss


# ------------------------------------------------------------------------------ 3. SISDR mode unchanged, WSD only changes the loss
@gpu
@pytest.mark.parametrize("route", ["log", "mel", "p0"])
def test_sisdr_mode_is_unchanged_and_wsd_changes_only_the_loss(se, route):
    B, T = 4, 16000
    lengths, wavs = _ragged(B, T, seed=5, hop=256)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    eng = _engine(se, 512, 256, route)
    a = eng.eval_step(lengths, wavs)
    n_a = eng.launches_per_step
    b = eng.eval_step(lengths, wavs, criterion=se.SISDR())
    n_b = eng.launches_per_step
    w = eng.eval_step(lengths, wavs, criterion=se.WSD())
    n_w = eng.launches_per_step
    torch.cuda.synchronize()
    assert n_a == n_b and n_w == n_a + 1
    for key in ("wav_predicted", "gain", "sisdr", "mask"):
        assert torch.equal(a[key], b[key]), key
    assert torch.allclose(a["loss_per_utt"], b["loss_per_utt"], rtol=1e-6, atol=0)   # (float64 atomics: any order)
    for key in ("wav_predicted", "gain", "sisdr"):
        scale = a[key].abs().max()
        assert (w[key] - a[key]).abs().max() <= 1e-6 * scale, key
    assert not torch.allclose(w["loss_per_utt"], a["loss_per_utt"])


# ------------------------------------------------------------------------------ 4. the drop-in modules
@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (400, 160)])
def test_batch_mean_equals_the_drop_in_objective(se, n_fft, hop):
    B, T = 6, 16000
    lengths, wavs = _ragged(B, T, seed=9, hop=hop)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    eng = _engine(se, n_fft, hop)
    crit = se.WSD(alpha=0.7, db_interval=20.0)
    out = eng.eval_step(lengths, wavs, criterion=crit)
    c = eng.pre.get_feat_config
    linear_inp, linear_tar = eng.pre(wavs, [c("linear", 0), c("linear", 1)])
    ref, _ = crit(linear_inp=linear_inp, offset=out["mask"], linear_tar=linear_tar, stft_lengths=lengths // hop + 1)
    assert out["loss_per_utt"].mean().item() == pytest.approx(ref.item(), rel=1e-4)


# ------------------------------------------------------------------------------ 5. captured replays
@gpu
@pytest.mark.parametrize("route", ["log", "p0"])
def test_captured_replays_reset_the_maximum(se, route):
    B, T = 4, 16000
    eng = _engine(se, 512, 256, route)
    crit = se.WSD()
    l1, w1 = _ragged(B, T, seed=21, hop=256)
    l2, w2 = _ragged(B, T, seed=22, hop=256)
    w2 *= 1e-2                                                                 # 40 dB quieter: a stale maximum unvoices it
    eager = [eng.eval_step(l.cuda(), w.cuda(), criterion=crit) for l, w in ((l1, w1), (l2, w2))]
    eager = [{k: v.clone() for k, v in e.items() if v is not None} for e in eager]
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    st = eng.capture_bound(l1.cuda(), w1.cuda(), metric_acc=acc, criterion=crit)
    got = []
    for l, w in ((l1, w1), (l2, w2)):
        st["lengths"].copy_(l)
        st["wavs"].copy_(w)
        st["graph"].replay()
        torch.cuda.synchronize()
        got.append((st["loss_per_utt"].clone(), st["sisdr"].clone()))
        assert st["ws"][-1].item() == 0.0                                       # maximum and counter left at zero
    for (loss, sisdr), e in zip(got, eager):
        torch.testing.assert_close(loss, e["loss_per_utt"], rtol=1e-5, atol=0)
        torch.testing.assert_close(sisdr, e["sisdr"], rtol=1e-5, atol=1e-5)
    # had the first batch's maximum survived, the quiet batch would be thresholded against it
    ref_stale, _, _ = _terms64(w2, eager[1]["mask"], l2, 512, 256, 0.5, 30.0,
                               emax=_power64(w1, 1, 512, 256).sum(-1).max(), guard=False)
    assert np.abs(ref_stale - got[1][0].cpu().double().numpy()).max() > 1e-3 * got[1][0].abs().max().item()
    want = [sum(e[k].double().sum().item() for e in eager) for k in ("loss_per_utt", "sisdr")]
    assert acc[0].item() == pytest.approx(want[0], rel=1e-5)
    assert acc[1].item() == pytest.approx(want[1], rel=1e-5, abs=1e-4)
    assert acc[2].item() == 2 * B


# ------------------------------------------------------------------------------ 6. data parallelism
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_batch():
    """7 utterances; utterance 5 (rank 1's shard under the 4 / 3 split) is 40 dB louder than the others."""
    lengths, wavs = _ragged(7, 16000, seed=31, hop=256)
    wavs[5] *= 100.0
    return lengths, wavs


def _gloo_worker(rank, world_size, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp
    lengths, wavs = dp.shard_batch(*_dp_batch(), rank, world_size)
    out = _engine(se, 512, 256).eval_step(lengths.cuda(), wavs.cuda(), criterion=se.WSD())
    torch.cuda.synchronize()
    ret[rank] = out["loss_per_utt"].cpu()
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_two_ranks_threshold_against_the_global_maximum(se):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_gloo_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    lengths, wavs = _dp_batch()
    out = _engine(se, 512, 256).eval_step(lengths.cuda(), wavs.cuda(), criterion=se.WSD())
    whole = out["loss_per_utt"].cpu()
    for rank, (lo, hi) in enumerate([(0, 4), (4, 7)]):
        np.testing.assert_allclose(ret[rank].numpy(), whole[lo:hi].numpy(), rtol=2e-5, atol=0)
    # rank 0 thresholding against its own maximum would report another loss
    ref, energy, _ = _terms64(wavs, out["mask"], lengths, 512, 256, 0.5, 30.0)
    local, _, _ = _terms64(wavs[:4], out["mask"][:4], lengths[:4], 512, 256, 0.5, 30.0, guard=False)
    assert energy[:4].max() < energy.max()
    assert np.abs(local - ref[:4]).max() > 10 * 1e-4 * np.abs(ref[:4]).max()


def _nccl_worker(rank, world_size, port, ret):
    """A world-size-1 NCCL group standing in for N ranks: ``dp.world`` reports two, so the step forks its side stream and
    ``dp.global_max`` issues a real NCCL all-reduce(MAX) there -- eagerly and inside the captured graph."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK="0", WORLD_SIZE="1")
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp
    streams = []

    def global_max(t):
        streams.append(torch.cuda.current_stream().cuda_stream)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t

    dp.world, dp.global_max = (lambda: (0, 2)), global_max
    lengths, wavs = _ragged(4, 16000, seed=41, hop=256)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    eng = _engine(se, 512, 256)
    crit = se.WSD()
    eager = [eng.eval_step(lengths, wavs, criterion=crit)["loss_per_utt"].cpu() for _ in range(3)]
    n_eager = len(streams)
    acc = torch.zeros(3, device="cuda", dtype=torch.float64)
    st = eng.capture_bound(lengths, wavs, metric_acc=acc, criterion=crit)
    for _ in range(3):
        st["graph"].replay()
    torch.cuda.synchronize()
    side = [s.cuda_stream for s in eng._side_streams.values()]
    ret[0] = (eager, st["loss_per_utt"].cpu(), acc.cpu(), n_eager, len(streams), all(s in side for s in streams))
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_captured_wsd_eval_all_reduces_the_maximum_on_a_side_stream(se):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_nccl_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    eager, graph, acc, n_eager, n_all, on_side = ret[0]
    assert n_eager == 3 and n_all == 6 and on_side      # one per eager step; 2 warm-ups + the capture; all on the side stream
    for e in eager[1:]:
        torch.testing.assert_close(e, eager[0], rtol=1e-6, atol=0)
    torch.testing.assert_close(graph, eager[0], rtol=1e-5, atol=0)
    assert acc[0].item() == pytest.approx(3 * eager[0].double().sum().item(), rel=1e-5)
    assert acc[2].item() == 12


# ------------------------------------------------------------------------------ 7. errors and the no-loss mode
@gpu
def test_unsupported_criterion_raises_and_no_loss_without_want_spec_loss(se):
    lengths, wavs = _ragged(2, 8000, seed=1, hop=256)
    eng = _engine(se, 512, 256)
    with pytest.raises(RuntimeError, match="SISDR.*WSD"):
        eng.eval_step(lengths.cuda(), wavs.cuda(), criterion=se.L1())
    out = eng.eval_step(lengths.cuda(), wavs.cuda(), want_spec_loss=False, criterion=se.WSD())
    assert out["loss_per_utt"] is None and torch.isfinite(out["sisdr"]).all()


# ------------------------------------------------------------------------------ 8. CPU: which geometries have the fused route
def test_wsd_eval_route_is_host_logic():
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    for n_fft, hop in ((512, 256), (1024, 256), (400, 160)):
        assert lib.se_mask_istft_wsd_supported(n_fft, hop) == 1
    for n_fft, hop in ((512, 128), (256, 128)):
        assert lib.se_mask_istft_wsd_supported(n_fft, hop) == 0
