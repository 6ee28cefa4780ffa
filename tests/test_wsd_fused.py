"""objective.WSD split at its batch maximum (se_wsd_energy -> all-reduce(max) -> se_wsd_mask_step), its backward folded into
the TMA weight-gradient kernel (se_linear_head_bwd_wsd), the fused WSD training step, and data parallelism: every rank
thresholds voicing against the loudest frame of the GLOBAL batch, as the single-process reference does."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import signal_path as sp

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def _spectra(B, F, K, seed):
    """Heavy-tailed power spectra with a 40 dB spread of frame levels (some frames far below the voicing threshold) and
    X - S of both signs."""
    g = torch.Generator().manual_seed(seed)
    tar = (torch.rand(B, F, K, generator=g) ** 4) * 3.0
    tar *= 10.0 ** (-4.0 * torch.rand(B, F, 1, generator=g))
    tar[:, F // 3:F // 2] *= 1e-4
    inp = tar + (torch.rand(B, F, K, generator=g) - 0.3).clamp_min(-0.2) * tar.mean(-1, keepdim=True)
    off = torch.rand(B, F, K, generator=g)
    return g, inp, off, tar


def _terms64(inp, off, tar, frames, alpha, db, emax=None):
    """Per-utterance terms alpha * sd_u + (1 - alpha) * rn_u in float64 (objective.py:127-153 before the batch mean)."""
    inp, off, tar = inp.double(), off.double(), tar.double()
    m = (torch.arange(tar.shape[1])[None, :] < frames[:, None]).double()[..., None]
    energy = tar.sum(-1, keepdim=True)
    top = energy.max() if emax is None else torch.tensor(float(emax), dtype=torch.float64)
    voiced = (10 * torch.log10(energy + 1e-10) > 10 * torch.log10(top + 1e-10) - db).double()
    sd = ((tar - off * tar) * voiced * m).pow(2).sum((1, 2))
    rn = (off * (inp - tar).clamp_min(0) * m).pow(2).sum((1, 2))
    return alpha * sd + (1 - alpha) * rn


# ------------------------------------------------------------------------------ kernels vs the autograd op
@gpu
@pytest.mark.parametrize("B,F,K,alpha,db,hop", [(3, 40, 201, 0.3, 50.0, 160), (5, 120, 257, 0.5, 30.0, 0), (2, 33, 129, 0.9, 10.0, 256)])
def test_split_kernels_match_the_wsd_op(se, B, F, K, alpha, db, hop):
    """wsd_energy + wsd_mask_step on row-padded tensors (NaN in the pad columns; float4 and scalar variants) against se.WSD on
    the unpadded ones: ragged lengths as sample lengths with hop or as frame counts, frames below the threshold."""
    from speech_enhancement_by_s3prl_b200 import ops
    g, inp, off, tar = _spectra(B, F, K, seed=B * F + K)
    frames = torch.randint(F // 2, F + 1, (B,), generator=g)
    frames[0] = F
    lens = ((frames - 1) * hop + torch.randint(0, hop, (B,), generator=g)) if hop else frames
    ref_off = off.cuda().requires_grad_(True)
    loss_ref, _ = se.WSD(alpha=alpha, db_interval=db)(inp.cuda(), ref_off, tar.cuda(), stft_lengths=frames.cuda())
    loss_ref.backward()
    masks = (torch.arange(F)[None, :] < frames[:, None]).long()
    assert loss_ref.item() == pytest.approx(sp.wsd(inp, off, tar, masks, alpha=alpha, db_interval=db).item(), rel=2e-5)
    terms = _terms64(inp, off, tar, frames, alpha, db)
    g_ref = ref_off.grad
    for LD in (K, ops.round4(K)):
        pad = lambda x: torch.nn.functional.pad(x, (0, LD - K), value=float("nan")).contiguous().cuda()
        energy, emax = ops.wsd_energy(pad(tar), K)
        assert energy.shape == (B, F) and emax.shape == (1,) and emax.dtype == torch.float32
        assert (energy.cpu() - tar.sum(-1)).abs().max().item() < 1e-5 * tar.sum(-1).max().item()
        assert emax.item() == energy.max().item()                              # a plain float: what all_reduce(MAX) combines
        loss, loss_u, g_off, sums2 = ops.wsd_mask_step(pad(off), pad(inp), pad(tar), lens.cuda(), hop, K, energy, emax, alpha, db)
        assert loss.dim() == 0 and loss.item() == pytest.approx(loss_ref.item(), rel=1e-5)
        np.testing.assert_allclose(loss_u.cpu().double().numpy(), terms.numpy(), rtol=1e-5, atol=0)
        assert sums2.shape == (B, 2) and sums2.dtype == torch.float64
        assert g_off.shape == (B, F, LD) and torch.isfinite(g_off).all() and (g_off[..., K:] == 0).all()
        scale = g_ref.abs().max().item()
        assert (g_off[..., :K] - g_ref).abs().max().item() < 2e-5 * scale
        for b in range(B):
            assert (g_off[b, int(frames[b]):] == 0).all()                      # padded frames carry no gradient
        loss1, loss_u1, none, _ = ops.wsd_mask_step(pad(off), pad(inp), pad(tar), lens.cuda(), hop, K, energy, emax, alpha, db,
                                                    want_grad=False)
        assert none is None and loss1.item() == pytest.approx(loss.item(), rel=1e-6)


@gpu
def test_wsd_energy_maximum_of_any_sign(se):
    """The maximum buffer orders sums of any sign as floats (atomicMax of the bits for non-negative sums, atomicMin for
    negative ones, in any arrival order): all-negative rows, mixed signs, one non-negative row among negatives."""
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(5)
    B, F, K = 6, 700, 129
    base = torch.rand(B, F, K, generator=g) + 0.01
    cases = {"all negative": -base, "mixed": torch.randn(B, F, K, generator=g), "one non-negative row": -base.clone()}
    cases["one non-negative row"][4, 321] = 0.001
    for name, tar in cases.items():
        pad = torch.nn.functional.pad(tar, (0, ops.round4(K) - K), value=float("nan")).contiguous().cuda()
        energy, emax = ops.wsd_energy(pad, K)
        assert (energy.cpu() - tar.sum(-1)).abs().max().item() < 1e-4 * tar.sum(-1).abs().max().item(), name
        assert emax.item() == energy.max().item(), name


# ------------------------------------------------------------------------------ the backward folded into the weight gradient
@gpu
@pytest.mark.parametrize("B,F,D,act,cmvn,hop", [(4, 101, 257, "Sigmoid", True, 256), (48, 300, 201, "Sigmoid", True, 160),
                                                (5, 64, 129, "ReLU", False, 0), (7, 50, 201, "ReLU", True, 160)])
def test_head_backward_with_wsd_folded_in(se, B, F, D, act, cmvn, hop):
    """se_linear_head_bwd_wsd equals se_wsd_mask_step's grad_offset followed by se_linear_head_bwd_fused on the same padded
    operands, and float64 autograd of the reference objective through the head."""
    from speech_enhancement_by_s3prl_b200 import ops
    alpha, db = 0.3, 30.0
    g, inp, off, tar = _spectra(B, F, D, seed=B + F + D)
    LD = ops.round4(D)
    pad = lambda x: torch.nn.functional.pad(x, (0, LD - D), value=float("nan")).contiguous().cuda()
    feats = pad(torch.randn(B, F, D, generator=g) * 2 - 3)
    if act == "ReLU":
        off = (off - 0.3).clamp_min(0.0)
    off, inp, tar = pad(off), pad(inp), pad(tar)
    frames = torch.randint(1, F + 1, (B,), generator=g)
    frames[0] = F
    lens = (((frames - 1) * hop + torch.randint(0, max(hop, 1), (B,), generator=g)) if hop else frames).cuda()
    frames = frames.cuda()
    assert ops.linear_head_bwd_wsd_supported(B, F, D, D, LD, LD, LD, LD)
    sums = ops.feature_sums(feats, D) if cmvn else None
    energy, emax = ops.wsd_energy(tar, D)
    loss, _, g_off, _ = ops.wsd_mask_step(off, inp, tar, lens, hop, D, energy, emax, alpha, db)
    gw0, gb0 = ops.linear_head_bwd_fused(feats, D, sums, 1e-6, off, g_off, D, act)
    gw1, gb1 = ops.linear_head_bwd_wsd(feats, D, sums, 1e-6, off, inp, tar, lens, hop, energy, emax, D, act, alpha, db)
    torch.cuda.synchronize()
    assert torch.isfinite(gw1).all() and torch.isfinite(gb1).all()
    sw, sb = gw0.abs().max().item(), gb0.abs().max().item()
    assert (gw1 - gw0).abs().max().item() < 2e-4 * sw and (gb1 - gb0).abs().max().item() < 2e-4 * sb
    # float64 autograd of the reference formula (objective.py:127-153) through the head
    o64, x64, t64 = (v[..., :D].double() for v in (off, inp, tar))
    xh = feats[..., :D].double()
    if cmvn:
        xh = (xh - xh.mean(1, keepdim=True)) / (xh.std(1, keepdim=True) + 1e-6)
    o64.requires_grad_(True)
    masks = (torch.arange(F, device="cuda")[None, :] < frames[:, None]).double()
    l64 = sp.wsd(x64, o64, t64, masks, alpha=alpha, db_interval=db)
    assert l64.item() == pytest.approx(loss.item(), rel=1e-4)
    l64.backward()
    dz = o64.grad
    if act == "Sigmoid":
        dz = dz * o64.detach() * (1 - o64.detach())
    elif act == "ReLU":
        dz = dz * (o64.detach() > 0).double()
    gw_ref = torch.einsum("bfn,bfk->nk", dz, xh)
    assert (gw1.double() - gw_ref).abs().max().item() < 3e-3 * gw_ref.abs().max().item()
    assert (gb1.double() - dz.sum((0, 1))).abs().max().item() < 3e-3 * dz.sum((0, 1)).abs().max().item()


# ------------------------------------------------------------------------------ engine: fused WSD step vs the autograd route
def _pre(se, n_fft):
    n_freq, win_ms, hop_ms = {400: (201, 25, 10), 512: (257, 32, 16)}[n_fft]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    return pre


def _both_routes(se, pre, lengths, wavs, D_in, D_out, feat_cfg=None):
    out = []
    for fused in (True, False):
        torch.manual_seed(11)
        head = se.LinearResidual(input_size=D_in, output_size=D_out, precision=1).cuda()
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1, feat_cfg=feat_cfg)
        eng.fused_training = fused
        crit = se.WSD()
        assert eng.fused_training_supported(crit, wavs.shape[0], wavs.shape[2]) == fused
        opt = torch.optim.SGD(head.parameters(), lr=0.0)                      # lr 0: gradients only
        loss = eng.train_step(lengths, wavs, crit, opt, None)
        torch.cuda.synchronize()
        out.append((loss.item(), head.linear.weight.grad.clone(), head.linear.bias.grad.clone()))
    return out


def _assert_routes_agree(out):
    (l_f, gw_f, gb_f), (l_a, gw_a, gb_a) = out
    assert np.isfinite(l_f) and l_f == pytest.approx(l_a, rel=1e-4)          # TF32 head in both
    for g_f, g_a in ((gw_f, gw_a), (gb_f, gb_a)):
        scale = g_a.abs().max().item()
        assert scale > 0
        assert (g_f - g_a).abs().max().item() < 4e-3 * scale                  # TF32 operands on both sides, different summation
        assert (g_f - g_a).abs().mean().item() < 4e-4 * scale


@gpu
@pytest.mark.parametrize("B,T,ragged", [(4, 16000, False), (6, 32000, True)])
def test_fused_wsd_training_step_matches_autograd_path(se, B, T, ragged):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_parity import synth
    lens = torch.LongTensor([T - 997 * i for i in range(B)]) if ragged else None
    lengths, wavs = synth(B, T, seed=B + T, lengths=lens)
    _assert_routes_agree(_both_routes(se, _pre(se, 512), lengths.cuda(), wavs.cuda(), 257, 257))


@gpu
def test_fused_wsd_training_step_at_the_configs2_shape(se):
    """48 utterances of 3-10 s at 400 / 160 (one K1 launch for both channels, the folded backward)."""
    from speech_enhancement_by_s3prl_b200 import synth
    lengths, wavs = synth.batch(48, 10.0, min_seconds=3.0)
    _assert_routes_agree(_both_routes(se, _pre(se, 400), lengths.cuda(), wavs.cuda(), 201, 201))


@gpu
def test_fused_wsd_training_step_with_a_mel_feature_config(se):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_parity import synth
    pre = _pre(se, 400)
    lengths, wavs = synth(4, 8000, seed=3, lengths=torch.LongTensor([8000, 6000, 4321, 7999]))
    cfg = pre.get_feat_config("mel", 0, log=True, delta=2)
    _assert_routes_agree(_both_routes(se, pre, lengths.cuda(), wavs.cuda(), 120, 201, feat_cfg=cfg))


@gpu
def test_wsd_train_step_graph_follows_eager_fused_steps(se):
    """The captured fused WSD step with ClipAdam (3 eager warm-ups + 5 replays) lands where eight eager fused steps land."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_parity import synth
    pre = _pre(se, 512)
    lengths, wavs = synth(4, 16000, seed=31, lengths=torch.LongTensor([16000, 12000, 16000, 9000]))
    lengths, wavs = lengths.cuda(), wavs.cuda()
    finals = []
    for graph in (False, True):
        torch.manual_seed(5)
        head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        crit = se.WSD()
        opt = se.ClipAdam(head.parameters(), lr=1e-3)
        w0 = head.linear.weight.detach().clone()
        for _ in range(5 if graph else 8):
            loss = eng.train_step_graph(lengths, wavs, crit, opt, 1.0) if graph else eng.train_step(lengths, wavs, crit, opt, 1.0)
        torch.cuda.synchronize()
        assert opt.steps_taken() == [8]
        finals.append((loss.item(), head.linear.weight.detach().clone(), w0))
    (l_e, w_e, w0), (l_g, w_g, _) = finals
    assert (w_e - w0).abs().max().item() > 1e-3                               # it trained
    assert l_g == pytest.approx(l_e, rel=1e-3)
    assert (w_e - w_g).abs().max().item() < 2e-3                              # 8 Adam steps of lr 1e-3: updates of ~8e-3


# ------------------------------------------------------------------------------ data parallelism (two ranks on one GPU, gloo)
ALPHA, DB = 0.5, 30.0


def _dp_data():
    """Global batch of 7 utterances; utterance 5 (rank 1's shard under the 4 / 3 split) holds the loudest frame."""
    B, F, K = 7, 60, 201
    g, inp, off, tar = _spectra(B, F, K, seed=7)
    tar[5] *= 30.0
    inp[5] *= 30.0
    frames = torch.randint(F // 2, F + 1, (B,), generator=g)
    frames[0] = F
    return inp, off, tar, frames


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(rank, world_size, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp, ops
    inp, off, tar, frames = _dp_data()
    lo, hi = dp.shard_bounds(7, rank, world_size)
    K = tar.shape[2]
    pad = lambda x: torch.nn.functional.pad(x[lo:hi], (0, ops.round4(K) - K), value=float("nan")).contiguous().cuda()
    energy, emax = ops.wsd_energy(pad(tar), K)
    local = emax.clone()
    dp.global_max(emax)
    step = lambda m: ops.wsd_mask_step(pad(off), pad(inp), pad(tar), frames[lo:hi].cuda(), 0, K, energy, m, ALPHA, DB, want_grad=False)
    _, terms, _, _ = step(emax)
    _, terms_local, _, _ = step(local)
    vec = dp.reduce_sums(torch.stack([terms.double().sum(), torch.tensor(float(hi - lo), dtype=torch.float64, device="cuda")]))
    # the fused training step on an even 4 / 4 split of 8 utterances: averaged head gradients
    from speech_enhancement_by_s3prl_b200 import synth
    lengths, wavs = synth.batch(8, 2.0, min_seconds=1.0)
    lengths, wavs = dp.shard_batch(lengths, wavs, rank, world_size)
    grads = _engine_grads(se, lengths.cuda(), wavs.cuda())
    ret[rank] = (terms.cpu(), terms_local.cpu(), (vec[0] / vec[1]).item(), emax.item(), local.item(), grads)
    dist.destroy_process_group()


def _engine_grads(se, lengths, wavs):
    pre = _pre(se, 512)
    torch.manual_seed(11)
    head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = se.WSD(alpha=ALPHA, db_interval=DB)
    assert eng.fused_training_supported(crit, wavs.shape[0], wavs.shape[2])
    eng.train_step(lengths, wavs, crit, torch.optim.SGD(head.parameters(), lr=0.0), None)
    torch.cuda.synchronize()
    return head.linear.weight.grad.cpu(), head.linear.bias.grad.cpu()


@gpu
@pytest.mark.timeout(600)
def test_two_ranks_threshold_against_the_global_batch_maximum(se):
    import torch.multiprocessing as mp
    from speech_enhancement_by_s3prl_b200 import ops, synth
    world_size = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dp_worker, args=(world_size, _free_port(), ret), nprocs=world_size, join=True)
    # single process, whole batch
    inp, off, tar, frames = _dp_data()
    K = tar.shape[2]
    energy, emax = ops.wsd_energy(tar.cuda(), K)
    _, terms_sp, _, _ = ops.wsd_mask_step(off.cuda(), inp.cuda(), tar.cuda(), frames.cuda(), 0, K, energy, emax, ALPHA, DB, want_grad=False)
    terms_sp = terms_sp.cpu()
    masks = (torch.arange(tar.shape[1])[None, :] < frames[:, None]).long()
    ref = sp.wsd(inp, off, tar, masks, alpha=ALPHA, db_interval=DB).item()
    for rank, (lo, hi) in enumerate([(0, 4), (4, 7)]):
        terms, terms_local, global_loss, gmax, local, _ = ret[rank]
        assert gmax == emax.item()
        np.testing.assert_allclose(terms.numpy(), terms_sp[lo:hi].numpy(), rtol=1e-5, atol=0)
        assert global_loss == pytest.approx(ref, rel=1e-5)
    # rank 0's own maximum is lower: thresholding against it (what the single-process kernels did per shard) gives another loss
    terms0, terms0_local, _, gmax, local0, _ = ret[0]
    assert local0 < gmax
    assert (terms0_local - terms_sp[0:4]).abs().max().item() > 10 * 1e-5 * terms_sp[0:4].abs().max().item()   # 10x the tolerance above
    # averaged gradients of the even split equal the single-process gradients of the whole batch
    lengths, wavs = synth.batch(8, 2.0, min_seconds=1.0)
    gw_sp, gb_sp = _engine_grads(se, lengths.cuda(), wavs.cuda())
    for rank in range(world_size):
        gw, gb = ret[rank][5]
        assert (gw - gw_sp).abs().max().item() < 1e-4 * gw_sp.abs().max().item()
        assert (gb - gb_sp).abs().max().item() < 1e-4 * gb_sp.abs().max().item()


# ------------------------------------------------------------------------------ the captured step's side-stream collective (NCCL)
def _nccl_worker(rank, world_size, port, ret):
    """A world-size-1 NCCL group standing in for N ranks: ``dp.world`` reports two ranks, so the fused WSD step forks its side
    stream, and ``dp.global_max`` issues a real NCCL all-reduce(MAX) there -- eagerly and inside the captured graph."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK="0", WORLD_SIZE="1")
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1)
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import dp, synth
    streams = []

    def global_max(t):
        streams.append(torch.cuda.current_stream().cuda_stream)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t

    dp.world, dp.global_max = (lambda: (0, 2)), global_max
    lengths, wavs = synth.batch(4, 1.0, min_seconds=0.6)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    pre = _pre(se, 512)
    finals = []
    for graph in (False, True):
        torch.manual_seed(5)
        head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        crit, opt = se.WSD(), se.ClipAdam(head.parameters(), lr=1e-3)
        w0 = head.linear.weight.detach().clone()
        del streams[:]
        for _ in range(5 if graph else 8):
            loss = eng.train_step_graph(lengths, wavs, crit, opt, 1.0) if graph else eng.train_step(lengths, wavs, crit, opt, 1.0)
        torch.cuda.synchronize()
        side = [s.cuda_stream for s in eng._side_streams.values()]
        finals.append((loss.item(), (head.linear.weight.detach() - w0).cpu(), opt.steps_taken(), len(streams),
                       all(s in side for s in streams)))
    ret[0] = finals
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_captured_wsd_step_all_reduces_the_maximum_on_a_side_stream(se):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_nccl_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    (l_e, dw_e, steps_e, n_e, side_e), (l_g, dw_g, steps_g, n_g, side_g) = ret[0]
    assert steps_e == steps_g == [8]
    assert n_e == 8 and side_e                       # one all-reduce per eager step, each on the engine's side stream
    assert n_g == 4 and side_g                       # three eager warm-ups + the capture (replays re-run the captured one)
    assert dw_e.abs().max().item() > 1e-3            # it trained
    assert l_g == pytest.approx(l_e, rel=1e-3)
    assert (dw_e - dw_g).abs().max().item() < 2e-3   # 8 Adam steps of lr 1e-3: updates of ~8e-3


# ------------------------------------------------------------------------------ CPU: launch planning
def test_wsd_fold_launch_planning_is_host_logic():
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    assert lib.se_linear_head_bwd_wsd_supported(48, 1001, 201, 201, 204, 204, 204, 204) == 1          # configs[2]
    assert lib.se_linear_head_bwd_wsd_supported(48, 1001, 120, 201, 120, 204, 204, 204) == 1          # mel 120 -> 201
    assert lib.se_linear_head_bwd_wsd_supported(48, 1001, 201, 201, 201, 204, 204, 204) == 0          # rows not 16-byte multiples
    assert lib.se_linear_head_bwd_wsd_supported(48, 1001, 201, 201, 204, 204, 204, 201) == 0
    assert lib.se_linear_head_bwd_wsd_supported(64, 16, 257, 257, 260, 260, 260, 260) == 0            # shorter than one 32-row block
