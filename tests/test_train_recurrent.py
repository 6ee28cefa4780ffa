"""The training step with recurrent heads (EnhancementEngine.train_step with model.LSTM + objective.L1 and model.Residual +
objective.SISDR / WSD): the fused route -- K1, the cuDNN body in torch autograd, the projection on the TMA head, the objective's step
kernel (se_l1_mask_step for L1), act'(z) in place, the weight gradient on the split-K TMA kernel, dH = dZ W on the TMA head with the
persistent W^T copy, cuDNN BPTT -- against the autograd route and a float64 oracle, ClipAdam over every parameter of the head, the
captured step and data parallelism.  The GPU tests run cuDNN without TF32, so that the body is the same fp32 computation on both
routes and the differences come from the TF32 projection alone."""
import os
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
GEOS = {512: (257, 32), 400: (201, 25), 1024: (513, 64)}


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


@pytest.fixture(autouse=True)
def _no_cudnn_tf32():
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        yield


def _pre(se, n_fft, hop, device="cuda"):
    n_freq, win_ms = GEOS[n_fft]
    pre = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop // 16, n_freq=n_freq).to(device)
    pre.channel_inp, pre.channel_tar = 0, 1
    return pre


def _head(se, kind, n_freq, hidden, layers, bidir=False, cmvn=False, activation=None, device="cuda"):
    torch.manual_seed(7)
    if kind == "LSTM":
        head = se.LSTM(input_size=n_freq, output_size=n_freq, hidden_size=hidden, num_layers=layers, bidirectional=bidir,
                       activation=activation or "Identity", precision=1)
    else:
        head = se.Residual(input_size=n_freq, output_size=n_freq, hidden_size=hidden, num_layers=layers, bidirectional=bidir,
                           cmvn=cmvn, activation=activation or "Sigmoid", precision=1)
    return head.to(device)


def _crit(se, name):
    return {"L1": se.L1(), "SISDR": se.SISDR(), "WSD": se.WSD(alpha=0.4, db_interval=30.0)}[name]


def _ragged(B, T, hop, seed):
    return synth(B, T, seed=seed, lengths=torch.LongTensor([T - (1777 * i) % (T // 2) - (hop // 3 if i else 0) for i in range(B)]))


def _grads_of_route(se, eng, head, lengths, wavs, crit, fused):
    eng.fused_training = fused
    assert eng.fused_training_supported(crit, wavs.shape[0], wavs.shape[2]) == fused
    loss = eng.train_step(lengths, wavs, crit, torch.optim.SGD(head.parameters(), lr=0.0), None)   # lr 0: gradients only
    torch.cuda.synchronize()
    return loss.item(), {n: p.grad.detach().clone() for n, p in head.named_parameters()}


def _both_routes(se, kind, crit_name, n_fft, hop, hidden, layers, bidir, cmvn, lengths, wavs):
    pre = _pre(se, n_fft, hop)
    head = _head(se, kind, GEOS[n_fft][0], hidden, layers, bidir, cmvn)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = _crit(se, crit_name)
    return [_grads_of_route(se, eng, head, lengths, wavs, crit, fused) for fused in (True, False)]


def _assert_grads_agree(got, ref, max_rel=4e-3, mean_rel=4e-4):
    for name, g_ref in ref.items():
        g = got[name]
        scale = g_ref.abs().max().item()
        assert scale > 0 and torch.isfinite(g).all(), name
        err = (g - g_ref).abs()
        assert err.max().item() < max_rel * scale, f"{name}: max error {err.max().item() / scale:.2e} of max|g|"
        assert err.mean().item() < mean_rel * scale, f"{name}: mean error {err.mean().item() / scale:.2e} of max|g|"


# ------------------------------------------------------------------------------ 1. fused route vs the autograd route
@gpu
@pytest.mark.parametrize("kind,crit,n_fft,hop,hidden,layers,bidir,cmvn", [
    ("LSTM", "L1", 512, 256, 64, 2, False, False),
    ("LSTM", "L1", 400, 160, 32, 3, True, False),
    ("LSTM", "L1", 1024, 256, 64, 2, False, False),
    ("LSTM", "L1", 512, 128, 48, 2, True, False),            # a geometry without register-resident kernels
    ("Residual", "SISDR", 512, 256, 64, 2, False, False),
    ("Residual", "SISDR", 400, 160, 32, 2, True, True),
    ("Residual", "WSD", 512, 256, 64, 3, False, True),
    ("Residual", "WSD", 1024, 256, 32, 2, False, False),
    ("Residual", "WSD", 512, 128, 64, 2, True, False),
])
def test_fused_recurrent_step_matches_autograd_route(se, kind, crit, n_fft, hop, hidden, layers, bidir, cmvn):
    T = 20000
    lengths, wavs = _ragged(5, T, hop, seed=n_fft + hop + hidden)
    (l_f, g_f), (l_a, g_a) = _both_routes(se, kind, crit, n_fft, hop, hidden, layers, bidir, cmvn, lengths.cuda(), wavs.cuda())
    assert np.isfinite(l_f) and l_f == pytest.approx(l_a, rel=2e-4)
    assert set(g_f) == set(g_a) and any(n.startswith("lstm.") for n in g_f)
    _assert_grads_agree(g_f, g_a)


# ------------------------------------------------------------------------------ 2. float64 oracle at a small size
def _oracle_grads(eng, lengths, wavs, crit_name, crit, monkeypatch):
    """oracle.signal_path.recurrent_head in float64 on float64 spectra, the oracle's objective, autograd: gradients per parameter
    name of the engine's head, and the loss."""
    head = eng.head
    kind = type(head).__name__
    n_fft, hop = eng.n_fft, eng.hop
    w = eng.pre._frame_window.double().cpu().numpy()
    x = wavs.double().numpy()
    X, C = stft_f64.stft(x[:, 0], n_fft, hop, w), stft_f64.stft(x[:, 1], n_fft, hop, w)
    linear_inp, linear_tar = torch.from_numpy(np.abs(X) ** 2), torch.from_numpy(np.abs(C) ** 2)
    feats = torch.log(linear_inp + eng.pre.eps)
    F = feats.shape[1]
    masks = (torch.arange(F)[None, :] < torch.clamp(lengths // hop + 1, max=F)[:, None]).double()
    state = {k: v.detach().double().cpu().clone().requires_grad_(k.startswith("scaling_layer"))
             for k, v in head.state_dict().items()}
    made = []

    class _Recorded(torch.nn.LSTM):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            made.append(self)

    monkeypatch.setattr(torch.nn, "LSTM", _Recorded)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        pred, extra = sp.recurrent_head(kind, state, feats, linear_inp, bidirectional=head.bidirectional, activation=head.activation,
                                        cmvn=getattr(head, "cmvn", False), eps=getattr(head, "eps", 1e-6))
        if crit_name == "L1":
            loss = sp.l1_logspectral(extra["log_predicted"], linear_tar, masks, eps=crit.eps)
        elif crit_name == "SISDR":
            loss, _ = sp.sisdr_spectral(pred, linear_tar, masks, eps=crit.eps)
        else:
            loss = sp.wsd(linear_inp, extra["offset"], linear_tar, masks, alpha=crit.alpha, db_interval=crit.db_interval, eps=crit.eps)
        loss.backward()
    finally:
        torch.set_default_dtype(prev)
        monkeypatch.undo()
    grads = {"lstm." + n: p.grad for n, p in made[0].named_parameters()}
    grads.update({k: v.grad for k, v in state.items() if k.startswith("scaling_layer")})
    return loss.item(), grads


@gpu
@pytest.mark.parametrize("kind,crit_name,bidir,cmvn", [("LSTM", "L1", False, False), ("LSTM", "L1", True, False),
                                                       ("Residual", "SISDR", False, True), ("Residual", "WSD", True, False)])
def test_fused_recurrent_step_matches_the_float64_oracle(se, monkeypatch, kind, crit_name, bidir, cmvn):
    n_fft, hop, T = 512, 256, 12000
    lengths, wavs = _ragged(3, T, hop, seed=17)
    pre = _pre(se, n_fft, hop)
    head = _head(se, kind, 257, 32, 2, bidir, cmvn)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    crit = _crit(se, crit_name)
    loss, got = _grads_of_route(se, eng, head, lengths.cuda(), wavs.cuda(), crit, True)
    loss64, ref = _oracle_grads(eng, lengths, wavs, crit_name, crit, monkeypatch)
    assert loss == pytest.approx(loss64, rel=1e-3)
    assert set(got) == set(ref)
    for name, g64 in ref.items():
        g = got[name].double().cpu().flatten()
        g64 = g64.flatten()
        cos = torch.dot(g, g64) / (g.norm() * g64.norm())
        assert cos.item() > 0.9999, f"{name}: cosine {cos.item():.6f}"
        assert (g - g64).abs().max().item() < 1e-2 * g64.abs().max().item(), name


# ------------------------------------------------------------------------------ 3. which kernels run
def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events()                    # kernels and copies, not the optimizer's record_function ranges
            if e.device_type == torch.autograd.DeviceType.CUDA and not getattr(e, "is_user_annotation", False)]


@gpu
def test_route_check_by_kernel_names(se):
    lengths, wavs = _ragged(4, 16000, 256, seed=3)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    # torch's Adam kernels on a recurrent head's parameters (the positive control of the check below)
    head = _head(se, "LSTM", 257, 64, 2)
    for p in head.parameters():
        p.grad = torch.ones_like(p)
    adam = torch.optim.Adam(head.parameters(), lr=1e-4)
    torch_adam = {n for n in _kernel_names(adam.step) if "multi_tensor_apply" in n or "Adam" in n}
    assert torch_adam
    for kind, crit_name in (("LSTM", "L1"), ("Residual", "WSD")):
        pre = _pre(se, 512, 256)
        head = _head(se, kind, 257, 64, 2)
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        crit, opt = _crit(se, crit_name), se.ClipAdam(head.parameters(), lr=1e-4)
        assert eng.fused_training_supported(crit, 4, 16000)
        names = _kernel_names(lambda: eng.train_step(lengths, wavs, crit, opt, 1.0))
        has = lambda s: any(s in n for n in names)
        assert has("linear_head_fused_kernel") and has("linear_head_bwd_tma_kernel"), (kind, names)
        assert has("adam_update_kernel") and has("act_grad_kernel") == (kind == "Residual")
        assert has("l1_mask_step_kernel") == (crit_name == "L1")
        assert not has("linear_head_tc_kernel") and not has("linear_head_bwd_tc_kernel"), (kind, names)
        assert not torch_adam & set(names), (kind, torch_adam & set(names))
        torch_named = [n for n in names if "Adam" in n and "AdamArgs" not in n]      # (ClipAdam's kernels take AdamArgs)
        assert not torch_named, (kind, torch_named)
    # pairs without a fused route keep the autograd route through the drop-in modules
    pre = _pre(se, 512, 256)
    for kind, crit_name in (("LSTM", "SISDR"), ("Residual", "L1")):
        head = _head(se, kind, 257, 64, 2)
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        crit = _crit(se, crit_name)
        assert not eng.fused_training_supported(crit, 4, 16000)
        if kind == "LSTM":
            names = _kernel_names(lambda: eng.train_step(lengths, wavs, crit, torch.optim.SGD(head.parameters(), lr=0.0), None))
            assert any("linear_head_tc_kernel" in n for n in names) and not any("linear_head_fused_kernel" in n for n in names)


# ------------------------------------------------------------------------------ 4. ClipAdam over the whole recurrent head
@gpu
@pytest.mark.parametrize("bidir,n_tensors", [(False, 14), (True, 26)])
def test_clip_adam_over_a_recurrent_head(se, bidir, n_tensors):
    from speech_enhancement_by_s3prl_b200 import ops
    pre = _pre(se, 512, 256)
    head_ref, head = _head(se, "LSTM", 257, 32, 3, bidir), _head(se, "LSTM", 257, 32, 3, bidir)
    params_ref, params = list(head_ref.parameters()), list(head.parameters())
    assert len(params) == n_tensors
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    eng._padded_weight_t()
    o_ref = torch.optim.Adam(params_ref, lr=3e-3, betas=(0.9, 0.98))
    opt = se.ClipAdam(params, lr=3e-3, betas=(0.9, 0.98))
    g = torch.Generator().manual_seed(9)
    proj = head.scaling_layer[0]
    K, H = proj.weight.shape

    def check_buffers():
        w = ops.round_tf32(proj.weight.detach())
        assert torch.equal(eng._wpad[:, :H], w) and (eng._wpad[:, H:] == 0).all()
        assert torch.equal(eng._wtpad[:, :K], w.t()) and (eng._wtpad[:, K:] == 0).all()

    for it in range(5):
        grads = [torch.randn(p.shape, generator=g).cuda() * (0.1 + it) for p in params]
        for p, q, gr in zip(params_ref, params, grads):
            p.grad, q.grad = gr.clone(), gr.clone()
        torch.nn.utils.clip_grad_norm_(params_ref, 1.0)
        o_ref.step()
        eng._clip_and_step(opt, 1.0)
        for p, q in zip(params_ref, params):
            assert (p - q).abs().max().item() < 2e-6
        check_buffers()
    assert opt.steps_taken() == [5] and opt.steps_skipped() == [0]
    before = [p.detach().clone() for p in params]
    for q in params:
        q.grad = torch.randn(q.shape, generator=g).cuda()
    params[5].grad[0] = float("nan")
    eng._clip_and_step(opt, 1.0)
    assert opt.steps_taken() == [5] and opt.steps_skipped() == [1]
    assert all(torch.equal(p, b) for p, b in zip(params, before))
    check_buffers()


# ------------------------------------------------------------------------------ 5. the captured step
@gpu
@pytest.mark.parametrize("kind,crit_name", [("LSTM", "L1"), ("Residual", "WSD")])
def test_captured_recurrent_step_follows_eager_fused_steps(se, kind, crit_name):
    lengths, wavs = _ragged(4, 16000, 256, seed=31)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    pre = _pre(se, 512, 256)
    finals = []
    for graph in (False, True):
        head = _head(se, kind, 257, 64, 2)
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
        crit, opt = _crit(se, crit_name), se.ClipAdam(head.parameters(), lr=1e-3)
        assert eng.fused_training_supported(crit, 4, 16000)
        p0 = [p.detach().clone() for p in head.parameters()]
        for _ in range(5 if graph else 8):              # graph: 3 eager warm-ups inside capture_train + 5 replays
            loss = eng.train_step_graph(lengths, wavs, crit, opt, 1.0) if graph else eng.train_step(lengths, wavs, crit, opt, 1.0)
        torch.cuda.synchronize()
        assert opt.steps_taken() == [8]
        finals.append((loss.item(), [p.detach().clone() for p in head.parameters()], p0, eng, head))
    (l_e, p_e, p0, _, _), (l_g, p_g, _, eng, head) = finals
    assert max((a - b).abs().max().item() for a, b in zip(p_e, p0)) > 1e-3            # it trained
    assert l_g == pytest.approx(l_e, rel=1e-3)
    for a, b in zip(p_e, p_g):
        assert (a - b).abs().max().item() < 2e-3                                       # 8 Adam steps of lr 1e-3
    # the evaluation step that follows reads the trained projection: the same mask as an engine with fresh weight buffers
    out = eng.eval_step(lengths, wavs, criterion=_crit(se, crit_name))
    fresh = se.EnhancementEngine(pre, head, log_features=True, precision=1).eval_step(lengths, wavs, criterion=_crit(se, crit_name))
    torch.cuda.synchronize()
    assert torch.equal(out["mask"], fresh["mask"])


# ------------------------------------------------------------------------------ 6. two gloo ranks on uneven shards
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
    from speech_enhancement_by_s3prl_b200 import dp
    lengths, wavs = _ragged(5, 16000, 256, seed=23)
    lengths, wavs = dp.shard_batch(lengths, wavs, rank, world_size)                  # 3 / 2 utterances
    out = {}
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        for kind, crit_name in (("LSTM", "L1"), ("Residual", "WSD")):
            out[kind] = _both_routes(se, kind, crit_name, 512, 256, 32, 2, False, kind == "Residual", lengths.cuda(), wavs.cuda())
    ret[rank] = {k: [(l, {n: g.cpu() for n, g in gr.items()}) for l, gr in v] for k, v in out.items()}
    dist.destroy_process_group()


@gpu
@pytest.mark.timeout(600)
def test_two_ranks_on_uneven_shards(se):
    import torch.multiprocessing as mp
    world_size = 2
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(world_size, _free_port(), ret), nprocs=world_size, join=True)
    for rank in range(world_size):
        for kind in ("LSTM", "Residual"):
            (l_f, g_f), (l_a, g_a) = ret[rank][kind]
            assert l_f == pytest.approx(l_a, rel=2e-4), (rank, kind)                  # each rank's own loss (local mean)
            _assert_grads_agree(g_f, g_a)
    for kind in ("LSTM", "Residual"):                                                  # all-reduced: the same on both ranks
        for name, g in ret[0][kind][0][1].items():
            assert torch.equal(g, ret[1][kind][0][1][name]), (kind, name)
        assert ret[0][kind][0][0] != ret[1][kind][0][0]                                # the local losses differ


# ------------------------------------------------------------------------------ CPU
def test_clip_adam_refuses_a_group_of_33_tensors():
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import optim
    assert optim._MAX_TENSORS == 32
    params = [torch.nn.Parameter(torch.zeros(2)) for _ in range(33)]
    for p in params:
        p.grad = torch.ones(2)
    with pytest.raises(RuntimeError, match="at most 32 tensors"):
        se.ClipAdam(params).clip_and_step(1.0)


def test_fused_training_supported_table():
    """Which (head, objective, precision, switch) pairs take the fused training route; host logic only."""
    import speech_enhancement_by_s3prl_b200 as se
    pre = _pre(se, 512, 256, device="cpu")
    B, T = 4, 16000

    def supported(head, crit, precision=1, fused=True, feat_cfg=None):
        eng = se.EnhancementEngine(pre, head, log_features=True, precision=precision, feat_cfg=feat_cfg)
        eng.fused_training = fused
        return eng.fused_training_supported(crit, B, T)

    L1, SISDR, WSD = se.L1(), se.SISDR(), se.WSD()
    lstm = _head(se, "LSTM", 257, 64, 3, device="cpu")
    bilstm = _head(se, "LSTM", 257, 64, 3, bidir=True, device="cpu")
    res = _head(se, "Residual", 257, 64, 2, device="cpu")
    res_cmvn = _head(se, "Residual", 257, 64, 2, cmvn=True, device="cpu")
    assert supported(lstm, L1) and supported(bilstm, L1)
    assert supported(res, SISDR) and supported(res, WSD) and supported(res_cmvn, SISDR) and supported(res_cmvn, WSD)
    assert not supported(lstm, SISDR) and not supported(lstm, WSD) and not supported(lstm, None)
    assert not supported(res, L1)
    assert not supported(lstm, L1, precision=0) and not supported(res, WSD, precision=0)
    assert not supported(lstm, L1, fused=False) and not supported(res, SISDR, fused=False)
    assert not supported(_head(se, "LSTM", 257, 30, 2, device="cpu"), L1)              # hidden width not a multiple of 4
    assert not supported(_head(se, "LSTM", 257, 33, 2, bidir=True, device="cpu"), L1)  # 66
    assert supported(_head(se, "LSTM", 257, 34, 2, bidir=True, device="cpu"), L1)      # 68
    assert not supported(_head(se, "LSTM", 200, 64, 2, device="cpu"), L1)              # input width is not the feature's
    assert not supported(se.Linear(input_size=257, output_size=257, precision=1), SISDR)
    assert supported(se.LinearResidual(input_size=257, output_size=257, precision=1), SISDR)
    # the environment switch
    old = os.environ.get("SE_B200_FUSED_TRAIN")
    os.environ["SE_B200_FUSED_TRAIN"] = "0"
    try:
        assert not se.EnhancementEngine(pre, lstm, log_features=True, precision=1).fused_training_supported(L1, B, T)
    finally:
        if old is None:
            del os.environ["SE_B200_FUSED_TRAIN"]
        else:
            os.environ["SE_B200_FUSED_TRAIN"] = old
