"""GPU (-m gpu): the CUDA path, called through the C ABI (ctypes) and through the drop-in
classes, against the CPU oracle on the same seeded inputs and against the golden fixtures.

Tolerances (BASELINE.json north_star): spectra within 1e-4 relative in fp32; reconstructed
waveforms within 0.01 dB SI-SDR.  "Relative" for a power spectrum is taken against the
largest bin of the utterance (bins 120 dB below it hold rounding noise in the oracle too).
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import signal_path as sp
from oracle.preprocessor import OnlinePreprocessor as OraclePre

pytestmark = pytest.mark.gpu

SPEC_RTOL = 1e-4
SISDR_TOL_DB = 0.01
CFGS = {256: (129, 16, 8), 400: (201, 25, 10), 512: (257, 32, 16), 1024: (513, 64, 16), 2048: (1025, 128, 32)}


@pytest.fixture(scope="module")
def se():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import speech_enhancement_by_s3prl_b200 as pkg
    return pkg


def make_pair(se, n_fft):
    n_freq, win_ms, hop_ms = CFGS[n_fft]
    ora = OraclePre(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq)
    mine = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).cuda()
    for p in (ora, mine):
        p.channel_inp, p.channel_tar = 0, 1
    return ora, mine


def synth(B, T, seed, lengths=None):
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(T) / 16000.0
    clean = torch.zeros(B, T)
    for b in range(B):
        f0 = 100 + 40 * b
        for h in range(1, 6):
            clean[b] += torch.sin(2 * np.pi * f0 * h * t + h) / h
        clean[b] *= 0.02 * (1 + 0.5 * torch.sin(2 * np.pi * 2.5 * t))
    noise = torch.randn(B, T, generator=g) * 0.01
    wavs = torch.stack([clean + noise, clean, noise], 1).contiguous()
    if lengths is None:
        lengths = torch.full((B,), T, dtype=torch.int64)
    for b, n in enumerate(lengths.tolist()):
        wavs[b, :, n:] = 0                                   # collate_fn zero-pads (dataset.py:175)
    return lengths, wavs


def rel_to_max(a, b):
    a, b = a.double(), b.double()
    scale = b.abs().amax(dim=(-1, -2), keepdim=True)
    return ((a - b).abs() / scale).max().item()


def sisdr_db(a, b):
    return sp.sisdr_eval(a, b)


# ------------------------------------------------------------------------------ STFT
ORACLE_STFT = [(512, 16000, 16), (512, 16001, 16), (512, 300, 16), (512, 4096, 16), (400, 16000, 10), (400, 7777, 10),
               (1024, 20000, 16), (256, 3000, 8), (2048, 30000, 32), (512, 16000, 10), (512, 9999, 8)]


@pytest.mark.parametrize("n_fft,T,hop_ms", ORACLE_STFT,
                         ids=[f"{n}-{t}" + ("" if h == CFGS[n][2] else f"-hop{h}") for n, t, h in ORACLE_STFT])
def test_stft_matches_oracle(se, n_fft, T, hop_ms):
    """Every n_fft against the oracle; n_fft 512 also at hops (160, 128) that have no register-resident kernel."""
    n_freq, win_ms, _ = CFGS[n_fft]
    ora = OraclePre(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq)
    mine = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).cuda()
    _, wavs = synth(3, T, seed=T)
    c = ora.get_feat_config
    cfgs = [c("linear", 0), c("phase", 0), c("linear", 1, log=True), c("linear", 2)]
    ref = ora(wavs, cfgs)
    got = [g.cpu() for g in mine(wavs.cuda(), cfgs)]
    hop = ora._win_args["hop_length"]
    assert got[0].shape == ref[0].shape == (3, T // hop + 1, n_fft // 2 + 1)
    assert rel_to_max(got[0], ref[0]) < SPEC_RTOL
    assert rel_to_max(got[3], ref[3]) < SPEC_RTOL
    strong = ref[0] > 1e-5 * ref[0].amax()
    dphi = torch.angle(torch.polar(torch.ones_like(ref[1]), got[1] - ref[1]))
    assert dphi[strong].abs().max() < 2e-3
    big = ref[2] > ref[2].max() + np.log(1e-6)                # log amplifies the rounding noise of empty bins
    assert (got[2] - ref[2])[big].abs().max() < 1e-2
    assert torch.isfinite(got[2]).all()


def test_stft_through_raw_c_abi(se):
    """ctypes straight into libse_b200.so, no Python wrapper classes in between."""
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    ora, _ = make_pair(se, 512)
    _, wavs = synth(2, 5000, seed=9)
    d = wavs.cuda()
    win = torch.hann_window(512).cuda()
    power = torch.empty(2, 5000 // 256 + 1, 257, device="cuda")
    rc = lib.se_stft(d.data_ptr() + 4 * 5000, 2, 3 * 5000, 5000, 512, 256, win.data_ptr(), 1e-10, power.data_ptr(), None, None,
                     torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    ref = ora(wavs, [ora.get_feat_config("linear", 1)])[0]
    assert rel_to_max(power.cpu(), ref) < SPEC_RTOL


def test_abi_error_codes_on_device(se):
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    x = torch.zeros(1, 1, 200, device="cuda")
    with pytest.raises(RuntimeError, match="reflect"):
        ops.stft(x, 0, 512, 256, torch.hann_window(512).cuda())         # T <= n_fft/2, as torch.stft refuses
    with pytest.raises(RuntimeError, match="n_fft"):
        ops.stft(torch.zeros(1, 1, 2000, device="cuda"), 0, 384, 128, torch.hann_window(384).cuda())
    # entry points of the training / sampling rows: integer codes through the raw C ABI, text through se_last_error
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(4096, device="cuda")
    dbl = torch.zeros(64, device="cuda", dtype=torch.float64)
    p = buf.data_ptr()
    assert lib.se_sisdr_mask_fwd(None, 0, p, 3, p, 8, None, 1, 4, 8, 1e-10, dbl.data_ptr(), None, st) == -1   # ld_inp < K
    assert "stride" in _lib.last_error()
    assert lib.se_sisdr_mask_bwd(None, 0, p, 8, p, 8, None, 1, 4, 8, 1e-10, dbl.data_ptr(), None, p, 8, st) == -1   # grad_out null
    assert lib.se_head_grad_embeddings_workspace(2, 16, 257, 257) == 0                    # fewer than 32 frames per utterance
    assert lib.se_linear_head_bwd_tc_workspace(2, 64, 300, 257) == 0                       # D_in beyond the B tile
    rc = lib.se_head_grad_embeddings(p, 257, None, None, None, 257, 1e-6, p, p, 257, 2, 16, 257, 257, 2, p, 4096, p, st)
    assert rc == -2 and "range" in _lib.last_error()                                      # SE_ERR_UNSUPPORTED
    ptrs = (ctypes.c_void_p * 9)(*([p] * 9))
    sizes = (ctypes.c_int64 * 9)(*([4] * 9))
    ints = torch.zeros(2, device="cuda", dtype=torch.int32)
    for n in (0, 9):
        assert lib.se_adam_clip_step(ptrs, ptrs, ptrs, ptrs, sizes, n, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, dbl.data_ptr(),
                                     ints.data_ptr(), st) == -1
    assert lib.se_match_scores(p, 0, p, 1, 8, 1e-12, dbl.data_ptr(), p, p, st) == -1
    noisy, out = torch.randn(2000, device="cuda"), torch.empty(2000, device="cuda")
    power, win = torch.rand(8, 257, device="cuda"), torch.hann_window(512, device="cuda")
    assert lib.se_mask_istft_ex(noisy.data_ptr(), None, 2000, power.data_ptr(), 257, None, 1, 2000, 512, 256, win.data_ptr(),
                                out.data_ptr(), 2000, 2000, None, 4, st) == 0                # SE_FLAG_MASK_IS_POWER runs
    assert torch.isfinite(out).all()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------ iSTFT
@pytest.mark.parametrize("n_fft,T", [(512, 16000), (512, 16100), (400, 16000), (400, 7777), (1024, 20000)])
def test_istft_matches_oracle(se, n_fft, T):
    ora, mine = make_pair(se, n_fft)
    _, wavs = synth(2, T, seed=T + 1)
    c = ora.get_feat_config
    lin, ph = ora(wavs, [c("linear", 0), c("phase", 0)])
    g = torch.Generator().manual_seed(1)
    lin = lin * torch.rand(lin.shape, generator=g)
    ref = ora.istft(lin, ph)
    got = mine.istft(lin.cuda(), ph.cuda()).cpu()
    assert got.shape == ref.shape
    assert (got - ref).abs().max() < 5e-6 * max(1.0, ref.abs().max().item() / 0.05)
    for b in range(2):
        assert sisdr_db(got[b], ref[b]) > 90.0


def test_stft_istft_round_trip_full_size(se):
    """Config-2 size (64 x 4 s): size-independent property, no oracle needed."""
    _, mine = make_pair(se, 512)
    _, wavs = synth(64, 64000, seed=5)
    d = wavs.cuda()
    c = mine.get_feat_config
    lin, ph = mine(d, [c("linear", 0), c("phase", 0)])
    back = mine.istft(lin, ph)
    assert back.shape == (64, 64000)
    assert (back - d[:, 0, :64000]).abs().max().item() < 5e-6
    # linearity of the analysis: STFT power of 2x is 4x
    lin2 = mine(d * 2, [c("linear", 0)])[0]
    assert rel_to_max(lin2.cpu(), 4 * lin.cpu()) < 1e-6


# ------------------------------------------------------------------------------ fused mask -> iSTFT
@pytest.mark.parametrize("n_fft,T", [(512, 16000), (512, 9999), (400, 16000), (1024, 20000)])
def test_mask_istft_matches_unfused_oracle(se, n_fft, T):
    from speech_enhancement_by_s3prl_b200 import ops
    ora, mine = make_pair(se, n_fft)
    B = 4
    lengths = torch.LongTensor([T, T - 1234, T // 2 + 7, T // 3])
    lengths, wavs = synth(B, T, seed=T + 2, lengths=lengths)
    hop = ora._win_args["hop_length"]
    K, F = n_fft // 2 + 1, T // hop + 1
    g = torch.Generator().manual_seed(3)
    mask = torch.rand(B, F, K, generator=g)
    c = ora.get_feat_config
    lin, ph, lin_t = ora(wavs, [c("linear", 0), c("phase", 0), c("linear", 1)])
    ref = ora.istft(lin * mask, ph)
    ref = torch.cat([ref, ref.new_zeros(B, T - ref.shape[1])], 1)
    wav, sums = ops.mask_istft(wavs.cuda(), 0, 1, mask.cuda(), lengths.cuda(), n_fft, hop, mine._frame_window, pad_to=T)
    wav, sums = wav.cpu(), sums.cpu()
    assert (wav - ref).abs().max() < 5e-6
    masks = sp.length_masks(sp.stft_lengths(lengths, hop))
    _, per_utt = sp.sisdr_spectral(lin * mask, lin_t, masks)
    gain, sisdr, loss = ops.finalize_metrics(sums.cuda(), lengths.cuda(), T, wav=None)
    np.testing.assert_allclose(loss.cpu().numpy(), per_utt.numpy(), atol=2e-3)
    for b in range(B):
        n = int(lengths[b])
        assert sisdr[b].item() == pytest.approx(sisdr_db(ref[b, :n], wavs[b, 1, :n]), abs=SISDR_TOL_DB)


# ------------------------------------------------------------------------------ objectives
def test_objectives_match_reference_golden(se, golden_dir):
    g = np.load(os.path.join(golden_dir, "signal_path_ref.npz"))
    T_ = lambda k: torch.from_numpy(g[k]).cuda()
    masks = T_("masks")
    pred = T_("predicted").requires_grad_(True)
    loss, _ = se.SISDR()(predicted=pred, linear_tar=T_("linear_tar"), stft_length_masks=masks, junk=1)
    assert loss.item() == pytest.approx(float(g["SISDR"]), abs=1e-4)
    loss.backward()
    np.testing.assert_allclose(pred.grad.cpu().numpy(), g["SISDR_grad"], rtol=2e-4, atol=1e-7)
    lp = T_("log_predicted").requires_grad_(True)
    l1, _ = se.L1()(log_predicted=lp, linear_tar=T_("linear_tar"), stft_length_masks=masks, loss=None)
    assert l1.item() == pytest.approx(float(g["L1"]), rel=1e-5)
    l1.backward()
    np.testing.assert_allclose(lp.grad.cpu().numpy(), g["L1_grad"], rtol=1e-5, atol=1e-9)
    w, _ = se.WSD(alpha=0.3, db_interval=50)(T_("linear_inp"), T_("offset"), T_("linear_tar"), masks)
    assert w.item() == pytest.approx(float(g["WSD"]), rel=1e-5)


def test_objectives_match_oracle_at_scale(se):
    g = torch.Generator().manual_seed(11)
    B, F, K = 6, 251, 257
    pred = (torch.randn(B, F, K, generator=g) + 0.3).abs() * torch.rand(B, F, K, generator=g)
    pred[0, :5] = -1.0                                     # relu branch
    tar = torch.rand(B, F, K, generator=g) * 2
    frames = torch.LongTensor([251, 200, 1, 77, 251, 130])
    masks = sp.length_masks(frames)
    masks = torch.cat([masks, masks.new_zeros(B, F - masks.shape[1])], 1)
    p_ref = pred.clone().requires_grad_(True)
    ref, _ = sp.sisdr_spectral(p_ref, tar, masks)
    ref.backward()
    p = pred.cuda().requires_grad_(True)
    loss, _ = se.SISDR()(predicted=p, linear_tar=tar.cuda(), stft_lengths=frames.cuda())
    loss.backward()
    assert loss.item() == pytest.approx(ref.item(), abs=1e-4)
    np.testing.assert_allclose(p.grad.cpu().numpy(), p_ref.grad.numpy(), rtol=1e-3, atol=1e-8)
    assert (p.grad[0, :5] == 0).all() and torch.isfinite(p.grad).all()
    lp_ref = torch.randn(B, F, K, generator=g).requires_grad_(True)
    r1 = sp.l1_logspectral(lp_ref, tar, masks)
    r1.backward()
    lp = lp_ref.detach().cuda().requires_grad_(True)
    l1, _ = se.L1()(log_predicted=lp, linear_tar=tar.cuda(), stft_length_masks=masks.cuda())
    l1.backward()
    assert l1.item() == pytest.approx(r1.item(), rel=1e-5)
    np.testing.assert_allclose(lp.grad.cpu().numpy(), lp_ref.grad.numpy(), rtol=1e-5, atol=1e-10)


# ------------------------------------------------------------------------------ waveform helpers
def test_waveform_helpers_match_reference_golden(se, golden_dir):
    g = np.load(os.path.join(golden_dir, "signal_path_ref.npz"))
    T_ = lambda k: torch.from_numpy(g[k])
    assert se.sisdr_eval(T_("ev_src"), T_("ev_tar")) == pytest.approx(float(g["sisdr_eval"]), abs=1e-3)
    assert se.sisdr_eval(T_("ev_src").cuda(), T_("ev_src").cuda()) == pytest.approx(float(g["sisdr_eval_self"]), abs=0.5)
    lengths = T_("nd_len").cuda()
    masks = se.get_length_masks(lengths)
    assert masks.dtype == torch.int64 and masks.shape == (3, 50)
    np.testing.assert_array_equal(masks.cpu().numpy(), sp.length_masks(T_("nd_len")).numpy())
    a, r = T_("nd_audio").cuda(), T_("nd_ref").cuda()
    np.testing.assert_allclose(se.masked_normalize_decibel(a, -25, masks).cpu().numpy(), g["nd_scalar"], rtol=2e-5)
    np.testing.assert_allclose(se.masked_normalize_decibel(a, r, masks).cpu().numpy(), g["nd_tensor"], rtol=2e-5)
    np.testing.assert_allclose(se.masked_normalize_decibel(a, r, lengths).cpu().numpy(), g["nd_tensor"], rtol=2e-5)
    np.testing.assert_array_equal(se.get_length_masks(T_("stft_len").cuda()).cpu().numpy(), g["masks"])


# ------------------------------------------------------------------------------ heads
def test_heads_match_reference_golden(se, golden_dir):
    g = np.load(os.path.join(golden_dir, "signal_path_ref.npz"))
    T_ = lambda k: torch.from_numpy(g[k]).cuda()
    head = se.LinearResidual(input_size=9, output_size=9).cuda()
    head.load_state_dict({"linear.weight": T_("lr_weight"), "linear.bias": T_("lr_bias")})
    pred, res = head(features=T_("lr_feats"), linears=T_("lr_linears"))
    np.testing.assert_allclose(pred.detach().cpu().numpy(), g["lr_predicted"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(res["offset"].detach().cpu().numpy(), g["lr_offset"], rtol=1e-4, atol=1e-6)
    lin = se.Linear(9, 9, activation="ReLU").cuda()
    lin.load_state_dict({"linear.weight": T_("li_weight"), "linear.bias": T_("li_bias")})
    np.testing.assert_allclose(lin(features=T_("lr_feats"))[0].detach().cpu().numpy(), g["li_predicted"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("D,act,cmvn", [(257, "Sigmoid", True), (201, "ReLU", False), (513, "Sigmoid", True), (120, "Identity", True)])
def test_head_forward_backward_match_torch_fp32(se, D, act, cmvn):
    g = torch.Generator().manual_seed(D)
    B, F, K = 3, 101, (D if D != 120 else 201)
    feats = torch.randn(B, F, D, generator=g) * 2 - 3
    linears = torch.rand(B, F, K, generator=g)
    torch.manual_seed(1)
    head = se.LinearResidual(input_size=D, output_size=K, activation=act, cmvn=cmvn).cuda()
    w = head.linear.weight.detach().cpu().clone().requires_grad_(True)
    b = head.linear.bias.detach().cpu().clone().requires_grad_(True)
    ref_pred, ref_off = sp.linear_residual_head(feats, linears, w, b, activation=act, cmvn=cmvn)
    upstream = torch.randn(B, F, K, generator=g)
    (ref_pred * upstream).sum().backward()
    pred, res = head(features=feats.cuda(), linears=linears.cuda())
    (pred * upstream.cuda()).sum().backward()
    np.testing.assert_allclose(res["offset"].detach().cpu().numpy(), ref_off.detach().numpy(), rtol=1e-4, atol=2e-6)
    np.testing.assert_allclose(pred.detach().cpu().numpy(), ref_pred.detach().numpy(), rtol=1e-4, atol=2e-6)
    scale = w.grad.abs().max().item()
    np.testing.assert_allclose(head.linear.weight.grad.cpu().numpy(), w.grad.numpy(), rtol=1e-3, atol=1e-4 * scale)
    np.testing.assert_allclose(head.linear.bias.grad.cpu().numpy(), b.grad.numpy(), rtol=1e-3, atol=1e-4 * b.grad.abs().max().item())


# ------------------------------------------------------------------------------ features (K1b)
def _floor_mask(ref_feat, base, order, floor_nats=16.0):
    """Elements of a log feature (B, F, (order+1) * base) whose value -- and, for the delta columns, every one of the five
    taps (and the taps of those taps) it is made of -- lies within `floor_nats` (16 nats = 70 dB) of the largest value."""
    logs = ref_feat[..., :base]
    ok = logs > logs.amax() - floor_nats
    cols = [ok]
    for _ in range(order):
        prev = cols[-1].float()
        pad = torch.nn.functional.pad(prev.transpose(1, 2), (2, 2), mode="replicate")
        cols.append((torch.nn.functional.avg_pool1d(pad, 5, stride=1).transpose(1, 2) > 0.999))
    return torch.cat(cols, dim=-1)


@pytest.mark.parametrize("n_fft", [400, 512, 1024])
def test_mel_delta_cmvn_features_match_oracle(se, n_fft):
    """Feature configs of pretrain_sample.yaml:54-65 / pseudo_noise.yaml:10-15 through the fused K1b kernel (mel -> log ->
    deltas -> CMVN sums in one launch) and the generic log / delta / CMVN kernels: MAXIMUM error against the oracle over all
    elements above a stated floor (70 dB below the largest value: below it the logarithm of a near-cancelled bin is
    rounding noise in the oracle as well); the floor must leave > 99 % of the elements in."""
    ora, mine = make_pair(se, n_fft)
    _, wavs = synth(3, 12000, seed=21)
    c = ora.get_feat_config
    # log / CMVN features on the channels that have a noise floor (0 = noisy, 2 = noise)
    cfgs = [c("mel", 0, log=True, delta=2), c("mel", 2, log=True, delta=1, cmvn=True), c("linear", 0, log=True, delta=1),
            c("linear", 2, log=True, cmvn=True), c("mel", 1), c("mel", 0, log=True), c("mel", 2, delta=1)]
    ref = ora(wavs, cfgs)
    got = [g.cpu() for g in mine(wavs.cuda(), cfgs)]
    K = n_fft // 2 + 1
    assert got[0].shape[-1] == 120 and got[1].shape[-1] == 80 and got[2].shape[-1] == 2 * K
    for r, g_ in zip(ref, got):
        assert r.shape == g_.shape
    # (feature, base width, delta order, max abs error): log-mel sums 5-40 positive bins, log-linear is one bin
    for idx, base, order, tol in ((0, 40, 2, 5e-4), (5, 40, 0, 5e-4), (2, K, 1, 2e-3)):
        mask = _floor_mask(ref[idx], base, order)
        assert mask.float().mean().item() > 0.99
        assert (got[idx] - ref[idx]).abs()[mask].max().item() < tol
    # CMVN over time (unbiased std + eps): the normalised values are O(1); mask from the un-normalised log feature
    un = ora(wavs, [c("mel", 2, log=True, delta=1), c("linear", 2, log=True)])
    for idx, base, order, src, tol in ((1, 40, 1, un[0], 2e-3), (3, K, 0, un[1], 5e-3)):
        mask = _floor_mask(src, base, order)
        assert mask.float().mean().item() > 0.99
        assert (got[idx] - ref[idx]).abs()[mask].max().item() < tol
        assert got[idx].mean(1).abs().max().item() < 1e-3                    # zero mean over time per (utterance, column)
    assert rel_to_max(got[4], ref[4]) < SPEC_RTOL                             # mel energies (no log): relative to the largest band
    assert rel_to_max(got[6], ref[6]) < SPEC_RTOL


def test_no_wav_call_and_cpu_inputs(se):
    """run_downstream.py:163 (no-argument call) and runner.py:50-51 (CPU copy fed CPU audio)."""
    _, mine = make_pair(se, 400)
    c = mine.get_feat_config
    outs = mine(feat_list=[c("mel", 0, log=True, delta=1, cmvn=True), c("linear", 1)])
    assert outs[0].shape == (1, 101, 80) and outs[1].shape == (1, 101, 201)
    import copy
    cpu_pre = copy.deepcopy(mine).cpu()
    out = cpu_pre(torch.randn(1, 1, 4000) * 0.1, [c("linear", 0, log=True)])[0]
    assert out.device.type == "cpu" and out.shape == (1, 26, 201)


# ------------------------------------------------------------------------------ whole step
def _load_runner_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "runner_evaluate_ref.npz"))
    items = [torch.from_numpy(g[f"item{i}"]) for i in range(len(g["lengths"]))]
    return g, items


@pytest.mark.parametrize("use_graph", [False, True])
def test_eval_step_matches_reference_runner_evaluate(se, golden_dir, use_graph):
    """Fused engine vs the loss / SI-SDR the reference's own Runner.evaluate() produced."""
    g, items = _load_runner_golden(golden_dir)
    _, mine = make_pair(se, 512)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    head.load_state_dict({"linear.weight": torch.from_numpy(g["weight"]), "linear.bias": torch.from_numpy(g["bias"])})
    eng = se.EnhancementEngine(mine, head, log_features=True)
    losses, scores = [], []
    for i in range(0, len(items), 2):
        lengths, wavs = sp.collate(items[i:i + 2])
        if use_graph:
            out = eng.eval_step_graph(lengths.cuda(), wavs.cuda())
        else:
            out = eng.eval_step(lengths.cuda(), wavs.cuda())
        losses.append(out["loss_per_utt"].mean().item())
        scores.append(out["sisdr"].mean().item())
        if i == 0:
            enh = out["wav_predicted"][0].cpu()
            ref = torch.from_numpy(g["enhanced0"])
            assert sisdr_db(enh[:len(ref)], ref) > 60.0
            np.testing.assert_allclose(enh[:len(ref)].numpy(), g["enhanced0"], atol=2e-5)
    assert np.mean(losses) == pytest.approx(float(g["loss"]), abs=2e-3)
    assert np.mean(scores) == pytest.approx(float(g["scores"][0]), abs=SISDR_TOL_DB)


def test_eval_step_matches_oracle_ragged_batch(se):
    ora, mine = make_pair(se, 512)
    B, T = 5, 24000
    lengths = torch.LongTensor([24000, 20011, 16000, 9000, 5120])
    lengths, wavs = synth(B, T, seed=77, lengths=lengths)
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    c = ora.get_feat_config
    ora.feat_list = [c("linear", 0, log=True), c("linear", 0, log=True), c("linear", 0), c("phase", 0), c("linear", 1), c("phase", 1)]
    ref = sp.eval_step(ora, dict(weight=head.linear.weight.detach().cpu(), bias=head.linear.bias.detach().cpu()), lengths, wavs)
    out = se.EnhancementEngine(mine, head).eval_step(lengths.cuda(), wavs.cuda())
    np.testing.assert_allclose(out["sisdr"].cpu().numpy(), ref["sisdr"].numpy(), atol=SISDR_TOL_DB)
    assert out["loss_per_utt"].mean().item() == pytest.approx(ref["loss"].item(), abs=2e-3)
    for b in range(B):
        n = int(lengths[b])
        assert sisdr_db(out["wav_predicted"][b, :n].cpu(), ref["wav_predicted"][b, :n]) > 50.0


def test_dropin_call_sequence_matches_oracle(se):
    """The reference's own call sequence (runner.py:556-575) on the drop-in classes."""
    ora, mine = make_pair(se, 400)
    B, T = 3, 16000
    lengths = torch.LongTensor([16000, 12345, 8000])
    lengths, wavs = synth(B, T, seed=5, lengths=lengths)
    c = ora.get_feat_config
    fl = [c("mel", 0, log=True, delta=1, cmvn=True), c("linear", 0, log=True), c("linear", 0), c("phase", 0), c("linear", 1), c("phase", 1)]
    ora.feat_list = fl
    mine.feat_list = fl
    torch.manual_seed(3)
    head = se.LinearResidual(input_size=201, output_size=201).cuda()
    hw = dict(weight=head.linear.weight.detach().cpu(), bias=head.linear.bias.detach().cpu())
    ref = sp.eval_step(ora, hw, lengths, wavs)
    d_wavs, d_len = wavs.cuda(), lengths.cuda()
    with torch.no_grad():
        feats_up, feats_down, linear_inp, phase_inp, linear_tar, phase_tar = mine(d_wavs)
        predicted, model_results = head(features=feats_down, linears=linear_inp)
        wav_predicted = se.decode_wav(mine, predicted, phase_inp, d_len, d_wavs[:, mine.channel_tar, :])
        stft_len = d_len // mine._win_args["hop_length"] + 1
        masks = se.get_length_masks(stft_len)
        loss, _ = se.SISDR()(**dict(predicted=predicted, linear_tar=linear_tar, stft_length_masks=masks, wavs=d_wavs), **model_results)
    assert loss.item() == pytest.approx(ref["loss"].item(), abs=2e-3)
    for b in range(B):
        n = int(lengths[b])
        mine_db = se.sisdr_eval(wav_predicted[b, :n].cpu(), wavs[b, 1, :n])
        assert mine_db == pytest.approx(ref["sisdr"][b].item(), abs=SISDR_TOL_DB)


def test_train_step_gradients_match_oracle(se):
    ora, mine = make_pair(se, 400)
    B, T = 4, 8000
    lengths = torch.LongTensor([8000, 6000, 4000, 7999])
    lengths, wavs = synth(B, T, seed=8, lengths=lengths)
    torch.manual_seed(5)
    head = se.LinearResidual(input_size=201, output_size=201).cuda()
    w = head.linear.weight.detach().cpu().clone().requires_grad_(True)
    b = head.linear.bias.detach().cpu().clone().requires_grad_(True)
    c = ora.get_feat_config
    feats, lin_i, lin_t = ora(wavs, [c("linear", 0, log=True), c("linear", 0), c("linear", 1)])
    pred, _ = sp.linear_residual_head(feats, lin_i, w, b)
    masks = sp.length_masks(sp.stft_lengths(lengths, 160))
    ref_loss, _ = sp.sisdr_spectral(pred, lin_t, masks)
    ref_loss.backward()
    eng = se.EnhancementEngine(mine, head)
    loss = eng.train_step(lengths.cuda(), wavs.cuda(), se.SISDR())
    loss.backward()
    assert loss.item() == pytest.approx(ref_loss.item(), abs=2e-3)
    gw = head.linear.weight.grad.cpu()
    assert torch.nn.functional.cosine_similarity(gw.flatten(), w.grad.flatten(), dim=0).item() > 0.9999
    np.testing.assert_allclose(gw.numpy(), w.grad.numpy(), rtol=5e-2, atol=2e-3 * w.grad.abs().max().item())


@pytest.mark.parametrize("precision", [0, 1])
def test_pseudo_noise_config_end_to_end_matches_oracle_autograd(se, precision):
    """BASELINE configs[2] (config/pseudo_noise.yaml: n_fft 400 / hop 160, baseline feature mel + log + delta 2 = 120-d):
    preprocessor -> LinearResidual(120 -> 201) -> SISDR, and the projection-as-log-spectrum route Linear(120 -> 201,
    Identity) -> L1, forward and backward, against the oracle preprocessor + torch autograd on the same ragged batch."""
    ora, mine = make_pair(se, 400)
    B, T = 4, 8000
    lengths = torch.LongTensor([8000, 6000, 4321, 7999])
    lengths, wavs = synth(B, T, seed=12, lengths=lengths)
    c = ora.get_feat_config
    cfgs = [c("mel", 0, log=True, delta=2), c("linear", 0), c("linear", 1)]
    feats_r, lin_i_r, lin_t_r = ora(wavs, cfgs)
    feats, lin_i, lin_t = mine(wavs.cuda(), cfgs)
    assert feats.shape == (B, T // 160 + 1, 120)
    masks = sp.length_masks(sp.stft_lengths(lengths, 160))
    frames = (lengths // 160 + 1).cuda()
    # ---- LinearResidual + SISDR (runner.py:453-459 with --downstream LinearResidual --objective SISDR)
    torch.manual_seed(5)
    head = se.LinearResidual(input_size=120, output_size=201, precision=precision).cuda()
    w = head.linear.weight.detach().cpu().clone().requires_grad_(True)
    b = head.linear.bias.detach().cpu().clone().requires_grad_(True)
    pred_r, _ = sp.linear_residual_head(feats_r, lin_i_r, w, b)
    ref_loss, _ = sp.sisdr_spectral(pred_r, lin_t_r, masks)
    ref_loss.backward()
    predicted, extra = head(features=feats, linears=lin_i)
    loss, _ = se.SISDR()(predicted=predicted, linear_tar=lin_t, stft_lengths=frames, **extra)
    loss.backward()
    assert loss.item() == pytest.approx(ref_loss.item(), abs=2e-3 if precision == 0 else 5e-3)
    for got, want in ((head.linear.weight.grad.cpu(), w.grad), (head.linear.bias.grad.cpu(), b.grad)):
        assert torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0).item() > 0.9995
        np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=5e-2, atol=(2e-3 if precision == 0 else 1e-2) * want.abs().max().item())
    # ---- Linear (Identity) as log-spectrum predictor + L1 (objective.py:109-117)
    torch.manual_seed(6)
    lin = se.Linear(120, 201, activation="Identity", precision=precision).cuda()
    w2 = lin.linear.weight.detach().cpu().clone().requires_grad_(True)
    b2 = lin.linear.bias.detach().cpu().clone().requires_grad_(True)
    ref_l1 = sp.l1_logspectral(sp.linear_head(feats_r, w2, b2, "Identity"), lin_t_r, masks)
    ref_l1.backward()
    log_pred, _ = lin(features=feats)
    l1, _ = se.L1()(log_predicted=log_pred, linear_tar=lin_t, stft_lengths=frames)
    l1.backward()
    assert l1.item() == pytest.approx(ref_l1.item(), rel=2e-4 if precision == 0 else 2e-3)
    for got, want in ((lin.linear.weight.grad.cpu(), w2.grad), (lin.linear.bias.grad.cpu(), b2.grad)):
        assert torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0).item() > 0.999
        np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=5e-2, atol=(2e-3 if precision == 0 else 2e-2) * want.abs().max().item())


@pytest.mark.parametrize("route", ["autograd-fp32-torch-adam", "fused-tf32-clipadam", "fused-tf32-clipadam-graph"])
def test_training_steps_match_reference_runner_train(se, golden_dir, route):
    """runner.py:431-471 pinned by the reference ITSELF: tests/golden/runner_train_ref.npz holds the loss of every step and the
    final weights of four optimizer steps of the unmodified ``Runner.train()`` (LinearResidual + SISDR, Adam lr 1e-3, clipping
    1.0).  The engine's training step -- autograd route with torch's Adam, the fused route with ClipAdam, and the fused route
    replayed from a CUDA graph -- follows the same trajectory."""
    g = np.load(os.path.join(golden_dir, "runner_train_ref.npz"))
    items = [torch.from_numpy(g[f"item{i}"]) for i in range(len(g["lengths"]))]
    lengths, wavs = sp.collate(items)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    _, mine = make_pair(se, 512)
    precision = 0 if route.startswith("autograd") else 1
    head = se.LinearResidual(input_size=257, output_size=257, precision=precision).cuda()
    with torch.no_grad():
        head.linear.weight.copy_(torch.from_numpy(g["w0"]))
        head.linear.bias.copy_(torch.from_numpy(g["b0"]))
    eng = se.EnhancementEngine(mine, head, log_features=True, precision=precision)
    crit, steps, clip = se.SISDR(), int(g["steps"]), float(g["grad_clip"])
    losses = []
    if route.startswith("autograd"):
        opt = torch.optim.Adam(head.parameters(), lr=float(g["lr"]), betas=(0.9, 0.999))
        for _ in range(steps):
            losses.append(eng.train_step(lengths, wavs, crit, opt, clip).item())
    else:
        opt = se.ClipAdam(head.parameters(), lr=float(g["lr"]), betas=(0.9, 0.999))
        assert eng.fused_training_supported(crit, wavs.shape[0], wavs.shape[2])
        if route.endswith("graph"):
            st = eng.capture_train(lengths, wavs, crit, opt, clip)       # three eager warm-up steps happen in here:
            with torch.no_grad():                                        # rewind to the golden's starting point
                head.linear.weight.copy_(torch.from_numpy(g["w0"]))
                head.linear.bias.copy_(torch.from_numpy(g["b0"]))
                for p in head.parameters():
                    opt.state[p]["exp_avg"].zero_()
                    opt.state[p]["exp_avg_sq"].zero_()
                opt.param_groups[0]["_ws"][1].zero_()
            eng._padded_weight(force=True)
            for _ in range(steps):
                st["graph"].replay()
                losses.append(st["loss"].item())
        else:
            for _ in range(steps):
                losses.append(eng.train_step(lengths, wavs, crit, opt, clip).item())
    torch.cuda.synchronize()
    np.testing.assert_allclose(losses, g["losses"], atol=2e-3 if precision == 0 else 5e-3)
    dw = head.linear.weight.detach().cpu().numpy() - g["w1"]
    db = head.linear.bias.detach().cpu().numpy() - g["b1"]
    moved = np.abs(g["w1"] - g["w0"])
    print(route, "max |dw|", np.abs(dw).max(), "mean |dw|", np.abs(dw).mean(), "moved max / mean", moved.max(), moved.mean())
    if precision == 0:
        assert np.abs(dw).max() < 5e-5 and np.abs(db).max() < 5e-5 and moved.max() > 1e-3
    else:
        # TF32 operands in the weight-gradient GEMM: Adam's m / sqrt(v) turns the rounding noise of a near-zero gradient into a
        # full-size step for that element, so single weights may differ by a step or two while the bulk follows the trajectory
        assert np.abs(dw).mean() < 0.02 * moved.mean() and np.abs(dw).max() < 0.6 * moved.max()
        assert np.abs(db).mean() < 0.05 * np.abs(g["b1"] - g["b0"]).mean()
        update = (head.linear.weight.detach().cpu().numpy() - g["w0"]).ravel()
        assert np.dot(update, (g["w1"] - g["w0"]).ravel()) / (np.linalg.norm(update) * np.linalg.norm(g["w1"] - g["w0"])) > 0.995


def test_engine_training_step_with_a_feature_config(se):
    """EnhancementEngine(feat_cfg=...): the training step on the pseudo_noise.yaml baseline feature (mel + log + delta 2).
    The autograd route equals the hand-written chain on the drop-in modules; the FUSED route (K1b kernel -> sums -> TMA head ->
    SISDR forward / backward kernels -> split-K head backward, no autograd graph) gives the same loss and gradients up to the
    TF32 operands of its weight-gradient GEMM; and the step replays from a CUDA graph with ClipAdam."""
    _, mine = make_pair(se, 400)
    lengths, wavs = synth(4, 8000, seed=3, lengths=torch.LongTensor([8000, 6000, 4321, 7999]))
    lengths, wavs = lengths.cuda(), wavs.cuda()
    c = mine.get_feat_config
    cfg = c("mel", 0, log=True, delta=2)
    torch.manual_seed(5)
    head = se.LinearResidual(input_size=120, output_size=201, precision=1).cuda()
    eng = se.EnhancementEngine(mine, head, precision=1, feat_cfg=cfg)
    assert eng.fused_training_supported(se.SISDR(), 4, 8000)
    assert not se.EnhancementEngine(mine, head, precision=1, feat_cfg=c("mel", 0, log=True, delta=2, cmvn=True)).fused_training_supported(se.SISDR(), 4, 8000)
    eng.fused_training = False                              # autograd route through the custom ops
    loss = eng.train_step(lengths, wavs, se.SISDR())
    loss.backward()
    g_w, g_b = head.linear.weight.grad.clone(), head.linear.bias.grad.clone()
    head.zero_grad()
    feats, lin_i, lin_t = mine(wavs, [cfg, c("linear", 0), c("linear", 1)])
    predicted, extra = head(features=feats, linears=lin_i)
    ref, _ = se.SISDR()(predicted=predicted, linear_tar=lin_t, stft_lengths=lengths // 160 + 1, **extra)
    ref.backward()
    assert loss.item() == pytest.approx(ref.item(), abs=1e-6) and torch.equal(g_w, head.linear.weight.grad)
    del loss, ref, predicted, extra, feats                  # (eager autograd graphs hold default-stream nodes: drop them before capturing)
    head.zero_grad(set_to_none=True)
    eng.fused_training = True                               # fused route: gradients land in .grad without an autograd graph
    loss_f = eng._fused_forward_backward(lengths, wavs, se.SISDR())
    torch.cuda.synchronize()
    assert loss_f.item() == pytest.approx(float((g_w * 0).sum()) + loss_f.item())          # finite
    for got, want in ((head.linear.weight.grad, g_w), (head.linear.bias.grad, g_b)):
        assert torch.nn.functional.cosine_similarity(got.flatten(), want.flatten(), dim=0).item() > 0.99999
        assert (got - want).abs().max().item() < 2e-3 * want.abs().max().item()
    # evaluation step on the same feature config: the hand-written chain on the drop-in modules gives the same metrics
    with torch.no_grad():
        out = eng.eval_step(lengths, wavs)
        feats, lin_i, ph_i = mine(wavs, [cfg, c("linear", 0), c("phase", 0)])
        predicted, _ = head(features=feats, linears=lin_i)
        wav_ref = se.decode_wav(mine, predicted, ph_i, lengths)            # (level differs: SI-SDR is scale-invariant)
    for b in range(4):
        n = int(lengths[b])
        assert abs(sp.sisdr_eval(wav_ref[b, :n].cpu(), wavs[b, 1, :n].cpu()) - out["sisdr"][b].item()) < 0.02
    torch.manual_seed(5)
    head_g = se.LinearResidual(input_size=120, output_size=201, precision=1).cuda()
    eng_g = se.EnhancementEngine(mine, head_g, precision=1, feat_cfg=cfg)
    w0 = head_g.linear.weight.detach().clone()
    opt = se.ClipAdam(head_g.parameters(), lr=1e-3)
    crit = se.SISDR()                                       # (the captured step is cached per objective / optimizer object)
    for _ in range(5):
        out = eng_g.train_step_graph(lengths, wavs, crit, opt, 1.0)
    torch.cuda.synchronize()
    assert opt.steps_taken() == [8] and torch.isfinite(out).all() and not torch.equal(w0, head_g.linear.weight.detach())


# ------------------------------------------------------------------------------ fast paths vs generic tile kernels
GEO = {512: (257, 32, 16, 256), 1024: (513, 64, 16, 256), 400: (201, 25, 10, 160)}


@pytest.mark.parametrize("n_fft,T", [(512, 16000), (512, 16001), (512, 12345), (512, 700), (512, 1500), (512, 64000),
                                     (1024, 16000), (1024, 16001), (1024, 12345), (1024, 1500), (1024, 64000), (400, 16000),
                                     (400, 16001), (400, 7777), (400, 350), (400, 64000)])
def test_fast_geometries_stft_equals_generic_path(se, n_fft, T):
    """Register-resident STFT (fastgeo.cu: 512/256, 1024/256, 400/160) against the generic tile path and the oracle: odd T
    (unaligned rows: element-wise reflect loads), runs shorter than the halo, several utterances."""
    from speech_enhancement_by_s3prl_b200 import _lib
    n_freq, win_ms, hop_ms, hop = GEO[n_fft]
    mine = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).cuda()
    ora = OraclePre(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq)
    _, wavs = synth(3, T, seed=T + n_fft)
    c = mine.get_feat_config
    cfgs = [c("linear", 0), c("phase", 0), c("linear", 1, log=True), c("linear", 2)]
    lib = _lib.load()
    fast = [t.cpu() for t in mine(wavs.cuda(), cfgs)]
    try:
        lib.se_set_option(0, 1)
        slow = [t.cpu() for t in mine(wavs.cuda(), cfgs)]
    finally:
        lib.se_set_option(0, 0)
    ref = ora(wavs, cfgs)
    assert fast[0].shape == ref[0].shape == (3, T // hop + 1, n_freq)
    assert rel_to_max(fast[0], slow[0]) < 2e-6 and rel_to_max(fast[3], slow[3]) < 2e-6
    assert rel_to_max(fast[0], ref[0]) < SPEC_RTOL
    loud = slow[2] > slow[2].amax() - 7.0                                          # log-power of bins within 30 dB of the largest one
    assert (fast[2] - slow[2]).abs()[loud].max() < 2e-3
    strong = ref[0] > 1e-5 * ref[0].amax()
    dphi = torch.angle(torch.polar(torch.ones_like(ref[1]), fast[1] - ref[1]))
    assert dphi[strong].abs().max() < 2e-3


@pytest.mark.parametrize("n_fft,T,B", [(512, 16000, 3), (512, 16001, 2), (512, 9999, 3), (512, 1100, 2), (512, 64000, 5),
                                       (1024, 16000, 3), (1024, 16001, 2), (1024, 9999, 3), (1024, 2100, 2), (1024, 64000, 5),
                                       (1024, 160000, 2), (400, 16000, 3), (400, 16001, 2), (400, 9999, 3), (400, 1100, 2),
                                       (400, 64000, 5), (400, 160000, 2)])
def test_fast_geometries_mask_istft_equals_generic_path(se, n_fft, T, B):
    """Fused mask -> iSTFT of fastgeo.cu (overlap-add carry in registers, 2-4 frames per sample, emit windows, virtual
    flush frames, edge envelopes) against the generic tile path: waveform, all six sums, ragged lengths, power mode."""
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    n_freq, win_ms, hop_ms, hop = GEO[n_fft]
    mine = se.OnlinePreprocessor(win_ms=win_ms, hop_ms=hop_ms, n_freq=n_freq).cuda()
    lengths = torch.LongTensor([T, max(300, T - 777), T // 2 + 3, T, T // 3 + 1][:B])
    lengths, wavs = synth(B, T, seed=T + 5, lengths=lengths)
    g = torch.Generator().manual_seed(4)
    mask = torch.rand(B, T // hop + 1, n_freq, generator=g).cuda()
    lib = _lib.load()
    args = (wavs.cuda(), 0, 1, mask, lengths.cuda(), n_fft, hop, mine._frame_window)
    wav_f, sums_f = ops.mask_istft(*args, pad_to=T)
    pw_f, _ = ops.mask_istft(*args, pad_to=T, mask_is_power=True)
    try:
        lib.se_set_option(0, 1)
        wav_s, sums_s = ops.mask_istft(*args, pad_to=T)
        pw_s, _ = ops.mask_istft(*args, pad_to=T, mask_is_power=True)
    finally:
        lib.se_set_option(0, 0)
    wav_tol, sums_rtol = (2e-6, 2e-5) if n_fft == 512 else (3e-6, 3e-5)
    assert wav_f.shape == wav_s.shape == (B, T)
    assert (wav_f - wav_s).abs().max().item() < wav_tol
    # power mode gives every bin the magnitude sqrt(mask), also bins whose noisy phase is rounding noise: looser bound
    assert (pw_f - pw_s).abs().max().item() < 2e-4 * pw_s.abs().max().item()
    np.testing.assert_allclose(sums_f.cpu().numpy(), sums_s.cpu().numpy(), rtol=sums_rtol, atol=1e-9)
    # padded mask rows (the fused step's layout), and no clean / sums / lengths
    LD = (n_freq + 3) // 4 * 4
    mask_p = torch.zeros(B, T // hop + 1, LD, device="cuda")
    mask_p[..., :n_freq] = mask
    wav_p, sums_p = ops.mask_istft(wavs.cuda(), 0, 1, mask_p, lengths.cuda(), n_fft, hop, mine._frame_window, pad_to=T, mask_padded=True)
    assert torch.equal(wav_p, wav_f)
    wav_n, none = ops.mask_istft(wavs.cuda(), 0, None, mask, None, n_fft, hop, mine._frame_window, pad_to=T, want_sums=False)
    assert none is None and (wav_n - wav_s).abs().max().item() < wav_tol


@pytest.mark.parametrize("n_fft,B,T", [(512, 1, 960000), (512, 200, 1100), (512, 3, 257), (512, 2, 1281), (1024, 1, 960000),
                                       (1024, 200, 1100), (1024, 3, 1281), (1024, 2, 1535), (400, 1, 480000), (400, 300, 700),
                                       (400, 3, 801), (400, 2, 959), (400, 5, 201)])
def test_fast_geometries_edge_shapes_match_oracle(se, n_fft, B, T):
    """Edge shapes of the register-resident kernels against the CPU oracle: one long utterance (60 s / 30 s: thousands of
    runs per utterance), hundreds of tiny ones (every run shorter than its halo; fewer than six frames falls back to the
    generic path), T just above n_fft/2 (torch.stft's minimum), first / last samples covered by fewer frames than the interior."""
    from speech_enhancement_by_s3prl_b200 import ops
    ora, mine = make_pair(se, n_fft)
    hop = mine._win_args["hop_length"]
    K = n_fft // 2 + 1
    g = torch.Generator().manual_seed(n_fft + B + T)
    wavs = torch.randn(B, 3, T, generator=g) * 0.05
    lengths = torch.randint(max(n_fft // 2 + 1, T // 2), T + 1, (B,), generator=g)
    lengths[0] = T
    for b, n in enumerate(lengths.tolist()):
        wavs[b, :, n:] = 0
    c = ora.get_feat_config
    lin_r, ph_r = ora(wavs[:4], [c("linear", 0), c("phase", 0)])
    lin = mine(wavs[:4].cuda(), [c("linear", 0)])[0].cpu()
    assert lin.shape == lin_r.shape == (min(B, 4), T // hop + 1, K)
    assert rel_to_max(lin, lin_r) < SPEC_RTOL
    mask = torch.rand(B, T // hop + 1, K, generator=g)
    wav, sums = ops.mask_istft(wavs.cuda(), 0, 1, mask.cuda(), lengths.cuda(), n_fft, hop, mine._frame_window, pad_to=T)
    torch.cuda.synchronize()
    assert wav.shape == (B, T) and torch.isfinite(wav).all() and torch.isfinite(sums).all()
    ref = ora.istft(lin_r * mask[:4], ph_r)                                  # (4, hop * (F - 1))
    n_out = ref.shape[1]
    assert (wav[:4, :n_out].cpu() - ref).abs().max().item() < 5e-6 * max(1.0, ref.abs().max().item() / 0.05)
    assert wav[:, n_out:].abs().max().item() == 0.0 if n_out < T else True     # zero-padded to T (runner.py:268)
    for b in range(min(B, 4)):
        n = int(lengths[b])
        y, cl = wav[b, :n].double().cpu(), wavs[b, 1, :n].double()
        np.testing.assert_allclose(sums[b, :3].cpu().numpy(), [float((y * cl).sum()), float((cl * cl).sum()), float((y * y).sum())],
                                   rtol=2e-4, atol=1e-7)


# ------------------------------------------------------------------------------ tensor-core head (tcgen05, TF32)
@pytest.mark.parametrize("B,F,Din,Dout,act,cmvn", [(3, 101, 257, 257, "Sigmoid", True), (2, 300, 201, 201, "ReLU", False),
                                                   (1, 77, 513, 513, "Sigmoid", True), (2, 128, 120, 201, "Identity", True),
                                                   (64, 251, 257, 257, "Sigmoid", True)])
def test_tensor_core_head_matches_fp32_head(se, B, F, Din, Dout, act, cmvn):
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(Din + F)
    feats = (torch.randn(B, F, Din, generator=g) * 2 - 3).cuda()
    linears = torch.rand(B, F, Dout, generator=g).cuda()
    torch.manual_seed(2)
    lin = torch.nn.Linear(Din, Dout).cuda()
    mean = std = None
    if cmvn:
        mean, std = ops.cmvn_stats(feats)
    off0, pred0 = ops.linear_head_fused(feats, lin.weight, lin.bias, act, mean, std, 1e-6, linears=linears, precision=0)
    off1, pred1 = ops.linear_head_fused(feats, lin.weight, lin.bias, act, mean, std, 1e-6, linears=linears, precision=1)
    torch.cuda.synchronize()
    # TF32 operands (10-bit mantissa, round-to-nearest), fp32 accumulation
    scale = max(1.0, feats.abs().max().item() * 0.1)              # error scales with |x| |w| sqrt(Din)
    assert (off1 - off0).abs().max().item() < 3e-3 * scale
    assert (pred1 - pred0).abs().max().item() < 3e-3 * scale
    assert (off1 - off0).abs().mean().item() < 3e-4 * scale


def test_eval_step_with_tensor_core_head_keeps_sisdr_parity(se, golden_dir):
    g, items = _load_runner_golden(golden_dir)
    _, mine = make_pair(se, 512)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    head.load_state_dict({"linear.weight": torch.from_numpy(g["weight"]), "linear.bias": torch.from_numpy(g["bias"])})
    eng = se.EnhancementEngine(mine, head, log_features=True, precision=1)
    losses, scores = [], []
    for i in range(0, len(items), 2):
        lengths, wavs = sp.collate(items[i:i + 2])
        out = eng.eval_step(lengths.cuda(), wavs.cuda())
        losses.append(out["loss_per_utt"].mean().item())
        scores.append(out["sisdr"].mean().item())
    assert np.mean(losses) == pytest.approx(float(g["loss"]), abs=5e-3)
    assert np.mean(scores) == pytest.approx(float(g["scores"][0]), abs=SISDR_TOL_DB)


# ------------------------------------------------------------------------------ fused step: K1 with CMVN sums, TMA head
@pytest.mark.parametrize("n_fft,B,T,logp", [(512, 3, 16000, True), (512, 5, 9999, True), (512, 2, 64000, False),
                                            (512, 64, 4096, True), (400, 2, 16000, True), (400, 5, 9999, False),
                                            (400, 64, 4000, True), (1024, 3, 16000, True), (1024, 2, 9999, False),
                                            (1024, 64, 8192, True)])
def test_stft_features_and_cmvn_sums(se, n_fft, B, T, logp):
    from speech_enhancement_by_s3prl_b200 import ops
    _, mine = make_pair(se, n_fft)
    hop = mine._win_args["hop_length"]
    K = n_fft // 2 + 1
    _, wavs = synth(B, T, seed=T + B)
    wavs = wavs.cuda()
    feats, sums = ops.stft_features(wavs, 0, n_fft, hop, mine._frame_window, logpower=logp)
    ref = ops.stft(wavs, 0, n_fft, hop, mine._frame_window, power=not logp, logpower=logp)["logpower" if logp else "power"]
    torch.cuda.synchronize()
    assert torch.equal(feats[..., :K], ref)                                     # same kernel body: bit-identical features
    s1 = ref.double().sum(1)
    s2 = (ref.double() ** 2).sum(1)
    # the fused kernel adds up a run's few frames in fp32 before the double-precision combine: ~1e-7 relative per partial
    F = ref.shape[1]
    a1 = 1e-6 * (s2.max().item() * F) ** 0.5
    np.testing.assert_allclose(sums[:, :K, 0].cpu().numpy(), s1.cpu().numpy(), rtol=2e-6, atol=a1)
    np.testing.assert_allclose(sums[:, :K, 1].cpu().numpy(), s2.cpu().numpy(), rtol=2e-6)
    # and the standalone sums entry point (double precision throughout)
    sums2 = ops.feature_sums(feats, K)
    np.testing.assert_allclose(sums2[:, :K, 0].cpu().numpy(), s1.cpu().numpy(), rtol=1e-9, atol=1e-3 * a1)
    np.testing.assert_allclose(sums2[:, :K, 1].cpu().numpy(), s2.cpu().numpy(), rtol=1e-9)
    # what the head derives from the sums: mean / unbiased std against torch
    mean = (sums[:, :K, 0] / F).float()
    var = ((sums[:, :K, 1] - sums[:, :K, 0] ** 2 / F) / (F - 1)).clamp_min(0)
    assert (mean - ref.mean(1)).abs().max().item() < 1e-5 * max(1.0, ref.abs().max().item())
    np.testing.assert_allclose(var.sqrt().float().cpu().numpy(), ref.std(1).cpu().numpy(), rtol=2e-5, atol=1e-7)


@pytest.mark.parametrize("B,F,Din,Dout,act,cmvn", [(3, 101, 257, 257, "Sigmoid", True), (2, 300, 201, 201, "ReLU", False),
                                                   (2, 128, 120, 201, "Identity", True), (64, 251, 257, 257, "Sigmoid", True),
                                                   (1, 9, 257, 257, "Sigmoid", True), (700, 40, 129, 129, "Sigmoid", True),
                                                   (2, 77, 513, 513, "Sigmoid", True), (64, 251, 513, 513, "Sigmoid", True),
                                                   (3, 40, 513, 300, "ReLU", False), (2, 33, 120, 513, "Identity", True),
                                                   (96, 251, 257, 257, "Sigmoid", True), (40, 777, 257, 257, "ReLU", True),
                                                   (30, 1001, 201, 201, "Sigmoid", True), (9, 3751, 513, 513, "Sigmoid", True)])
def test_tma_head_matches_fp32_head(se, B, F, Din, Dout, act, cmvn):
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(Din + F)
    LDx = ops.round4(Din)
    feats = torch.full((B, F, LDx), float("nan"))                            # padding columns must never leak into the result
    feats[..., :Din] = torch.randn(B, F, Din, generator=g) * 2 - 3
    feats = feats.cuda()
    torch.manual_seed(2)
    lin = torch.nn.Linear(Din, Dout).cuda()
    dense = feats[..., :Din].contiguous()
    mean = std = sums = None
    if cmvn:
        mean, std = ops.cmvn_stats(dense)
        sums = ops.feature_sums(feats, Din)
    off0, _ = ops.linear_head_fused(dense, lin.weight, lin.bias, act, mean, std, 1e-6, precision=0)
    assert ops.linear_head_tma_supported(B, F, Din, Dout, LDx, LDx, ops.round4(Dout))
    wpad = ops.round_tf32(ops.pad_weight(lin.weight.detach()))
    off1 = ops.linear_head_tma(feats, Din, wpad, lin.bias, act, sums, 1e-6)[..., :Dout]
    torch.cuda.synchronize()
    scale = max(1.0, dense.abs().max().item() * 0.1)
    assert torch.isfinite(off1).all()
    assert (off1 - off0).abs().max().item() < 3e-3 * scale
    assert (off1 - off0).abs().mean().item() < 3e-4 * scale


def test_round_tf32_matches_cvt_rna(se):
    from speech_enhancement_by_s3prl_b200 import ops
    w = torch.randn(1000).cuda()
    r = ops.round_tf32(w)
    assert ((r.view(torch.int32) & 0x1FFF) == 0).all()
    assert ((r - w).abs() <= w.abs() * 2.0 ** -11 * 1.0001).all()


# ------------------------------------------------------------------------------ recurrent heads (a7): projection + multiply / exp
RECURRENT = {"lstm_uni": ("LSTM", dict(bidirectional=False, activation="Identity")),
             "lstm_bi": ("LSTM", dict(bidirectional=True, activation="Identity")),
             "res_uni": ("Residual", dict(bidirectional=False, activation="Sigmoid", cmvn=False)),
             "res_bi_cmvn": ("Residual", dict(bidirectional=True, activation="Sigmoid", cmvn=True)),
             "res_relu": ("Residual", dict(bidirectional=False, activation="ReLU", cmvn=True))}


@pytest.mark.parametrize("tag", sorted(RECURRENT))
@pytest.mark.parametrize("precision", [0, 1])
def test_recurrent_heads_match_reference_golden(se, golden_dir, tag, precision):
    """model.py:37-91 -- LSTM / Residual with the REFERENCE's state dict: outputs, and the gradients of every parameter
    (the projection's from the head kernels' wgrad, the LSTM's through the head kernels' input gradient), against what
    the reference's own classes produced (oracle/make_golden.py::make_recurrent_heads)."""
    gold = np.load(os.path.join(golden_dir, "recurrent_heads_ref.npz"))
    cls, kw = RECURRENT[tag]
    head = getattr(se, cls)(input_size=9, output_size=9, hidden_size=12, num_layers=2, precision=precision, **kw).cuda()
    state = {k[len(tag) + 7:]: torch.from_numpy(gold[k]) for k in gold.files if k.startswith(f"{tag}_param_")}
    head.load_state_dict(state)                                             # same parameter names as the reference (strict)
    feats, linears = torch.from_numpy(gold["feats"]).cuda(), torch.from_numpy(gold["linears"]).cuda()
    tol = 1e-4 if precision == 0 else 3e-3                                  # values are O(1); precision 1: TF32 operands in the projection
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):        # the cuDNN LSTM body in fp32: the bounds test the projection
        predicted, res = head(features=feats, linears=linears)
        assert (predicted.cpu() - torch.from_numpy(gold[f"{tag}_predicted"])).abs().max().item() < tol * 5
        for k, v in res.items():
            assert (v.detach().cpu() - torch.from_numpy(gold[f"{tag}_{k}"])).abs().max().item() < tol
        loss = (predicted * torch.linspace(0.5, 1.5, 9, device="cuda")).pow(2).mean() + 0.1 * predicted.mean()
        assert loss.item() == pytest.approx(float(gold[f"{tag}_loss"]), rel=tol * 10)
        loss.backward()
    for name, p in head.named_parameters():
        want = torch.from_numpy(gold[f"{tag}_grad_{name}"])
        assert p.grad is not None, name
        scale = max(want.abs().max().item(), 1e-4)
        assert (p.grad.cpu() - want).abs().max().item() < (2e-4 if precision == 0 else 2e-2) * scale, name


# ------------------------------------------------------------------------------ the bench configuration at full size
@pytest.fixture(scope="module")
def bench_case(se):
    """BASELINE.json configs[1]: 64 x 4 s, 16 kHz, n_fft 512 / hop 256, LinearResidual(257) on log-power -- the exact batch
    bench.py times, with ragged lengths added for half of the utterances.  The oracle runs it in well under a second."""
    from speech_enhancement_by_s3prl_b200 import synth as synth_mod
    ora, mine = make_pair(se, 512)
    lengths, wavs = synth_mod.batch(64, 4.0)
    g = torch.Generator().manual_seed(9)
    lengths = lengths.clone()
    cut = torch.randint(20000, 64000, (32,), generator=g)
    lengths[::2] = cut
    for b, n in enumerate(lengths.tolist()):
        wavs[b, :, n:] = 0                                                  # collate_fn zero-pads (dataset.py:175)
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    c = ora.get_feat_config
    ora.feat_list = [c("linear", 0, log=True), c("linear", 0, log=True), c("linear", 0), c("phase", 0), c("linear", 1), c("phase", 1)]
    with torch.no_grad():
        ref = sp.eval_step(ora, dict(weight=head.linear.weight.detach().cpu(), bias=head.linear.bias.detach().cpu()), lengths, wavs)
    return dict(mine=mine, head=head, lengths=lengths, wavs=wavs, ref=ref)


@pytest.mark.parametrize("mode", ["eager", "graph", "host_pipeline"])
def test_bench_configuration_matches_oracle_at_full_size(se, bench_case, mode):
    bc = bench_case
    eng = se.EnhancementEngine(bc["mine"], bc["head"], log_features=True, precision=1)       # the path bench.py times
    lengths, wavs, ref = bc["lengths"], bc["wavs"], bc["ref"]
    if mode == "eager":
        out = eng.eval_step(lengths.cuda(), wavs.cuda())
        sisdr, loss = out["sisdr"].cpu(), out["loss_per_utt"].mean().item()
    elif mode == "graph":
        st = eng.capture_bound(lengths.cuda(), wavs.cuda())
        for _ in range(3):                                                  # replays must not accumulate into the workspaces
            st["graph"].replay()
        torch.cuda.synchronize()
        sisdr, loss = st["sisdr"].cpu(), st["loss_per_utt"].mean().item()
        out = st
    else:
        pipe = eng.host_pipeline(64, 3, 64000, depth=2)
        lp, wp = lengths.clone().pin_memory(), wavs.clone().pin_memory()
        for _ in range(3):
            pipe.submit(lp, wp)
        res = pipe.drain()
        assert len(res) == 3
        for r in res[1:]:                                                   # every slot of the pipeline gives the same answer
            # (equal up to the order of the double-precision atomics that combine the per-run sums)
            assert (r[0] - res[0][0]).abs().max().item() < 1e-5 and (r[1] - res[0][1]).abs().max().item() < 1e-5
        sisdr, loss = res[0][1], res[0][0].mean().item()
        out = None
    np.testing.assert_allclose(sisdr.numpy(), ref["sisdr"].numpy(), atol=SISDR_TOL_DB)
    assert loss == pytest.approx(ref["loss"].item(), abs=5e-3)              # TF32 head: 10-bit mantissa operands
    if out is not None:
        for b in (0, 1, 31, 63):
            n = int(lengths[b])
            assert sisdr_db(out["wav_predicted"][b, :n].cpu(), ref["wav_predicted"][b, :n]) > 40.0


def test_host_pipeline_pcm16_input_and_waveform_output(se, bench_case):
    """int16 PCM host batches (2 bytes per sample over PCIe, widened on the device: exact) give what the fp32 pipeline gives
    on the dequantised batch, and want_wav returns the level-matched enhanced waveforms the device step produced."""
    bc = bench_case
    eng = se.EnhancementEngine(bc["mine"], bc["head"], log_features=True, precision=1)
    lengths = bc["lengths"]
    pcm = (bc["wavs"] * 32768.0).round().clamp_(-32768, 32767).to(torch.int16)
    deq = pcm.to(torch.float32) / 32768.0
    assert (deq - bc["wavs"]).abs().max().item() <= 0.5 / 32768 + 1e-9
    pipe16 = eng.host_pipeline(64, 3, 64000, depth=2, pcm16=True, want_wav=True)
    pipe32 = eng.host_pipeline(64, 3, 64000, depth=2)
    assert pipe16.h2d_bytes == 64 * 2 * 64000 * 2 + 64 * 8 and pipe16.d2h_bytes == 2 * 64 * 4 + 64 * 64000 * 4
    lp = lengths.clone().pin_memory()
    for _ in range(2):
        pipe16.submit(lp, pcm.clone().pin_memory())
        pipe32.submit(lp, deq.clone().pin_memory())
    r16, r32 = pipe16.drain(), pipe32.drain()
    assert len(r16) == 2 and len(r16[0]) == 3 and len(r32[0]) == 2
    for a, b in zip(r16, r32):
        assert (a[0] - b[0]).abs().max().item() < 1e-5 and (a[1] - b[1]).abs().max().item() < 1e-5
    np.testing.assert_allclose(r16[0][1].numpy(), bc["ref"]["sisdr"].numpy(), atol=0.05)          # 16-bit quantisation of the inputs
    out = eng.eval_step(lengths.cuda(), deq.cuda())
    assert (r16[1][2] - out["wav_predicted"].cpu()).abs().max().item() < 1e-6
    with pytest.raises(RuntimeError):
        pipe16.submit(lp, deq.clone().pin_memory())                                                # fp32 batch into the int16 pipeline


def test_fused_step_properties_at_full_size(se, bench_case):
    """Size-independent properties of the fused kernels on the full bench batch (no oracle involved)."""
    from speech_enhancement_by_s3prl_b200 import ops
    mine, wavs = bench_case["mine"], bench_case["wavs"].cuda()
    B, _, T = wavs.shape
    F, K = T // 256 + 1, 257
    win = mine._frame_window
    # (1) an all-ones mask reconstructs the noisy waveform: iSTFT(STFT(x)) = x through the fused mask->iSTFT kernel
    ones = torch.ones(B, F, K, device=wavs.device)
    wav, sums = ops.mask_istft(wavs, 0, 0, ones, None, 512, 256, win, pad_to=T)
    assert (wav - wavs[:, 0]).abs().max().item() < 5e-6
    # ... and its sums are the waveform's energy three times over (y = c = noisy), spectral sums tie: st = tt = ss
    e = (wavs[:, 0].double() ** 2).sum(1)
    for col in (0, 1, 2):
        np.testing.assert_allclose(sums[:, col].cpu().numpy(), e.cpu().numpy(), rtol=2e-5)
    np.testing.assert_allclose(sums[:, 3].cpu().numpy(), sums[:, 4].cpu().numpy(), rtol=1e-5)
    np.testing.assert_allclose(sums[:, 5].cpu().numpy(), sums[:, 4].cpu().numpy(), rtol=1e-5)
    # (2) a constant mask g scales the output by sqrt(g) (the mask multiplies the POWER spectrum, model.py:33)
    wav_q, _ = ops.mask_istft(wavs, 0, None, ones * 0.25, None, 512, 256, win, pad_to=T, want_sums=False)
    assert (wav_q - 0.5 * wav).abs().max().item() < 5e-6
    # (3) Parseval on the analysis side: sum_k c_k |X_k|^2 = N * sum_n (w_n x_n)^2 per frame, checked in aggregate
    feats, st_sums = ops.stft_features(wavs, 0, 512, 256, win, logpower=False)
    p = feats[..., :K].double()
    wgt = torch.full((K,), 2.0, dtype=torch.float64, device=p.device)
    wgt[0] = wgt[-1] = 1.0
    lhs = (p * wgt).sum((1, 2))
    x = torch.nn.functional.pad(wavs[:, 0:1].double(), (256, 256), mode="reflect")[:, 0]
    frames = x.unfold(1, 512, 256)[:, :F]
    rhs = 512.0 * ((frames * win.double()) ** 2).sum((1, 2))
    np.testing.assert_allclose(lhs.cpu().numpy(), rhs.cpu().numpy(), rtol=2e-5)
    # (4) the CMVN sums of K1 are the column sums of what it wrote
    np.testing.assert_allclose(st_sums[:, :K, 0].cpu().numpy(), p.sum(1).cpu().numpy(), rtol=5e-6, atol=1e-9)


# ------------------------------------------------------------------------------ fused WSD objective (SURVEY 8f, rank 1)
@pytest.mark.parametrize("B,F,K,alpha,db", [(3, 40, 201, 0.3, 50.0), (5, 120, 257, 0.5, 30.0), (2, 33, 129, 0.9, 10.0)])
def test_wsd_matches_oracle_and_autograd(se, B, F, K, alpha, db):
    g = torch.Generator().manual_seed(B * F + K)
    tar = (torch.rand(B, F, K, generator=g) ** 4) * 3.0                         # heavy-tailed power spectra
    tar[:, F // 3:F // 2] *= 1e-4                                               # some frames well below the voicing threshold
    inp = tar + (torch.rand(B, F, K, generator=g) - 0.3).clamp_min(-0.2) * 0.5  # X - S of both signs
    off = torch.rand(B, F, K, generator=g)
    lens = torch.randint(F // 2, F + 1, (B,), generator=g)
    lens[0] = F
    masks = (torch.arange(F)[None, :] < lens[:, None]).long()
    ref_off = off.clone().requires_grad_(True)
    ref = sp.wsd(inp, ref_off, tar, masks, alpha=alpha, db_interval=db)
    ref.backward()
    mine_off = off.cuda().requires_grad_(True)
    loss, _ = se.WSD(alpha=alpha, db_interval=db)(inp.cuda(), mine_off, tar.cuda(), masks.cuda())
    loss.backward()
    assert loss.item() == pytest.approx(ref.item(), rel=2e-5)
    scale = ref_off.grad.abs().max().item()
    assert (mine_off.grad.cpu() - ref_off.grad).abs().max().item() < 2e-5 * scale
    assert torch.count_nonzero(mine_off.grad.cpu()[masks == 0]).item() == 0     # padded frames carry no gradient
    # frame counts instead of masks (what the fused step passes)
    loss2, _ = se.WSD(alpha=alpha, db_interval=db)(inp.cuda(), off.cuda(), tar.cuda(), stft_lengths=lens.cuda())
    assert loss2.item() == pytest.approx(loss.item(), rel=1e-6)
    # the one-call form se_wsd_fwd through the C ABI: the oracle's loss, and the energies / batch maximum of se_wsd_energy
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    inp_d, off_d, tar_d, lens_d = inp.cuda(), off.cuda(), tar.cuda(), lens.cuda()
    energy, emax = ops.wsd_energy(tar_d, K)
    ws_energy, ws_max, loss3 = torch.empty(B * F, device="cuda"), torch.empty(1, device="cuda"), torch.empty(1, device="cuda")
    ws_sums2 = torch.empty(B, 2, device="cuda", dtype=torch.float64)
    rc = _lib.load().se_wsd_fwd(inp_d.data_ptr(), off_d.data_ptr(), tar_d.data_ptr(), lens_d.data_ptr(), B, F, K, alpha, db, 1e-10,
                                ws_energy.data_ptr(), ws_max.data_ptr(), ws_sums2.data_ptr(), loss3.data_ptr(),
                                torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _lib.last_error()
    assert loss3.item() == pytest.approx(ref.item(), rel=2e-5)
    assert torch.equal(ws_max, emax) and torch.equal(ws_energy, energy.flatten())


# ------------------------------------------------------------------------------ on-device batch synthesis (SURVEY 8f, rank 3)
def test_mix_batch_matches_reference_recipe(se):
    """dataset.py:128-179 on the GPU: normalise -> tile/crop noise -> scale to SNR -> mix -> stack -> zero-pad."""
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(3)
    s_lens = [16000, 9001, 12345, 4000, 16000]
    n_lens = [5000, 20000, 12345, 3999, 48000]                                  # tiled, cropped, equal, tiled by one + rest, cropped
    snrs = torch.tensor([3.0, -8.0, 0.0, 8.0, 5.0])
    Ts, Tn = max(s_lens), max(n_lens)
    speech, noise = torch.zeros(5, Ts), torch.zeros(5, Tn)
    items = []
    for b, (ls, ln) in enumerate(zip(s_lens, n_lens)):
        sp_b = 0.3 * torch.randn(ls, generator=g) * (1 + torch.sin(torch.arange(ls) / 700.0))
        nz_b = 0.05 * torch.randn(ln, generator=g)
        speech[b, :ls], noise[b, :ln] = sp_b, nz_b
        s_n, n_n = sp.normalize_wav_decibel(sp_b), sp.normalize_wav_decibel(nz_b)
        noisy, scaled = sp.add_noise(s_n[None], n_n[None], snrs[b:b + 1], eps=1e-8)
        items.append(torch.stack([noisy[0], s_n, scaled[0]], dim=-1))
    ref_len, ref_wavs = sp.collate(items)
    lengths, wavs = ops.mix_batch(speech.cuda(), torch.tensor(s_lens).cuda(), noise.cuda(), torch.tensor(n_lens).cuda(), snrs.cuda())
    assert torch.equal(lengths.cpu(), ref_len) and wavs.shape == ref_wavs.shape
    assert (wavs.cpu() - ref_wavs).abs().max().item() < 2e-6 * ref_wavs.abs().max().item() + 1e-7
    # the requested SNR is met on every utterance (SURVEY 8c known-answer check)
    for b, ls in enumerate(s_lens):
        clean, sc = wavs[b, 1, :ls].double(), wavs[b, 2, :ls].double()
        assert 10 * torch.log10(clean.pow(2).sum() / sc.pow(2).sum()).item() == pytest.approx(snrs[b].item(), abs=1e-3)
        assert torch.count_nonzero(wavs[b, :, ls:]).item() == 0


def test_train_step_graph_matches_eager_training(se):
    """Five optimisation steps replayed from the captured training graph land on the same weights as five eager steps."""
    _, mine = make_pair(se, 512)
    lengths, wavs = synth(4, 16000, seed=21, lengths=torch.LongTensor([16000, 12000, 16000, 9000]))
    lengths, wavs = lengths.cuda(), wavs.cuda()
    results = []
    for use_graph in (False, True):
        torch.manual_seed(5)
        head = se.LinearResidual(input_size=257, output_size=257).cuda()
        eng = se.EnhancementEngine(mine, head, log_features=True, precision=0)
        opt = torch.optim.Adam(head.parameters(), lr=1e-3, capturable=True)
        obj = se.SISDR()
        init = head.linear.weight.detach().clone()
        for _ in range(5):
            loss = eng.train_step_graph(lengths, wavs, obj, opt, grad_clip=1.0) if use_graph else eng.train_step(lengths, wavs, obj, opt, 1.0)
        torch.cuda.synchronize()
        results.append((head.linear.weight.detach().clone(), loss.item(), init))
    (w_e, l_e, init), (w_g, l_g, _) = results
    # the graph's capture runs three warm-up steps first: compare against eight eager steps' trajectory instead of weights --
    # what must hold is that graph replays keep optimising from wherever they start and match eager numerics step for step
    assert (w_e - init).abs().max().item() > 1e-4 and (w_g - init).abs().max().item() > 1e-4
    assert np.isfinite(l_g) and l_g < l_e + 0.5


@pytest.mark.parametrize("n_fft,B,T,chans", [(400, 5, 16000, (0, 1)), (1024, 3, 20000, (0, 1)), (400, 4, 7777, (2, 0)), (512, 3, 9999, (0, 1)),
                                             (512, 5, 16000, (2, 1))])
def test_stft_features_pair_equals_two_launches(se, n_fft, B, T, chans):
    """se_stft_features_pair (input-channel power + log-power + CMVN sums and target-channel power in ONE launch of the
    register-resident kernels) is bit-identical to se_stft_features2 + the target channel's own launch."""
    from speech_enhancement_by_s3prl_b200 import ops
    _, mine = make_pair(se, n_fft)
    hop = mine._win_args["hop_length"]
    lengths, wavs = synth(B, T, seed=n_fft + B)
    wavs = wavs.cuda()
    window = mine._frame_window
    K, LD = n_fft // 2 + 1, ops.round4(n_fft // 2 + 1)
    ci, ct = chans
    p0, l0, s0 = ops.stft_features2(wavs, ci, n_fft, hop, window, True, True, 1e-10)
    t0 = ops.stft_padded(wavs, ct, n_fft, hop, window, logpower=False)
    p1, l1, t1, s1 = ops.stft_features_pair(wavs, ci, ct, n_fft, hop, window, 1e-10)
    torch.cuda.synchronize()
    assert p1.shape == t1.shape == l1.shape == (B, T // hop + 1, LD) and p1.is_contiguous() and t1.is_contiguous()
    assert torch.equal(p1[..., :K], p0[..., :K]) and torch.equal(l1[..., :K], l0[..., :K]) and torch.equal(t1[..., :K], t0[..., :K])
    assert torch.allclose(s1[:, :K], s0[:, :K], rtol=1e-12, atol=1e-9)           # double-precision atomics: order-dependent last bits


# ------------------------------------------------------------------------------ tensor-core head backward (tcgen05 split-K)
@pytest.mark.parametrize("B,F,Din,Dout,act,cmvn", [(3, 101, 257, 257, "Sigmoid", True), (64, 251, 257, 257, "Sigmoid", True),
                                                   (2, 300, 201, 201, "ReLU", False), (5, 64, 120, 201, "Identity", True),
                                                   (9, 40, 129, 300, "Sigmoid", True)])
def test_tensor_core_head_backward_matches_torch(se, B, F, Din, Dout, act, cmvn):
    """The backward kernel in isolation: same offset / grad_offset into the fp32 SIMT kernel, the tcgen05 kernel and torch."""
    from speech_enhancement_by_s3prl_b200 import ops
    assert ops._lib.load().se_linear_head_bwd_tc_workspace(B, F, Din, Dout) > 0
    g = torch.Generator().manual_seed(Din + F + B)
    feats = (torch.randn(B, F, Din, generator=g) * 2 - 3).cuda()
    offset = torch.rand(B, F, Dout, generator=g).cuda()
    if act == "ReLU":
        offset = (offset - 0.3).clamp_min(0.0)                                # exact zeros where the unit is off
    grad_offset = torch.randn(B, F, Dout, generator=g).cuda()
    weight = torch.randn(Dout, Din, generator=g).cuda()
    mean = std = None
    if cmvn:
        mean, std = ops.cmvn_stats(feats)
    code = ops.ACT[act]
    gw0, gb0 = torch.ops.se_b200.linear_head_bwd(feats, mean, std, 1e-6, weight, offset, grad_offset, code, 0)
    gw1, gb1 = torch.ops.se_b200.linear_head_bwd(feats, mean, std, 1e-6, weight, offset, grad_offset, code, 1)
    torch.cuda.synchronize()
    # torch reference in float64
    xh = feats.double()
    if cmvn:
        xh = (xh - mean.double()[:, None, :]) / (std.double()[:, None, :] + 1e-6)
    dz = grad_offset.double()
    if act == "Sigmoid":
        dz = dz * offset.double() * (1 - offset.double())
    elif act == "ReLU":
        dz = dz * (offset > 0).double()
    gw_ref = torch.einsum("bfn,bfk->nk", dz, xh)
    gb_ref = dz.sum((0, 1))
    sw, sb = gw_ref.abs().max().item(), gb_ref.abs().max().item()
    assert (gw0.double() - gw_ref).abs().max().item() < 2e-4 * sw             # fp32 kernel
    assert torch.isfinite(gw1).all() and torch.isfinite(gb1).all()
    # TF32 operands (2^-11 relative rounding each) in a length B*F reduction of random-sign terms
    assert (gw1.double() - gw_ref).abs().max().item() < 2e-3 * sw
    assert (gw1.double() - gw_ref).abs().mean().item() < 2e-4 * sw
    assert (gb1.double() - gb_ref).abs().max().item() < 2e-3 * sb


@pytest.mark.parametrize("B,F,Din,Dout,act,cmvn", [(3, 101, 257, 257, "Sigmoid", True), (64, 251, 257, 257, "Sigmoid", True),
                                                   (48, 1001, 201, 201, "Sigmoid", True), (256, 251, 257, 257, "ReLU", True),
                                                   (300, 40, 129, 129, "Sigmoid", True), (5, 64, 120, 201, "Identity", False),
                                                   (2, 33, 256, 256, "Sigmoid", True), (7, 95, 201, 128, "Sigmoid", True)])
def test_tma_head_backward_on_padded_operands_matches_torch(se, B, F, Din, Dout, act, cmvn):
    """se_linear_head_bwd_fused on the engine's row-padded tensors (16-byte rows: the TMA / MN-major tcgen05 kernel; NaN in the
    padding columns must not leak) against torch in float64.  Batches that need more splits than one wave of CTAs are in
    tests/test_head_gemm_f64.py."""
    from speech_enhancement_by_s3prl_b200 import ops
    assert ops.linear_head_bwd_fused_supported(B, F, Din, Dout)
    g = torch.Generator().manual_seed(Din + F + B)
    LDx, LDo = ops.round4(Din), ops.round4(Dout)
    feats = torch.full((B, F, LDx), float("nan"))
    feats[..., :Din] = torch.randn(B, F, Din, generator=g) * 2 - 3
    offset = torch.full((B, F, LDo), float("nan"))
    offset[..., :Dout] = torch.rand(B, F, Dout, generator=g)
    if act == "ReLU":
        offset[..., :Dout] = (offset[..., :Dout] - 0.3).clamp_min(0.0)
    grad = torch.full((B, F, LDo), float("nan"))
    grad[..., :Dout] = torch.randn(B, F, Dout, generator=g)
    feats, offset, grad = feats.cuda(), offset.cuda(), grad.cuda()
    sums = ops.feature_sums(feats, Din) if cmvn else None
    gw, gb = ops.linear_head_bwd_fused(feats, Din, sums, 1e-6, offset, grad, Dout, act)
    torch.cuda.synchronize()
    xh = feats[..., :Din].double()
    if cmvn:
        xh = (xh - xh.mean(1, keepdim=True)) / (xh.std(1, keepdim=True) + 1e-6)
    o, dz = offset[..., :Dout].double(), grad[..., :Dout].double()
    if act == "Sigmoid":
        dz = dz * o * (1 - o)
    elif act == "ReLU":
        dz = dz * (o > 0).double()
    gw_ref = torch.einsum("bfn,bfk->nk", dz, xh)
    gb_ref = dz.sum((0, 1))
    sw, sb = gw_ref.abs().max().item(), gb_ref.abs().max().item()
    assert gw.shape == (Dout, Din) and torch.isfinite(gw).all() and torch.isfinite(gb).all()
    assert (gw.double() - gw_ref).abs().max().item() < 2e-3 * sw
    assert (gw.double() - gw_ref).abs().mean().item() < 2e-4 * sw
    assert (gb.double() - gb_ref).abs().max().item() < 2e-3 * sb


@pytest.mark.parametrize("B,F,D,act,cmvn,hop", [(4, 101, 257, "Sigmoid", True, 256), (48, 300, 201, "Sigmoid", True, 160),
                                                (5, 64, 129, "ReLU", False, 0), (130, 40, 257, "Sigmoid", True, 128)])
def test_head_backward_with_the_objective_folded_in(se, B, F, D, act, cmvn, hop):
    """se_linear_head_bwd_sisdr (d loss / d offset rebuilt inside the TMA weight-gradient kernel) equals se_sisdr_mask_bwd followed by
    se_linear_head_bwd_fused on the same operands -- ragged lengths, padded frames, sample lengths or frame counts."""
    from speech_enhancement_by_s3prl_b200 import ops
    g = torch.Generator().manual_seed(B + F + D)
    LD = ops.round4(D)
    pad = lambda x: torch.nn.functional.pad(x, (0, LD - D), value=float("nan")).contiguous().cuda()
    feats = pad(torch.randn(B, F, D, generator=g) * 2 - 3)
    off = torch.rand(B, F, D, generator=g)
    if act == "ReLU":
        off = (off - 0.3).clamp_min(0.0)
    off, inp, tar = pad(off), pad(torch.randn(B, F, D, generator=g) ** 2), pad(torch.randn(B, F, D, generator=g) ** 2)
    frames = torch.randint(1, F + 1, (B,), generator=g)
    frames[0] = F
    lens = (((frames - 1) * hop + torch.randint(0, max(hop, 1), (B,), generator=g)) if hop else frames).cuda()
    frames = frames.cuda()
    assert ops.linear_head_bwd_sisdr_supported(B, F, D, D, LD, LD, LD, LD)
    sums = ops.feature_sums(feats, D) if cmvn else None
    loss, loss_u, g_off, sums3 = ops.sisdr_mask_step(off, inp, tar, lens, hop, D)
    gw0, gb0 = ops.linear_head_bwd_fused(feats, D, sums, 1e-6, off, g_off, D, act)
    loss1, _, none, sums3b = ops.sisdr_mask_step(off, inp, tar, lens, hop, D, want_grad=False)
    assert none is None and abs(loss.item() - loss1.item()) < 1e-6                  # (the sums are double-precision atomics: order-dependent last bits)
    assert torch.allclose(sums3, sums3b, rtol=1e-12, atol=0)
    gw1, gb1 = ops.linear_head_bwd_sisdr(feats, D, sums, 1e-6, off, inp, tar, lens, hop, sums3, D, act)
    torch.cuda.synchronize()
    assert torch.isfinite(gw1).all() and torch.isfinite(gb1).all()
    # same TF32 operands up to the last bit of the re-derived gradient: far inside the TF32 rounding of either
    sw, sb = gw0.abs().max().item(), gb0.abs().max().item()
    assert (gw1 - gw0).abs().max().item() < 2e-4 * sw and (gb1 - gb0).abs().max().item() < 2e-4 * sb
    if act == "ReLU":
        return                                   # (autograd of sqrt(relu(0)) is 0 * inf = NaN; the kernels define that gradient as 0)
    # and against float64 autograd of the reference formulas
    o64, x64, t64 = (v[..., :D].double() for v in (off, inp, tar))
    xh = feats[..., :D].double()
    if cmvn:
        xh = (xh - xh.mean(1, keepdim=True)) / (xh.std(1, keepdim=True) + 1e-6)
    o64.requires_grad_(True)
    m = (torch.arange(F, device="cuda")[None, :] < frames[:, None]).double()[..., None]
    src, tgt = (o64 * x64).clamp_min(0).sqrt() * m, t64.clamp_min(0).sqrt() * m
    al = (src * tgt).sum((1, 2)) / ((tgt ** 2).sum((1, 2)) + 1e-10)
    num = ((al[:, None, None] * tgt) ** 2).sum((1, 2))
    den = ((al[:, None, None] * tgt - src) ** 2).sum((1, 2)) + 1e-10
    l64 = (-10 * torch.log10(num / den + 1e-10)).mean()
    assert abs(l64.item() - loss.item()) < 1e-4
    l64.backward()
    dz = o64.grad
    if act == "Sigmoid":
        dz = dz * o64.detach() * (1 - o64.detach())
    elif act == "ReLU":
        dz = dz * (o64.detach() > 0).double()
    gw_ref = torch.einsum("bfn,bfk->nk", dz, xh)
    assert (gw1.double() - gw_ref).abs().max().item() < 3e-3 * gw_ref.abs().max().item()


def test_tensor_core_head_trains_like_fp32_head(se):
    """End to end through autograd: a few Adam steps with the tensor-core forward + backward track the fp32 head's loss."""
    _, mine = make_pair(se, 512)
    lengths, wavs = synth(4, 16000, seed=31)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    losses = []
    for precision in (0, 1):
        torch.manual_seed(5)
        head = se.LinearResidual(input_size=257, output_size=257, precision=precision).cuda()
        eng = se.EnhancementEngine(mine, head, log_features=True, precision=precision)
        opt = torch.optim.Adam(head.parameters(), lr=1e-3)
        for _ in range(6):
            loss = eng.train_step(lengths, wavs, se.SISDR(), opt, 1.0)
        losses.append(loss.item())
    assert losses[1] == pytest.approx(losses[0], abs=0.05)


# ------------------------------------------------------------------------------ K1 -> K3 spectrum workspace (512/256)
@pytest.mark.parametrize("B,T,ragged", [(4, 16000, False), (6, 32000, True), (64, 64000, False)])
def test_fused_training_step_matches_autograd_path(se, B, T, ragged):
    """K1(power + log-power + sums) -> TMA head -> SISDR on offset * linear_inp -> its backward -> split-K weight gradient
    against the drop-in modules under autograd (runner.py:431-460), and both against the CPU oracle's gradient at small size."""
    from speech_enhancement_by_s3prl_b200 import ops
    ora, mine = make_pair(se, 512)
    lens = torch.LongTensor([T - 997 * i for i in range(B)]) if ragged else None
    lengths, wavs = synth(B, T, seed=B + T, lengths=lens)
    lengths_d, wavs_d = lengths.cuda(), wavs.cuda()
    grads, losses = [], []
    for fused in (True, False):
        torch.manual_seed(11)
        head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
        eng = se.EnhancementEngine(mine, head, log_features=True, precision=1)
        eng.fused_training = fused
        assert eng.fused_training_supported(se.SISDR(), B, T) == fused
        opt = torch.optim.SGD(head.parameters(), lr=0.0)                      # lr 0: gradients only
        loss = eng.train_step(lengths_d, wavs_d, se.SISDR(), opt, None)
        torch.cuda.synchronize()
        grads.append((head.linear.weight.grad.clone(), head.linear.bias.grad.clone()))
        losses.append(loss.item())
    assert losses[0] == pytest.approx(losses[1], abs=2e-4)                    # TF32 head in both
    for g_f, g_a in zip(*grads):
        scale = g_a.abs().max().item()
        assert (g_f - g_a).abs().max().item() < 4e-3 * scale                  # TF32 operands on both sides, different summation
        assert (g_f - g_a).abs().mean().item() < 4e-4 * scale
    if B <= 6:
        # fp32 oracle on CPU (same weights)
        torch.manual_seed(11)
        init = se.LinearResidual(input_size=257, output_size=257)
        w = init.linear.weight.detach().clone().requires_grad_(True)
        b = init.linear.bias.detach().clone().requires_grad_(True)
        c = ora.get_feat_config
        feats, lin_i, lin_t = ora(wavs, [c("linear", 0, log=True), c("linear", 0), c("linear", 1)])
        pred, _ = sp.linear_residual_head(feats, lin_i, w, b)
        masks = sp.length_masks(sp.stft_lengths(lengths, 256))
        ref_loss, _ = sp.sisdr_spectral(pred, lin_t, masks)
        ref_loss.backward()
        assert losses[0] == pytest.approx(ref_loss.item(), abs=2e-3)
        gw = grads[0][0].cpu()
        assert torch.nn.functional.cosine_similarity(gw.flatten(), w.grad.flatten(), dim=0).item() > 0.9999
        assert (gw - w.grad).abs().max().item() < 1e-2 * w.grad.abs().max().item()


def test_sisdr_mask_kernels_match_unfused_objective(se):
    """se_sisdr_mask_fwd / _bwd (strided, float4 and scalar variants) and the dense sisdr_spec against the float64 oracle of
    objective.SISDR on predicted = offset * linear_inp."""
    from speech_enhancement_by_s3prl_b200 import ops
    B, F, K = 5, 77, 257
    g = torch.Generator().manual_seed(2)
    off = torch.rand(B, F, K, generator=g).cuda()
    inp = (torch.randn(B, F, K, generator=g) ** 2).cuda()
    tar = (torch.randn(B, F, K, generator=g) ** 2).cuda()
    inp[0, 3, 5] = 0.0                                                         # predicted == 0: zero gradient, no NaN
    frames = torch.LongTensor([77, 60, 1, 77, 33]).cuda()
    off64 = off.double().cpu().requires_grad_(True)
    _, ref_u = sp.sisdr_spectral(off64 * inp.double().cpu(), tar.double().cpu(), sp.length_masks(frames.cpu()))
    ref_u.mean().backward()
    loss_ref, g_ref = ref_u.detach(), off64.grad.cuda()
    pred = (off * inp).requires_grad_(True)                                    # the dense entry points (autograd route)
    loss_dense = ops.sisdr_spec(pred, tar, frames, 1e-10)
    loss_dense.mean().backward()
    np.testing.assert_allclose(loss_dense.detach().cpu().numpy(), loss_ref.cpu().numpy(), rtol=1e-5, atol=1e-5)
    assert (pred.grad * inp - g_ref).abs().max().item() < 1e-5 * g_ref.abs().max().item()
    for LD in (K, 260):                                                        # scalar and float4 variants
        pad = lambda x: torch.nn.functional.pad(x, (0, LD - K), value=float("nan")).contiguous()
        loss, sums3 = ops.sisdr_mask_fwd(pad(off), pad(inp), pad(tar), frames, K)
        np.testing.assert_allclose(loss.cpu().numpy(), loss_ref.cpu().numpy(), rtol=1e-5, atol=1e-5)
        go = torch.full((B,), 1.0 / B, device="cuda")
        gr = ops.sisdr_mask_bwd(pad(off), pad(inp), pad(tar), frames, K, sums3, go)
        assert gr.shape == (B, F, LD) and torch.isfinite(gr).all() and (gr[..., K:] == 0).all()
        scale = g_ref.abs().max().item()
        assert (gr[..., :K] - g_ref).abs().max().item() < 1e-5 * scale
        assert (gr[1, 60:] == 0).all() and (gr[2, 1:] == 0).all()
        loss_p, _ = ops.sisdr_mask_fwd(None, pad(off * inp), pad(tar), frames, K)   # offset = None: predicted given
        np.testing.assert_allclose(loss_p.cpu().numpy(), loss_ref.cpu().numpy(), rtol=1e-5, atol=1e-5)
        # the training step's three-launch form: frames = lengths // hop + 1 in the kernels, batch-mean loss, uniform 1 / B gradient
        hop = 160
        lens = (frames - 1) * hop + torch.LongTensor([0, 159, 7, 80, 1]).cuda()
        l_mean, l_u, g_step, _ = ops.sisdr_mask_step(pad(off), pad(inp), pad(tar), lens, hop, K)
        assert l_mean.dim() == 0 and abs(l_mean.item() - loss_ref.mean().item()) < 1e-5
        np.testing.assert_allclose(l_u.cpu().numpy(), loss.cpu().numpy(), rtol=0, atol=0)
        assert torch.equal(g_step, gr)


# ------------------------------------------------------------------------------ clip + Adam in two launches
@pytest.mark.parametrize("max_norm,wd", [(1.0, 0.0), (None, 0.0), (0.05, 0.01)])
def test_clip_adam_matches_torch_clip_and_adam(se, max_norm, wd):
    g = torch.Generator().manual_seed(3)
    shapes = [(257, 257), (257,), (3, 5, 7)]
    init = [torch.randn(*s, generator=g) for s in shapes]
    p_ref = [torch.nn.Parameter(t.clone().cuda()) for t in init]
    p_new = [torch.nn.Parameter(t.clone().cuda()) for t in init]
    o_ref = torch.optim.Adam(p_ref, lr=3e-3, betas=(0.9, 0.98), eps=1e-8, weight_decay=wd)
    o_new = se.ClipAdam(p_new, lr=3e-3, betas=(0.9, 0.98), eps=1e-8, weight_decay=wd)
    for it in range(5):
        grads = [torch.randn(*s, generator=g).cuda() * (0.1 + it) for s in shapes]
        for p, q, gr in zip(p_ref, p_new, grads):
            p.grad, q.grad = gr.clone(), gr.clone()
        if max_norm is not None:
            torch.nn.utils.clip_grad_norm_(p_ref, max_norm)
        o_ref.step()
        o_new.clip_and_step(max_norm)
        for p, q in zip(p_ref, p_new):
            assert (p.grad - q.grad).abs().max().item() <= 1e-6 * max(1.0, p.grad.abs().max().item())
            assert (p - q).abs().max().item() < 2e-6
    assert o_new.steps_taken() == [5]
    # mirrors: the update kernel keeps a row-padded, TF32-rounded copy of a 2-D parameter current (what the head kernels read)
    from speech_enhancement_by_s3prl_b200 import ops
    buf = torch.full((257, 260), 7.0, device="cuda")
    for q, gr in zip(p_new, grads):
        q.grad = gr.clone()
    o_new.clip_and_step(max_norm, mirrors={p_new[0]: buf}, mirror_tf32=True)
    assert torch.equal(buf[:, :257], ops.round_tf32(p_new[0].detach())) and (buf[:, 257:] == 7.0).all()
    buf32 = torch.zeros(257, 260, device="cuda")
    for q, gr in zip(p_new, grads):
        q.grad = gr.clone()
    o_new.clip_and_step(max_norm, mirrors={p_new[0]: buf32})
    assert torch.equal(buf32[:, :257], p_new[0].detach())
    with pytest.raises(RuntimeError):
        o_new.clip_and_step(max_norm, mirrors={p_new[1]: buf32})              # a 1-D parameter has no row-padded copy
    with pytest.raises(RuntimeError):
        cpu_p = torch.nn.Parameter(torch.zeros(3))
        cpu_p.grad = torch.ones(3)
        se.ClipAdam([cpu_p]).step()


def test_train_step_graph_with_clip_adam(se):
    """The whole training step -- fused forward / backward + ClipAdam -- replayed from a CUDA graph tracks eager torch Adam."""
    _, mine = make_pair(se, 512)
    lengths, wavs = synth(4, 16000, seed=31)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    finals = []
    for mode in ("torch-eager", "clipadam-graph"):
        torch.manual_seed(5)
        head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
        eng = se.EnhancementEngine(mine, head, log_features=True, precision=1)
        crit = se.SISDR()
        if mode == "torch-eager":
            opt = torch.optim.Adam(head.parameters(), lr=1e-3)
            for _ in range(8):
                loss = eng.train_step(lengths, wavs, crit, opt, 1.0)
        else:
            opt = se.ClipAdam(head.parameters(), lr=1e-3)
            for _ in range(5):                      # train_step_graph itself takes 3 eager warm-up steps before capturing
                loss = eng.train_step_graph(lengths, wavs, crit, opt, 1.0)
            assert opt.steps_taken() == [8]
        torch.cuda.synchronize()
        finals.append((loss.item(), head.linear.weight.detach().clone()))
    assert finals[0][0] == pytest.approx(finals[1][0], abs=0.02)
    assert (finals[0][1] - finals[1][1]).abs().max().item() < 2e-3       # 8 Adam steps of lr 1e-3: updates of ~8e-3


def test_eval_after_graph_training_uses_current_weights(se):
    """ADVICE r1 (high): the padded / TF32 weight copy the kernels read is ONE buffer refreshed in place, so evaluation --
    eager, through a cached graph captured BEFORE training, and through the host pipeline -- sees the weights that
    train_step_graph replays produced (which never bump the parameter's version)."""
    _, mine = make_pair(se, 512)
    lengths, wavs = synth(4, 16000, seed=77)
    lengths, wavs = lengths.cuda(), wavs.cuda()
    torch.manual_seed(9)
    head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
    eng = se.EnhancementEngine(mine, head, log_features=True, precision=1)
    before = eng.eval_step_graph(lengths, wavs)["sisdr"].clone()          # eval graph captured with the initial weights
    pipe = eng.host_pipeline(4, 3, 16000, depth=1)
    opt = se.ClipAdam(head.parameters(), lr=5e-3)
    for _ in range(12):
        eng.train_step_graph(lengths, wavs, se.SISDR(), opt, 1.0)
    torch.cuda.synchronize()
    fresh_head = se.LinearResidual(input_size=257, output_size=257, precision=1).cuda()
    fresh_head.load_state_dict(head.state_dict())
    want = se.EnhancementEngine(mine, fresh_head, log_features=True, precision=1).eval_step(lengths, wavs)["sisdr"]
    assert (want - before).abs().max().item() > 0.05                     # training moved the metric: the check has teeth
    got_eager = eng.eval_step(lengths, wavs)["sisdr"]
    got_graph = eng.eval_step_graph(lengths, wavs)["sisdr"]
    pipe.submit(lengths.cpu().pin_memory(), wavs.cpu().pin_memory())
    got_pipe = pipe.drain()[0][1].cuda()
    for got in (got_eager, got_graph, got_pipe):
        assert (got - want).abs().max().item() < 1e-4
    # ... and after an eager update with a torch optimizer (version bump path)
    opt2 = torch.optim.SGD(head.parameters(), lr=0.5)
    eng.train_step(lengths, wavs, se.SISDR(), opt2, 1.0)
    fresh_head.load_state_dict(head.state_dict())
    want2 = se.EnhancementEngine(mine, fresh_head, log_features=True, precision=1).eval_step(lengths, wavs)["sisdr"]
    assert (eng.eval_step_graph(lengths, wavs)["sisdr"] - want2).abs().max().item() < 1e-4


@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
def test_clip_adam_skips_nan_and_inf_gradient_norms(se, bad):
    """runner.py:467-470: a NaN / inf gradient norm skips optimizer.step(); the parameters and moments survive the batch."""
    torch.manual_seed(1)
    p = torch.nn.Parameter(torch.randn(33, 7).cuda())
    q = torch.nn.Parameter(torch.randn(5).cuda())
    opt = se.ClipAdam([p, q], lr=1e-2)
    p.grad, q.grad = torch.randn_like(p), torch.randn_like(q)
    opt.clip_and_step(1.0)
    snap = [t.detach().clone() for t in (p, q, opt.state[p]["exp_avg"], opt.state[p]["exp_avg_sq"])]
    p.grad, q.grad = torch.randn_like(p), torch.randn_like(q)
    p.grad[3, 2] = bad
    for max_norm in (1.0, None):                                         # the guard also holds without clipping
        opt.clip_and_step(max_norm)
    torch.cuda.synchronize()
    for a, b in zip(snap, (p, q, opt.state[p]["exp_avg"], opt.state[p]["exp_avg_sq"])):
        assert torch.equal(a, b.detach())
    assert opt.steps_taken() == [1] and opt.steps_skipped() == [2]
    p.grad, q.grad = torch.randn_like(p), torch.randn_like(q)            # the next healthy batch trains again
    opt.clip_and_step(1.0)
    assert opt.steps_taken() == [2] and torch.isfinite(p).all() and not torch.equal(snap[0], p.detach())
    # generic optimizers: the engine keeps the runner's host-side check
    _, mine = make_pair(se, 512)
    head = se.LinearResidual(input_size=257, output_size=257).cuda()
    eng = se.EnhancementEngine(mine, head)
    w0 = head.linear.weight.detach().clone()
    for prm in head.parameters():
        prm.grad = torch.full_like(prm, bad)
    eng._clip_and_step(torch.optim.SGD(head.parameters(), lr=0.1), 1.0)
    assert torch.equal(w0, head.linear.weight.detach())


# ------------------------------------------------------------------------------ active sampling: gradient embeddings + matching
def test_matching_matches_reference_formula(se):
    g = torch.Generator().manual_seed(9)
    for nq, nk, P in [(32, 12, 66306), (3, 5, 1000), (1, 1, 7)]:
        q = torch.randn(nq, P, generator=g).cuda() * 3
        k = torch.randn(nk, P, generator=g).cuda() * 0.1
        k[0] = 0.0                                                             # a zero gradient scores 0 (eps in the norm)
        got = se.matching(q, k)
        qn = q.double() / (q.double().pow(2).sum(-1, keepdim=True).pow(0.5) + 1e-12)      # sampler.py:113-116
        kn = k.double() / (k.double().pow(2).sum(-1, keepdim=True).pow(0.5) + 1e-12)
        ref = torch.mm(kn, qn.mean(0).unsqueeze(1)).reshape(-1)
        assert (got.double() - ref).abs().max().item() < 2e-6
        assert torch.equal(se.thresholding(got), got > 0)
    with pytest.raises(RuntimeError):
        se.matching(torch.zeros(2, 3), torch.zeros(2, 3))


@pytest.mark.parametrize("n_fft,cmvn,act", [(400, True, "Sigmoid"), (512, True, "Sigmoid"), (400, False, "ReLU")])
def test_scoring_batched_equals_per_utterance_loop(se, n_fft, cmvn, act):
    """Per-utterance gradient embeddings in one pass (se_head_grad_embeddings) against the reference's loop of backward
    calls (sampler.py:77-110) on the drop-in modules, and against the CPU oracle's autograd."""
    from speech_enhancement_by_s3prl_b200 import sampler_ops
    ora, mine = make_pair(se, n_fft)
    hop = mine._win_args["hop_length"]
    K = n_fft // 2 + 1
    B, T = 5, 12000
    lengths, wavs = synth(B, T, seed=n_fft, lengths=torch.LongTensor([12000, 9000, 12000, 5000, 11111]))
    torch.manual_seed(4)
    head = se.LinearResidual(input_size=K, output_size=K, activation=act, cmvn=cmvn).cuda()
    crit = se.SISDR()
    c = mine.get_feat_config
    feats, lin_i, lin_t = mine(wavs.cuda(), [c("linear", 0, log=True), c("linear", 0), c("linear", 1)])
    frames = lengths.cuda() // hop + 1
    assert sampler_ops._batched_ok(head, crit, feats)
    fast = sampler_ops.scoring_batched(head, crit, feats, lin_i, lin_t, frames)
    loop = sampler_ops.scoring_loop(head, crit, feats, lin_i, lin_t, frames)
    assert fast.shape == loop.shape == (B, K * K + K)
    for u in range(B):
        scale = loop[u].abs().max().item()
        assert (fast[u] - loop[u]).abs().max().item() < 2e-3 * scale          # TF32 operands in the batched kernel
        assert torch.nn.functional.cosine_similarity(fast[u], loop[u], dim=0).item() > 0.99999
    # mean=True: gradient of the batch-mean loss
    fast_m = sampler_ops.scoring_batched(head, crit, feats, lin_i, lin_t, frames, mean=True)
    loop_m = sampler_ops.scoring_loop(head, crit, feats, lin_i, lin_t, frames, mean=True)
    assert fast_m.shape == (1, K * K + K)
    assert torch.nn.functional.cosine_similarity(fast_m[0], loop_m[0], dim=0).item() > 0.99999
    # the public entry point takes the batch
    top = se.scoring(mine, head, crit, lengths.cuda(), wavs.cuda())
    assert (top - fast).abs().max().item() <= 1e-6 * fast.abs().max().item()
    # oracle (CPU autograd, fp32) for one utterance
    if cmvn and act == "Sigmoid":
        w = head.linear.weight.detach().cpu().clone().requires_grad_(True)
        b = head.linear.bias.detach().cpu().clone().requires_grad_(True)
        oc = ora.get_feat_config
        f_o, li_o, lt_o = ora(wavs[1:2], [oc("linear", 0, log=True), oc("linear", 0), oc("linear", 1)])
        pred, _ = sp.linear_residual_head(f_o, li_o, w, b)
        masks = sp.length_masks(sp.stft_lengths(lengths[1:2], hop))[:, :pred.shape[1]]
        if masks.shape[1] < pred.shape[1]:
            masks = torch.nn.functional.pad(masks, (0, pred.shape[1] - masks.shape[1]))
        ref_loss, _ = sp.sisdr_spectral(pred, lt_o, masks)
        ref_loss.backward()
        ref = torch.cat([w.grad.reshape(-1), b.grad.reshape(-1)])
        assert torch.nn.functional.cosine_similarity(fast[1].cpu(), ref, dim=0).item() > 0.9999
        # scores: the sampler's decision is the sign / ranking of the match
        s_fast = se.matching(fast[:2], fast[2:])
        s_loop = se.matching(loop[:2], loop[2:])
        assert (s_fast - s_loop).abs().max().item() < 2e-3


@pytest.mark.parametrize("n_fft,cmvn,act", [(400, True, "Sigmoid"), (512, True, "Sigmoid"), (256, False, "ReLU")])
def test_scoring_fused_pass_equals_per_utterance_loop(se, n_fft, cmvn, act):
    """se.scoring with the tensor-core head takes the engine's padded pipeline (K1 with fused log / CMVN sums, TMA head, the
    objective's backward folded into the per-utterance weight-gradient kernel): rows against the reference's loop of backward
    calls (sampler.py:77-110) on an fp32 copy of the head, ragged lengths."""
    from speech_enhancement_by_s3prl_b200 import sampler_ops
    _, mine = make_pair(se, n_fft)
    hop = mine._win_args["hop_length"]
    K = n_fft // 2 + 1
    B, T = 5, 12000
    lengths, wavs = synth(B, T, seed=n_fft + 1, lengths=torch.LongTensor([12000, 9000, 12000, 5000, 11111]))
    lengths, wavs = lengths.cuda(), wavs.cuda()
    torch.manual_seed(4)
    head32 = se.LinearResidual(input_size=K, output_size=K, activation=act, cmvn=cmvn).cuda()
    head = se.LinearResidual(input_size=K, output_size=K, activation=act, cmvn=cmvn, precision=1).cuda()
    head.load_state_dict(head32.state_dict())
    crit = se.SISDR()
    assert sampler_ops._fused_ok(mine, head, crit, B, T, True) and not sampler_ops._fused_ok(mine, head32, crit, B, T, True)
    fast = se.scoring(mine, head, crit, lengths, wavs)
    c = mine.get_feat_config
    feats, lin_i, lin_t = mine(wavs, [c("linear", 0, log=True), c("linear", 0), c("linear", 1)])
    # ReLU: a unit within TF32 rounding of its threshold switches between the fp32 and the TF32 forward, and its whole gradient row
    # with it -- compare that case against the loop on the TF32 head itself
    loop = sampler_ops.scoring_loop(head if act == "ReLU" else head32, crit, feats, lin_i, lin_t, lengths // hop + 1)
    assert fast.shape == loop.shape == (B, K * K + K) and torch.isfinite(fast).all()
    for u in range(B):
        scale = loop[u].abs().max().item()
        assert (fast[u] - loop[u]).abs().max().item() < 3e-3 * scale          # TF32 operands in the head and in the gradient kernel
        assert torch.nn.functional.cosine_similarity(fast[u], loop[u], dim=0).item() > 0.99999
    fast_m = se.scoring(mine, head, crit, lengths, wavs, mean=True)
    assert fast_m.shape == (1, K * K + K) and (fast_m[0] - fast.mean(0)).abs().max().item() <= 1e-6 * fast.abs().max().item()
    s_fast, s_loop = se.matching(fast[:2], fast[2:]), se.matching(loop[:2], loop[2:])
    assert (s_fast - s_loop).abs().max().item() < 3e-3


# ------------------------------------------------------------------------------ pseudo-wave generation (runner.py:266-305)
def test_scoring_matches_reference_sampler_golden(se, golden_dir):
    """sampler.py:59-116 pinned by the reference ITSELF: tests/golden/scoring_ref.npz holds what the unmodified
    ``sampler.scoring`` / ``sampler.matching`` returned for the reference ``model.LSTM`` + ``objective.L1`` (run_active.sh's
    combination).  The drop-in ``scoring`` (all parameters: the loop, with the projection and its input gradient on the head
    kernels), the batched projection-only path and ``matching`` must reproduce it."""
    from speech_enhancement_by_s3prl_b200 import sampler_ops
    gold = np.load(os.path.join(golden_dir, "scoring_ref.npz"))
    _, mine = make_pair(se, 400)
    lengths, wavs = torch.from_numpy(gold["lengths"]).cuda(), torch.from_numpy(gold["wavs"]).cuda()
    head = se.LSTM(input_size=201, output_size=201, hidden_size=24, num_layers=2).cuda()
    head.load_state_dict({str(n): torch.from_numpy(gold[f"param_{n}"]) for n in gold["param_names"]})
    want, want_mean = torch.from_numpy(gold["per_utt"]), torch.from_numpy(gold["mean"])
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):        # the cuDNN LSTM body in fp32
        got = se.scoring(mine, head, se.L1(), lengths, wavs).cpu()
        got_mean = se.scoring(mine, head, se.L1(), lengths, wavs, mean=True).cpu()
        proj = se.scoring(mine, head, se.L1(), lengths, wavs, projection_only=True).cpu()
    assert got.shape == want.shape and got_mean.shape == want_mean.shape
    for u in range(want.shape[0]):
        assert torch.nn.functional.cosine_similarity(got[u], want[u], dim=0).item() > 0.99999
        assert (got[u] - want[u]).abs().max().item() < 2e-3 * want[u].abs().max().item()
    assert torch.nn.functional.cosine_similarity(got_mean[0], want_mean[0], dim=0).item() > 0.99999
    n_proj = 201 * 24 + 201                                                  # scaling_layer.0.{weight, bias} come last
    assert proj.shape == (want.shape[0], n_proj)
    for u in range(want.shape[0]):
        ref_u = want[u, -n_proj:]
        assert torch.nn.functional.cosine_similarity(proj[u], ref_u, dim=0).item() > 0.99999
        assert (proj[u] - ref_u).abs().max().item() < 2e-3 * ref_u.abs().max().item()
    match = se.matching(got[:2].cuda(), got[2:].cuda()).cpu()
    np.testing.assert_allclose(match.numpy(), gold["match"], atol=2e-4)
    np.testing.assert_allclose(se.matching(want[:2].cuda(), want[2:].cuda()).cpu().numpy(), gold["match"], atol=1e-5)


@pytest.mark.parametrize("kind", ["Linear", "LSTM"])
def test_scoring_l1_batched_equals_loop_and_oracle(se, kind):
    """BASELINE configs[4] names the L1 spectral objective (run_active.sh: --downstream LSTM with the L1-trained checkpoint):
    per-utterance gradient embeddings of the projection layer in one pass against the reference's loop of backward calls
    (sampler.py:77-110) on the drop-in modules, and against the CPU oracle's autograd for one utterance."""
    from speech_enhancement_by_s3prl_b200 import sampler_ops
    ora, mine = make_pair(se, 400)
    K, B, T = 201, 5, 12000
    lengths, wavs = synth(B, T, seed=77, lengths=torch.LongTensor([12000, 9000, 12000, 5000, 11111]))
    torch.manual_seed(4)
    if kind == "Linear":
        head = se.Linear(K, K, activation="Identity").cuda()
    else:
        head = se.LSTM(input_size=K, output_size=K, hidden_size=64, num_layers=2).cuda()
    crit = se.L1()
    c = mine.get_feat_config
    feats, lin_i, lin_t = mine(wavs.cuda(), [c("linear", 0, log=True), c("linear", 0), c("linear", 1)])
    frames = lengths.cuda() // 160 + 1
    assert sampler_ops._batched_l1_ok(head, crit, feats, projection_only=True)
    assert sampler_ops._batched_l1_ok(head, crit, feats, projection_only=False) == (kind == "Linear")
    fast = sampler_ops.scoring_batched_l1(head, crit, feats, lin_t, frames)
    loop = sampler_ops.scoring_loop(head, crit, feats, lin_i, lin_t, frames, projection_only=True)
    P = (64 if kind == "LSTM" else K) * K + K
    assert fast.shape == loop.shape == (B, P)
    for u in range(B):
        assert (fast[u] - loop[u]).abs().max().item() < 2e-3 * loop[u].abs().max().item()      # TF32 operands in the batched kernel
        assert torch.nn.functional.cosine_similarity(fast[u], loop[u], dim=0).item() > 0.99999
    fast_m = sampler_ops.scoring_batched_l1(head, crit, feats, lin_t, frames, mean=True)
    loop_m = sampler_ops.scoring_loop(head, crit, feats, lin_i, lin_t, frames, mean=True, projection_only=True)
    assert fast_m.shape == (1, P) and torch.nn.functional.cosine_similarity(fast_m[0], loop_m[0], dim=0).item() > 0.99999
    top = se.scoring(mine, head, crit, lengths.cuda(), wavs.cuda(), projection_only=True)
    assert (top - fast).abs().max().item() <= 1e-6 * fast.abs().max().item()
    if kind == "LSTM":                                  # all parameters (the reference's default): the loop, LSTM layers included
        full = se.scoring(mine, head, crit, lengths[:2].cuda(), wavs[:2].cuda())
        assert full.shape == (2, sum(p.numel() for p in head.parameters()))
    else:                                               # oracle autograd (CPU, fp32) for one utterance
        w = head.linear.weight.detach().cpu().clone().requires_grad_(True)
        b = head.linear.bias.detach().cpu().clone().requires_grad_(True)
        oc = ora.get_feat_config
        f_o, lt_o = ora(wavs[1:2], [oc("linear", 0, log=True), oc("linear", 1)])
        masks = sp.length_masks(sp.stft_lengths(lengths[1:2], 160))
        masks = torch.nn.functional.pad(masks, (0, f_o.shape[1] - masks.shape[1]))
        sp.l1_logspectral(sp.linear_head(f_o, w, b, "Identity"), lt_o, masks).backward()
        ref = torch.cat([w.grad.reshape(-1), b.grad.reshape(-1)])
        assert torch.nn.functional.cosine_similarity(fast[1].cpu(), ref, dim=0).item() > 0.999


@pytest.mark.parametrize("n_fft", [512, 400, 1024])
def test_pseudo_wav_matches_decode_wav_of_the_oracle(se, n_fft):
    """_pseudo_clean / _pseudo_noise: a predicted power spectrum with the noisy phase -> waveform at -25 dB.  The fused path
    (no phase tensor) against the oracle's preprocessor.istft(linears, phase_inp) + pad + masked_normalize_decibel, on a
    zero-padded ragged batch (frames of exact zeros take the atan2(0, 0) = 0 branch)."""
    ora, mine = make_pair(se, n_fft)
    B, T = 4, 20000
    lengths, wavs = synth(B, T, seed=n_fft + 1, lengths=torch.LongTensor([20000, 15000, 9000, 20000]))
    c = ora.get_feat_config
    _, lin_i, phase_i, lin_t = ora(wavs, [c("linear", 0), c("linear", 0), c("phase", 0), c("linear", 1)])
    g = torch.Generator().manual_seed(1)
    predicted = lin_t * (0.5 + torch.rand(lin_t.shape, generator=g)) + 1e-6       # what a SpecHead (ReLU output) would emit
    ref = sp.decode_wav(ora, predicted, phase_i, lengths, target_level=-25)
    got = se.pseudo_wav(mine, predicted.cuda(), wavs.cuda(), lengths.cuda(), target_level=-25)
    assert got.shape == ref.shape
    for b in range(B):
        n = int(lengths[b])
        assert sisdr_db(got[b, :n].cpu(), ref[b, :n]) > 60.0                     # same waveform to ~1e-3 relative
        level = 10 * torch.log10(got[b, :n].pow(2).mean()).item()
        assert level == pytest.approx(-25.0, abs=1e-3)
    # the unfused drop-in sequence gives the same answer (decode_wav on K1's phase)
    feats = mine(wavs.cuda(), [mine.get_feat_config("phase", 0)])
    unfused = se.decode_wav(mine, predicted.cuda(), feats[0], lengths.cuda(), target_level=-25)
    assert (unfused - got).abs().max().item() < 2e-4 * got.abs().max().item()


# ------------------------------------------------------------------------------ BASELINE.json configs[3]: long-form utterances
@pytest.mark.parametrize("n_fft,secs", [(1024, 60.0), (512, 60.0), (400, 20.0)])
def test_long_form_eval_step_matches_oracle(se, n_fft, secs):
    """60 s utterances (960 000 samples; the reference's own length masks stop at 50 s, runner.py:32) through the fused
    evaluation step at n_fft 1024 / hop 256 -- the long-form configuration -- and the other geometries, against the oracle."""
    from speech_enhancement_by_s3prl_b200 import synth as synth_mod
    ora, mine = make_pair(se, n_fft)
    K = n_fft // 2 + 1
    lengths, wavs = synth_mod.batch(2, secs)
    T = wavs.shape[2]
    lengths = lengths.clone()
    lengths[1] = T - 12345
    wavs[1, :, T - 12345:] = 0
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=K, output_size=K).cuda()
    c = ora.get_feat_config
    ora.feat_list = [c("linear", 0, log=True), c("linear", 0, log=True), c("linear", 0), c("phase", 0), c("linear", 1), c("phase", 1)]
    with torch.no_grad():
        ref = sp.eval_step(ora, dict(weight=head.linear.weight.detach().cpu(), bias=head.linear.bias.detach().cpu()), lengths, wavs)
    for precision in (0, 1):
        eng = se.EnhancementEngine(mine, head, log_features=True, precision=precision)
        out = eng.eval_step(lengths.cuda(), wavs.cuda())
        np.testing.assert_allclose(out["sisdr"].cpu().numpy(), ref["sisdr"].numpy(), atol=SISDR_TOL_DB)
        assert out["loss_per_utt"].mean().item() == pytest.approx(ref["loss"].item(), abs=5e-3)
        for b in range(2):
            n = int(lengths[b])
            assert sisdr_db(out["wav_predicted"][b, :n].cpu(), ref["wav_predicted"][b, :n]) > 40.0
        assert out["wav_predicted"].shape == (2, T)
