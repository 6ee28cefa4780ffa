"""The fused evaluation step's workspace: ONE float64 vector [stat_sums (B, round4(K), 2) | sums (B, 6) | criterion state]
laid out by ops.step_workspace_views, the predicate of the register-resident kernels, the library's check that a self-cleaning
K1 call matches that layout, and that every captured route leaves the whole workspace zeroed for its next replay."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_parity import synth  # noqa: E402

gpu = pytest.mark.gpu
SE_OPT_FORCE_GENERIC, SE_ERR_BAD_ARG = 0, -1
FAST = ((512, 256), (1024, 256), (400, 160))


# ------------------------------------------------------------------------------ CPU: the layout
@pytest.mark.parametrize("B,n_fft", [(1, 512), (3, 400), (4, 1024), (7, 256), (2, 2048)])
def test_workspace_views_tile_the_buffer(B, n_fft):
    from speech_enhancement_by_s3prl_b200 import ops
    K = n_fft // 2 + 1
    LD = (K + 3) // 4 * 4
    for crit, extra in (("sisdr", 0), ("wsd", 1), ("l1", 2)):
        n = ops.step_workspace_doubles(B, n_fft, crit)
        assert n == B * (2 * LD + 6) + extra
        ws = torch.arange(n, dtype=torch.float64)
        stat_sums, sums, state = ops.step_workspace_views(ws, B, n_fft)
        assert stat_sums.shape == (B, LD, 2) and sums.shape == (B, 6) and state.shape == (extra,)
        assert all(v.dtype == torch.float64 and v.is_contiguous() for v in (stat_sums, sums, state))
        assert stat_sums.storage_offset() == 0
        assert sums.storage_offset() == B * 2 * LD
        assert state.storage_offset() == B * (2 * LD + 6)
        # no gap, no overlap: the views laid end to end are the buffer
        assert torch.equal(torch.cat([stat_sums.reshape(-1), sums.reshape(-1), state]), ws)
        for v in (stat_sums, sums, state):
            assert v.untyped_storage().data_ptr() == ws.untyped_storage().data_ptr()


def test_workspace_views_refuse_other_buffers():
    from speech_enhancement_by_s3prl_b200 import ops
    n = ops.step_workspace_doubles(2, 512)
    for bad in (torch.zeros(n + 3, dtype=torch.float64), torch.zeros(n - 1, dtype=torch.float64), torch.zeros(n),
                torch.zeros(2 * n, dtype=torch.float64)[::2]):
        with pytest.raises(AssertionError):
            ops.step_workspace_views(bad, 2, 512)


# ------------------------------------------------------------------------------ CPU: one predicate for the fast path
def test_register_resident_predicates_agree():
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    lib = _lib.load()
    exports = (lib.se_stft_features_pair_supported, lib.se_mask_istft_wsd_supported, lib.se_mask_istft_l1_supported)
    table = [(n_fft, hop) for n_fft in (256, 400, 512, 1024, 2048) for hop in (64, 128, 160, 200, 256, 512)]
    try:
        for force in (0, 1):
            assert lib.se_set_option(SE_OPT_FORCE_GENERIC, force) == 0
            for n_fft, hop in table:
                want = int(not force and (n_fft, hop) in FAST)
                assert [f(n_fft, hop) for f in exports] == [want] * 3, (force, n_fft, hop)
                # K3's register-resident kernel also needs six frames
                assert ops.mask_istft_register_resident(n_fft, hop, 5 * hop) == bool(want)
                assert not ops.mask_istft_register_resident(n_fft, hop, 5 * hop - 1)
    finally:
        lib.se_set_option(SE_OPT_FORCE_GENERIC, 0)


# ------------------------------------------------------------------------------ GPU: the library checks the layout
@gpu
@pytest.mark.parametrize("n_fft,hop", [(512, 256), (512, 128)])
def test_self_clean_needs_the_workspace_layout(n_fft, hop):
    """A self-cleaning K1 zeroes the K3 sums right after the statistics; with rows of the statistics wider than round4(K) it
    would look for them elsewhere than K3 does, so the call is refused and touches nothing.  The buffer holds either reading
    of the layout."""
    from speech_enhancement_by_s3prl_b200 import _lib, ops
    lib = _lib.load()
    B, T = 3, 16000
    K, F = n_fft // 2 + 1, T // hop + 1
    LD = ops.round4(K)
    wavs = synth(B, T, seed=3)[1].cuda()
    window = torch.hann_window(n_fft, device="cuda")
    feat = torch.empty(B, F, LD, device="cuda")
    flags = ops.FLAG_SUMS_ZEROED | ops.FLAG_WS_SELF_CLEAN
    st = torch.cuda.current_stream().cuda_stream
    for ld_stats, rc_want in ((LD + 4, SE_ERR_BAD_ARG), (LD, 0)):
        buf = torch.full((B * (2 * ld_stats + 6),), 7.0, device="cuda", dtype=torch.float64)
        stat_sums, sums = buf[:B * 2 * ld_stats], buf[B * 2 * ld_stats:]
        stat_sums.zero_()
        rc = lib.se_stft_features(wavs.data_ptr(), B, wavs.shape[1] * T, T, n_fft, hop, window.data_ptr(), 1e-10, 1, feat.data_ptr(),
                                  LD, buf.data_ptr(), ld_stats, flags, st)
        torch.cuda.synchronize()
        assert rc == rc_want, _lib.last_error()
        if rc_want:
            assert "ld_stats" in _lib.last_error()
            assert torch.all(stat_sums == 0) and torch.all(sums == 7.0)          # untouched
        else:
            assert torch.all(sums == 0) and torch.any(stat_sums != 0)           # K3's sums cleaned, the statistics written


# ------------------------------------------------------------------------------ GPU: every route leaves the workspace zeroed
def _engine(se, head_kind):
    pre = se.OnlinePreprocessor(win_ms=32, hop_ms=16, n_freq=257).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(7)
    if head_kind == "LinearResidual":
        head = se.LinearResidual(input_size=257, output_size=257, activation="Sigmoid", precision=1)
    elif head_kind == "LSTM":
        head = se.LSTM(input_size=257, output_size=257, hidden_size=32, num_layers=2, activation="Identity", precision=1)
    else:
        head = se.Residual(input_size=257, output_size=257, hidden_size=32, num_layers=2, activation="Sigmoid", precision=1)
    return se.EnhancementEngine(pre, head.cuda().eval(), log_features=True, precision=1)


@gpu
@pytest.mark.parametrize("head_kind,crit", [("LinearResidual", "SISDR"), ("LinearResidual", "WSD"), ("LSTM", "L1"),
                                            ("Residual", "WSD")])
def test_steps_leave_the_workspace_clean(head_kind, crit):
    """After every eager step and every replay the statistics and the criterion's state are zero again.  The K3 sums are what
    K3' read; the next step's K1 zeroes them before its K3 adds to them, so every step finds them clean: they repeat instead of
    accumulating."""
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import ops
    eng = _engine(se, head_kind)
    criterion = getattr(se, crit)()
    B, T = 4, 16000
    lengths, wavs = synth(B, T, seed=11, lengths=torch.LongTensor([T - 1777 * i for i in range(B)]))
    lengths, wavs = lengths.cuda(), wavs.cuda()

    def check(ws, step, first):
        torch.cuda.synchronize()
        stat_sums, sums, state = ops.step_workspace_views(ws, B, eng.n_fft)
        assert torch.count_nonzero(stat_sums).item() == 0 and torch.count_nonzero(state).item() == 0
        assert torch.isfinite(step["loss_per_utt"]).all()
        if first:
            torch.testing.assert_close(sums, first[0], rtol=1e-9, atol=0)
            torch.testing.assert_close(step["loss_per_utt"], first[1], rtol=1e-6, atol=0)
        else:
            first += [sums.clone(), step["loss_per_utt"].clone()]

    ws, first = eng.step_workspace(B, wavs.device, criterion), []
    for _ in range(3):
        check(ws, eng.eval_step(lengths, wavs, ws=ws, criterion=criterion), first)
    st = eng.capture_bound(lengths, wavs, criterion=criterion)
    assert st["ws"].numel() == ws.numel()
    for _ in range(3):
        st["graph"].replay()
        check(st["ws"], st, first)
