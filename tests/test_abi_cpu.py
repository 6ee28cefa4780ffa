"""CPU: the C-ABI library builds/loads and exports every symbol include/se_b200.h declares;
host-side logic (sharding, tile planning, drop-in module plumbing) without any GPU compute."""
import copy
import os
import pickle
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "se_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(?:int|int64_t)\s+(se_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 18
    for name in names:
        assert hasattr(lib, name), f"{name} declared in se_b200.h but not exported"
    assert set(names) == set(_lib.EXPORTS), "ctypes signature table and header disagree"
    assert lib.se_version() >= 100


def test_errors_are_reported_not_thrown():
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    rc = lib.se_stft(None, 1, 1, 1, 512, 256, None, 1e-10, None, None, None, None)
    assert rc == -1 and "null" in _lib.last_error()
    with pytest.raises(RuntimeError):
        _lib.check(rc, "se_stft")


def test_no_cpu_fallback():
    from speech_enhancement_by_s3prl_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.stft(torch.zeros(1, 1, 1000), 0, 512, 256, torch.hann_window(512))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sisdr_wave(torch.zeros(1, 100), torch.zeros(1, 100))


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "speech_enhancement_by_s3prl_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_preprocessor_module_plumbing():
    """deepcopy / .cpu() / pickle (runner.py:65, 232) and get_feat_config."""
    from speech_enhancement_by_s3prl_b200 import OnlinePreprocessor
    pre = OnlinePreprocessor(sample_rate=16000, win_ms=25, hop_ms=10, n_freq=201, n_mels=40, n_mfcc=13,
                             roots=["x"], max_time=10000, target_level=-25, noise_proportion=0.5, snrs=[3])
    assert pre._win_args == {"n_fft": 400, "hop_length": 160, "win_length": 400}
    assert pre._sample_rate == 16000 and pre._window.shape == (400,)
    clone = pickle.loads(pickle.dumps(copy.deepcopy(pre).cpu()))
    assert clone._win_args == pre._win_args
    cfg = OnlinePreprocessor.get_feat_config("linear", 1, log=True)
    assert cfg == {"feat_type": "linear", "channel": 1, "log": True, "delta": 0, "cmvn": False}
    pre.channel_inp, pre.channel_tar = 0, 1
    with pytest.raises(ValueError):
        OnlinePreprocessor(n_freq=300)


def test_heads_keep_reference_construction_contract():
    """eval(args.downstream)(input_size=, output_size=, **all_cli_args) -- run_downstream.py:208-210."""
    from speech_enhancement_by_s3prl_b200 import Linear, LinearResidual, LSTM, Residual
    junk = dict(gpu=True, seed=1337, objective="SISDR", n_jobs=4)
    torch.manual_seed(1337)
    h = LinearResidual(input_size=257, output_size=257, cmvn=True, **junk)
    torch.manual_seed(1337)
    ref = torch.nn.Linear(257, 257)
    assert torch.equal(h.linear.weight, ref.weight)             # same init stream as the reference head
    assert set(h.state_dict()) == {"linear.weight", "linear.bias"}
    assert set(Linear(40, 201, activation="ReLU").state_dict()) == {"linear.weight", "linear.bias"}
    lstm = LSTM(input_size=201, output_size=201, hidden_size=32, num_layers=2, activation="ReLU", **junk)
    assert "scaling_layer.0.weight" in lstm.state_dict() and "lstm.weight_hh_l1" in lstm.state_dict()
    res = Residual(input_size=201, output_size=201, hidden_size=32, num_layers=1, bidirectional=True, cmvn=True)
    assert res.scaling_layer[0].in_features == 64


def test_shard_bounds_partition_the_batch():
    from speech_enhancement_by_s3prl_b200 import dp
    for n in (1, 7, 64, 1024):
        for w in (1, 2, 3, 8):
            spans = [dp.shard_bounds(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_launch_planning_is_host_logic():
    """The `_supported` / `_workspace` entry points are pure host planning (148 SMs assumed without a device): the shapes of the
    BASELINE configs are inside the fast paths, the stated limits are enforced, and the workspaces have the documented sizes."""
    from speech_enhancement_by_s3prl_b200 import _lib
    lib = _lib.load()
    # TMA / tcgen05 head: configs[1] (257), configs[2] (201, mel 120 -> 201), configs[3] (513); rows must be 16-byte multiples
    for B, F, Din, Dout in [(64, 251, 257, 257), (48, 1001, 201, 201), (48, 1001, 120, 201), (128, 3751, 513, 513)]:
        r4 = lambda v: (v + 3) // 4 * 4
        assert lib.se_linear_head_fused_supported(B, F, Din, Dout, r4(Din), r4(Din), r4(Dout)) == 1
    assert lib.se_linear_head_fused_supported(64, 251, 257, 257, 257, 260, 260) == 0          # ldx not a multiple of 4 floats
    assert lib.se_linear_head_fused_supported(64, 251, 600, 257, 600, 600, 260) == 0          # more than 544 input features
    assert lib.se_linear_head_fused_supported(64, 4, 257, 257, 260, 260, 260) == 0            # fewer than 8 frames
    # split-K weight gradient: one wave of (row split, 128-row output tile) CTAs, partials (splits, m_rows, 272)
    def splits(R, per_wave):                                                                   # rows per split: a multiple of 32
        rows = -(-(-(-R // per_wave)) // 32) * 32
        return -(-R // rows)
    assert lib.se_linear_head_bwd_tc_workspace(64, 251, 257, 257) == splits(64 * 251, 74) * 257 * 272   # 2 tiles + 1 leftover row
    assert lib.se_linear_head_bwd_tc_workspace(48, 1001, 201, 201) == splits(48 * 1001, 74) * 256 * 272
    assert lib.se_linear_head_bwd_tc_workspace(1024, 251, 257, 257) > 0                        # large batches: more splits than one wave
    assert lib.se_linear_head_bwd_tc_workspace(64, 16, 257, 257) == 0                          # utterances shorter than one 32-row block
    assert lib.se_linear_head_bwd_tc_workspace(64, 251, 513, 513) == 0                         # D_in + 1 > 272 columns of tensor memory
    # per-utterance gradients (sampler.py:95-108): one split per utterance, up to four while the grid stays below one wave
    assert lib.se_head_grad_embeddings_workspace(44, 1001, 201, 201) == 44 * 256 * 272
    assert lib.se_head_grad_embeddings_workspace(12, 1001, 201, 201) == 12 * 4 * 256 * 272
    # the objective folded into the weight gradient needs TMA-able (16-byte) rows
    assert lib.se_linear_head_bwd_sisdr_supported(48, 1001, 201, 201, 204, 204, 204, 204) == 1
    assert lib.se_linear_head_bwd_sisdr_supported(48, 1001, 201, 201, 201, 204, 204, 204) == 0
    assert lib.se_head_grad_embeddings_sisdr_supported(44, 1001, 201, 201, 204, 204, 204, 204) == 1
    # one K1 launch for both channels exists for the register-resident geometries of fastgeo.cu only
    assert lib.se_stft_features_pair_supported(400, 160) == 1 and lib.se_stft_features_pair_supported(1024, 256) == 1
    assert lib.se_stft_features_pair_supported(512, 256) == 1 and lib.se_stft_features_pair_supported(400, 200) == 0
