"""GPU (-m gpu): bench.py --dump-outputs writes what the last timed step of the headline pass returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_last_timed_step(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    steps, ring = 3, 8
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                          "--ring", str(ring), "--skip-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         cwd=ROOT, capture_output=True, text=True)
    assert run.returncode == 0, run.stderr[-4000:]
    line = json.loads(run.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps

    arrays = {fn[:-4]: np.load(tmp_path / fn) for fn in os.listdir(tmp_path)}
    assert set(arrays) == {"loss_per_utt", "sisdr", "gain", "wav_predicted", "mask", "pass_sums"}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    sums = arrays.pop("pass_sums")
    assert sums.dtype == np.float64
    B, T, F, K = 64, 64000, 251, 257
    assert arrays["wav_predicted"].shape == (B, T) and arrays["mask"].shape == (B, F, K)
    for name in ("loss_per_utt", "sisdr", "gain"):
        assert arrays[name].shape == (B,)
    for a in arrays.values():
        assert a.dtype == np.float32 and np.isfinite(a).all()
    assert sums[2] == steps * B
    dp = line["check"]["device_pass"]
    np.testing.assert_allclose(sums[:2] / sums[2], [dp["mean_loss"], dp["mean_sisdr_db"]], rtol=1e-12)

    # the last of `steps` steps ran ring slot (steps - 1) % ring: rank 0's host batch of that index, on the same head
    import speech_enhancement_by_s3prl_b200 as se
    from speech_enhancement_by_s3prl_b200 import synth
    sys.path.insert(0, ROOT)
    import bench
    slot = (steps - 1) % ring
    assert slot < 4                                   # the first four slots are host batches, not shifted copies
    lengths, wavs = synth.batch(B, bench.SECONDS, first_index=slot * B)
    pre = se.OnlinePreprocessor(**bench.PRE_KW).cuda()
    pre.channel_inp, pre.channel_tar = 0, 1
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=K, output_size=K).cuda()
    out = se.EnhancementEngine(pre, head, log_features=True, precision=1).eval_step(lengths.cuda(), wavs.cuda())
    np.testing.assert_allclose(arrays["sisdr"], out["sisdr"].cpu().numpy(), atol=1e-3)
    np.testing.assert_allclose(arrays["loss_per_utt"], out["loss_per_utt"].cpu().numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(arrays["wav_predicted"], out["wav_predicted"].cpu().numpy(), atol=1e-5)
