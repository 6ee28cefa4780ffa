"""Drop-in metrics (reference evaluation.py) plus their batched device forms.

The reference evaluates its metrics one utterance at a time on CPU slices through joblib
(runner.py:587-602).  ``sisdr_eval(src, tar)``, ``stoi_eval`` and ``estoi_eval`` keep that
signature (1-D tensors, returns a Python float) but compute on the GPU; the ``*_batch`` forms
do the whole batch at once and are what the fused evaluation step uses.
"""
import torch

from . import ops


def sisdr_eval_batch(src, tar, lengths=None, eps=1e-10):
    """src, tar: (B, T) CUDA tensors, lengths (B,) int64 -> (B,) SI-SDR in dB."""
    return ops.sisdr_wave(src, tar, lengths, eps)


def sisdr_eval(src, tar, sr=16000, eps=1e-10):
    if not torch.cuda.is_available():
        raise RuntimeError("se_b200.sisdr_eval needs a CUDA device (no CPU fallback)")
    dev = src.device if src.is_cuda else torch.device("cuda", torch.cuda.current_device())
    s = src.reshape(1, -1).to(dev, torch.float32).contiguous()
    t = tar.reshape(1, -1).to(dev, torch.float32).contiguous()
    return ops.sisdr_wave(s, t, None, eps).item()


def _row(t, dev):
    return t.reshape(1, -1).to(dev, torch.float32).contiguous()


def stoi_eval_batch(src, tar, lengths=None, sr=16000, acc=None):
    """src (estimate), tar (clean reference): (B, T) CUDA tensors, lengths (B,) int64 -> (stoi, estoi), each (B,) fp32.
    acc: float64 (3,) device tensor += [sum STOI, sum ESTOI, B]."""
    return ops.stoi(src, tar, lengths, fs=sr, acc=acc)


def _one(src, tar, sr, extended):
    if not torch.cuda.is_available():
        raise RuntimeError("se_b200.stoi_eval needs a CUDA device (no CPU fallback)")
    dev = src.device if src.is_cuda else torch.device("cuda", torch.cuda.current_device())
    s, e = ops.stoi(_row(src, dev), _row(tar, dev), None, fs=sr, want_stoi=not extended, want_estoi=extended)
    return (e if extended else s).item()


def stoi_eval(src, tar, sr=16000):
    """pystoi.stoi(tar, src, sr): src is the estimate and tar the clean reference, which is pystoi's first argument."""
    return _one(src, tar, sr, False)


def estoi_eval(src, tar, sr=16000):
    """pystoi.stoi(tar, src, sr, extended=True): src is the estimate and tar the clean reference (pystoi's x)."""
    return _one(src, tar, sr, True)
