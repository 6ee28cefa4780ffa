"""Drop-in objectives (reference objective.py).  Instantiated by name with the config block
(``eval(f'{args.objective}(**cfg)')`` runner.py:83) and called with every local variable of
the training step as keyword arguments (runner.py:458, 575; sampler.py:90), so each
``forward`` names what it consumes and swallows the rest in ``**kwargs``.

Instead of the (B, F) int64 ``stft_length_masks`` the kernels take per-utterance frame
counts; they are recovered from the masks (prefix masks, runner.py:216-220) or passed
directly as ``stft_lengths`` by callers that have them.
"""
import torch
import torch.nn as nn

from . import ops


def _frames(stft_length_masks=None, stft_lengths=None):
    if stft_lengths is not None:
        return stft_lengths.to(torch.int64)
    return stft_length_masks.sum(dim=-1).to(torch.int64)


class SISDR(nn.Module):
    """objective.py:81-100 -- SI-SDR between spectral magnitudes sqrt(relu(power)); mean over the batch."""

    def __init__(self, eps=1e-10, **kwargs):
        super().__init__()
        self.eps = eps

    def forward(self, predicted, linear_tar, stft_length_masks=None, stft_lengths=None, **kwargs):
        per_utt = ops.sisdr_spec(predicted, linear_tar, _frames(stft_length_masks, stft_lengths), self.eps)
        return per_utt.mean(), {}


class L1(nn.Module):
    """objective.py:103-117 -- mean |log_predicted - log(linear_tar + eps)| over the valid elements of the batch."""

    def __init__(self, eps=1e-10, **kwargs):
        super().__init__()
        self.eps = eps

    def forward(self, log_predicted, linear_tar, stft_length_masks=None, stft_lengths=None, **kwargs):
        acc = ops.l1_logspec_sums(log_predicted, linear_tar, _frames(stft_length_masks, stft_lengths), self.eps)
        return (acc[0] / acc[1]).to(torch.float32), {}


class WSD(nn.Module):
    """objective.py:120-153 -- weighted speech distortion: alpha * speech distortion on voiced frames + (1 - alpha) *
    residual noise, both summed per utterance over valid frames and averaged over the batch.  Fused forward and
    backward (w.r.t. ``offset``); ``linear_inp`` / ``linear_tar`` are data and get no gradient, as in the reference's use.
    The voicing threshold comes from the loudest frame of the whole batch, all-reduced across data-parallel ranks
    (``dp.global_max``): while a process group of world size > 1 is initialized, every rank must call it for every batch."""

    def __init__(self, alpha=0.5, db_interval=30, eps=1e-10, **kwargs):
        super().__init__()
        self.alpha, self.db_interval, self.eps = alpha, db_interval, eps

    def forward(self, linear_inp, offset, linear_tar, stft_length_masks=None, stft_lengths=None, **kwargs):
        loss = ops.wsd(linear_inp, offset, linear_tar, _frames(stft_length_masks, stft_lengths), self.alpha, self.db_interval,
                       self.eps)
        return loss, {}
