"""Gradient clipping + Adam for the mask head in two launches (runner.py:463-466).

The reference clips with ``torch.nn.utils.clip_grad_norm_`` and steps a torch / BertAdam optimizer
(runner.py:114-115, 463-466): about fifteen small launches for two small tensors, which is most of a
training step once forward and backward are fused.  ``ClipAdam`` keeps ``torch.optim.Adam``'s update
rule (L2 ``weight_decay``, bias correction, no amsgrad) and state names, and adds
``clip_and_step(max_norm)``; all of its state is on the device, so the step replays from a CUDA graph.  A step whose
gradient norm is NaN / inf is skipped on the device, as the runner does on the host (runner.py:467-470).
"""
import ctypes

import torch

from . import _lib

_MAX_TENSORS = 32          # per parameter group (se_adam_clip_step_mirror): e.g. a bidirectional 3-layer LSTM head + projection, 26


class ClipAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def _group_state(self, group):
        ps = [p for p in group["params"] if p.grad is not None]
        if not ps:
            return ps, None
        if len(ps) > _MAX_TENSORS:
            raise RuntimeError(f"ClipAdam handles at most {_MAX_TENSORS} tensors per parameter group")
        for p in ps:
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and p.grad.is_contiguous()):
                raise RuntimeError("ClipAdam needs contiguous fp32 CUDA parameters and gradients (there is no CPU fallback)")
            st = self.state[p]
            if not st:
                st["exp_avg"] = torch.zeros_like(p)
                st["exp_avg_sq"] = torch.zeros_like(p)
        ws = group.get("_ws")
        if ws is None or ws[0].device != ps[0].device:
            ws = (torch.zeros(1, device=ps[0].device, dtype=torch.float64), torch.zeros(3, device=ps[0].device, dtype=torch.int32))
            group["_ws"] = ws
        return ps, ws

    @torch.no_grad()
    def clip_and_step(self, max_norm=None, mirrors=None, mirror_tf32=False):
        """``clip_grad_norm_(params, max_norm)`` (skipped for None / <= 0) followed by ``Adam.step()``, per parameter group.
        mirrors: {parameter: (rows, LD) fp32 buffer} -- the update kernel also writes the new value of a 2-D parameter
        (rows, cols <= LD) into its row-padded buffer, rounded to TF32 if ``mirror_tf32`` (the copy the TMA / tensor-core head
        reads: it follows the parameters inside the same launch instead of three more)."""
        lib = _lib.load()
        for group in self.param_groups:
            ps, ws = self._group_state(group)
            if not ps:
                continue
            n = len(ps)
            arr = ctypes.c_void_p * n
            sizes = (ctypes.c_int64 * n)(*[p.numel() for p in ps])
            mir = [None] * n
            if mirrors:
                for i, p in enumerate(ps):
                    buf = next((b for q, b in mirrors.items() if q is p), None)
                    if buf is not None:
                        if p.dim() != 2 or buf.dim() != 2 or buf.shape[0] != p.shape[0] or buf.shape[1] < p.shape[1] or \
                                buf.dtype != torch.float32 or buf.device != p.device or buf.stride(1) != 1:
                            raise RuntimeError("ClipAdam: a mirror must be a (rows, LD >= cols) fp32 buffer on the parameter's device")
                        mir[i] = buf
            cols = (ctypes.c_int64 * n)(*[(p.shape[1] if mir[i] is not None else 0) for i, p in enumerate(ps)])
            lds = (ctypes.c_int64 * n)(*[(mir[i].stride(0) if mir[i] is not None else 0) for i in range(n)])
            with torch.cuda.device(ps[0].device):
                rc = lib.se_adam_clip_step_mirror(arr(*[p.data_ptr() for p in ps]), arr(*[p.grad.data_ptr() for p in ps]),
                                                  arr(*[self.state[p]["exp_avg"].data_ptr() for p in ps]),
                                                  arr(*[self.state[p]["exp_avg_sq"].data_ptr() for p in ps]), sizes, n,
                                                  float(group["lr"]), float(group["betas"][0]), float(group["betas"][1]),
                                                  float(group["eps"]), float(group["weight_decay"]),
                                                  float(max_norm) if max_norm is not None else 0.0,
                                                  arr(*[(b.data_ptr() if b is not None else None) for b in mir]), cols, lds,
                                                  1 if mirror_tf32 else 0, ws[0].data_ptr(), ws[1].data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "se_adam_clip_step_mirror")
            for p in ps:                            # the kernel wrote through raw pointers: let version-keyed caches see it
                torch.autograd.graph.increment_version(p)
                torch.autograd.graph.increment_version(p.grad)

    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self.clip_and_step(None)
        return loss

    def steps_skipped(self):
        """Steps whose gradient norm was NaN / inf and that therefore left the parameters untouched (runner.py:467-470)."""
        return [int(g["_ws"][1][2].item()) if g.get("_ws") is not None else 0 for g in self.param_groups]

    def steps_taken(self):
        """Device-side step counts, one per parameter group (synchronises)."""
        return [int(g["_ws"][1][0].item()) if g.get("_ws") is not None else 0 for g in self.param_groups]
