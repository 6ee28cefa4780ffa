"""B200-native (sm_100a) enhancement signal path: drop-in replacements for the hot path of
leo19941227/Speech-Enhancement-by-S3PRL -- ``OnlinePreprocessor`` (STFT / features / iSTFT),
the ``Linear`` / ``LinearResidual`` mask heads, the ``SISDR`` / ``L1`` objectives,
``sisdr_eval``, ``stoi_eval`` / ``estoi_eval`` and ``masked_normalize_decibel`` -- on hand-written CUDA kernels behind the C
ABI of ``include/se_b200.h`` (``libse_b200.so``), plus the fused evaluation / training step
(``engine.EnhancementEngine``).  There is no CPU fallback: the kernels must be present.
"""
from .preprocessor import OnlinePreprocessor                      # noqa: F401
from .model import Linear, LinearResidual, LSTM, Residual          # noqa: F401
from .objective import SISDR, L1, WSD, WaveSISDR                   # noqa: F401
from .evaluation import sisdr_eval, sisdr_eval_batch, stoi_eval, estoi_eval, stoi_eval_batch  # noqa: F401
from .utils import masked_mean, masked_normalize_decibel           # noqa: F401
from .runner_ops import get_length_masks, decode_wav, pseudo_wav, stft_lengths  # noqa: F401
from .engine import EnhancementEngine                              # noqa: F401
from .optim import ClipAdam                                        # noqa: F401
from .sampler_ops import scoring, matching, thresholding           # noqa: F401

__version__ = "0.1.0"
