"""acoustic_echo_cancellation_b200 -- B200-native stage-1 linear echo canceller.

Host side of the drop-in for the data-parallel hot path of
SZU-Speech/Acoustic-Echo-Cancellation (STFT -> partitioned FDAF -> iSTFT -> feature
output).  Importing the package does not load CUDA; the first call into
``libaec_b200.so`` does, and raises if the library has not been built -- there is no
CPU fallback.  See DESIGN.md / INTEGRATION.md.
"""
from ._lib import ALGO_KALMAN, ALGO_NLMS, ALGO_PBFDAF, ALGO_PBFKF, AecError, LIB_PATH  # noqa: F401
from .stage1 import (HOST_PORTABLE, HOST_WRITE_COMBINED, DelayConfig, HostPipeline, Stage1Config,  # noqa: F401
                     Stage1Stream, align_far, estimate_delay, fp32_peak_tflops, is_pinned, launch_count, num_frames, out_samples,
                     pinned_empty, stage1_aec, stage1_aec_features)
from .spectral import ConvSTFT, ConviSTFT, batch_shift, erb_filterbank, stage2_features  # noqa: F401
from .stage2 import AecStream, LittleNetInference, Stage2Stream  # noqa: F401

__all__ = [
    "ALGO_KALMAN", "ALGO_NLMS", "ALGO_PBFDAF", "ALGO_PBFKF", "AecError", "LIB_PATH", "HostPipeline", "Stage1Config", "fp32_peak_tflops",
    "launch_count", "num_frames", "out_samples", "pinned_empty", "is_pinned", "HOST_WRITE_COMBINED",
    "HOST_PORTABLE", "stage1_aec", "stage1_aec_features", "ConvSTFT", "ConviSTFT",
    "erb_filterbank", "stage2_features", "batch_shift", "LittleNetInference", "DelayConfig", "estimate_delay",
    "align_far", "Stage1Stream", "Stage2Stream", "AecStream",
]
