"""adapted_b200 -- B200-native (sm_100a) boundary-detection hot path, drop-in for KleistLab/ADAPTed v0.2.4.

Host code is python over a C-ABI CUDA library (``include/adapted_b200.h``); see DESIGN.md.
"""
from .config import SigProcConfig, get_chemistry_specific_config, load_config, start_peak_config  # noqa: F401
from .records import DetectResults, ReadResult  # noqa: F401

__version__ = "0.1.0"


def __getattr__(name):
    # the detectors need the CUDA library; import them lazily so that config / records stay usable for tooling
    if name in ("combined_detect_llr2", "combined_detect_cnn", "combined_detect_start_peak", "detect_reads",
                "c_llr_trace", "c_llr_trace_batch", "global_med_mad", "downscale_signal"):
        from . import detect

        return getattr(detect, name)
    if name == "StreamSession":
        from .stream import StreamSession

        return StreamSession
    raise AttributeError(name)
