"""ctypes binding of libadapted_b200.so (include/adapted_b200.h).

The library is the product: if it is missing or no CUDA device is present every compute call raises --
there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any, Dict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# ADB_LIB_PATH: load another build of the same library (A/B runs of kernel variants)
SO_PATH = os.environ.get("ADB_LIB_PATH") or os.path.join(HERE, "csrc", "libadapted_b200.so")

ADB_MAX_CAND = 16
ADB_MAX_OPEN_PORES = 48
SIG_F32, SIG_I16 = 0, 1
CNN_NPARAMS = 58882

STATUS_TEXT = {
    0: "ok", -1: "CUDA error", -2: "invalid argument", -3: "MAD normalization failed: scale is 0",
    -4: "attempt to get argmin of an empty sequence", -5: "unsupported configuration",
    -6: "open-pore list longer than the record keeps and no overflow row supplied",
}

D2 = C.c_double * 2


class AdbConfig(C.Structure):
    _fields_ = [
        ("max_obs_trace", C.c_int32), ("min_obs_adapter", C.c_int32), ("max_obs_adapter", C.c_int32),
        ("min_obs_polya", C.c_int32), ("downscale_factor", C.c_int32), ("primary_method", C.c_int32),
        ("sig_norm_outlier_thresh", C.c_double),
        ("adapter_peak_prominence", C.c_double), ("adapter_peak_rel_height", C.c_double),
        ("adapter_peak_width", C.c_int32),
        ("polya_cand_k", C.c_int32), ("fallback_to_llr_short_reads", C.c_int32),
        ("mvs_detect_check", C.c_int32), ("mvs_detect_overwrite", C.c_int32), ("search_window", C.c_int32),
        ("pA_mean_window", C.c_int32), ("pA_var_window", C.c_int32), ("median_shift_window", C.c_int32),
        ("polyA_window", C.c_int32), ("pA_mean_range_empty", C.c_int32), ("pA_mean_scale_range_empty", C.c_int32),
        ("pA_mean_range", D2), ("pA_var_range", D2), ("median_shift_range", D2), ("polyA_med_range", D2),
        ("polyA_local_range", D2), ("pA_mean_scale_range", D2),
        ("detect_open_pores", C.c_int32), ("real_signal_check", C.c_int32), ("mean_window", C.c_int32),
        ("max_obs_local_range", C.c_int32),
        ("mean_start_range", D2), ("mean_end_range", D2), ("local_range", D2), ("adapter_mad_range", D2),
        ("detect_med_shift", C.c_int32), ("med_shift_window", C.c_int32), ("med_shift_range", D2),
        ("sp_downscale_factor", C.c_int32), ("start_peak_max_idx", C.c_int32), ("sp_offset1", C.c_int32),
        ("sp_offset2", C.c_int32), ("open_pore_pa", C.c_double),
        ("sig_preload_size", C.c_int32), ("_pad", C.c_int32),
    ]


class AdbStreamConfig(C.Structure):
    _fields_ = [
        ("min_obs_adapter", C.c_int32), ("min_obs_post_loc", C.c_int32), ("search_increment_step", C.c_int32),
        ("pA_mean_window", C.c_int32), ("pA_var_window", C.c_int32), ("median_shift_window", C.c_int32),
        ("polyA_window", C.c_int32), ("_pad", C.c_int32),
        ("pA_mean_range", D2), ("pA_var_range", D2), ("median_shift_range", D2), ("polyA_med_range", D2),
        ("polyA_local_range", D2),
    ]


class AdbBatch(C.Structure):
    _fields_ = [
        ("signal", C.c_void_p), ("sig_type", C.c_int32), ("n_reads", C.c_int32), ("m", C.c_int32),
        ("batch_size", C.c_int32), ("offsets", C.c_void_p), ("full_lens", C.c_void_p),
        ("calib_offset", C.c_void_p), ("calib_scale", C.c_void_p),
    ]


class AdbSvbBatch(C.Structure):
    _fields_ = [
        ("comp", C.c_void_p), ("comp_offsets", C.c_void_p), ("n_samples", C.c_void_p),
        ("n_reads", C.c_int32), ("m", C.c_int32), ("batch_size", C.c_int32), ("_pad", C.c_int32),
        ("full_lens", C.c_void_p), ("calib_offset", C.c_void_p), ("calib_scale", C.c_void_p),
    ]


class AdbFileJob(C.Structure):
    _fields_ = [
        ("paths", C.POINTER(C.c_char_p)), ("n_paths", C.c_int32), ("minibatch_size", C.c_int32),
        ("keep", C.POINTER(C.c_void_p)), ("out_dir", C.c_char_p),
        ("batch_size_output", C.c_int32), ("chunk_batches", C.c_int32), ("bidx_pass", C.c_int32), ("bidx_fail", C.c_int32),
        ("n_copy_threads", C.c_int32), ("n_format_threads", C.c_int32), ("write_csv", C.c_int32), ("_pad", C.c_int32),
    ]


class AdbFileStats(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("reads", "n_pass", "n_fail", "lost", "files", "comp_bytes", "h2d_bytes")] + [
        (k, C.c_double) for k in ("seconds", "read_s", "gpu_wait_s", "write_s")]


# numpy mirror of adb_record (512 bytes)
RECORD_DTYPE = np.dtype([
    ("success", "<i4"), ("fail_code", "<i4"), ("mvs_fail_mask", "<i4"), ("valid", "<u4"),
    ("signal_len", "<i4"), ("preloaded", "<i4"),
    ("adapter_start", "<i4"), ("adapter_end", "<i4"), ("polya_end", "<i4"),
    ("primary_adapter_end", "<i4"), ("primary_polya_end", "<i4"), ("mvs_adapter_end", "<i4"),
    ("n_cand", "<i4"), ("cand", "<i4", (ADB_MAX_CAND,)),
    ("n_open_pores", "<i4"), ("open_pores", "<i4", (ADB_MAX_OPEN_PORES,)),
    ("sp_idx", "<i4"), ("sp_next_idx", "<i4"), ("sp_open_pore_idx", "<i4"), ("sp_flag", "<i4"),
    ("sp_pa", "<f4"), ("sp_next_pa", "<f4"),
    ("stats", "<f8", (3, 4)), ("mvs", "<f8", (5,)), ("real", "<f8", (3,)), ("med_shift", "<f8"),
    ("_reserved", "u1", (8,)),
])
assert RECORD_DTYPE.itemsize == 512

_lib = None


class AdbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"adapted_b200 [{STATUS_TEXT.get(status, status)}]: {message}")
        self.status = status


def load() -> C.CDLL:
    """Load the CUDA library; raises (loudly) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build it with `python -m adapted_b200.csrc.build` "
            "(adapted_b200 is CUDA-only and has no CPU fallback)")
    L = C.CDLL(SO_PATH)
    vp, ip = C.c_void_p, C.c_int
    L.adb_abi_version.restype = ip
    L.adb_last_error.restype = C.c_char_p
    L.adb_device_count.restype = ip
    L.adb_record_size.restype = ip
    L.adb_config_size.restype = ip
    L.adb_ctx_create.argtypes = [ip, C.POINTER(vp)]
    L.adb_ctx_destroy.argtypes = [vp]
    L.adb_ctx_destroy.restype = None
    L.adb_ctx_launch_count.argtypes = [vp]
    L.adb_ctx_launch_count.restype = C.c_int64
    L.adb_ctx_set_option.argtypes = [vp, C.c_char_p, ip]
    L.adb_ctx_set_option.restype = ip
    L.adb_ctx_query.argtypes = [vp, C.c_char_p]
    L.adb_ctx_query.restype = C.c_int64
    L.adb_detect_host.argtypes = [vp, C.POINTER(AdbBatch), C.POINTER(AdbConfig), vp, vp, vp]
    L.adb_detect_dev.argtypes = [vp, C.POINTER(AdbBatch), C.POINTER(AdbConfig), vp, vp, vp, vp]
    L.adb_detect_pipelined_host.argtypes = [vp, C.POINTER(AdbBatch), C.POINTER(AdbConfig), vp, vp, vp, C.c_int32]
    L.adb_ctx_set_timing.argtypes = [vp, ip]
    L.adb_ctx_get_timing.argtypes = [vp, vp]
    L.adb_llr_trace_host.argtypes = [vp, vp, vp, C.c_int32, vp, vp, vp, vp]
    L.adb_llr_detect_host.argtypes = [vp, vp, vp, C.c_int32, vp, vp]
    L.adb_llr_detect_host.restype = ip
    L.adb_global_med_mad_host.argtypes = [vp, C.POINTER(AdbBatch), C.c_int32, vp]
    L.adb_downscale_host.argtypes = [vp, C.POINTER(AdbBatch), C.c_int32, C.c_int32, vp]
    L.adb_cnn_scores_host.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp]
    L.adb_mvs_stream_detect_host.argtypes = [vp, C.POINTER(AdbBatch), C.POINTER(AdbStreamConfig), vp]
    L.adb_mvs_stream_detect_host.restype = ip
    L.adb_stream_session_create.argtypes = [vp, C.POINTER(AdbStreamConfig), C.c_int32, C.c_int32, C.POINTER(vp)]
    L.adb_stream_session_create.restype = ip
    L.adb_stream_session_destroy.argtypes = [vp]
    L.adb_stream_session_destroy.restype = None
    L.adb_stream_session_push.argtypes = [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.adb_stream_session_push.restype = ip
    L.adb_stream_session_create_f32.argtypes = [vp, C.POINTER(AdbStreamConfig), C.c_int32, C.c_int32, C.POINTER(vp)]
    L.adb_stream_session_create_f32.restype = ip
    L.adb_stream_session_push_f32.argtypes = [vp, C.c_int32, vp, vp, vp, vp, vp, vp]
    L.adb_stream_session_push_f32.restype = ip
    L.adb_stream_session_create_dev.argtypes = [vp, C.POINTER(AdbStreamConfig), C.c_int32, C.c_int32, C.c_int32,
                                                C.POINTER(vp)]
    L.adb_stream_session_create_dev.restype = ip
    L.adb_stream_session_push_dev.argtypes = [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.adb_stream_session_push_dev.restype = ip
    L.adb_stream_session_reason.argtypes = [C.c_int32]
    L.adb_stream_session_reason.restype = C.c_char_p
    L.adb_format_csv.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, C.c_char_p, C.c_int32, vp, C.c_int64]
    L.adb_format_csv.restype = C.c_int64
    L.adb_format_csv_ex.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, C.c_char_p, C.c_int32, vp, vp, vp, vp, C.c_int64]
    L.adb_format_csv_ex.restype = C.c_int64
    L.adb_open_pores_host.argtypes = [vp, C.POINTER(AdbBatch), vp, C.c_int32, vp, vp, vp, vp, C.c_int64]
    L.adb_open_pores_host.restype = ip
    L.adb_find_peaks_host.argtypes = [vp, vp, vp, C.c_int32, vp, vp]
    L.adb_find_peaks_host.restype = ip
    L.adb_svb16_decode_host.argtypes = [vp, C.POINTER(AdbSvbBatch), vp]
    L.adb_svb16_decode_host.restype = ip
    L.adb_detect_pipelined_svb_host.argtypes = [vp, C.POINTER(AdbSvbBatch), C.POINTER(AdbConfig), vp, vp, vp, C.c_int32]
    L.adb_detect_pipelined_svb_host.restype = ip
    L.adb_zstd_decompress_host.argtypes = [vp, vp, vp, C.c_int32, vp, vp, vp]
    L.adb_zstd_decompress_host.restype = ip
    L.adb_detect_pipelined_vbz_host.argtypes = [vp, C.POINTER(AdbSvbBatch), C.POINTER(AdbConfig), vp, vp, vp, C.c_int32]
    L.adb_detect_pipelined_vbz_host.restype = ip
    L.adb_detect_files.argtypes = [vp, C.POINTER(AdbFileJob), C.POINTER(AdbConfig), vp, C.POINTER(AdbFileStats)]
    L.adb_detect_files.restype = ip
    for f in ("adb_detect_pipelined_host", "adb_ctx_set_timing", "adb_ctx_get_timing", "adb_ctx_create", "adb_detect_host", "adb_detect_dev", "adb_llr_trace_host",
              "adb_global_med_mad_host", "adb_downscale_host", "adb_cnn_scores_host"):
        getattr(L, f).restype = ip
    assert L.adb_record_size() == RECORD_DTYPE.itemsize, "adb_record layout mismatch"
    assert L.adb_config_size() == C.sizeof(AdbConfig), "adb_config layout mismatch"
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise AdbError(rc, load().adb_last_error().decode())


def fill_config(flat: Dict[str, Any]) -> AdbConfig:
    cfg = AdbConfig()
    for name, _ in AdbConfig._fields_:
        if name == "_pad":
            continue
        v = flat[name]
        if isinstance(v, tuple):
            setattr(cfg, name, D2(float(v[0]), float(v[1])))
        else:
            setattr(cfg, name, v)
    return cfg


def fill_stream_config(flat: Dict[str, Any]) -> AdbStreamConfig:
    cfg = AdbStreamConfig()
    for name, _ in AdbStreamConfig._fields_:
        if name == "_pad":
            continue
        v = flat[name]
        setattr(cfg, name, D2(float(v[0]), float(v[1])) if isinstance(v, tuple) else v)
    return cfg


class Context:
    """Per-device context (adb_ctx): scratch arena + stream.  One per process and GPU."""

    def __init__(self, device: int = 0):
        L = load()
        self._h = C.c_void_p()
        check(L.adb_ctx_create(int(device), C.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    @property
    def launches(self) -> int:
        return int(load().adb_ctx_launch_count(self._h))

    def set_option(self, name: str, value: int) -> None:
        check(load().adb_ctx_set_option(self._h, name.encode(), int(value)))

    def query(self, name: str) -> int:
        return int(load().adb_ctx_query(self._h, name.encode()))

    def close(self) -> None:
        if getattr(self, "_h", None):
            load().adb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Dict[int, Context] = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
