"""Drop-in minibatch detectors: same names, arguments and error behaviour as the reference's seam functions
(adapted/detect/combined.py:122-355), executed by the CUDA library.

    combined_detect_llr2(batch_of_signals, full_signal_lens, spc)          -> List[DetectResults]
    combined_detect_cnn(batch_of_signals, full_signal_lens, model, spc)    -> List[DetectResults] | DetectResults
    combined_detect_start_peak(batch_of_signals, full_signal_lens, spc)    -> List[DetectResults]

``batch_of_signals`` is the reference's float32 [N, m] NaN-padded pA matrix; ``spc`` may be this package's
:class:`adapted_b200.config.SigProcConfig` or the reference's own object; ``model`` may be the reference's
``BoundariesCNN`` (any object with ``state_dict()``), a state-dict-like mapping, or a flat float32 array.

:func:`detect_reads` is the native ingest: ragged int16 ADC + per-read calibration, any number of
minibatches per call.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, List, Optional, Sequence, Union

import numpy as np

from . import _lib
from .config import flatten_config
from .records import DetectResults, records_to_results

_CNN_KEYS = ("0.weight", "0.bias", "2.weight", "2.bias", "4.weight", "4.bias", "6.weight", "6.bias")


def flatten_cnn_weights(model: Any) -> np.ndarray:
    """state dict of BoundariesCNN (adapted/detect/cnn.py:16-52) -> flat float32[58882] in ABI order."""
    if isinstance(model, np.ndarray):
        w = np.ascontiguousarray(model, dtype=np.float32).ravel()
    else:
        sd = model.state_dict() if hasattr(model, "state_dict") else model
        if len(sd) == 0:
            raise ValueError("Model weights were not loaded")  # cnn.py:90-91
        parts = []
        for k in _CNN_KEYS:
            v = sd[k]
            v = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
            parts.append(np.ascontiguousarray(v, dtype=np.float32).ravel())
        w = np.concatenate(parts)
    if w.size != _lib.CNN_NPARAMS:
        raise ValueError(f"expected {_lib.CNN_NPARAMS} CNN parameters, got {w.size}")
    return w


def _dense_batch(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray):
    x = np.ascontiguousarray(batch_of_signals, dtype=np.float32)
    if x.ndim != 2:
        raise ValueError("batch_of_signals must be a 2-D float32 array")
    lens = np.ascontiguousarray(full_signal_lens, dtype=np.int32)
    n, m = x.shape
    if lens.ndim != 1 or lens.size != n:
        raise ValueError(f"full_signal_lens must hold one length per row ({n}), got {lens.size}")
    b = _lib.AdbBatch(signal=x.ctypes.data, sig_type=_lib.SIG_F32, n_reads=n, m=m, batch_size=max(n, 1),
                      offsets=None, full_lens=lens.ctypes.data, calib_offset=None, calib_scale=None)
    return b, (x, lens)


def _check_ragged(adc: np.ndarray, offsets: np.ndarray, n: int, coff: np.ndarray, cscale: np.ndarray) -> None:
    """The device trusts the ragged description (a read's sample count is offsets[r + 1] - offsets[r]): refuse
    inconsistent ones here instead of faulting on the GPU."""
    if n == 0 and offsets.size <= 1:
        return
    if offsets.ndim != 1 or offsets.size != n + 1:
        raise ValueError(f"offsets must hold n_reads + 1 = {n + 1} entries, got {offsets.size}")
    if coff.size != n or cscale.size != n:
        raise ValueError("one calibration offset and scale per read")
    if n and (offsets[0] < 0 or np.any(offsets[1:] < offsets[:-1]) or offsets[-1] > adc.size):
        raise ValueError("offsets must be non-negative, non-decreasing and end inside the ADC blob")


def _raise_minibatch_error(status: int) -> None:
    # Failures the reference raises outside its per-read try (SURVEY.md A.11): same exception type and text.
    if status == -3:
        raise ValueError("MAD normalization failed: scale is 0")
    if status == -4:
        raise ValueError("attempt to get argmin of an empty sequence")
    if status != 0:
        raise _lib.AdbError(status, "minibatch failed")


def combined_detect_llr2(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray, spc: Any,
                         device: int = 0) -> List[Any]:
    """adapted/detect/combined.py:122-227 on the GPU."""
    b, keep = _dense_batch(batch_of_signals, full_signal_lens)
    if b.n_reads == 0:
        return []
    flat = flatten_config(spc)
    flat["primary_method"] = 0
    recs, status, cfg = _run_flat(b, flat, None, device, keep)
    _raise_minibatch_error(int(status[0]))
    return records_to_results(recs, 0, "", open_pore_overflow(b, recs, device))


def combined_detect_cnn(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray, model: Any, spc: Any,
                        device: int = 0) -> Union[List[Any], Any]:
    """adapted/detect/combined.py:230-309 on the GPU (returns a bare object for N == 1, like :309)."""
    b, keep = _dense_batch(batch_of_signals, full_signal_lens)
    w = flatten_cnn_weights(model)
    flat = flatten_config(spc)
    flat["primary_method"] = 1
    recs, status, cfg = _run_flat(b, flat, w, device, keep)
    _raise_minibatch_error(int(status[0]))
    res = records_to_results(recs, 1, None, open_pore_overflow(b, recs, device))
    return res if len(res) > 1 else res[0]


def combined_detect_start_peak(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray, spc: Any,
                               device: int = 0) -> List[Any]:
    """adapted/detect/combined.py:312-355 on the GPU."""
    b, keep = _dense_batch(batch_of_signals, full_signal_lens)
    if b.n_reads == 0:
        return []
    flat = flatten_config(spc)
    flat["primary_method"] = 2
    recs, status, cfg = _run_flat(b, flat, None, device, keep)
    if int(status[0]) == -4:
        raise ValueError("attempt to get argmax of an empty sequence")  # start_peak.py:25-29, outside the try
    _raise_minibatch_error(int(status[0]))
    return records_to_results(recs, 2, None, open_pore_overflow(b, recs, device))


def open_pore_overflow(batch: _lib.AdbBatch, recs: np.ndarray, device: int = 0) -> Optional[dict]:
    """Full open-pore lists (find_open_pores, adapted/detect/anomalies.py:15-35) of the reads of ``batch`` whose list
    does not fit the fixed-size record, computed on the GPU (adb_open_pores_host): {record index: int32 positions}, or
    None when no read overflows (the ordinary case).  ``batch`` must still describe the HOST buffers of the call that
    produced ``recs``."""
    over = np.flatnonzero((recs["n_open_pores"] > _lib.ADB_MAX_OPEN_PORES) & ((recs["valid"] & (1 << 6)) != 0)
                          & ((recs["valid"] & (1 << 11)) != 0)).astype(np.int32)
    if over.size == 0:
        return None
    seg0 = np.zeros(over.size, dtype=np.int32)                            # validate_boundaries scans from adapter_start = 0
    seg1 = np.ascontiguousarray(recs["primary_adapter_end"][over], dtype=np.int32)   # ... to the primary adapter end
    offs = np.zeros(over.size + 1, dtype=np.int64)
    L, ctx = _lib.load(), _lib.default_context(device)
    _lib.check(L.adb_open_pores_host(ctx.handle, C.byref(batch), over.ctypes.data, int(over.size), seg0.ctypes.data,
                                     seg1.ctypes.data, offs.ctypes.data, None, 0))
    pos = np.zeros(max(int(offs[-1]), 1), dtype=np.int32)
    _lib.check(L.adb_open_pores_host(ctx.handle, C.byref(batch), over.ctypes.data, int(over.size), seg0.ctypes.data,
                                     seg1.ctypes.data, offs.ctypes.data, pos.ctypes.data, int(pos.size)))
    return {int(i): pos[offs[k]:offs[k + 1]] for k, i in enumerate(over)}


def overflow_tables(overflow: Optional[dict], n_records: int):
    """{record index: positions} -> the (op_index, op_offsets, op_pos) arrays of adb_format_csv_ex."""
    if not overflow:
        return None
    index = np.full(n_records, -1, dtype=np.int32)
    offs = np.zeros(len(overflow) + 1, dtype=np.int64)
    parts = []
    for k, (i, p) in enumerate(sorted(overflow.items())):
        index[i] = k
        parts.append(np.asarray(p, dtype=np.int32))
        offs[k + 1] = offs[k] + parts[-1].size
    return index, offs, np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(1, np.int32))


def _run_flat(batch: _lib.AdbBatch, flat: dict, weights: Optional[np.ndarray], device: int, keep):
    cfg = _lib.fill_config(flat)
    ctx = _lib.default_context(device)
    n_batches = (batch.n_reads + batch.batch_size - 1) // batch.batch_size
    recs = np.zeros(batch.n_reads, dtype=_lib.RECORD_DTYPE)
    status = np.zeros(max(n_batches, 1), dtype=np.int32)
    wptr = weights.ctypes.data if weights is not None else None
    _lib.check(_lib.load().adb_detect_host(ctx.handle, C.byref(batch), C.byref(cfg), wptr, recs.ctypes.data,
                                           status.ctypes.data))
    del keep
    return recs, status, cfg


def detect_reads(adc: np.ndarray, offsets: np.ndarray, full_lens: np.ndarray, calib_offset: np.ndarray,
                 calib_scale: np.ndarray, spc: Any, model: Any = None, minibatch_size: int = 1000,
                 device: int = 0, return_records: bool = False, return_overflow: bool = False):
    """Native ingest: ragged int16 ADC reads (pod5-equivalent information) -> per-read results.

    Reads are processed in consecutive minibatches of ``minibatch_size`` (parser.py:95-99), which is the unit
    the reference normalises / post-processes over.  Returns (results, batch_status) where a non-zero
    batch_status marks a minibatch the reference would have lost (its reads are returned as None).
    """
    adc = np.ascontiguousarray(adc, dtype=np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    lens = np.ascontiguousarray(full_lens, dtype=np.int32)
    coff = np.ascontiguousarray(calib_offset, dtype=np.float32)
    cscale = np.ascontiguousarray(calib_scale, dtype=np.float32)
    n = lens.size
    _check_ragged(adc, offsets, n, coff, cscale)
    flat = flatten_config(spc)
    w = flatten_cnn_weights(model) if flat["primary_method"] == 1 else None
    b = _lib.AdbBatch(signal=adc.ctypes.data, sig_type=_lib.SIG_I16, n_reads=n, m=int(flat["sig_preload_size"]),
                      batch_size=int(minibatch_size), offsets=offsets.ctypes.data, full_lens=lens.ctypes.data,
                      calib_offset=coff.ctypes.data, calib_scale=cscale.ctypes.data)
    if n == 0:
        if return_records:
            empty = (np.zeros(0, _lib.RECORD_DTYPE), np.zeros(0, np.int32))
            return empty + (None,) if return_overflow else empty
        return ([], np.zeros(0, np.int32))
    recs, status, cfg = _run_flat(b, flat, w, device, (adc, offsets, lens, coff, cscale))
    over = open_pore_overflow(b, recs, device)
    if return_records:
        # return_overflow: also the full open-pore lists of the records beyond ADB_MAX_OPEN_PORES ({index: positions})
        return (recs, status, over) if return_overflow else (recs, status)
    res = records_to_results(recs, flat["primary_method"], "" if flat["primary_method"] == 0 else None, over)
    for bi, s in enumerate(status):
        if s != 0:
            for i in range(bi * minibatch_size, min((bi + 1) * minibatch_size, n)):
                res[i] = None
    return res, status


def svb16_decode(comp: np.ndarray, comp_offsets: np.ndarray, n_samples: np.ndarray, m: Optional[int] = None,
                 device: int = 0):
    """svb16 + zig-zag + delta decode on the GPU (adb_svb16_decode_host) -> (adc int16, offsets int64 [n + 1])."""
    comp = np.ascontiguousarray(comp, dtype=np.uint8)
    coff = np.ascontiguousarray(comp_offsets, dtype=np.int64)
    ns = np.ascontiguousarray(n_samples, dtype=np.int32)
    n = ns.size
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(ns, out=off[1:])
    out = np.zeros(int(off[-1]), dtype=np.int16)
    if n == 0:
        return out, off
    if coff.size != n + 1 or np.any(coff[1:] < coff[:-1]) or coff[0] < 0 or coff[-1] + 16 > comp.size or np.any(coff % 16):
        raise ValueError("comp_offsets must hold n + 1 non-decreasing 16-byte aligned offsets inside the blob (16 bytes of slack)")
    lens = ns.copy()
    zeros = np.zeros(n, np.float32)
    b = _lib.AdbSvbBatch(comp=comp.ctypes.data, comp_offsets=coff.ctypes.data, n_samples=ns.ctypes.data, n_reads=n,
                         m=int(m if m else max(int(ns.max()), 1)), batch_size=max(n, 1), full_lens=lens.ctypes.data,
                         calib_offset=zeros.ctypes.data, calib_scale=zeros.ctypes.data)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_svb16_decode_host(ctx.handle, C.byref(b), out.ctypes.data))
    return out, off


def zstd_decompress(frames: np.ndarray, frame_offsets: np.ndarray, capacities: np.ndarray, device: int = 0):
    """zstd decode on the GPU (adb_zstd_decompress_host): frame i = frames[frame_offsets[i]: frame_offsets[i + 1]]
    decodes into a slot of capacities[i] bytes.  Returns (out uint8, status int32 [n]): slot i is
    out[o[i]: o[i] + capacities[i]] with o the exclusive prefix sum of the capacities; status[i] is the decoded size or
    a negative ADB_ZSTD_E_* code."""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    foff = np.ascontiguousarray(frame_offsets, dtype=np.int64)
    cap = np.ascontiguousarray(capacities, dtype=np.int64)
    n = cap.size
    if foff.size != n + 1 or (n and (foff[0] < 0 or np.any(foff[1:] < foff[:-1]) or foff[-1] > frames.size)) or np.any(cap < 0):
        raise ValueError("frame_offsets must hold n + 1 non-decreasing offsets inside `frames`; capacities >= 0")
    doff = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(cap, out=doff[1:])
    out = np.zeros(int(doff[-1]), dtype=np.uint8)
    status = np.zeros(n, dtype=np.int32)
    if n == 0:
        return out, status
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_zstd_decompress_host(ctx.handle, frames.ctypes.data, foff.ctypes.data, n, out.ctypes.data,
                                                    doff.ctypes.data, status.ctypes.data))
    return out, status


def detect_reads_vbz(frames: np.ndarray, frame_offsets: np.ndarray, n_samples: np.ndarray, full_lens: np.ndarray,
                     calib_offset: np.ndarray, calib_scale: np.ndarray, spc: Any, model: Any = None,
                     minibatch_size: int = 1000, chunk_minibatches: int = 16, device: int = 0):
    """VBZ ingest: one zstd frame per read over its svb16 stream (adapted_b200.svb16.vbz_encode_reads) travels to the
    GPU as it is, is decoded there (zstd, then svb16) and detected (adb_detect_pipelined_vbz_host).  Returns
    (records, batch_status), as detect_reads_svb does for the same reads."""
    return detect_reads_svb(frames, frame_offsets, n_samples, full_lens, calib_offset, calib_scale, spc, model,
                            minibatch_size, chunk_minibatches, device, _vbz=True)


def detect_reads_svb(comp: np.ndarray, comp_offsets: np.ndarray, n_samples: np.ndarray, full_lens: np.ndarray,
                     calib_offset: np.ndarray, calib_scale: np.ndarray, spc: Any, model: Any = None,
                     minibatch_size: int = 1000, chunk_minibatches: int = 16, device: int = 0, _vbz: bool = False):
    """Compressed ingest: svb16 streams (adapted_b200.svb16) travel to the GPU compressed, are decoded there and
    detected (adb_detect_pipelined_svb_host).  Returns (records, batch_status)."""
    comp = np.ascontiguousarray(comp, dtype=np.uint8)
    coff = np.ascontiguousarray(comp_offsets, dtype=np.int64)
    ns = np.ascontiguousarray(n_samples, dtype=np.int32)
    lens = np.ascontiguousarray(full_lens, dtype=np.int32)
    co = np.ascontiguousarray(calib_offset, dtype=np.float32)
    cs = np.ascontiguousarray(calib_scale, dtype=np.float32)
    n = lens.size
    flat = flatten_config(spc)
    m = int(flat["sig_preload_size"])
    if ns.size != n or co.size != n or cs.size != n or (n and (coff.size != n + 1 or np.any(coff[1:] < coff[:-1]) or coff[0] < 0
                                                              or coff[-1] + (0 if _vbz else 16) > comp.size
                                                              or (not _vbz and np.any(coff % 16)))):
        raise ValueError("inconsistent compressed batch description")
    if n and (ns.min() < 0 or ns.max() > m):
        raise ValueError("n_samples must lie in [0, sig_preload_size]")
    w = flatten_cnn_weights(model) if flat["primary_method"] == 1 else None
    n_batches = (n + minibatch_size - 1) // minibatch_size
    recs = np.zeros(n, dtype=_lib.RECORD_DTYPE)
    status = np.zeros(max(n_batches, 1), dtype=np.int32)
    if n == 0:
        return recs, status[:0]
    b = _lib.AdbSvbBatch(comp=comp.ctypes.data, comp_offsets=coff.ctypes.data, n_samples=ns.ctypes.data, n_reads=n, m=m,
                         batch_size=int(minibatch_size), full_lens=lens.ctypes.data, calib_offset=co.ctypes.data,
                         calib_scale=cs.ctypes.data)
    cfg = _lib.fill_config(flat)
    ctx = _lib.default_context(device)
    entry = _lib.load().adb_detect_pipelined_vbz_host if _vbz else _lib.load().adb_detect_pipelined_svb_host
    _lib.check(entry(ctx.handle, C.byref(b), C.byref(cfg), w.ctypes.data if w is not None else None,
                     recs.ctypes.data, status.ctypes.data, int(chunk_minibatches)))
    return recs, status


# ---- streaming poly(A) detector (adapted/detect/mvs.py:341-426) --------------------------------------------------------

def mean_var_shift_polyA_detect_batch(batch_of_signals: np.ndarray, signal_lens: np.ndarray, params: Any = None,
                                      device: int = 0) -> np.ndarray:
    """mean_var_shift_polyA_detect for every row of a dense float32 [N, m] matrix (row i = its first signal_lens[i]
    samples): poly(A) start per read, 0 where the reference returns 0."""
    from .config import flatten_streaming_config
    from .stream import resolve_stream_params

    params = resolve_stream_params(params)
    b, keep = _dense_batch(batch_of_signals, signal_lens)
    out = np.zeros(b.n_reads, dtype=np.int32)
    if b.n_reads == 0:
        return out
    cfg = _lib.fill_stream_config(flatten_streaming_config(params))
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_mvs_stream_detect_host(ctx.handle, C.byref(b), C.byref(cfg), out.ctypes.data))
    del keep
    return out


def mean_var_shift_polyA_detect(calibrated_signal: np.ndarray, params: Any = None, device: int = 0) -> int:
    """Same signature as the reference's function: one calibrated signal -> poly(A) start or 0."""
    x = np.ascontiguousarray(calibrated_signal, dtype=np.float32).reshape(1, -1)
    if x.shape[1] == 0:
        return 0
    return int(mean_var_shift_polyA_detect_batch(x, np.array([x.shape[1]], np.int32), params, device)[0])


def mean_var_shift_polyA_detect_i16(adc: np.ndarray, offsets: np.ndarray, calib_offset: np.ndarray,
                                    calib_scale: np.ndarray, params: Any = None, window: Optional[int] = None,
                                    device: int = 0) -> np.ndarray:
    """Ragged int16 form (what a read-until cache holds): read i = adc[offsets[i]:offsets[i+1]], calibrated on the
    device; `window` bounds the samples looked at per read (default: the longest read)."""
    from .config import flatten_streaming_config
    from .stream import resolve_stream_params

    params = resolve_stream_params(params)
    adc = np.ascontiguousarray(adc, dtype=np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    lens = np.ascontiguousarray(np.diff(offsets), dtype=np.int32)
    coff = np.ascontiguousarray(calib_offset, dtype=np.float32)
    cscale = np.ascontiguousarray(calib_scale, dtype=np.float32)
    n = lens.size
    _check_ragged(adc, offsets, n, coff, cscale)
    out = np.zeros(n, dtype=np.int32)
    if n == 0:
        return out
    m = int(window) if window else int(lens.max())
    b = _lib.AdbBatch(signal=adc.ctypes.data, sig_type=_lib.SIG_I16, n_reads=n, m=m, batch_size=n,
                      offsets=offsets.ctypes.data, full_lens=lens.ctypes.data, calib_offset=coff.ctypes.data,
                      calib_scale=cscale.ctypes.data)
    cfg = _lib.fill_stream_config(flatten_streaming_config(params))
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_mvs_stream_detect_host(ctx.handle, C.byref(b), C.byref(cfg), out.ctypes.data))
    return out


# ---- kernel-level mirrors of the Cython module (adapted/detect/_c_llr.pyx) ---------------------------------------

def c_llr_trace(raw_signal, start, end, min_obs, border_trim, stride=1, adapter_early_stopping=0,
                adapter_early_stop_window=500, adapter_early_stop_stride=100, polya_early_stopping=0,
                polya_early_stop_window=50, polya_early_stop_stride=10, return_c_c2=0, device: int = 0):
    """_c_llr.pyx:202-236 on the GPU (one trace)."""
    out = c_llr_trace_batch([raw_signal], [(start, end, min_obs, border_trim, stride, adapter_early_stopping,
                                            adapter_early_stop_window, adapter_early_stop_stride,
                                            polya_early_stopping, polya_early_stop_window,
                                            polya_early_stop_stride)], bool(return_c_c2), device)
    return out[0]


def c_llr_trace_batch(signals, params, return_c_c2: bool = False, device: int = 0):
    sigs = [np.ascontiguousarray(s, dtype=np.float64) for s in signals]
    offs = np.zeros(len(sigs) + 1, dtype=np.int64)
    np.cumsum([s.size for s in sigs], out=offs[1:])
    blob = np.concatenate(sigs) if sigs else np.zeros(0)
    p = np.ascontiguousarray(np.asarray(params, dtype=np.int64).reshape(len(sigs), 11))
    for row in p:
        stride = max(int(row[4]), 1)
        if (row[8] > 0 or row[5] > 0) and (row[7] <= 0 or row[7] % stride != 0):
            raise AssertionError("early_stop_stride % stride != 0")  # _c_llr.pyx:102,139
        if row[8] > 0 and (row[10] <= 0 or row[10] % stride != 0):
            raise AssertionError("early_stop_stride % stride != 0")  # _c_llr.pyx:140
    g = np.empty_like(blob)
    c = np.empty_like(blob) if return_c_c2 else None
    c2 = np.empty_like(blob) if return_c_c2 else None
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_llr_trace_host(
        ctx.handle, blob.ctypes.data, offs.ctypes.data, len(sigs), p.ctypes.data, g.ctypes.data,
        c.ctypes.data if return_c_c2 else None, c2.ctypes.data if return_c_c2 else None))
    out = []
    for i in range(len(sigs)):
        sl = slice(offs[i], offs[i + 1])
        out.append((g[sl], c[sl], c2[sl]) if return_c_c2 else g[sl])
    return out


def c_llr_detect_batch(signals, min_obs_adapter, border_trim, min_obs_polya=None, device: int = 0) -> np.ndarray:
    """The legacy three-split detectors for many signals: int64 [n, 4] = adapter_start, adapter_end, polya_end and
    the length of the tuple the reference function returns (see include/adapted_b200.h)."""
    sigs = [np.ascontiguousarray(s, dtype=np.float64) for s in signals]
    n = len(sigs)
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum([s.size for s in sigs], out=offs[1:])
    blob = np.concatenate(sigs) if sigs else np.zeros(0)
    p = np.empty((n, 3), dtype=np.int64)
    p[:, 0], p[:, 1] = min_obs_adapter, border_trim
    p[:, 2] = -1 if min_obs_polya is None else min_obs_polya
    out = np.zeros((n, 4), dtype=np.int64)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_llr_detect_host(ctx.handle, blob.ctypes.data, offs.ctypes.data, n, p.ctypes.data,
                                               out.ctypes.data))
    return out


def c_llr_detect_adapter(raw_signal, min_obs_adapter, border_trim, device: int = 0):
    """_c_llr.pyx:239-288 on the GPU -> (adapter_start, adapter_end)"""
    r = c_llr_detect_batch([raw_signal], min_obs_adapter, border_trim, None, device)[0]
    return int(r[0]), int(r[1])


def c_llr_detect_adapter_polya(raw_signal, min_obs_adapter, border_trim, min_obs_polya, device: int = 0):
    """_c_llr.pyx:290-363 on the GPU -> (adapter_start, adapter_end, polya_end), or (0, 0) for an empty signal"""
    r = c_llr_detect_batch([raw_signal], min_obs_adapter, border_trim, min_obs_polya, device)[0]
    return (0, 0) if r[3] == 2 else (int(r[0]), int(r[1]), int(r[2]))


def c_llr_boundary_traces(raw_signal, min_obs_adapter, border_trim, device: int = 0):
    """c_llr_detect_adapter_trace / c_llr_boundary_traces (_c_llr.pyx:368-388, 415-434): the gains of the three
    splits; the traces come from the GPU gain kernel, the arg-max between them from numpy like in the reference."""
    return _legacy_traces(raw_signal, min_obs_adapter, border_trim, None, device)


c_llr_detect_adapter_trace = c_llr_boundary_traces


def c_llr_detect_adapter_polya_trace(raw_signal, min_obs_adapter, border_trim, min_obs_polya, device: int = 0):
    """_c_llr.pyx:390-413"""
    return _legacy_traces(raw_signal, min_obs_adapter, border_trim, min_obs_polya, device)


def _legacy_traces(raw_signal, moa, bt, mop, device):
    x = np.ascontiguousarray(raw_signal, dtype=np.float64)
    length = x.size - 1
    g_first = c_llr_trace(x, 0, length, moa + bt, bt, device=device)
    x_first = int(np.argmax(g_first))
    g_head, g_tail = c_llr_trace_batch([x, x], [(0, x_first, bt, moa, 1, 0, 0, 0, 0, 0, 0),
                                                (x_first, length, moa, bt, 1, 0, 0, 0, 0, 0, 0)], device=device)
    if mop is None:
        return g_first, g_head, g_tail
    x_last = int(np.argmax(g_tail))
    g_polya = c_llr_trace(x, x_last, length, mop, bt, device=device)
    return g_first, g_head, g_tail, g_polya


def find_peaks_device(traces, mode: int = 0, distance: int = 0, prominence: float = 0.0, width: float = 0.0,
                      rel_height: float = 0.5, want: int = 32, nan_to_num: bool = False, device: int = 0):
    """Peak picking of the GPU kernels on given float64 traces (adb_find_peaks_host; kernel-level test entry).
    mode 0: the first ``want`` peaks of scipy.signal.find_peaks(trace, distance, prominence, width, rel_height);
    mode 1: adapter_end_from_trace (llr.py:204-259) -> index or -1; mode 2: detect_full_polya_trace_peak_with_spike
    (llr.py:406-479) -> index or 0.  Returns one int64 array (mode 0) or int (modes 1, 2) per trace."""
    tr = [np.ascontiguousarray(t, dtype=np.float64) for t in traces]
    n = len(tr)
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum([t.size for t in tr], out=offs[1:])
    blob = np.concatenate(tr) if tr else np.zeros(0)
    if blob.size == 0:
        blob = np.zeros(1)
    par = np.zeros((n, 8), dtype=np.float64)
    par[:] = [mode, distance, prominence, width, rel_height, want, float(bool(nan_to_num)), 0]
    out = np.zeros((n, 33), dtype=np.int32)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_find_peaks_host(ctx.handle, blob.ctypes.data, offs.ctypes.data, n, par.ctypes.data, out.ctypes.data))
    if mode == 0:
        return [out[i, 1: 1 + out[i, 0]].astype(np.int64) for i in range(n)]
    return [int(out[i, 1]) for i in range(n)]


def cnn_scores(x: np.ndarray, model: Any, device: int = 0) -> np.ndarray:
    """BoundariesCNN forward (adapted/detect/cnn.py:16-52,85-98) on prepared inputs x[n, L] -> scores[n, 2, L_out]."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n, L = x.shape
    L1 = (L + 6 - 7) // 3 + 1
    Lout = (L1 - 1) * 3 - 6 + 7
    w = flatten_cnn_weights(model)
    out = np.zeros((n, 2, Lout), dtype=np.float32)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_cnn_scores_host(ctx.handle, x.ctypes.data, n, L, w.ctypes.data, out.ctypes.data))
    return out


def global_med_mad(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray, max_obs_trace: int, device: int = 0):
    """med_mad(batch[:, :max_obs_trace], with_nan=True), adapted/detect/normalize.py:15-22."""
    b, keep = _dense_batch(batch_of_signals, full_signal_lens)
    out = np.zeros(2, dtype=np.float32)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_global_med_mad_host(ctx.handle, C.byref(b), int(max_obs_trace), out.ctypes.data))
    del keep
    return float(out[0]), float(out[1])


def global_med_mad_i16(adc: np.ndarray, offsets: np.ndarray, full_lens: np.ndarray, calib_offset: np.ndarray,
                       calib_scale: np.ndarray, m: int, max_obs_trace: int, minibatch_size: int, device: int = 0,
                       exact: bool = False):
    """Same statistic on ragged int16 reads, one (med, mad) per minibatch.  Returns (med_mad [n_batches, 2],
    number of minibatches the sampled one-pass select handed to the exact multi-pass select).  ``exact=True``
    forces the multi-pass select."""
    adc = np.ascontiguousarray(adc, dtype=np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    lens = np.ascontiguousarray(full_lens, dtype=np.int32)
    coff = np.ascontiguousarray(calib_offset, dtype=np.float32)
    cscale = np.ascontiguousarray(calib_scale, dtype=np.float32)
    n = lens.size
    b = _lib.AdbBatch(signal=adc.ctypes.data, sig_type=_lib.SIG_I16, n_reads=n, m=int(m), batch_size=int(minibatch_size),
                      offsets=offsets.ctypes.data, full_lens=lens.ctypes.data, calib_offset=coff.ctypes.data,
                      calib_scale=cscale.ctypes.data)
    n_batches = (n + minibatch_size - 1) // minibatch_size
    out = np.zeros((n_batches, 2), dtype=np.float32)
    ctx = _lib.default_context(device)
    ctx.set_option("exact_global_select", 1 if exact else 0)
    try:
        _lib.check(_lib.load().adb_global_med_mad_host(ctx.handle, C.byref(b), int(max_obs_trace), out.ctypes.data))
        fallbacks = 0 if exact else ctx.query("global_select_fallbacks")
    finally:
        ctx.set_option("exact_global_select", 0)
    return out, fallbacks


def downscale_signal(batch_of_signals: np.ndarray, full_signal_lens: np.ndarray, factor: int, col0: int = 0,
                     device: int = 0) -> np.ndarray:
    """downscale_signal(batch[:, col0:], factor), adapted/detect/downscale.py:37-41."""
    b, keep = _dense_batch(batch_of_signals, full_signal_lens)
    ncols = (max(b.m - col0, 0) + factor - 1) // factor
    out = np.zeros((b.n_reads, ncols), dtype=np.float32)
    ctx = _lib.default_context(device)
    _lib.check(_lib.load().adb_downscale_host(ctx.handle, C.byref(b), int(col0), int(factor), out.ctypes.data))
    del keep
    return out
