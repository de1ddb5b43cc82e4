"""Read-until sessions of the streaming poly(A) detector (mean_var_shift_polyA_detect, adapted/detect/mvs.py:341-426).

A read-until client asks the detector again every time a channel delivers a chunk.  :class:`StreamSession` keeps the
cache of every channel on the GPU together with the detector's running state, so a push costs work for the appended
samples, not for the whole cache.  The caches hold int16 ADC codes, calibrated per read, and the answers are exactly
those of :func:`adapted_b200.detect.mean_var_shift_polyA_detect_i16` on them; or, with ``dtype=np.float32``,
calibrated float32 pA, and the answers are exactly those of :func:`adapted_b200.detect.mean_var_shift_polyA_detect`
(include/adapted_b200.h, adapted_b200/csrc/adb_stream_session.cuh).

    with StreamSession(StreamingConfig(), n_slots=512, max_samples=100_000) as s:
        start, settled = s.push([3, 7], [chunk3, chunk7], reset=[True, False], calib_offset=[-221.0, 0.0],
                                calib_scale=[0.1755, 0.0])
    with StreamSession(StreamingConfig(), n_slots=512, max_samples=100_000, dtype=np.float32) as s:
        start, settled = s.push([3, 7], [pa3, pa7], reset=[True, False])

A session created with ``device_push=True`` takes its pushes from CUDA tensors instead and enqueues them on a stream,
without a host synchronise (:meth:`StreamSession.push_device`).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Optional, Sequence, Tuple

import numpy as np

from . import _lib


def resolve_stream_params(params: Any = None) -> Any:
    """A StreamingConfig (this package's or the reference's), a SigProcConfig with a [streaming] section, or None
    (the defaults) -> the StreamingConfig-like object, resolved as mean_var_shift_polyA_detect_i16 does."""
    from .config import StreamingConfig

    if hasattr(params, "streaming"):  # a whole SigProcConfig: its optional [streaming] section
        params = params.streaming
    return StreamingConfig() if params is None else params


SESSION_DTYPES = (np.dtype(np.int16), np.dtype(np.float32))


def session_dtype(dtype: Any) -> np.dtype:
    """np.int16 or np.float32 (any spelling numpy accepts) -> that dtype; anything else raises ValueError"""
    try:
        dt = np.dtype(dtype)
    except TypeError:
        dt = None
    if dt not in SESSION_DTYPES:
        raise ValueError(f"a session holds int16 ADC or float32 pA samples, not {dtype!r}")
    return dt


def pack_chunks(slots: Sequence[int], chunks: Any, dtype: Any = np.int16) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(slots, chunks) -> (slots int32 [n], samples `dtype` [total], offsets int64 [n + 1]).

    `chunks` is either a list of per-slot arrays or an ``(samples, offsets)`` tuple with chunk k at
    samples[offsets[k]:offsets[k + 1]]; samples are cast to `dtype` (int16 ADC or float32 pA).  Offsets must lie
    inside `samples`; their order is checked by the library."""
    dt = session_dtype(dtype)
    sl = np.ascontiguousarray(np.asarray(slots).reshape(-1), dtype=np.int32)
    n = sl.size
    if isinstance(chunks, tuple):
        if len(chunks) != 2:
            raise ValueError("chunks given as a tuple must be the pair (samples, offsets)")
        adc = np.ascontiguousarray(np.asarray(chunks[0]).reshape(-1), dtype=dt)
        offsets = np.ascontiguousarray(np.asarray(chunks[1]).reshape(-1), dtype=np.int64)
        if offsets.size != n + 1:
            raise ValueError(f"offsets must hold len(slots) + 1 = {n + 1} entries, got {offsets.size}")
        if n and (offsets.min() < 0 or offsets.max() > adc.size):
            raise ValueError("chunk offsets must lie inside the samples")
        return sl, adc, offsets
    parts = [np.ascontiguousarray(np.asarray(c).reshape(-1), dtype=dt) for c in chunks]
    if len(parts) != n:
        raise ValueError(f"one chunk per slot: {n} slots, {len(parts)} chunks")
    offsets = np.zeros(n + 1, dtype=np.int64)
    if n:
        offsets[1:] = np.cumsum([p.size for p in parts])
    adc = np.concatenate(parts) if n else np.zeros(0, dt)
    return sl, np.ascontiguousarray(adc, dtype=dt), offsets


def _per_entry(values: Optional[Sequence], n: int, dtype) -> Optional[np.ndarray]:
    """one value per pushed slot (a scalar applies to all); None stays None"""
    if values is None:
        return None
    return np.ascontiguousarray(np.broadcast_to(np.asarray(values, dtype=dtype), (n,)))


class StreamSession:
    """`n_slots` channels, each caching at most `max_samples` samples of the read on it, on GPU `device`: int16 ADC
    codes (`dtype` np.int16) or calibrated float32 pA (np.float32).

    :meth:`push` appends one chunk to each of the given slots (after starting a new read on those marked in `reset`;
    an int16 read comes with its calibration pA = (float32(adc) + offset) * scale) and returns per slot the poly(A)
    start on its whole cache (0: none yet) and whether that answer is final.

    With `device_push` the session takes :meth:`push_device` instead: the same pushes from CUDA tensors, enqueued on a
    stream, answers in CUDA tensors."""

    def __init__(self, params: Any = None, n_slots: int = 512, max_samples: int = 100_000, device: int = 0,
                 dtype: Any = np.int16, device_push: bool = False):
        from .config import flatten_streaming_config

        self._h = None
        self.dtype = session_dtype(dtype)
        self.device_push = bool(device_push)
        self.device = int(device)
        self.params = resolve_stream_params(params)
        self.n_slots, self.max_samples = int(n_slots), int(max_samples)
        self._cfg = _lib.fill_stream_config(flatten_streaming_config(self.params))
        self._ctx = _lib.default_context(device)
        h = C.c_void_p()
        lib = _lib.load()
        f32 = self.dtype == np.float32
        if self.device_push:
            _lib.check(lib.adb_stream_session_create_dev(self._ctx.handle, C.byref(self._cfg), self.n_slots,
                                                         self.max_samples, _lib.SIG_F32 if f32 else _lib.SIG_I16,
                                                         C.byref(h)))
        else:
            create = lib.adb_stream_session_create_f32 if f32 else lib.adb_stream_session_create
            _lib.check(create(self._ctx.handle, C.byref(self._cfg), self.n_slots, self.max_samples, C.byref(h)))
        self._h = h

    def push(self, slots: Sequence[int], chunks: Any, reset: Optional[Sequence[bool]] = None,
             calib_offset: Optional[Sequence[float]] = None,
             calib_scale: Optional[Sequence[float]] = None) -> Tuple[np.ndarray, np.ndarray]:
        """-> (polya_start int32 [n], settled bool [n]) for the n pushed slots, in the order given.  A zero-length
        chunk returns the current answer.  Raises AdbError (the session stays usable) for a slot out of range or
        twice in one push, decreasing offsets, an append to a slot never reset, a bad calibration, or a float32 sample
        that is not finite.  A float32 session casts the chunks to float32 and takes no calibration (ValueError)."""
        if not self._h:
            raise ValueError("the session is closed")
        if self.device_push:
            raise ValueError("a device-push session takes push_device(), not push()")
        f32 = self.dtype == np.float32
        if f32 and (calib_offset is not None or calib_scale is not None):
            raise ValueError("a float32 session holds calibrated pA: calib_offset / calib_scale do not apply")
        sl, samples, offsets = pack_chunks(slots, chunks, self.dtype)
        n = sl.size
        out = np.zeros(n, dtype=np.int32)
        done = np.zeros(n, dtype=np.uint8)
        rs = _per_entry(reset, n, np.uint8)
        ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
        lib = _lib.load()
        if f32:
            _lib.check(lib.adb_stream_session_push_f32(self._h, n, ptr(sl), ptr(offsets), ptr(samples), ptr(rs),
                                                       ptr(out), ptr(done)))
        else:
            co = _per_entry(calib_offset, n, np.float32)
            cs = _per_entry(calib_scale, n, np.float32)
            _lib.check(lib.adb_stream_session_push(self._h, n, ptr(sl), ptr(offsets), ptr(samples), ptr(rs), ptr(co),
                                                   ptr(cs), ptr(out), ptr(done)))
        return out, done.astype(bool)

    def push_device(self, slots: Any, chunk_offsets: Any, samples: Any, reset: Any = None, calib_offset: Any = None,
                    calib_scale: Any = None, stream: Any = None, out: Any = None) -> Tuple[Any, Any, Any]:
        """:meth:`push` from CUDA tensors on the session's device, enqueued on `stream` (torch's current stream by
        default) with no host synchronise -> (polya_start int32 [n], settled bool [n], status int32 [2]), CUDA tensors
        written in stream order.

        slots int32 [n]; chunk_offsets int64 [n + 1], chunk k is samples[chunk_offsets[k]:chunk_offsets[k + 1]];
        samples int16 ADC or float32 pA as the session holds, 1-D; reset bool or uint8 [n] (None: no entry resets);
        calib_offset / calib_scale float32 [n] (int16 sessions only).  All contiguous.  `out` optionally gives the
        three output tensors to write instead of new ones.

        The data is checked on the device: status is {0, 0} for an accepted push, {-2, reason} for one the host push
        would refuse, which then changes neither the session nor polya_start / settled (see
        :meth:`raise_for_status`).  Arguments of the wrong dtype, device, layout or shape raise ValueError before
        anything is enqueued."""
        import torch

        if not self._h:
            raise ValueError("the session is closed")
        if not self.device_push:
            raise ValueError("push_device() needs a session created with device_push=True")
        f32 = self.dtype == np.float32
        if f32 and (calib_offset is not None or calib_scale is not None):
            raise ValueError("a float32 session holds calibrated pA: calib_offset / calib_scale do not apply")
        dev = torch.device("cuda", self.device)
        given = []

        def arg(t, name, dtypes, size=None):
            if t is None:
                return
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"{name} must be a torch tensor, got {type(t).__name__}")
            if t.dtype not in dtypes:
                raise ValueError(f"{name} must be {' or '.join(str(d) for d in dtypes)}, got {t.dtype}")
            if t.dim() != 1 or (size is not None and t.numel() != size):
                want = f"[{size}]" if size is not None else "1-D"
                raise ValueError(f"{name} must have shape {want}, got {list(t.shape)}")
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
            given.append((name, t))

        if slots is None or chunk_offsets is None or samples is None:
            raise ValueError("slots, chunk_offsets and samples are required")
        arg(slots, "slots", (torch.int32,))
        n = slots.numel()
        if n > self.n_slots:
            raise ValueError(f"{n} entries for {self.n_slots} slots: a push names each slot at most once")
        arg(chunk_offsets, "chunk_offsets", (torch.int64,), n + 1)
        arg(samples, "samples", (torch.float32,) if f32 else (torch.int16,))
        arg(reset, "reset", (torch.uint8, torch.bool), n)
        arg(calib_offset, "calib_offset", (torch.float32,), n)
        arg(calib_scale, "calib_scale", (torch.float32,), n)
        if out is not None:
            if len(out) != 3:
                raise ValueError("out must be the three tensors (polya_start, settled, status)")
            arg(out[0], "polya_start", (torch.int32,), n)
            arg(out[1], "settled", (torch.bool, torch.uint8), n)
            arg(out[2], "status", (torch.int32,), 2)
        for name, t in given:
            if t.device != dev:
                raise ValueError(f"{name} must be on {dev}, got {t.device}")
        if out is None:
            out = (torch.empty(n, dtype=torch.int32, device=dev), torch.empty(n, dtype=torch.bool, device=dev),
                   torch.empty(2, dtype=torch.int32, device=dev))
        if stream is None:
            stream = torch.cuda.current_stream(dev)
        ptr = lambda t: None if t is None or t.numel() == 0 else t.data_ptr()  # noqa: E731
        _lib.check(_lib.load().adb_stream_session_push_dev(
            self._h, n, ptr(slots), ptr(chunk_offsets), ptr(samples), ptr(reset), ptr(calib_offset), ptr(calib_scale),
            ptr(out[0]), ptr(out[1]), ptr(out[2]), stream.cuda_stream))
        return tuple(out)

    @staticmethod
    def raise_for_status(status: Any) -> None:
        """Waits for the push that writes `status` (push_device's third result) and raises ValueError with the host
        push's message if it was refused."""
        import torch

        torch.cuda.synchronize(status.device)  # the push may have run on any stream
        code, reason = (int(v) for v in status.cpu())
        if code != 0:
            text = _lib.load().adb_stream_session_reason(reason)
            raise ValueError(text.decode() if text else f"push refused (status {code}, reason {reason})")

    def close(self) -> None:
        if getattr(self, "_h", None):
            _lib.load().adb_stream_session_destroy(self._h)
            self._h = None

    def __enter__(self) -> "StreamSession":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
