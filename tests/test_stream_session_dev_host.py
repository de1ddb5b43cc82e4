"""Host logic of device-push sessions (no GPU): StreamSession.push_device refuses arguments of the wrong dtype, device,
layout, shape or session kind before the library is asked to enqueue anything."""
import numpy as np
import pytest

from adapted_b200.stream import StreamSession

torch = pytest.importorskip("torch")


@pytest.fixture
def no_library(monkeypatch):
    from adapted_b200 import _lib

    def refuse(*a, **k):
        raise AssertionError("the library was reached")

    monkeypatch.setattr(_lib, "load", refuse)
    monkeypatch.setattr(_lib, "default_context", refuse)


def _session(dtype=np.int16, device_push=True, n_slots=4):
    """a session object as __init__ leaves it, without a library behind it"""
    s = object.__new__(StreamSession)
    s._h, s.dtype, s.device_push, s.device, s.n_slots = "handle", np.dtype(dtype), device_push, 0, n_slots
    return s


@pytest.fixture
def sessions(no_library):
    made = []

    def make(*a, **k):
        made.append(_session(*a, **k))
        return made[-1]

    yield make
    for s in made:
        s._h = None  # nothing to free


def _args(n=2, dtype=torch.int16, device="cpu"):
    return (torch.arange(n, dtype=torch.int32, device=device), torch.arange(n + 1, dtype=torch.int64, device=device),
            torch.zeros(2 * n, dtype=dtype, device=device))


def test_session_kinds_do_not_mix(sessions):
    with pytest.raises(ValueError, match="device_push=True"):
        sessions(device_push=False).push_device(*_args())
    with pytest.raises(ValueError, match="push_device"):
        sessions().push([0], [np.zeros(3, np.int16)])


@pytest.mark.parametrize("which,bad", [
    (0, torch.arange(2, dtype=torch.int64)),                  # slots: dtype
    (1, torch.arange(3, dtype=torch.int32)),                  # chunk_offsets: dtype
    (1, torch.arange(2, dtype=torch.int64)),                  # chunk_offsets: n entries instead of n + 1
    (2, torch.zeros(4, dtype=torch.float32)),                 # samples of the other session kind
    (2, torch.zeros(2, 2, dtype=torch.int16)),                # samples: 2-D
    (2, torch.zeros(8, dtype=torch.int16)[::2]),              # samples: not contiguous
    (2, np.zeros(4, np.int16)),                               # not a tensor
    (0, None),
])
def test_bad_array_refused(sessions, which, bad):
    args = list(_args())
    args[which] = bad
    with pytest.raises(ValueError):
        sessions().push_device(*args)


@pytest.mark.parametrize("kw", [
    dict(reset=torch.zeros(2, dtype=torch.int32)),
    dict(reset=torch.zeros(3, dtype=torch.uint8)),
    dict(calib_offset=torch.zeros(2, dtype=torch.float64)),
    dict(calib_scale=torch.ones(1, dtype=torch.float32)),
    dict(out=(torch.zeros(2, dtype=torch.int32), torch.zeros(2, dtype=torch.bool))),
    dict(out=(torch.zeros(2, dtype=torch.int64), torch.zeros(2, dtype=torch.bool), torch.zeros(2, dtype=torch.int32))),
    dict(out=(torch.zeros(2, dtype=torch.int32), torch.zeros(2, dtype=torch.bool), torch.zeros(3, dtype=torch.int32))),
])
def test_bad_optional_array_refused(sessions, kw):
    with pytest.raises(ValueError):
        sessions().push_device(*_args(), **kw)


def test_host_tensors_refused(sessions):
    """well-formed arguments in host memory: refused for their device"""
    with pytest.raises(ValueError, match="cuda:0"):
        sessions().push_device(*_args())
    with pytest.raises(ValueError, match="cuda:0"):
        sessions(np.float32).push_device(*_args(dtype=torch.float32))


def test_more_entries_than_slots_refused(sessions):
    with pytest.raises(ValueError, match="at most once"):
        sessions(n_slots=4).push_device(*_args(5))


def test_float32_session_takes_no_calibration(sessions):
    s = sessions(np.float32)
    for kw in (dict(calib_offset=torch.zeros(2)), dict(calib_scale=torch.ones(2))):
        with pytest.raises(ValueError, match="calib"):
            s.push_device(*_args(dtype=torch.float32), **kw)


def test_closed_session_refused(sessions):
    s = sessions()
    s._h = None
    with pytest.raises(ValueError):
        s.push_device(*_args())
