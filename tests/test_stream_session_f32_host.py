"""Host logic of float32 read-until sessions (no GPU): packing of pushed pA chunks and the choice of sample type."""
import numpy as np
import pytest

from adapted_b200.stream import StreamSession, pack_chunks


def test_pack_f32_chunk_list():
    a, b = np.array([80.5, -3.25, 1e-3], np.float32), np.array([107.0], np.float32)
    slots, pa, offsets = pack_chunks([4, 1, 9], [a, np.zeros(0, np.float32), b], dtype=np.float32)
    assert slots.dtype == np.int32 and list(slots) == [4, 1, 9]
    assert pa.dtype == np.float32 and pa.flags.c_contiguous
    assert np.array_equal(pa, np.array([80.5, -3.25, 1e-3, 107.0], np.float32))
    assert offsets.dtype == np.int64 and list(offsets) == [0, 3, 3, 4]


def test_pack_f32_pair_passes_through():
    pa = np.linspace(-5.0, 120.0, 10, dtype=np.float32)
    slots, got, offsets = pack_chunks(np.array([2, 3]), (pa, [1, 4, 10]), dtype=np.float32)
    assert list(slots) == [2, 3] and got.dtype == np.float32 and np.array_equal(got, pa) and list(offsets) == [1, 4, 10]


def test_pack_f32_casts_float64_as_the_stateless_call_does():
    x = np.array([0.1, 107.123456789, -2.0 ** -130, 1e300, np.nan])  # float64: rounded, underflow, overflow, NaN kept
    with np.errstate(over="ignore"):
        _, got, _ = pack_chunks([0], [x], dtype=np.float32)
        want = np.ascontiguousarray(x, dtype=np.float32)  # what mean_var_shift_polyA_detect hands to the library
        _, got2, _ = pack_chunks([0], (x, [0, 5]), dtype="float32")
    assert np.isinf(want[3])  # the library refuses it as a non-finite sample
    assert got.dtype == np.float32 and np.array_equal(got, want, equal_nan=True)
    got = got2
    assert np.array_equal(got, want, equal_nan=True)


def test_pack_f32_empty_push():
    slots, pa, offsets = pack_chunks([], [], dtype=np.float32)
    assert slots.size == 0 and pa.size == 0 and pa.dtype == np.float32 and list(offsets) == [0]


def test_pack_default_stays_int16():
    _, adc, _ = pack_chunks([0], [np.array([1.9, -2.0])])
    assert adc.dtype == np.int16 and list(adc) == [1, -2]


@pytest.mark.parametrize("dtype", [np.float64, np.int32, np.uint16, "float16", "no-such-type", None])
def test_unsupported_dtype_refused(dtype, monkeypatch):
    from adapted_b200 import _lib

    def no_library(*a, **k):
        raise AssertionError("the library was loaded for an unsupported dtype")

    monkeypatch.setattr(_lib, "load", no_library)
    monkeypatch.setattr(_lib, "default_context", no_library)
    with pytest.raises(ValueError):
        StreamSession(None, 4, 1000, dtype=dtype)
    with pytest.raises(ValueError):
        pack_chunks([0], [np.zeros(3)], dtype=dtype)
