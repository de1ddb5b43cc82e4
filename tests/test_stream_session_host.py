"""Host logic of adapted_b200.stream (no GPU): packing of pushed chunks and resolution of the detector parameters."""
import numpy as np
import pytest

from adapted_b200.config import SigProcConfig, StreamingConfig
from adapted_b200.stream import pack_chunks, resolve_stream_params


def test_pack_chunk_list():
    a, b = np.arange(5, dtype=np.int16), np.array([7, -3], dtype=np.int16)
    slots, adc, offsets = pack_chunks([4, 1, 9], [a, np.zeros(0, np.int16), b])
    assert slots.dtype == np.int32 and list(slots) == [4, 1, 9]
    assert adc.dtype == np.int16 and list(adc) == [0, 1, 2, 3, 4, 7, -3]
    assert offsets.dtype == np.int64 and list(offsets) == [0, 5, 5, 7]


def test_pack_pair_passes_through():
    adc = np.arange(10, dtype=np.int16)
    slots, got, offsets = pack_chunks(np.array([2, 3]), (adc, [1, 4, 10]))
    assert list(slots) == [2, 3] and np.array_equal(got, adc) and list(offsets) == [1, 4, 10]
    # the library checks the order of the offsets; the wrapper only keeps them inside the blob
    assert list(pack_chunks([0, 1], (adc, [0, 6, 3]))[2]) == [0, 6, 3]


def test_pack_empty_push():
    slots, adc, offsets = pack_chunks([], [])
    assert slots.size == 0 and adc.size == 0 and list(offsets) == [0]


@pytest.mark.parametrize("slots,chunks", [
    ([0, 1], [np.zeros(3, np.int16)]),                         # one chunk per slot
    ([0, 1], (np.zeros(4, np.int16), [0, 2])),                 # len(slots) + 1 offsets
    ([0, 1], (np.zeros(4, np.int16), [0, 2, 5])),              # past the end of adc
    ([0], (np.zeros(4, np.int16), [-1, 2])),                   # before its start
    ([0], (np.zeros(4, np.int16), [0, 2], "extra")),           # not a pair
])
def test_pack_refuses_inconsistent_chunks(slots, chunks):
    with pytest.raises(ValueError):
        pack_chunks(slots, chunks)


def test_resolve_params():
    assert resolve_stream_params(None) == StreamingConfig()
    p = StreamingConfig(min_obs_adapter=1000)
    assert resolve_stream_params(p) is p
    spc = SigProcConfig()
    spc.streaming = p
    assert resolve_stream_params(spc) is p
    assert resolve_stream_params(SigProcConfig()) == StreamingConfig()  # no [streaming] section: the defaults
