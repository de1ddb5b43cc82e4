"""Packed tiles of the tensor-core convolutions against the per-read tiles (option cnn_tc_per_read_tiles).

Packing the reads of a chunk end to end changes only which rows a tile covers: every output row still accumulates the
same 7 taps x 4 K-steps in the same order from the same operand values, and the epilogues do the same arithmetic.  The
scores -- and the records derived from them -- must therefore be BIT-IDENTICAL between the two tilings, for any chunk
size, any layer-1 length, and with reads that leave the fp16 range and are recomputed on the FP32 pipe next to reads
that are not."""
import numpy as np
import pytest

from adapted_b200.config import get_chemistry_specific_config
from adapted_b200.synth import make_reads
from oracle import detect_ref
from tests.golden_io import load_cnn_weights

pytestmark = pytest.mark.gpu


def _scores(x, w, per_read):
    from adapted_b200 import _lib
    from adapted_b200.detect import cnn_scores

    ctx = _lib.default_context(0)
    ctx.set_option("cnn_tc_per_read_tiles", per_read)
    try:
        return cnn_scores(x, w)
    finally:
        ctx.set_option("cnn_tc_per_read_tiles", 0)


def _records(b, spc, w, per_read, mbs=1000):
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads

    ctx = _lib.default_context(0)
    ctx.set_option("cnn_tc_per_read_tiles", per_read)
    try:
        recs, st = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w,
                                minibatch_size=mbs, return_records=True)
    finally:
        ctx.set_option("cnn_tc_per_read_tiles", 0)
    return np.asarray(recs).copy(), np.asarray(st).copy()


def _same_bits(a, b):
    assert a.shape == b.shape
    bad = np.flatnonzero((a.view(np.uint32) != b.view(np.uint32)).reshape(len(a), -1).any(axis=1))
    assert bad.size == 0, f"{bad.size} reads differ, first {bad[:5]}"


def _prepared(b, spc):
    dense = b.to_dense_pa()
    return np.concatenate([detect_ref.cnn_prepare(dense[i:i + 2000], spc.core) for i in range(0, len(dense), 2000)])


def test_rna004_shipped_window_scores_and_records():
    """20 000 RNA004 reads at the shipped window (L1 = 550): three chunks, the last one partial"""
    spc = get_chemistry_specific_config("rna004")
    w = load_cnn_weights()
    b = make_reads(20000, "rna004", spc.sig_preload_size, seed=71)
    x = _prepared(b, spc)
    assert x.shape[1] == 1650
    packed = _scores(x, w, 0)
    _same_bits(packed, _scores(x, w, 1))
    assert np.isfinite(packed).all()
    # the device pipeline: x written by the prep kernel with its zero tails, scores -> peaks -> validation -> records
    ra, sa = _records(b, spc, w, 0)
    rb, sb = _records(b, spc, w, 1)
    assert not sa.any() and not sb.any()
    assert np.array_equal(np.ascontiguousarray(ra).view(np.uint8), np.ascontiguousarray(rb).view(np.uint8))


def test_stress_read_mix_records():
    """bench.py --stress read mix: long poly(A) tails up to the preload limit, 10 % short reads"""
    spc = get_chemistry_specific_config("rna004")
    w = load_cnn_weights()
    b = make_reads(4000, "rna004", spc.sig_preload_size, seed=72, stress=True, short_frac=0.1)
    x = _prepared(b, spc)
    _same_bits(_scores(x, w, 0), _scores(x, w, 1))
    ra, sa = _records(b, spc, w, 0)
    rb, sb = _records(b, spc, w, 1)
    assert np.array_equal(sa, sb)
    assert np.array_equal(np.ascontiguousarray(ra).view(np.uint8), np.ascontiguousarray(rb).view(np.uint8))


@pytest.mark.parametrize("n", [1, 2, 7598 + 1])
def test_chunk_sizes(n):
    """a single read, two reads, and one read more than a chunk of the 1 650-sample window (a 1-read last chunk)"""
    rng = np.random.default_rng(n)
    w = load_cnn_weights()
    x = rng.normal(0, 1.5, size=(n, 1650)).astype(np.float32)
    x[::3, 1200:] = -5.0
    _same_bits(_scores(x, w, 0), _scores(x, w, 1))


# layer-1 lengths L1 = (L - 1) // 3 + 1: one off / at multiples of 128, the shipped 550, long preload windows
@pytest.mark.parametrize("L1", [127, 128, 129, 255, 256, 257, 550, 4000, 14545])
def test_layer1_lengths(L1):
    L = 3 * L1 - 1
    rng = np.random.default_rng(L1)
    w = load_cnn_weights()
    n = 7 if L1 < 4000 else 3
    x = rng.normal(0, 1.5, size=(n, L)).astype(np.float32)
    x[1, L // 2:] = -5.0
    packed = _scores(x, w, 0)
    _same_bits(packed, _scores(x, w, 1))
    want = detect_ref.cnn_forward(x, w)
    assert np.abs(packed - want).max() <= 2e-5 * np.abs(want).max() + 1e-4


def test_read_outside_fp16_range_is_recomputed_alone():
    """a read whose activations leave the fp16 range goes to the FP32 pipe; the reads sharing its tiles keep their
    tensor-core scores bit for bit (they come out the same as with a tame read in its place)"""
    rng = np.random.default_rng(73)
    w = load_cnn_weights()
    tame = rng.normal(0, 1.5, size=(12, 1650)).astype(np.float32)
    x = tame.copy()
    x[5, 700:720] = 3.0e6  # layer-1 outputs far above 65504
    packed = _scores(x, w, 0)
    _same_bits(packed, _scores(x, w, 1))
    want = detect_ref.cnn_forward(x, w)
    assert np.isfinite(packed).all()
    assert np.abs(packed[5] - want[5]).max() <= 2e-5 * np.abs(want[5]).max() + 1e-4
    keep = np.arange(12) != 5
    _same_bits(packed[keep], _scores(tame, w, 0)[keep])
