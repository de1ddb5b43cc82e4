"""The long-window read set of tests/test_gpu_long_window.py on the oracle alone (no GPU): with the window raised, the
oracle finds poly(A) ends beyond the shipped RNA004 window (17 500 samples), so the GPU tests cover ground the shipped
configurations cannot reach; and the long CNN read sets of the GPU tests contain reads that take the hail-mary LLR
fallback, whose prefix sums validate_kernel keeps in global memory once the window is no longer staged."""
import numpy as np

from oracle import detect_ref
from tests.golden_io import load_cnn_weights
from tests.test_gpu_long_window import CNN_SETS, SHIPPED_RNA004, _polya_ends, _subset, cnn_set, long_config, long_reads


def test_long_config_raises_only_the_window():
    for chem, m in (("rna004", 49500), ("rna002", 81500), ("rna004", 131072)):
        spc = long_config(chem, m)
        assert spc.sig_preload_size == m
        assert spc.core.max_obs_trace == m - 1500


def test_oracle_cnn_finds_polya_ends_beyond_the_shipped_window():
    m = 49500
    spc = long_config("rna004", m)
    b = long_reads("rna004", m, 40, seed=7900)
    res = detect_ref.detect_cnn(b.to_dense_pa(), b.full_lens, load_cnn_weights(), spc)
    pe = _polya_ends(res)
    assert pe.max() <= m
    assert np.sum(pe > SHIPPED_RNA004) >= 8, pe


def test_oracle_llr_finds_polya_ends_beyond_the_shipped_window():
    m = 81500
    spc = long_config("rna002", m)
    b = long_reads("rna002", m, 40, seed=7901)
    b = _subset(b, np.flatnonzero(b.full_lens >= spc.core.min_obs_adapter + 2 * spc.core.downscale_factor))
    res = detect_ref.detect_llr2(b.to_dense_pa(), b.full_lens, spc)
    pe = _polya_ends(res)
    assert pe.max() <= m
    assert np.sum(pe > SHIPPED_RNA004) >= 8, pe


def test_long_cnn_sets_take_the_hail_mary_fallback(monkeypatch):
    w = load_cnn_weights()
    orig = detect_ref.hail_mary_polya
    calls = []

    def counted(*args, **kw):
        pe = orig(*args, **kw)
        calls.append(pe)
        return pe

    monkeypatch.setattr(detect_ref, "hail_mary_polya", counted)
    for kind, m in CNN_SETS:
        if m <= SHIPPED_RNA004 + 1000:
            continue
        calls.clear()
        spc, b = cnn_set(kind, m)
        x = b.to_dense_pa()
        for i in range(0, b.n, 100):
            detect_ref.detect_cnn(x[i:i + 100].copy(), b.full_lens[i:i + 100], w, spc)
        # reads through the fallback, and some whose fallback trace finds a poly(A) end (validated a second time)
        assert len(calls) >= 3 and sum(pe > 0 for pe in calls) >= 1, (kind, m, calls)
