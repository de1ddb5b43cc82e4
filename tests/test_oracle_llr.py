"""The C restatement of the LLR gain loops (oracle/llr_gains.c) against the reference's own Cython kernel
(_c_llr.pyx): bit-identical for all dispatch branches.  Where a copy of the reference is present (its source, or a
prebuilt oracle/_ref) the kernel itself is called.  Elsewhere its results for the calls below come from
tests/golden/c_llr_calls.json.gz (golden_io.KernelCalls; arrays as digests that are equal exactly when the arrays are).
That file names its source: where it is the oracle's own earlier output rather than the reference's, these tests pin
the oracle against change instead of checking it against the reference, and they warn."""
import numpy as np
import pytest

from oracle import build_ref, detect_ref
from tests.golden_io import KernelCalls, array_digest, warn_if_oracle_source


@pytest.fixture(scope="module")
def ref():
    if build_ref.kernel_available():
        return KernelCalls(build_ref.load_c_llr())
    calls = KernelCalls()
    warn_if_oracle_source(calls.source, "tests/golden/c_llr_calls.json.gz")
    return calls


def _squiggle(rng, n):
    k1, k2 = sorted(rng.integers(20, n - 20, size=2))
    x = np.concatenate([rng.normal(-1.0, 1.0, k1), rng.normal(1.5, 0.3, k2 - k1), rng.normal(0.5, 1.4, n - k2)])
    return x.astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("seed", range(6))
def test_full_trace_bit_identical(ref, seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(60, 1700))
    x = _squiggle(rng, n)
    for start, head, tail in ((0, 5, 5), (int(rng.integers(1, n // 2)), 1, 1)):
        g_ref, c_ref, c2_ref = ref.c_llr_trace(x, start, n - 1, head, tail, 1, 0, 0, 0, 0, 0, 0, 1)
        g, c, c2 = detect_ref.llr_trace(x, start, n - 1, head, tail, 1, 0, 0, 0, 0, 0, 0, 1)
        assert array_digest(c) == c_ref and array_digest(c2) == c2_ref
        assert array_digest(g) == g_ref


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("stride", (1, 2, 5))
def test_early_stop_variants_bit_identical(ref, seed, stride):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(400, 1700))
    x = _squiggle(rng, n)
    for aes, pes, aw, as_, pw, ps in ((1, 0, 100, 20, 0, 0), (1, 0, 50, 10, 0, 0), (1, 1, 100, 20, 30, 10),
                                     (0, 1, 60, 10, 20, 10)):
        g_ref = ref.c_llr_trace(x, 0, n - 1, 5, 5, stride, aes, aw, as_, pes, pw, ps, 0)
        g = detect_ref.llr_trace(x, 0, n - 1, 5, 5, stride, aes, aw, as_, pes, pw, ps, 0)
        assert array_digest(g) == g_ref, (aes, pes, stride)
        # SURVEY a7: an early-stopped trace is a prefix of the full trace
        full = detect_ref.llr_trace(x, 0, n - 1, 5, 5, stride, 0, 0, 0, 0, 0, 0, 0)
        nz = np.flatnonzero(g)
        if nz.size:
            assert np.array_equal(g[: nz[-1] + 1], full[: nz[-1] + 1], equal_nan=True)


def test_degenerate_variances(ref):
    """constant stretches give var == 0 -> log = -inf / nan, propagated unguarded (SURVEY A.2)."""
    x = np.concatenate([np.zeros(30), np.ones(30), np.full(40, 2.0)])
    g_ref = ref.c_llr_trace(x, 0, x.size - 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0)
    g = detect_ref.llr_trace(x, 0, x.size - 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0)
    assert array_digest(g) == g_ref
    assert not np.isfinite(g[1:-2]).all()


def test_pairwise_sum_matches_numpy():
    from oracle._clib import lib
    import ctypes

    rng = np.random.default_rng(0)
    for n in (0, 1, 7, 8, 9, 127, 128, 129, 300, 1000, 1649):
        a = rng.normal(size=n) * 10 ** rng.uniform(-3, 3, size=n)
        got = lib().adb_oracle_pairwise_sum_f64(a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), n)
        assert got == (np.add.reduce(a) if n else 0.0)


def _four_level(rng, n):
    k = sorted(rng.integers(5, n - 5, size=3))
    lv, sd = rng.normal(0, 1.5, size=4), rng.uniform(0.2, 1.5, size=4)
    parts = [k[0], k[1] - k[0], k[2] - k[1], n - k[2]]
    x = np.concatenate([rng.normal(lv[i], sd[i], m) for i, m in enumerate(parts)])
    return x.astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("seed", range(4))
def test_legacy_three_split_detectors_match_reference_kernel(ref, seed):
    """_best_split / c_llr_detect_adapter[_polya] / the *_trace variants (_c_llr.pyx:40-64, 239-434): the oracle's
    restatement against the reference's compiled Cython module, tuples and traces bit for bit"""
    rng = np.random.default_rng(300 + seed)
    for _ in range(40):
        n = int(rng.integers(40, 1500))
        x = _four_level(rng, n)
        moa, bt, mop = int(rng.integers(3, 40)), int(rng.integers(1, 8)), int(rng.integers(2, 20))
        assert tuple(int(v) for v in ref.c_llr_detect_adapter(x, moa, bt)) == detect_ref.llr_detect_adapter(x, moa, bt)
        assert tuple(int(v) for v in ref.c_llr_detect_adapter_polya(x, moa, bt, mop)) == \
            detect_ref.llr_detect_adapter_polya(x, moa, bt, mop)
        for got, want in zip(detect_ref.llr_boundary_traces(x, moa, bt, mop), ref.c_llr_detect_adapter_polya_trace(x, moa, bt, mop)):
            assert array_digest(got) == want
        for got, want in zip(detect_ref.llr_boundary_traces(x, moa, bt), ref.c_llr_boundary_traces(x, moa, bt)):
            assert array_digest(got) == want
    # degenerate inputs: too short for any split -> (0, 0) from both functions
    x = _four_level(rng, 30)
    assert tuple(int(v) for v in ref.c_llr_detect_adapter(x, 40, 5)) == detect_ref.llr_detect_adapter(x, 40, 5) == (0, 0)
    assert tuple(int(v) for v in ref.c_llr_detect_adapter_polya(x, 40, 5, 3)) == detect_ref.llr_detect_adapter_polya(x, 40, 5, 3)
