"""The int16 fast paths (counting-based validate kernel, sampled global select, length-sorted moving statistics)
against the oracle AND against the general kernels they stand in for.

Every fast path keeps a hand-over to the general kernel for what it cannot do (codes outside [0, 0x7c00), further
poly(A) candidates, hail-mary fallback, ...).  These tests drive both sides of each hand-over."""
import numpy as np
import pytest

from adapted_b200.config import get_chemistry_specific_config, start_peak_config
from adapted_b200.synth import ReadBatch, make_reads
from oracle import detect_ref
from tests.golden_io import load_cnn_weights
from tests.helpers import diff_results

pytestmark = pytest.mark.gpu


def _detect(b, spc, mbs, model=None, **opts):
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads

    ctx = _lib.default_context(0)
    for k, v in opts.items():
        ctx.set_option(k, v)
    try:
        return detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=model, minibatch_size=mbs)
    finally:
        for k in opts:
            ctx.set_option(k, 0)


def _oracle_llr(b, spc, mbs):
    x = b.to_dense_pa()
    out = []
    for i in range(0, b.n, mbs):
        out += detect_ref.detect_llr2(x[i:i + mbs], b.full_lens[i:i + mbs], spc)
    return out


@pytest.mark.parametrize("seed,kw,cfg", [(601, {}, {}), (602, {"stress": True}, {}), (603, {"short_frac": 0.3}, {}),
                                         # the MVS check and the median-shift check together: validate_fast_kernel is the
                                         # production path (validate_hist_kernel has too few accumulators for their ranges)
                                         (604, {}, {"med_shift": {"detect_med_shift": True}})],
                         ids=["601-kw0", "602-kw1", "603-kw2", "604-med_shift"])
def test_llr_fast_and_general_validate_agree_with_oracle(seed, kw, cfg):
    spc = get_chemistry_specific_config("rna002")
    for group, fields in cfg.items():
        for k, v in fields.items():
            setattr(getattr(spc, group), k, v)
    b = make_reads(200, "rna002", spc.sig_preload_size, seed=seed, **kw)
    if kw.get("short_frac"):
        # keep the minibatch alive: the reference loses it on an empty downscaled row (SURVEY A.11)
        keep = b.full_lens >= spc.core.min_obs_adapter + 2 * spc.core.downscale_factor
        b = _subset(b, np.flatnonzero(keep))
    want = _oracle_llr(b, spc, b.n)
    fast, st = _detect(b, spc, b.n)
    assert not st.any()
    assert diff_results(fast, want) == []
    general, st = _detect(b, spc, b.n, no_fast_validate=1, exact_global_select=1)
    assert not st.any()
    assert diff_results(general, want) == []
    # order statistics are exact in both kernels: those fields must agree bit for bit between them
    assert diff_results(fast, general, exact_floats=False) == []
    for f, g in zip(fast, general):
        for k in ("adapter_med", "adapter_mad", "polya_med", "polya_mad", "rna_preloaded_med", "rna_preloaded_mad",
                  "mvs_detect_mean_at_loc", "mvs_detect_var_at_loc", "mvs_detect_polya_med",
                  "mvs_detect_polya_local_range", "mvs_detect_med_shift", "real_adapter_local_range",
                  "real_adapter_mean_start", "real_adapter_mean_end"):
            a, c = getattr(f, k), getattr(g, k)
            assert (a is None and c is None) or a == c or (a != a and c != c), (k, a, c)


def _subset(b: ReadBatch, idx) -> ReadBatch:
    chunks = [b.adc[b.offsets[i]:b.offsets[i + 1]] for i in idx]
    offs = np.zeros(len(idx) + 1, np.int64)
    np.cumsum([c.size for c in chunks], out=offs[1:])
    return ReadBatch(adc=np.concatenate(chunks), offsets=offs, full_lens=b.full_lens[idx], calib_offset=b.calib_offset[idx],
                     calib_scale=b.calib_scale[idx], truth=b.truth[idx], m=b.m)


def test_negative_adc_codes_are_handed_to_the_general_kernel():
    """codes below zero do not read as ordered half-precision patterns: the counting kernel must pass such reads on"""
    spc = get_chemistry_specific_config("rna002")
    b = make_reads(48, "rna002", spc.sig_preload_size, seed=611)
    # shift the ADC codes of every other read far below zero and compensate in the calibration offset (the pA values
    # move by a float32 rounding; the oracle is run on exactly what the device computes from these codes)
    adc = b.adc.astype(np.int32)
    coff = b.calib_offset.copy()
    for i in range(0, b.n, 2):
        adc[b.offsets[i]:b.offsets[i + 1]] -= 3000
        coff[i] += 3000.0
    assert adc.min() < 0 and adc.min() >= -32768
    b2 = ReadBatch(adc=adc.astype(np.int16), offsets=b.offsets, full_lens=b.full_lens, calib_offset=coff,
                   calib_scale=b.calib_scale, truth=b.truth, m=b.m)
    got, st = _detect(b2, spc, b2.n)
    assert not st.any()
    assert diff_results(got, _oracle_llr(b2, spc, b2.n)) == []


def test_heavy_ties_and_even_odd_lengths():
    """quantised two-level signals: every median / percentile / MAD sits on large ties, segment lengths of both
    parities; compares the fast kernel with the oracle on the float32 matrix"""
    from adapted_b200.detect import detect_reads

    spc = get_chemistry_specific_config("rna002")
    rng = np.random.default_rng(621)
    n, m = 24, spc.sig_preload_size
    chunks, lens = [], []
    for i in range(n):
        n_op, n_ad, n_pa = int(rng.integers(30, 90)), int(rng.integers(4001, 7000)), int(rng.integers(700, 3000))
        n_rna = int(rng.integers(8000, 30000))
        levels = [(220, 2, n_op), (80, 6, n_ad), (108, 2, n_pa), (95, 12, n_rna)]
        pa = np.concatenate([np.round(rng.normal(mu, sd, k) / 2.0) * 2.0 for mu, sd, k in levels])  # 2 pA grid
        lens.append(pa.size)
        chunks.append(pa[:m])
    coff = np.full(n, -220.0, np.float32)
    scale = np.full(n, 0.25, np.float32)
    adc = [np.rint(c / 0.25 + 220.0).astype(np.int16) for c in chunks]
    offs = np.zeros(n + 1, np.int64)
    np.cumsum([a.size for a in adc], out=offs[1:])
    b = ReadBatch(adc=np.concatenate(adc), offsets=offs, full_lens=np.asarray(lens, np.int32), calib_offset=coff,
                  calib_scale=scale, truth=np.zeros((n, 3), np.int32), m=m)
    got, st = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, minibatch_size=n)
    assert not st.any()
    assert diff_results(got, _oracle_llr(b, spc, n)) == []


@pytest.mark.parametrize("seed,kw", [(631, {}), (632, {"stress": True})])
def test_cnn_fast_validate_matches_general_kernel(seed, kw):
    """RNA004 / CNN primaries: first candidate in the counting kernel, failed reads (further candidates, hail mary)
    handed over -- the two kernels must produce the same results read for read"""
    spc = get_chemistry_specific_config("rna004")
    w = load_cnn_weights()
    b = make_reads(150, "rna004", spc.sig_preload_size, seed=seed, short_frac=0.1, **kw)
    fast, st = _detect(b, spc, b.n, model=w)
    general, st2 = _detect(b, spc, b.n, model=w, no_fast_validate=1)
    assert not st.any() and not st2.any()
    assert diff_results(fast, general) == []
    assert any(not r.success for r in fast) and any(r.success for r in fast)


def test_start_peak_int16_ingest_matches_oracle():
    """start-peak primary (median-shift check on, MVS off) through the int16 ingest -> counting kernel"""
    from adapted_b200.detect import detect_reads

    spc = start_peak_config("rna004")
    b = make_reads(60, "rna004", spc.sig_preload_size, seed=641)
    want = detect_ref.detect_start_peak(b.to_dense_pa(), b.full_lens, spc)
    got, st = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, minibatch_size=b.n)
    assert not st.any()
    assert diff_results(got, want) == []


@pytest.mark.parametrize("chem", ["rna002", "rna004"])
def test_pipelined_ingest_equals_one_shot(chem):
    """adb_detect_pipelined_host (ramped chunk schedule, chunks alternating between two contexts, one copy stream) gives
    byte-identical records to adb_detect_host on the same reads"""
    import ctypes as C

    from adapted_b200 import _lib
    from adapted_b200.config import flatten_config, get_chemistry_specific_config
    from adapted_b200.detect import flatten_cnn_weights
    from adapted_b200.synth import make_reads
    from tests.golden_io import load_cnn_weights

    spc = get_chemistry_specific_config(chem)
    flat = flatten_config(spc)
    mbs, n = 24, 24 * 9 + 7
    b = make_reads(n, chem, flat["sig_preload_size"], seed=55, short_frac=0.05 if chem == "rna004" else 0.0)
    cfg = _lib.fill_config(flat)
    w = flatten_cnn_weights(load_cnn_weights()) if flat["primary_method"] == 1 else None
    wptr = w.ctypes.data if w is not None else None
    batch = _lib.AdbBatch(signal=b.adc.ctypes.data, sig_type=_lib.SIG_I16, n_reads=n, m=flat["sig_preload_size"], batch_size=mbs,
                          offsets=b.offsets.ctypes.data, full_lens=b.full_lens.ctypes.data,
                          calib_offset=b.calib_offset.ctypes.data, calib_scale=b.calib_scale.ctypes.data)
    L = _lib.load()
    ctx = _lib.default_context(0)
    nb = (n + mbs - 1) // mbs
    one = np.zeros(n, dtype=_lib.RECORD_DTYPE)
    st1 = np.zeros(nb, np.int32)
    _lib.check(L.adb_detect_host(ctx.handle, C.byref(batch), C.byref(cfg), wptr, one.ctypes.data, st1.ctypes.data))
    for chunk in (1, 2, 3, 64):
        got = np.zeros(n, dtype=_lib.RECORD_DTYPE)
        st2 = np.full(nb, -99, np.int32)
        _lib.check(L.adb_detect_pipelined_host(ctx.handle, C.byref(batch), C.byref(cfg), wptr, got.ctypes.data,
                                               st2.ctypes.data, chunk))
        assert got.tobytes() == one.tobytes(), chunk
        assert np.array_equal(st1, st2), chunk


def test_cnn_tensor_core_and_fp32_pipe_agree():
    """A/B of the two convolution back ends through the whole CNN seam: the tcgen05 kernels (fp16 hi / lo split, fused
    layer 1 and transposed convolution) against the FP32-pipe kernels; records identical except where a primary
    coordinate moves by at most one downscaled step"""
    from tests.golden_io import load_cnn_weights
    from tests.test_gpu_cnn_path import _cnn_compare

    spc = get_chemistry_specific_config("rna004")
    w = load_cnn_weights()
    b = make_reads(300, "rna004", spc.sig_preload_size, seed=611, short_frac=0.1)
    tc, st = _detect(b, spc, 100, model=w)
    fp, st2 = _detect(b, spc, 100, model=w, cnn_fp32_pipe=1)
    assert not st.any() and not st2.any()
    _cnn_compare(tc, fp, spc.core.downscale_factor)


@pytest.mark.parametrize("seed,kw", [(631, {}), (632, {"stress": True}), (633, {"short_frac": 0.2})])
def test_cnn_candidate_follow_up_equals_general_kernel(seed, kw):
    """reads whose first poly(A) candidate fails: validate_cand_kernel (further candidates from the fast path) writes
    the same records, byte for byte, as the general validate kernel taking them over (option no_cand_followup), and
    both take noticeably many such reads"""
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads

    spc = get_chemistry_specific_config("rna004")
    w = load_cnn_weights()
    b = make_reads(3000, "rna004", spc.sig_preload_size, seed=seed, **kw)
    ctx = _lib.default_context(0)
    out = {}
    for opt in (0, 1):
        ctx.set_option("no_cand_followup", opt)
        try:
            recs, st = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w, minibatch_size=1000,
                                    return_records=True)
            out[opt] = (recs.copy(), ctx.query("validate_handovers"))
        finally:
            ctx.set_option("no_cand_followup", 0)
        assert not st.any()
    assert out[0][0].tobytes() == out[1][0].tobytes()
    assert out[0][1] < out[1][1], (out[0][1], out[1][1])  # reads left the general kernel
