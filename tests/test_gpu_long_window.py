"""Preload windows longer than the shipped configurations (long poly(A) tails): every detection entry point against the
oracle and against each other.

`core.max_obs_trace` is raised so that sig_preload_size = max_obs_trace + 1500 takes the values below.  Past the
shipped RNA004 window (17 500 samples) the CNN post-processing sizes its peak lists from the window; past the
shared-memory limit of the staged layout, validate_kernel reads the window straight from global memory (for float32
input at about 55 900 samples in LLR mode and 34 600 with the CNN path's hail-mary trace; for int16 at about 111 800
and 49 300).  Above 65 535 samples validate_hist_kernel stands down and int16 reads take the counting kernel or
validate_kernel.  Reads: the long-poly(A) stress set mixed with ordinary reads, a share of them short enough for the
hail-mary fallback."""
import numpy as np
import pytest

from adapted_b200.config import config_as_dict, config_from_dict, get_chemistry_specific_config
from adapted_b200.synth import ReadBatch, make_reads
from oracle import detect_ref
from tests.golden_io import load_cnn_weights
from tests.helpers import as_dict, diff_results
from tests.test_gpu_cnn_path import _cnn_compare

pytestmark = pytest.mark.gpu

SHIPPED_RNA004 = 17500


def long_config(chem: str, m: int):
    d = config_as_dict(get_chemistry_specific_config(chem))
    base = get_chemistry_specific_config(chem)
    d["core"]["max_obs_trace"] = m - (base.sig_preload_size - base.core.max_obs_trace)
    spc = config_from_dict(d)
    assert spc.sig_preload_size == m
    return spc


def _concat(parts) -> ReadBatch:
    offs = [np.zeros(1, np.int64)]
    base = 0
    for p in parts:
        offs.append(p.offsets[1:] + base)
        base += int(p.offsets[-1])
    return ReadBatch(np.concatenate([p.adc for p in parts]), np.concatenate(offs),
                     np.concatenate([p.full_lens for p in parts]), np.concatenate([p.calib_offset for p in parts]),
                     np.concatenate([p.calib_scale for p in parts]), np.concatenate([p.truth for p in parts]), parts[0].m)


def long_reads(chem: str, m: int, n: int, seed: int) -> ReadBatch:
    """long poly(A) tails (a fifth of them cut short) shuffled with ordinary reads and with reads that end inside the
    adapter / poly(A): those are short enough (full length < 2 max_obs_adapter) for the CNN path's hail-mary fallback"""
    stress = make_reads(n - n // 4 - n // 8, chem, m, seed=seed, stress=True, short_frac=0.2)
    plain = make_reads(n // 4, chem, m, seed=seed + 1)
    short = make_reads(n // 8, chem, m, seed=seed + 2, short_frac=1.0)
    b = _concat([stress, plain, short])
    perm = np.random.default_rng(seed).permutation(b.n)
    return _subset(b, perm)


def _subset(b: ReadBatch, idx) -> ReadBatch:
    parts = [b.adc[b.offsets[i]:b.offsets[i + 1]] for i in idx]
    offs = np.zeros(len(idx) + 1, np.int64)
    np.cumsum([p.size for p in parts], out=offs[1:])
    return ReadBatch(np.concatenate(parts), offs, b.full_lens[idx], b.calib_offset[idx], b.calib_scale[idx], b.truth[idx], b.m)


def _oracle(fn, x, lens, mbs, *args):
    out = []
    for i in range(0, len(lens), mbs):
        out += fn(x[i:i + mbs].copy(), lens[i:i + mbs], *args)
    return out


def _polya_ends(results):
    return np.array([(as_dict(r).get("polya_end") or 0) if r is not None else 0 for r in results])


def _assert_long_tails(got, want, m):
    """the window is used: a real share of the poly(A) ends lies beyond the shipped RNA004 window in both results"""
    for res in (got, want):
        pe = _polya_ends(res)
        assert pe.max() <= m
        assert np.mean(pe > SHIPPED_RNA004) >= 0.15, np.mean(pe > SHIPPED_RNA004)


# the CNN read sets of the tests below: (input, window) -> (reads, seed)
CNN_SETS = {("int16", 17600): (200, 7143), ("int16", 49500): (200, 7130), ("int16", 131072): (200, 7125),
            ("float32", 49500): (100, 7221), ("float32", 131072): (100, 7222), ("int16", 65000): (200, 7401)}


def cnn_set(kind: str, m: int):
    n, seed = CNN_SETS[(kind, m)]
    return long_config("rna004", m), long_reads("rna004", m, n, seed)


@pytest.mark.parametrize("m", [17600, 49500, 131072])
def test_cnn_int16_long_window_matches_oracle(m):
    from adapted_b200.detect import detect_reads

    spc, b = cnn_set("int16", m)
    w = load_cnn_weights()
    got, status = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w,
                               minibatch_size=100)
    assert not status.any()
    want = _oracle(detect_ref.detect_cnn, b.to_dense_pa(), b.full_lens, 100, w, spc)
    _cnn_compare(got, want, spc.core.downscale_factor)
    if m > SHIPPED_RNA004 + 1000:
        _assert_long_tails(got, want, m)


def test_cnn_topk_global_working_set_strides_over_reads():
    """131 072 samples: cnn_topk_kernel's working set lives in global scratch, one slice per CTA of a grid of 8 CTAs
    per SM that strides over the reads.  With more reads than CTAs, CTAs reuse their slice for a second read; the
    records of the first and the last two minibatches equal those of calls on just those reads (one read per CTA) and
    the oracle's."""
    import torch

    from adapted_b200.detect import detect_reads

    m = 131072
    spc = long_config("rna004", m)
    w = load_cnn_weights()
    ctas = torch.cuda.get_device_properties(0).multi_processor_count * 8
    n = (ctas + 299) // 100 * 100
    b = long_reads("rna004", m, n, seed=7701)
    full, st = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w,
                            minibatch_size=100, return_records=True)
    assert not st.any()
    for lo in (0, n - 200):
        idx = np.arange(lo, lo + 200)
        s = _subset(b, idx)
        part, st = detect_reads(s.adc, s.offsets, s.full_lens, s.calib_offset, s.calib_scale, spc, model=w,
                                minibatch_size=100, return_records=True)
        assert not st.any()
        assert part.tobytes() == full[idx].tobytes(), lo
    s = _subset(b, np.arange(n - 200, n))
    got, _ = detect_reads(s.adc, s.offsets, s.full_lens, s.calib_offset, s.calib_scale, spc, model=w, minibatch_size=100)
    want = _oracle(detect_ref.detect_cnn, s.to_dense_pa(), s.full_lens, 100, w, spc)
    _cnn_compare(got, want, spc.core.downscale_factor)


@pytest.mark.parametrize("m", [49500, 131072])
def test_cnn_float32_long_window_matches_oracle(m):
    from adapted_b200.detect import combined_detect_cnn

    spc, b = cnn_set("float32", m)
    w = load_cnn_weights()
    x = b.to_dense_pa()
    got = combined_detect_cnn(x, b.full_lens, w, spc)
    want = detect_ref.detect_cnn(x.copy(), b.full_lens, w, spc)
    _cnn_compare(got, want, spc.core.downscale_factor)
    _assert_long_tails(got, want, m)


def test_llr_float32_long_window_matches_oracle():
    from adapted_b200.detect import combined_detect_llr2

    m = 81500
    spc = long_config("rna002", m)
    b = long_reads("rna002", m, 100, seed=7301)
    # keep the minibatch alive: the reference loses it on an empty downscaled row
    b = _subset(b, np.flatnonzero(b.full_lens >= spc.core.min_obs_adapter + 2 * spc.core.downscale_factor))
    x = b.to_dense_pa()
    got = combined_detect_llr2(x, b.full_lens, spc)
    want = detect_ref.detect_llr2(x.copy(), b.full_lens, spc)
    assert diff_results(got, want) == []
    _assert_long_tails(got, want, m)


def test_llr_int16_long_window_matches_oracle():
    """131 072 samples: beyond the staged validate_kernel layout and beyond validate_hist_kernel's 16-bit counts"""
    from adapted_b200.detect import detect_reads

    m = 131072
    spc = long_config("rna002", m)
    b = long_reads("rna002", m, 200, seed=7302)
    b = _subset(b, np.flatnonzero(b.full_lens >= spc.core.min_obs_adapter + 2 * spc.core.downscale_factor))
    got, status = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, minibatch_size=100)
    assert not status.any()
    want = _oracle(detect_ref.detect_llr2, b.to_dense_pa(), b.full_lens, 100, spc)
    assert diff_results(got, want) == []
    _assert_long_tails(got, want, m)


def test_unstaged_general_kernel_equals_histogram_kernel():
    """65 000 samples, int16, RNA004: validate_hist_kernel still runs, the staged validate_kernel layout no longer fits.
    Every read through the unstaged validate_kernel == the default kernels, record for record."""
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads

    spc, b = cnn_set("int16", 65000)
    w = load_cnn_weights()
    args = (b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc)
    want, st0 = detect_reads(*args, model=w, minibatch_size=100, return_records=True)
    ctx = _lib.default_context(0)
    ctx.set_option("no_fast_validate", 1)
    try:
        got, st1 = detect_reads(*args, model=w, minibatch_size=100, return_records=True)
    finally:
        ctx.set_option("no_fast_validate", 0)
    assert not st0.any() and not st1.any()
    assert got.tobytes() == want.tobytes()


def test_compressed_ingest_long_window_equals_plain_ingest():
    from adapted_b200 import svb16
    from adapted_b200.detect import detect_reads, detect_reads_svb

    m = 49500
    spc = long_config("rna004", m)
    w = load_cnn_weights()
    b = long_reads("rna004", m, 230, seed=7501)
    want, st_want = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w,
                                 minibatch_size=100, return_records=True)
    comp, coff, ns = svb16.encode_reads(b.adc, b.offsets)
    got, st_got = detect_reads_svb(comp, coff, ns, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w,
                                   minibatch_size=100, chunk_minibatches=2)
    assert np.array_equal(st_got, st_want)
    assert got.tobytes() == want.tobytes()


def test_native_file_pipeline_long_window_equals_python_driver(tmp_path):
    import os

    from adapted_b200.ingest import detect_files, detect_files_native, write_container, write_container_v2

    m = 49500
    spc = long_config("rna004", m)
    w = load_cnn_weights()
    v1, v2 = [], []
    for k, n in enumerate((130, 95)):
        b = long_reads("rna004", m, n, seed=7601 + k)
        ids = [f"{k:02d}-{i:06d}-read" for i in range(n)]
        v1.append(write_container(str(tmp_path / f"v1_{k}"), b.adc, b.offsets, b.full_lens, b.calib_offset,
                                  b.calib_scale, ids))
        v2.append(write_container_v2(str(tmp_path / f"v2_{k}"), b.adc, b.offsets, b.full_lens, b.calib_offset,
                                     b.calib_scale, ids, compress=True))
    a, c = str(tmp_path / "py"), str(tmp_path / "native")
    s1 = detect_files(v1, a, spc, model=w, minibatch_size=100, batch_size_output=64, minibatches_per_call=2)
    s2 = detect_files_native(v2, c, spc, model=w, minibatch_size=100, batch_size_output=64, chunk_minibatches=2)
    keys = ("reads", "pass", "fail", "lost", "files")
    assert {k: s2[k] for k in keys} == {k: s1[k] for k in keys}
    assert s1["reads"] == 225

    def tables(root):
        out = {}
        for sub in ("boundaries", "failed_reads"):
            d = os.path.join(root, sub)
            for fn in sorted(os.listdir(d)) if os.path.isdir(d) else []:
                with open(os.path.join(d, fn), "rb") as f:
                    out[f"{sub}/{fn}"] = f.read()
        return out

    ta, tc = tables(a), tables(c)
    assert sorted(ta) == sorted(tc) and len(ta) == s1["files"]
    for k in ta:
        assert ta[k] == tc[k], k
