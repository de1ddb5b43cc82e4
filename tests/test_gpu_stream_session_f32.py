"""Float32 read-until sessions (adapted_b200.stream.StreamSession(..., dtype=np.float32)): after every push, each
pushed slot answers exactly what mean_var_shift_polyA_detect (adapted/detect/mvs.py:341-426) returns on that slot's
whole float32 cache -- the stateless GPU operator on a dense float32 matrix and the CPU oracle -- and an int16 session
fed the same reads as ADC agrees answer for answer.  `settled` is only reported for answers no later sample can
change.  The off-grid reads reach the float-key order statistics (ties, negative pA) that ADC input never does."""
import ctypes as C

import numpy as np
import pytest

from adapted_b200.config import StreamingConfig
from adapted_b200.synth import SCALE, calibrate, make_reads
from oracle import detect_ref
from tests.golden_io import load_stream_cases

pytestmark = pytest.mark.gpu

# the configurations of test_gpu_stream_session.py: the defaults, and one where most hits are rejected
REJECTING = dict(min_obs_adapter=1000, search_increment_step=250, polyA_local_range=(0.0, 9.1),
                 polyA_med_range=(101.7, 113.9), median_shift_range=(19.3, None))
CHUNK_SIZES = (0, 1, 7, 400, 1600, 4000, -1)  # -1: the rest of the read


def _f32(x):
    return np.asarray(x, dtype=np.float32)


def _adc_of(pa, offset):
    return np.clip(np.rint(pa / SCALE - offset), -32768, 32767).astype(np.int16)


def _stateless(caches, p, m):
    """the stateless float32 operator on a dense NaN-padded [n, m] matrix plus lengths"""
    from adapted_b200.detect import mean_var_shift_polyA_detect_batch

    x = np.full((len(caches), m), np.nan, np.float32)
    for i, c in enumerate(caches):
        x[i, : c.size] = c
    return mean_var_shift_polyA_detect_batch(x, np.array([c.size for c in caches], np.int32), p)


def _oracle(pa, p):
    return detect_ref.mvs_stream_detect(_f32(pa), p)


def _read_pool(chem, seed, n, m):
    """synthetic reads (a quarter of them short) as (adc, offset, scale, pA), plus reads without any poly(A) that only
    settle on a full cache"""
    b = make_reads(n, chem, m, seed=seed, short_frac=0.25)
    reads = [(b.adc[b.offsets[i]: b.offsets[i + 1]], float(b.calib_offset[i]), float(b.calib_scale[i])) for i in range(b.n)]
    rng = np.random.default_rng(seed + 1)
    for k in range(0, len(reads), 10):
        off = float(np.float32(rng.uniform(-240.0, -200.0)))
        reads[k] = (_adc_of(rng.normal(80.0, 7.0, m), off), off, float(np.float32(SCALE)))
    return [(a, co, cs, calibrate(a, co, cs)) for a, co, cs in reads]


@pytest.mark.parametrize("chem,overrides,seed", [("rna002", {}, 911), ("rna004", REJECTING, 912)],
                         ids=["default", "rejecting"])
def test_f32_session_random_schedule_matches_stateless_oracle_and_int16(chem, overrides, seed):
    from adapted_b200.stream import StreamSession

    p = StreamingConfig(**overrides)
    n_slots, max_samples, steps = 300, 20000, 70
    rng = np.random.default_rng(seed)
    reads = _read_pool(chem, seed, 1400, 30000)
    nxt = 0
    cur = [None] * n_slots  # [read index, samples sent]
    reported = {}  # (slot, read) -> answer once settled
    by_accept = by_full = oracle_checked = 0
    with StreamSession(p, n_slots, max_samples, dtype=np.float32) as s, StreamSession(p, n_slots, max_samples) as s16:
        for _ in range(steps):
            pushed = rng.permutation(n_slots)[: int(rng.integers(1, n_slots + 1))]
            adc_chunks, pa_chunks, reset, coff, cscale = [], [], [], [], []
            for sl in pushed:
                r = cur[sl]
                if r is None or r[1] >= reads[r[0]][0].size or rng.random() < 0.03:
                    r = cur[sl] = [nxt % len(reads), 0]
                    nxt += 1
                    reset.append(True)
                else:
                    reset.append(False)
                adc, co, cs, _ = reads[r[0]]
                size = int(rng.choice(CHUNK_SIZES))
                size = adc.size - r[1] if size < 0 else size
                adc_chunks.append(adc[r[1]: r[1] + size])
                pa_chunks.append(calibrate(adc_chunks[-1], co, cs))
                r[1] += adc_chunks[-1].size
                coff.append(co)
                cscale.append(cs)
            got, settled = s.push(pushed, pa_chunks, reset=reset)
            got16, settled16 = s16.push(pushed, adc_chunks, reset=reset, calib_offset=coff, calib_scale=cscale)
            assert np.array_equal(got, got16) and np.array_equal(settled, settled16)
            caches = [reads[cur[sl][0]][3][: min(cur[sl][1], max_samples)] for sl in pushed]
            want = _stateless(caches, p, max_samples)
            assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
            for j in rng.permutation(len(pushed))[:4]:
                assert got[j] == _oracle(caches[j], p)
                oracle_checked += 1
            for j, sl in enumerate(pushed):
                if not settled[j]:
                    continue
                key = (int(sl), cur[sl][0])
                if key in reported:
                    assert reported[key] == got[j]
                    continue
                reported[key] = got[j]
                assert got[j] == _oracle(reads[cur[sl][0]][3][:max_samples], p), \
                    "settled, but the whole read answers otherwise"
                if caches[j].size >= max_samples:
                    by_full += 1
                else:
                    assert got[j] > 0
                    by_accept += 1
    assert by_accept > 0 and by_full > 0 and oracle_checked > 0


def _off_grid_reads(rng, n):
    """float32 pA no ADC grid produces: noise around adapter and poly(A) levels.  Every second read is rounded to
    0.5 pA (many exact ties in every window); every third has a stretch around and below 0 pA (exact zeros, -0.0
    included) inside the median-shift window before its poly(A), long enough to carry that window's median."""
    reads = []
    for k in range(n):
        adapter = rng.normal(rng.uniform(70.0, 85.0), 7.0, int(rng.integers(3500, 9000)))
        polya = rng.normal(rng.uniform(100.0, 116.0), rng.uniform(1.2, 3.6), int(rng.integers(250, 2500)))
        body = rng.normal(rng.uniform(80.0, 96.0), 14.0, int(rng.integers(2000, 12000)))
        if k % 3 == 0:
            low = rng.normal(-4.0, 6.0, int(rng.integers(1100, 1800)))
            low[rng.integers(0, low.size, 40)] = 0.0
            low[rng.integers(0, low.size, 40)] = -0.0
            adapter = np.concatenate([adapter[:-1900], low, adapter[adapter.size - 1900 + low.size:]])
        pa = np.concatenate([adapter, polya, body])
        if k % 2 == 0:
            pa = np.round(pa * 2.0) / 2.0
        reads.append(_f32(pa))
    return reads


@pytest.mark.parametrize("overrides", [{}, REJECTING], ids=["default", "rejecting"])
def test_f32_session_off_grid_signal(overrides):
    """ties, negative pA and values off any ADC grid, fed chunk-wise: == the stateless operator and == the oracle on
    every read at every push"""
    from adapted_b200.stream import StreamSession

    p = StreamingConfig(**overrides)
    rng = np.random.default_rng(913 + len(overrides))
    reads = _off_grid_reads(rng, 48)
    n = len(reads)
    cap = max(r.size for r in reads)
    assert any((r < 0).any() for r in reads) and any(np.signbit(r[r == 0]).any() for r in reads)
    with StreamSession(p, n, cap, dtype=np.float32) as s:
        pos = np.zeros(n, np.int64)
        first = True
        while first or any(q < r.size for q, r in zip(pos, reads)):
            chunks = []
            for i, r in enumerate(reads):
                size = int(rng.choice((0, 13, 700, 1500, 3000)))
                chunks.append(r[pos[i]: pos[i] + size])
                pos[i] += chunks[-1].size
            got, _ = s.push(np.arange(n), chunks, reset=[first] * n)
            first = False
            caches = [r[:q] for r, q in zip(reads, pos)]
            assert np.array_equal(got, _stateless(caches, p, cap))
            want = [_oracle(c, p) for c in caches]
            assert list(got) == want, [(j, pos[j]) for j in range(n) if got[j] != want[j]][:4]
    # the data reaches the cases it is for: acceptances whose median before the hit is negative, and rejections
    w = p.median_shift_window
    assert any(g > 0 and np.median(r[max(g - w, 0): g]) < 0 for r, g in zip(reads, got))
    assert 0 < (got > 0).sum() < n


@pytest.mark.parametrize("case", load_stream_cases(), ids=lambda c: c["name"])
def test_f32_session_golden_fed_chunkwise(case):
    """the executed reference's answers on the golden caches, calibrated to float32 pA and delivered in chunks"""
    from adapted_b200.stream import StreamSession

    b = case["batch"]
    n = b.n
    rng = np.random.default_rng(len(case["name"]) + 1)
    pos = np.zeros(n, np.int64)
    lens = np.diff(b.offsets)
    pa = [calibrate(b.adc[b.offsets[i]: b.offsets[i + 1]], b.calib_offset[i], b.calib_scale[i]) for i in range(n)]
    with StreamSession(case["params"], n, case["m"], dtype=np.float32) as s:
        first = True
        while first or (pos < lens).any():
            chunks = []
            for i in range(n):
                size = int(rng.choice(CHUNK_SIZES))
                size = int(lens[i] - pos[i]) if size < 0 else size
                size = min(size, int(lens[i] - pos[i]))
                chunks.append(pa[i][pos[i]: pos[i] + size])
                pos[i] += size
            got, _ = s.push(np.arange(n), chunks, reset=np.full(n, first))
            first = False
    assert np.array_equal(got, case["want"])


def _flipping_read(rng):
    """adapter, a short poly(A)-like plateau, then a lower level, all off the ADC grid: on a short cache the plateau
    passes the median-shift check (post window clipped at the cache end), on the full post window it fails"""
    return _f32(np.concatenate([rng.normal(80.0, 7.0, 4000), rng.normal(108.0, 2.5, 500), rng.normal(86.0, 2.5, 6000)]))


def test_f32_session_follows_answers_that_change():
    """answers on clipped windows are taken again: an acceptance that a later push overturns is reproduced, at every
    push, exactly as the oracle answers on each prefix"""
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    rng = np.random.default_rng(915)
    reads = [_flipping_read(rng) for _ in range(4)]
    b = make_reads(12, "rna002", 20000, seed=916)
    reads += [calibrate(b.adc[b.offsets[i]: b.offsets[i + 1]], b.calib_offset[i], b.calib_scale[i]) for i in range(b.n)]
    n = len(reads)
    changed = 0
    with StreamSession(p, n, 20000, dtype=np.float32) as s:
        pos = [0] * n
        prev = [0] * n
        for step in range(200):
            size = 7 if step % 3 else 180
            chunks = [r[q: q + size] for r, q in zip(reads, pos)]
            pos = [q + c.size for q, c in zip(pos, chunks)]
            got, _ = s.push(np.arange(n), chunks, reset=[step == 0] * n)
            for i in range(n):
                want = _oracle(reads[i][: pos[i]], p)
                assert got[i] == want, (i, pos[i])
                if prev[i] != 0 and want != prev[i]:
                    changed += 1
                prev[i] = want
            if all(q >= r.size for q, r in zip(pos, reads)):
                break
    assert changed > 0, "no answer changed after having been non-zero: the data does not exercise the resume rule"


def test_f32_session_beyond_the_stateless_ceiling():
    """caches of 120 000 float32 samples, where the stateless float32 operator refuses the window, answer like the
    oracle; a read without poly(A) settles on a full cache"""
    from adapted_b200._lib import AdbError
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    rng = np.random.default_rng(917)
    reads = []
    for k in range(6):
        if k == 5:
            reads.append(_f32(rng.normal(80.0, 7.0, 130000)))  # no poly(A): settles on a full cache
            continue
        head = rng.normal(80.0, 7.0, 90000 + 5000 * k)  # nothing matches before the plateau
        reads.append(_f32(np.concatenate([head, rng.normal(108.0, 2.5, 3000), 95.0 + rng.normal(0.0, 14.0, 40000)])))
    n, cap = len(reads), 120000
    with pytest.raises(AdbError):
        _stateless([r[:cap] for r in reads], p, cap)
    with StreamSession(p, n, cap, dtype=np.float32) as s:
        pos = [0] * n
        for step in range(40):
            chunks = [r[q: q + 8000] for r, q in zip(reads, pos)]
            pos = [q + c.size for q, c in zip(pos, chunks)]
            got, settled = s.push(np.arange(n), chunks, reset=[step == 0] * n)
            if step % 4 == 3 or all(settled):
                want = [_oracle(r[: min(q, cap)], p) for r, q in zip(reads, pos)]
                assert list(got) == want
            if all(settled):
                break
    assert all(settled)
    assert (got[:5] > 90000).all() and got[5] == 0


def test_f32_session_argument_errors_leave_it_usable():
    from adapted_b200 import _lib
    from adapted_b200._lib import AdbError
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    with pytest.raises(AdbError) as e:
        StreamSession(StreamingConfig(pA_mean_window=0), 4, 1000, dtype=np.float32)
    assert e.value.status == -5
    for n_slots, cap in ((0, 1000), (4, 0)):
        with pytest.raises(AdbError) as e:
            StreamSession(p, n_slots, cap, dtype=np.float32)
        assert e.value.status == -2
    b = make_reads(2, "rna002", 20000, seed=918)
    a0 = b.adc[b.offsets[0]: b.offsets[1]]
    co, cs = float(b.calib_offset[0]), float(b.calib_scale[0])
    r0 = calibrate(a0, co, cs)
    assert r0.size > 9400
    r1 = _f32(np.random.default_rng(919).normal(80.0, 7.0, 30000))  # no poly(A)
    cap = 20000
    lib = _lib.load()
    with StreamSession(p, 6, cap, dtype=np.float32) as s, StreamSession(p, 6, cap) as s16:
        got, _ = s.push([1, 2], [r0[:9000], r0[:9000]], reset=[True, True])
        _, full = s.push([4], [r1[:cap]], reset=[True])  # settled on a full cache
        assert full[0]

        def poisoned(i, v):
            x = r0[9000:9400].copy()
            x[i] = v
            return x

        bad = []
        for v in (np.nan, np.inf, -np.inf):
            bad += [
                dict(slots=[1, 2], chunks=[poisoned(150, v), r0[9000:9400]]),   # in the first entry
                dict(slots=[1, 2], chunks=[r0[9000:9400], poisoned(0, v)]),     # in a later entry
                dict(slots=[2, 1], chunks=[r0[9000:9400], poisoned(399, v)]),
                dict(slots=[3], chunks=[poisoned(7, v)], reset=[True]),          # on a reset
                dict(slots=[4], chunks=[poisoned(20, v)]),                       # a settled read's chunk
                dict(slots=[1], chunks=[np.concatenate([r0[9000:], np.full(11000, 80.0, np.float32), [v]])]),  # clipped
            ]
        bad += [
            dict(slots=[6], chunks=[r0[:10]], reset=[True]),              # slot out of range
            dict(slots=[-1], chunks=[r0[:10]], reset=[True]),
            dict(slots=[1, 1], chunks=[r0[9000:9010], r0[9010:9020]]),   # the same slot twice
            dict(slots=[1, 2], chunks=(r0, np.array([9000, 9100, 9050]))),  # decreasing offsets
            dict(slots=[1, 3], chunks=[r0[9000:9010], r0[:10]]),          # slot 3 was never reset
        ]
        for kw in bad:
            with pytest.raises(AdbError) as e:
                s.push(kw["slots"], kw["chunks"], reset=kw.get("reset"))
            assert e.value.status == -2, kw
        # more entries than slots: the first refusal in check order
        many = [
            (dict(slots=[1] * 7, chunks=[r0[9000:9010]] * 7), "the same slot twice in one push"),
            (dict(slots=[1] * 7, chunks=(r0, np.array([0, 10, 20, 15, 30, 40, 50, 60]))),
             "chunk_offsets must be non-decreasing"),
            (dict(slots=[6] + [1] * 6, chunks=[r0[9000:9010]] * 7), "slot out of range"),
        ]
        for kw, msg in many:
            with pytest.raises(AdbError) as e:
                s.push(kw["slots"], kw["chunks"])
            assert e.value.status == -2 and str(e.value).endswith(": " + msg), (kw, str(e.value))
        # calibration belongs to int16 sessions
        for kw in (dict(calib_offset=co, calib_scale=cs), dict(calib_offset=[co]), dict(calib_scale=[cs])):
            with pytest.raises(ValueError):
                s.push([1], [r0[9000:9010]], **kw)
        # the wrong push kind, at the ABI: refused whatever the handle holds
        sl = np.array([1], np.int32)
        offs = np.array([0, 10], np.int64)
        out = np.zeros(1, np.int32)
        done = np.zeros(1, np.uint8)
        adc = np.ascontiguousarray(a0[9000:9010])
        one = np.ones(1, np.float32)
        assert lib.adb_stream_session_push(s._h, 1, sl.ctypes.data, offs.ctypes.data, adc.ctypes.data, None,
                                           one.ctypes.data, one.ctypes.data, out.ctypes.data, done.ctypes.data) == -2
        pa = np.ascontiguousarray(r0[9000:9010])
        assert lib.adb_stream_session_push_f32(s16._h, 1, sl.ctypes.data, offs.ctypes.data, pa.ctypes.data,
                                               np.ones(1, np.uint8).ctypes.data, out.ctypes.data,
                                               done.ctypes.data) == -2
        assert lib.adb_stream_session_push(s._h, 0, None, None, None, None, None, None, None, None) == -2
        assert lib.adb_stream_session_push_f32(s16._h, 0, None, None, None, None, None, None) == -2
        # nothing of the refused pushes reached either session: slots 1 and 2 still hold r0[:9000], slot 3 is not live
        again, _ = s.push([1, 2], [r0[:0], r0[:0]])
        assert list(again) == list(got) == [_oracle(r0[:9000], p)] * 2
        with pytest.raises(AdbError):
            s.push([3], [r0[:10]])
        with pytest.raises(AdbError):
            s16.push([1], [a0[:10]])  # the int16 session never started a read
        got, _ = s.push([1, 2], [r0[9000:], r0[9000:12000]])
        assert got[0] == _oracle(r0, p) and got[1] == _oracle(r0[:12000], p)
        got, settled = s.push([4], [r1[cap:cap + 10]])
        assert got[0] == 0 and settled[0]
