"""Read-until sessions of the streaming poly(A) detector (adapted_b200.stream.StreamSession): after every push, each
pushed slot answers exactly what mean_var_shift_polyA_detect (adapted/detect/mvs.py:341-426) returns on that slot's
whole cache -- the stateless GPU operator and the CPU oracle -- and `settled` is only reported for answers no later
sample can change."""
import numpy as np
import pytest

from adapted_b200.config import StreamingConfig
from adapted_b200.synth import SCALE, calibrate, make_reads
from oracle import detect_ref
from tests.golden_io import load_stream_cases

pytestmark = pytest.mark.gpu

# test_gpu_next_rows.py::test_stream_detector_matches_oracle_and_single_call: most hits are rejected
REJECTING = dict(min_obs_adapter=1000, search_increment_step=250, polyA_local_range=(0.0, 9.1),
                 polyA_med_range=(101.7, 113.9), median_shift_range=(19.3, None))
CHUNK_SIZES = (0, 1, 7, 400, 1600, 4000, -1)  # -1: the rest of the read


def _adc_of(pa, offset):
    return np.clip(np.rint(pa / SCALE - offset), -32768, 32767).astype(np.int16)


def _stateless(caches, coffs, cscales, p, window):
    from adapted_b200.detect import mean_var_shift_polyA_detect_i16

    offsets = np.zeros(len(caches) + 1, np.int64)
    offsets[1:] = np.cumsum([c.size for c in caches])
    blob = np.concatenate(caches) if caches else np.zeros(0, np.int16)
    return mean_var_shift_polyA_detect_i16(blob, offsets, np.asarray(coffs, np.float32), np.asarray(cscales, np.float32),
                                           p, window=window)


def _oracle(adc, coff, cscale, p):
    return detect_ref.mvs_stream_detect(calibrate(adc, coff, cscale), p)


def _read_pool(chem, seed, n, m):
    """synthetic reads (a quarter of them short), plus reads without any poly(A) that only settle on a full cache"""
    b = make_reads(n, chem, m, seed=seed, short_frac=0.25)
    reads = [(b.adc[b.offsets[i]: b.offsets[i + 1]], float(b.calib_offset[i]), float(b.calib_scale[i])) for i in range(b.n)]
    rng = np.random.default_rng(seed + 1)
    for k in range(0, len(reads), 10):
        off = float(np.float32(rng.uniform(-240.0, -200.0)))
        reads[k] = (_adc_of(rng.normal(80.0, 7.0, m), off), off, float(np.float32(SCALE)))
    return reads


@pytest.mark.parametrize("chem,overrides,seed", [("rna002", {}, 901), ("rna004", REJECTING, 902)],
                         ids=["default", "rejecting"])
def test_session_random_schedule_matches_stateless_and_oracle(chem, overrides, seed):
    from adapted_b200.stream import StreamSession

    p = StreamingConfig(**overrides)
    n_slots, max_samples, steps = 300, 20000, 70
    rng = np.random.default_rng(seed)
    reads = _read_pool(chem, seed, 1400, 30000)
    nxt = 0
    cur = [None] * n_slots  # [read index, samples sent]
    reported = {}  # (slot, read) -> answer once settled
    by_accept = by_full = oracle_checked = 0
    with StreamSession(p, n_slots, max_samples) as s:
        for _ in range(steps):
            pushed = rng.permutation(n_slots)[: int(rng.integers(1, n_slots + 1))]
            chunks, reset, coff, cscale = [], [], [], []
            for sl in pushed:
                r = cur[sl]
                if r is None or r[1] >= reads[r[0]][0].size or rng.random() < 0.03:
                    r = cur[sl] = [nxt % len(reads), 0]
                    nxt += 1
                    reset.append(True)
                else:
                    reset.append(False)
                adc, co, cs = reads[r[0]]
                size = int(rng.choice(CHUNK_SIZES))
                size = adc.size - r[1] if size < 0 else size
                chunks.append(adc[r[1]: r[1] + size])
                r[1] += chunks[-1].size
                coff.append(co)
                cscale.append(cs)
            got, settled = s.push(pushed, chunks, reset=reset, calib_offset=coff, calib_scale=cscale)
            caches = [reads[cur[sl][0]][0][: min(cur[sl][1], max_samples)] for sl in pushed]
            want = _stateless(caches, coff, cscale, p, max_samples)
            assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
            for j in rng.permutation(len(pushed))[:4]:
                assert got[j] == _oracle(caches[j], coff[j], cscale[j], p)
                oracle_checked += 1
            for j, sl in enumerate(pushed):
                if not settled[j]:
                    continue
                key = (int(sl), cur[sl][0])
                if key in reported:
                    assert reported[key] == got[j]
                    continue
                reported[key] = got[j]
                adc, co, cs = reads[cur[sl][0]]
                assert got[j] == _oracle(adc[:max_samples], co, cs, p), "settled, but the whole read answers otherwise"
                if caches[j].size >= max_samples:
                    by_full += 1
                else:
                    assert got[j] > 0
                    by_accept += 1
    assert by_accept > 0 and by_full > 0 and oracle_checked > 0


@pytest.mark.parametrize("case", load_stream_cases(), ids=lambda c: c["name"])
def test_session_golden_fed_chunkwise(case):
    """the executed reference's answers on the golden caches, with the caches delivered in chunks"""
    from adapted_b200.stream import StreamSession

    b = case["batch"]
    n = b.n
    rng = np.random.default_rng(len(case["name"]))
    pos = np.zeros(n, np.int64)
    lens = np.diff(b.offsets)
    with StreamSession(case["params"], n, case["m"]) as s:
        first = True
        while first or (pos < lens).any():
            chunks = []
            for i in range(n):
                size = int(rng.choice(CHUNK_SIZES))
                size = int(lens[i] - pos[i]) if size < 0 else size
                size = min(size, int(lens[i] - pos[i]))
                chunks.append(b.adc[b.offsets[i] + pos[i]: b.offsets[i] + pos[i] + size])
                pos[i] += size
            got, _ = s.push(np.arange(n), chunks, reset=np.full(n, first), calib_offset=b.calib_offset,
                            calib_scale=b.calib_scale)
            first = False
    assert np.array_equal(got, case["want"])


def _flipping_read(rng, offset):
    """adapter, a short poly(A)-like plateau, then a lower level: on a short cache the plateau passes the median-shift
    check (post window clipped at the cache end), on the full post window it fails"""
    pa = np.concatenate([rng.normal(80.0, 7.0, 4000), rng.normal(108.0, 2.5, 500), rng.normal(86.0, 2.5, 6000)])
    return _adc_of(pa, offset)


def test_session_follows_answers_that_change():
    """answers on clipped windows are taken again: an acceptance that a later push overturns is reproduced, at every
    push, exactly as the oracle answers on each prefix"""
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    rng = np.random.default_rng(905)
    off = float(np.float32(-220.0))
    reads = [_flipping_read(rng, off) for _ in range(4)]
    b = make_reads(12, "rna002", 20000, seed=906)
    reads += [b.adc[b.offsets[i]: b.offsets[i + 1]] for i in range(b.n)]
    offs = [off] * 4 + [float(x) for x in b.calib_offset]
    n = len(reads)
    changed = 0
    with StreamSession(p, n, 20000) as s:
        pos = [0] * n
        prev = [0] * n
        for step in range(200):
            size = 7 if step % 3 else 180
            chunks = [r[q: q + size] for r, q in zip(reads, pos)]
            pos = [q + c.size for q, c in zip(pos, chunks)]
            got, _ = s.push(np.arange(n), chunks, reset=[step == 0] * n, calib_offset=offs, calib_scale=SCALE)
            for i in range(n):
                want = _oracle(reads[i][: pos[i]], offs[i], SCALE, p)
                assert got[i] == want, (i, pos[i])
                if prev[i] != 0 and want != prev[i]:
                    changed += 1
                prev[i] = want
            if all(q >= r.size for q, r in zip(pos, reads)):
                break
    assert changed > 0, "no answer changed after having been non-zero: the data does not exercise the resume rule"


def test_session_beyond_the_stateless_ceiling():
    """caches of 150 000 int16 samples, where the stateless operator refuses the window, answer like the oracle"""
    from adapted_b200._lib import AdbError
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    rng = np.random.default_rng(907)
    off = float(np.float32(-215.0))
    reads = []
    for k in range(6):
        head = rng.normal(80.0, 7.0, 112000 + 5000 * k)  # nothing matches before the plateau
        if k == 5:
            reads.append(_adc_of(rng.normal(80.0, 7.0, 160000), off))  # no poly(A): settles on a full cache
            continue
        pa = np.concatenate([head, rng.normal(108.0, 2.5, 3000), 95.0 + rng.normal(0.0, 14.0, 40000)])
        reads.append(_adc_of(pa, off))
    n, cap = len(reads), 150000
    with pytest.raises(AdbError):
        _stateless([r[:cap] for r in reads], [off] * n, [SCALE] * n, p, cap)
    with StreamSession(p, n, cap) as s:
        pos = [0] * n
        for step in range(40):
            chunks = [r[q: q + 8000] for r, q in zip(reads, pos)]
            pos = [q + c.size for q, c in zip(pos, chunks)]
            got, settled = s.push(np.arange(n), chunks, reset=[step == 0] * n, calib_offset=off, calib_scale=SCALE)
            if step % 4 == 3 or all(settled):
                want = [_oracle(r[: min(q, cap)], off, SCALE, p) for r, q in zip(reads, pos)]
                assert list(got) == want
            if all(settled):
                break
    assert all(settled)
    assert (got[:5] > 110000).all() and got[5] == 0


def test_session_argument_errors_leave_it_usable():
    from adapted_b200._lib import AdbError
    from adapted_b200.stream import StreamSession

    p = StreamingConfig()
    with pytest.raises(AdbError) as e:
        StreamSession(StreamingConfig(pA_mean_window=0), 4, 1000)
    assert e.value.status == -5
    with pytest.raises(AdbError) as e:
        StreamSession(StreamingConfig(pA_var_window=5000), 4, 1000)
    assert e.value.status == -5
    for n_slots, cap in ((0, 1000), (4, 0)):
        with pytest.raises(AdbError) as e:
            StreamSession(p, n_slots, cap)
        assert e.value.status == -2
    b = make_reads(2, "rna002", 20000, seed=908)
    r0 = b.adc[b.offsets[0]: b.offsets[1]]
    co, cs = float(b.calib_offset[0]), float(b.calib_scale[0])
    with StreamSession(p, 4, 20000) as s:
        got, _ = s.push([1], [r0[:9000]], reset=[True], calib_offset=[co], calib_scale=[cs])
        bad = [
            dict(slots=[4], chunks=[r0[:10]], reset=[True]),             # slot out of range
            dict(slots=[-1], chunks=[r0[:10]], reset=[True]),
            dict(slots=[1, 1], chunks=[r0[9000:9010], r0[9010:9020]]),   # the same slot twice
            dict(slots=[1, 2], chunks=(r0, np.array([9000, 9100, 9050]))),  # decreasing offsets
            dict(slots=[1, 3], chunks=[r0[9000:9010], r0[:10]]),          # slot 3 was never reset
            dict(slots=[2], chunks=[r0[:10]], reset=[True], scale=float("nan")),
            dict(slots=[2], chunks=[r0[:10]], reset=[True], scale=float("inf")),
            dict(slots=[2], chunks=[r0[:10]], reset=[True], scale=0.0),
            dict(slots=[2], chunks=[r0[:10]], reset=[True], scale=-0.1755),
        ]
        for kw in bad:
            scale = kw.pop("scale", cs)
            with pytest.raises(AdbError) as e:
                s.push(kw["slots"], kw["chunks"], reset=kw.get("reset"), calib_offset=co, calib_scale=scale)
            assert e.value.status == -2, kw
        # nothing of the refused pushes reached the session: slot 1 still holds r0[:9000]
        again, _ = s.push([1], [r0[:0]])
        assert again[0] == got[0] == _oracle(r0[:9000], co, cs, p)
        got, _ = s.push([1], [r0[9000:]])
        assert got[0] == _oracle(r0, co, cs, p)
