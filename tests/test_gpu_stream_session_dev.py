"""Device-push read-until sessions (StreamSession(..., device_push=True).push_device): entries and chunks in device
memory, all work on the caller's stream.  After every push a device-push session answers exactly what a host-push
session fed the same pushes answers, refuses exactly what it refuses (with the same message, changing nothing), keeps
stream order without host synchronises, and replays from a captured CUDA graph."""
import re

import numpy as np
import pytest

from adapted_b200.config import StreamingConfig
from adapted_b200.synth import SCALE, calibrate, make_reads
from oracle import detect_ref
from tests.golden_io import load_stream_cases
from tests.test_gpu_stream_session import CHUNK_SIZES, REJECTING
from tests.test_gpu_stream_session_f32 import _adc_of, _read_pool

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DTYPES = (np.int16, np.float32)
SENTINEL = (-7, 77)  # outputs before a push; a refused push must leave them so


def _dev(a, dtype=None):
    return torch.from_numpy(np.array(a, dtype=dtype)).cuda()  # a writable contiguous copy


def _session(p, n_slots, cap, dtype, device_push):
    from adapted_b200.stream import StreamSession

    return StreamSession(p, n_slots, cap, dtype=dtype, device_push=device_push)


def _f32(dtype):
    return np.dtype(dtype) == np.float32


def _upload(s, slots, chunks, reset=None, coff=None, cscale=None):
    """the arguments of push_device for a push given as push() takes it"""
    from adapted_b200.stream import pack_chunks

    sl, samples, offsets = pack_chunks(slots, chunks, s.dtype)
    n = sl.size
    per = lambda v, dt: None if v is None else _dev(np.broadcast_to(np.asarray(v, dt), (n,)))  # noqa: E731
    kw = dict(reset=per(reset, np.uint8))
    if not _f32(s.dtype):
        kw.update(calib_offset=per(coff, np.float32), calib_scale=per(cscale, np.float32))
    return (_dev(sl), _dev(offsets), _dev(samples)), kw


def _push_both(h, d, slots, adc_chunks, pa_chunks, reset, coff, cscale):
    """the same push to a host-push session h and a device-push session d -> both answers, checked equal"""
    f32 = _f32(h.dtype)
    chunks = pa_chunks if f32 else adc_chunks
    cal = {} if f32 else dict(calib_offset=coff, calib_scale=cscale)
    want, wset = h.push(slots, chunks, reset=reset, **cal)
    args, kw = _upload(d, slots, chunks, reset, None if f32 else coff, None if f32 else cscale)
    got, gset, status = d.push_device(*args, **kw)
    d.raise_for_status(status)
    got, gset = got.cpu().numpy(), gset.cpu().numpy()
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
    assert np.array_equal(gset, wset)
    return want, wset


def _schedule(chem, seed, n_slots, steps, every_slot=False):
    """random read-until steps as in test_gpu_stream_session*.py: per step the pushed slots, their ADC and pA chunks,
    resets and calibrations, and the samples each pushed slot has received of its read"""
    rng = np.random.default_rng(seed)
    reads = _read_pool(chem, seed, 1400, 30000)
    nxt = 0
    cur = [None] * n_slots
    for _ in range(steps):
        pushed = np.arange(n_slots) if every_slot else rng.permutation(n_slots)[: int(rng.integers(1, n_slots + 1))]
        adc_chunks, pa_chunks, reset, coff, cscale = [], [], [], [], []
        for sl in pushed:
            r = cur[sl]
            if r is None or r[1] >= reads[r[0]][0].size or rng.random() < 0.03:
                r = cur[sl] = [nxt % len(reads), 0]
                nxt += 1
                reset.append(True)
            else:
                reset.append(False)
            adc, co, cs, pa = reads[r[0]]
            size = int(rng.choice(CHUNK_SIZES))
            size = adc.size - r[1] if size < 0 else size
            adc_chunks.append(adc[r[1]: r[1] + size])
            pa_chunks.append(pa[r[1]: r[1] + size])
            r[1] += adc_chunks[-1].size
            coff.append(co)
            cscale.append(cs)
        yield pushed, adc_chunks, pa_chunks, reset, coff, cscale, [cur[sl][1] for sl in pushed]


@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
@pytest.mark.parametrize("chem,overrides,seed", [("rna002", {}, 921), ("rna004", REJECTING, 922)],
                         ids=["default", "rejecting"])
def test_dev_session_random_schedule_matches_host_session(chem, overrides, seed, dtype):
    p = StreamingConfig(**overrides)
    n_slots, cap = 300, 20000
    by_accept = by_full = 0
    with _session(p, n_slots, cap, dtype, False) as h, _session(p, n_slots, cap, dtype, True) as d:
        for pushed, adc_c, pa_c, reset, coff, cscale, sent in _schedule(chem, seed, n_slots, 70):
            want, settled = _push_both(h, d, pushed, adc_c, pa_c, reset, coff, cscale)
            for j in np.flatnonzero(settled):
                if sent[j] >= cap:
                    by_full += 1
                else:
                    assert want[j] > 0
                    by_accept += 1
    assert by_accept > 0 and by_full > 0


@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
@pytest.mark.parametrize("case", load_stream_cases(), ids=lambda c: c["name"])
def test_dev_session_golden_fed_chunkwise(case, dtype):
    """the executed reference's answers on the golden caches, delivered in chunks through device pushes"""
    b = case["batch"]
    n = b.n
    f32 = _f32(dtype)
    rng = np.random.default_rng(len(case["name"]) + 2)
    pos = np.zeros(n, np.int64)
    lens = np.diff(b.offsets)
    sig = [b.adc[b.offsets[i]: b.offsets[i + 1]] for i in range(n)]
    if f32:
        sig = [calibrate(a, b.calib_offset[i], b.calib_scale[i]) for i, a in enumerate(sig)]
    with _session(case["params"], n, case["m"], dtype, True) as d:
        first = True
        while first or (pos < lens).any():
            chunks = []
            for i in range(n):
                size = int(rng.choice(CHUNK_SIZES))
                size = int(lens[i] - pos[i]) if size < 0 else size
                size = min(size, int(lens[i] - pos[i]))
                chunks.append(sig[i][pos[i]: pos[i] + size])
                pos[i] += size
            args, kw = _upload(d, np.arange(n), chunks, np.full(n, first), b.calib_offset, b.calib_scale)
            got, _, status = d.push_device(*args, **kw)
            d.raise_for_status(status)
            first = False
    assert np.array_equal(got.cpu().numpy(), case["want"])


# ---- refusals ------------------------------------------------------------------------------------------------------
def _host_raw(h, slots, samples, offsets, reset=None, coff=None, cscale=None):
    """a host push through the C ABI (offsets as given, unchecked by python) -> (status, message, polya_start,
    settled)"""
    from adapted_b200 import _lib

    lib = _lib.load()
    n = len(slots)
    sl = np.ascontiguousarray(slots, np.int32)
    offs = np.ascontiguousarray(offsets, np.int64)
    out = np.zeros(n, np.int32)
    done = np.zeros(n, np.uint8)
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    rs = None if reset is None else np.ascontiguousarray(reset, np.uint8)
    samples = None if samples is None else np.ascontiguousarray(samples)
    if _f32(h.dtype):
        rc = lib.adb_stream_session_push_f32(h._h, n, ptr(sl), ptr(offs), ptr(samples), ptr(rs), ptr(out), ptr(done))
    else:
        co = None if coff is None else np.ascontiguousarray(np.broadcast_to(np.float32(coff), (n,)))
        cs = None if cscale is None else np.ascontiguousarray(np.broadcast_to(np.float32(cscale), (n,)))
        rc = lib.adb_stream_session_push(h._h, n, ptr(sl), ptr(offs), ptr(samples), ptr(rs), ptr(co), ptr(cs),
                                         ptr(out), ptr(done))
    return rc, lib.adb_last_error().decode(), out, done


def _dev_raw(d, slots, samples, offsets, reset=None, coff=None, cscale=None):
    """the same push as a device push into outputs holding SENTINEL -> (status, polya_start, settled)"""
    n = len(slots)
    samples = np.ascontiguousarray(samples if samples is not None else np.zeros(0, d.dtype))
    kw = {}
    if reset is not None:
        kw["reset"] = _dev(reset, np.uint8)
    if coff is not None:
        kw["calib_offset"] = _dev(np.broadcast_to(np.float32(coff), (n,)))
    if cscale is not None:
        kw["calib_scale"] = _dev(np.broadcast_to(np.float32(cscale), (n,)))
    out = (torch.full((n,), SENTINEL[0], dtype=torch.int32, device="cuda"),
           torch.full((n,), SENTINEL[1], dtype=torch.uint8, device="cuda"),
           torch.full((2,), 99, dtype=torch.int32, device="cuda"))
    got = d.push_device(_dev(slots, np.int32), _dev(offsets, np.int64), _dev(samples), out=out, **kw)
    assert all(g is o for g, o in zip(got, out))
    return [int(v) for v in out[2].cpu()], out[0].cpu().numpy(), out[1].cpu().numpy()


def _bad_pushes(f32, r0, r1, cap):
    """(slots, samples, offsets, reset, calib scale or None) of pushes the host push refuses, on a session whose
    slots 1, 2 hold r0[:9000], slot 4 is settled on a full cache, and slots 0, 3, 5 never started a read; r0 is ADC
    or pA as the session holds, float32 chunks take non-finite values"""
    def cat(*parts):
        return np.concatenate([np.asarray(x, r0.dtype) for x in parts])

    def offs(*chunks):
        return np.concatenate([[0], np.cumsum([len(c) for c in chunks])])

    def push(slots, chunks, reset=None, scale=1.0):
        return (slots, cat(*chunks), offs(*chunks), reset, scale)

    a, b = r0[9000:9400], r0[9400:9800]
    bad = [
        push([6], [r0[:10]], [1]),                                       # slot out of range, first entry
        push([-1], [r0[:10]], [1]),
        push([1, 2, 6], [a, b, r0[:10]], [0, 0, 1]),                     # ... in a later entry
        push([1, 1], [r0[9000:9010], r0[9010:9020]]),                    # the same slot twice
        push([3, 2, 1, 2], [r0[:10], a, b, a], [1, 0, 0, 0]),            # ... next to a valid reset
        push([1, 3], [a, r0[:10]]),                                      # slot 3 never started a read
        push([0, 1, 3], [r0[:10], a, r0[:10]], [1, 0, 0]),
        push([1, 1, 9], [a, a, a]),                                      # the duplicate comes first
        push([9, 1, 1], [a, a, a]),                                      # the range error comes first
        (np.array([1, 2]), cat(r0[:300]), np.array([0, 200, 100]), None, 1.0),   # decreasing offsets
        (np.array([1, 1]), cat(r0[:300]), np.array([0, 200, 100]), None, 1.0),   # decreasing before duplicate
        (np.array([1, 2]), cat(r0[:300]), np.array([-1, 100, 200]), None, 1.0),  # negative first offset
        (np.array([1, 2]), None, np.array([0, 10, 20]), None, 1.0),              # null samples, non-empty chunks
    ]
    if not f32:
        for v in (np.nan, np.inf, 0.0, -0.1755):
            bad += [push([3], [r0[:10]], [1], scale=v), push([1, 3], [a, r0[:10]], [0, 1], scale=v)]
        bad += [push([3], [r0[:10]], [1], scale=None)]                   # a reset without calibration
    else:
        def poisoned(x, i, v):
            x = x.copy()
            x[i] = v
            return x

        for v in (np.nan, np.inf, -np.inf):
            bad += [
                push([1, 2], [poisoned(a, 150, v), b]),                  # in the first entry
                push([1, 2], [a, poisoned(b, 0, v)]),                    # in a later entry
                push([2, 1], [a, poisoned(b, 399, v)]),
                push([3, 5, 1], [r0[:10], r0[:20], poisoned(a, 7, v)], [1, 1, 0]),  # next to valid resets
                push([3], [poisoned(r0[:10], 7, v)], [1]),               # on a reset
                push([2, 4], [a, poisoned(r0[:20], 19, v)]),             # a settled read's chunk
                push([1], [cat(r0[9000:], np.full(cap, 80.0), [v])]),    # beyond max_samples
                push([1, 3], [poisoned(a, 3, v), r0[:10]]),              # never started comes first
            ]
    return bad


@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
def test_dev_session_refusals_match_host_and_change_nothing(dtype):
    from adapted_b200 import _lib

    f32 = _f32(dtype)
    p = StreamingConfig()
    bt = make_reads(2, "rna002", 20000, seed=923)
    a0 = bt.adc[bt.offsets[0]: bt.offsets[1]]
    co, cs = float(bt.calib_offset[0]), float(bt.calib_scale[0])
    r0 = calibrate(a0, co, cs) if f32 else a0
    assert r0.size > 9800
    cap = 20000
    r1 = np.random.default_rng(924).normal(80.0, 7.0, cap + 10).astype(np.float32)  # no poly(A)
    r1 = r1 if f32 else _adc_of(r1, co)
    with _session(p, 6, cap, dtype, False) as h, _session(p, 6, cap, dtype, True) as d:
        cal = {} if f32 else dict(coff=[co] * 2, cscale=[cs] * 2)
        for s in (h, d):
            s_push = _host_raw if s is h else _dev_raw
            res = s_push(s, [1, 2], np.concatenate([r0[:9000], r0[:9000]]), [0, 9000, 18000], [1, 1], **cal)
            assert res[0] == 0 or res[0] == [0, 0]
            res = s_push(s, [4], r1[:cap], [0, cap], [1], **({} if f32 else dict(coff=co, cscale=cs)))
            assert res[-1][0] == 1  # settled on a full cache
        lib = _lib.load()
        reasons = set()
        for slots, samples, offsets, reset, scale in _bad_pushes(f32, r0, r1, cap):
            ckw = {} if f32 or scale is None else dict(coff=co, cscale=scale)
            rc, msg, _, _ = _host_raw(h, slots, samples, offsets, reset, **ckw)
            assert rc == -2, (slots, offsets)
            status, got, done = _dev_raw(d, slots, samples, offsets, reset, **ckw)
            assert status[0] == -2 and lib.adb_stream_session_reason(status[1]).decode() == msg, (slots, status, msg)
            assert (got == SENTINEL[0]).all() and (done == SENTINEL[1]).all()
            with pytest.raises(ValueError, match="^" + re.escape(msg) + "$"):
                d.raise_for_status(torch.tensor(status, dtype=torch.int32, device="cuda"))
            reasons.add(status[1])
            # the next valid push answers as the host session, which never took the refused one either
            want = _host_raw(h, [1, 2, 4], r0[:0], [0, 0, 0, 0])
            status, got, done = _dev_raw(d, [1, 2, 4], r0[:0], [0, 0, 0, 0])
            assert status == [0, 0] and np.array_equal(got, want[2]) and np.array_equal(done, want[3])
        assert len(reasons) == (7 if f32 else 8), sorted(reasons)
        # slots 3 and 5 are still not started, slots 1 and 2 still hold r0[:9000]
        for s in (h, d):
            s_push = _host_raw if s is h else _dev_raw
            assert s_push(s, [3], r0[:10], [0, 10])[0] in (-2, [-2, 9])
        rest = np.concatenate([r0[9000:], r0[9000:12000]])
        want = _host_raw(h, [1, 2], rest, [0, r0.size - 9000, rest.size])
        status, got, done = _dev_raw(d, [1, 2], rest, [0, r0.size - 9000, rest.size])
        assert status == [0, 0] and np.array_equal(got, want[2]) and np.array_equal(done, want[3])
        assert got[0] == detect_ref.mvs_stream_detect(calibrate(a0, co, cs), p)




@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
def test_dev_session_refusals_the_host_sees(dtype):
    """n > n_slots, null pointers and the wrong session kind are refused at once (status untouched: nothing was
    enqueued), in python and at the C ABI"""
    from adapted_b200 import _lib

    lib = _lib.load()
    f32 = _f32(dtype)
    p = StreamingConfig()
    x = np.zeros(10, dtype)
    with _session(p, 4, 1000, dtype, False) as h, _session(p, 4, 1000, dtype, True) as d:
        sl, offs, smp = _dev(np.arange(5), np.int32), _dev(np.arange(6) * 2, np.int64), _dev(x)
        with pytest.raises(ValueError):
            d.push_device(sl, offs, smp)                                 # n > n_slots
        with pytest.raises(ValueError):
            d.push(np.arange(1), [x[:2]])                                # host push on a device-push session
        with pytest.raises(ValueError):
            h.push_device(sl[:1], offs[:2], smp)                         # device push on a host-push session
        if f32:
            with pytest.raises(ValueError):
                d.push_device(sl[:1], offs[:2], smp, calib_scale=_dev([1.0], np.float32))
        status = torch.full((2,), 99, dtype=torch.int32, device="cuda")
        out = torch.zeros(5, dtype=torch.int32, device="cuda")
        done = torch.zeros(5, dtype=torch.uint8, device="cuda")
        one = _dev([1.0], np.float32)
        ptrs = dict(slots=sl.data_ptr(), offs=offs.data_ptr(), samples=smp.data_ptr(), out=out.data_ptr(),
                    done=done.data_ptr(), status=status.data_ptr())

        def raw(s, n, **null):
            a = {k: (None if k in null else v) for k, v in ptrs.items()}
            cal = one.data_ptr() if f32 and "cal" in null else None
            return lib.adb_stream_session_push_dev(s._h, n, a["slots"], a["offs"], a["samples"], None, cal, cal,
                                                   a["out"], a["done"], a["status"], None)

        assert raw(d, 5) == -2                                           # n > n_slots
        for name in ("slots", "offs", "out", "done", "status"):
            assert raw(d, 1, **{name: True}) == -2, name
        assert raw(h, 1) == -2                                           # a host-push session
        if f32:
            assert raw(d, 1, cal=True) == -2
        hp, hoffs, hdone = np.zeros(1, np.int32), np.array([0, 1], np.int64), np.zeros(1, np.uint8)
        push_host = lib.adb_stream_session_push_f32 if f32 else lib.adb_stream_session_push
        hargs = (d._h, 1, hp.ctypes.data, hoffs.ctypes.data, x.ctypes.data, None)
        hout = (hp.ctypes.data, hdone.ctypes.data)
        assert (push_host(*hargs, *hout) if f32 else push_host(*hargs, None, None, *hout)) == -2
        torch.cuda.synchronize()
        assert status.tolist() == [99, 99]
        # an empty push is accepted and only writes the status
        got = d.push_device(sl[:0], offs[:1], smp[:0])
        assert got[0].numel() == 0 and got[2].tolist() == [0, 0]


def _xor_key(dtype):
    return 0x5A5A if not _f32(dtype) else 0x1234567


@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
def test_dev_session_stream_order(dtype):
    """pushes enqueued on a side stream for many steps with no host synchronise; each step's chunks are written into
    the same buffers by torch kernels on that stream just before its push; all answers == the host session's"""
    f32 = _f32(dtype)
    p = StreamingConfig()
    n_slots, cap, steps = 200, 20000, 40
    sched = list(_schedule("rna004", 925, n_slots, steps))
    side = torch.cuda.Stream()
    # every step's inputs, xor-ed, uploaded ahead; the kernels of each step undo the xor into the shared buffers
    staged, answers = [], []
    ibits = torch.int32 if f32 else torch.int16
    with _session(p, n_slots, cap, dtype, False) as h, _session(p, n_slots, cap, dtype, True) as d:
        for pushed, adc_c, pa_c, reset, coff, cscale, _ in sched:
            args, kw = _upload(d, pushed, pa_c if f32 else adc_c, reset, coff, cscale)
            sl, offs, smp = args
            staged.append((sl ^ 0x33, offs ^ 0x33, smp.view(ibits) ^ _xor_key(dtype), kw))
            cal = {} if f32 else dict(calib_offset=coff, calib_scale=cscale)
            answers.append(h.push(pushed, pa_c if f32 else adc_c, reset=reset, **cal))
        most = max(t[2].numel() for t in staged)
        buf_sl = torch.empty(n_slots, dtype=torch.int32, device="cuda")
        buf_offs = torch.empty(n_slots + 1, dtype=torch.int64, device="cuda")
        buf_smp = torch.empty(most, dtype=torch.float32 if f32 else torch.int16, device="cuda")
        torch.cuda.synchronize()
        outs = []
        with torch.cuda.stream(side):
            for sl_x, offs_x, smp_x, kw in staged:
                n, t = sl_x.numel(), smp_x.numel()
                torch.bitwise_xor(sl_x, 0x33, out=buf_sl[:n])
                torch.bitwise_xor(offs_x, 0x33, out=buf_offs[: n + 1])
                torch.bitwise_xor(smp_x, _xor_key(dtype), out=buf_smp.view(ibits)[:t])
                outs.append(d.push_device(buf_sl[:n], buf_offs[: n + 1], buf_smp[:t], **kw))
        side.synchronize()
        for (want, wset), (got, gset, status) in zip(answers, outs):
            assert status.tolist() == [0, 0]
            assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(gset.cpu().numpy(), wset)


@pytest.mark.parametrize("dtype", DTYPES, ids=["int16", "float32"])
def test_dev_session_graph_replay(dtype):
    """one push captured in a CUDA graph with static inputs and outputs, replayed over a schedule by refilling the
    inputs: no allocation and no synchronise inside a push"""
    f32 = _f32(dtype)
    p = StreamingConfig()
    n_slots, cap = 128, 20000
    sched = list(_schedule("rna002", 926, n_slots, 45, every_slot=True))
    most = max(sum(c.size for c in step[1]) for step in sched)
    sl_s = torch.zeros(n_slots, dtype=torch.int32, device="cuda")
    offs_s = torch.zeros(n_slots + 1, dtype=torch.int64, device="cuda")
    smp_s = torch.zeros(most, dtype=torch.float32 if f32 else torch.int16, device="cuda")
    rs_s = torch.zeros(n_slots, dtype=torch.uint8, device="cuda")
    co_s = torch.zeros(n_slots, dtype=torch.float32, device="cuda")
    cs_s = torch.ones(n_slots, dtype=torch.float32, device="cuda")
    cal = {} if f32 else dict(calib_offset=co_s, calib_scale=cs_s)
    with _session(p, n_slots, cap, dtype, False) as h, _session(p, n_slots, cap, dtype, True) as d:
        # loads every kernel of a push before the capture; refused (an append to slot 0, which holds no read), so it
        # changes nothing
        warm = d.push_device(sl_s, offs_s, smp_s, reset=rs_s, **cal)[2]
        assert warm.tolist() == [-2, 9]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            got, gset, status = d.push_device(sl_s, offs_s, smp_s, reset=rs_s, **cal)
        for pushed, adc_c, pa_c, reset, coff, cscale, _ in sched:
            chunks = pa_c if f32 else adc_c
            args, kw = _upload(d, pushed, chunks, reset, coff, cscale)
            sl_s.copy_(args[0])
            offs_s.copy_(args[1])
            smp_s[: args[2].numel()].copy_(args[2])
            rs_s.copy_(kw["reset"])
            if not f32:
                co_s.copy_(kw["calib_offset"])
                cs_s.copy_(kw["calib_scale"])
            g.replay()
            want, wset = h.push(pushed, chunks, reset=reset, **({} if f32 else dict(calib_offset=coff,
                                                                                       calib_scale=cscale)))
            assert status.tolist() == [0, 0]
            assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(gset.cpu().numpy(), wset)


@pytest.mark.parametrize("dtype,cap", [(np.int16, 150000), (np.float32, 120000)], ids=["int16", "float32"])
def test_dev_session_long_caches(dtype, cap):
    """caches beyond the stateless call's window, as in the host-push session tests: == the host session at every
    push, == the oracle at the end, every slot settled"""
    f32 = _f32(dtype)
    p = StreamingConfig()
    rng = np.random.default_rng(927)
    off = float(np.float32(-215.0))
    reads = []
    for k in range(6):
        if k == 5:
            pa = rng.normal(80.0, 7.0, cap + 10000)  # no poly(A): settles on a full cache
        else:
            head = rng.normal(80.0, 7.0, cap - 38000 + 5000 * k)
            pa = np.concatenate([head, rng.normal(108.0, 2.5, 3000), 95.0 + rng.normal(0.0, 14.0, 40000)])
        reads.append(pa.astype(np.float32) if f32 else _adc_of(pa, off))
    n = len(reads)
    with _session(p, n, cap, dtype, False) as h, _session(p, n, cap, dtype, True) as d:
        pos = [0] * n
        for step in range(40):
            chunks = [r[q: q + 8000] for r, q in zip(reads, pos)]
            pos = [q + c.size for q, c in zip(pos, chunks)]
            got, settled = _push_both(h, d, np.arange(n), chunks, chunks, [step == 0] * n, off, SCALE)
            if all(settled):
                break
    assert all(settled)
    sig = [r[:cap] if f32 else calibrate(r[:cap], off, SCALE) for r in reads]
    assert list(got) == [detect_ref.mvs_stream_detect(x, p) for x in sig]
    assert (got[:5] > cap - 40000).all() and got[5] == 0
