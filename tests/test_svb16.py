"""The compressed ingest format (svb16 + zig-zag + delta, pod5's VBZ minus zstd; restated, PARITY UNPINNED against
pod5 itself): encoder / numpy decoder round trips on the CPU, the CUDA decode kernel and the compressed pipelined
ingest on the GPU."""
import numpy as np
import pytest

from adapted_b200 import svb16
from adapted_b200.config import get_chemistry_specific_config
from adapted_b200.synth import make_reads


def _cases():
    rng = np.random.default_rng(0)
    out = {}
    b = make_reads(40, "rna004", 17500, seed=3, short_frac=0.3)
    out["synthetic"] = (b.adc, b.offsets)
    # every int16 value incl. the wrap-around deltas (-32768 -> 32767), empty reads, lengths around 8 / 32 / 128
    lens = [0, 1, 7, 8, 9, 31, 32, 33, 127, 128, 129, 255, 256, 257, 0, 1000, 4097]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    adc = rng.integers(-32768, 32768, size=int(off[-1])).astype(np.int16)
    adc[:4] = [-32768, 32767, -32768, 0]
    out["extremes"] = (adc, off)
    small = (rng.normal(0, 20, size=50000).cumsum() * 0.01 + rng.normal(0, 30, size=50000)).astype(np.int16)
    out["one_long_read"] = (small, np.array([0, 50000], np.int64))
    return out


@pytest.mark.parametrize("name", ["synthetic", "extremes", "one_long_read"])
def test_encode_decode_round_trip_numpy(name):
    adc, off = _cases()[name]
    comp, coff, ns = svb16.encode_reads(adc, off)
    assert coff[0] == 0 and np.all(coff % 16 == 0) and comp.size == coff[-1] + 16
    dec, doff = svb16.decode_reads(comp, coff, ns)
    assert np.array_equal(dec, adc) and np.array_equal(doff, off)


def test_known_answer_stream():
    """hand-computed stream: samples 3, 2, 300, -200 -> deltas 3, -1, 298, -500 -> zig-zag 6, 1, 596, 999"""
    comp, coff, ns = svb16.encode_reads(np.array([3, 2, 300, -200], np.int16), np.array([0, 4]))
    assert ns.tolist() == [4] and coff.tolist() == [0, 16]
    assert comp[:4].tolist() == [0b1100, 0, 0, 0]                       # keys: values 2 and 3 take two bytes
    assert comp[4:10].tolist() == [6, 1, 596 & 0xFF, 596 >> 8, 999 & 0xFF, 999 >> 8]


def test_torch_encoder_equals_numpy_encoder():
    import torch

    adc, off = _cases()["synthetic"]
    comp, coff, ns = svb16.encode_reads(adc, off)
    c2, o2, n2 = svb16.encode_reads_torch(torch.from_numpy(adc), torch.from_numpy(off), 17500, chunk=7)
    assert np.array_equal(c2.numpy(), comp) and np.array_equal(o2.numpy(), coff) and np.array_equal(n2.numpy(), ns)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["synthetic", "extremes", "one_long_read"])
def test_cuda_decode_round_trip(name):
    from adapted_b200.detect import svb16_decode

    adc, off = _cases()[name]
    comp, coff, ns = svb16.encode_reads(adc, off)
    dec, doff = svb16_decode(comp, coff, ns)
    assert np.array_equal(doff, off)
    assert np.array_equal(dec, adc)


def _pipelined(ctx, comp, coff, ns, b, spc, w, minibatch_size, chunk_minibatches, vbz=False):
    """adb_detect_pipelined_svb_host / _vbz_host called on `ctx` directly, without the checks of detect_reads_svb ->
    (status code, records, batch status)"""
    import ctypes as C

    from adapted_b200 import _lib
    from adapted_b200.config import flatten_config
    from adapted_b200.detect import flatten_cnn_weights

    flat = flatten_config(spc)
    comp, coff, ns = np.ascontiguousarray(comp, np.uint8), np.ascontiguousarray(coff, np.int64), np.ascontiguousarray(ns, np.int32)
    lens, co, cs = (np.ascontiguousarray(x, t) for x, t in ((b.full_lens, np.int32), (b.calib_offset, np.float32), (b.calib_scale, np.float32)))
    wf = flatten_cnn_weights(w) if flat["primary_method"] == 1 else None
    recs = np.zeros(lens.size, _lib.RECORD_DTYPE)
    status = np.zeros((lens.size + minibatch_size - 1) // minibatch_size, np.int32)
    sb = _lib.AdbSvbBatch(comp=comp.ctypes.data, comp_offsets=coff.ctypes.data, n_samples=ns.ctypes.data, n_reads=lens.size,
                          m=int(flat["sig_preload_size"]), batch_size=minibatch_size, full_lens=lens.ctypes.data,
                          calib_offset=co.ctypes.data, calib_scale=cs.ctypes.data)
    cfg = _lib.fill_config(flat)
    L = _lib.load()
    entry = L.adb_detect_pipelined_vbz_host if vbz else L.adb_detect_pipelined_svb_host
    rc = entry(ctx.handle, C.byref(sb), C.byref(cfg), wf.ctypes.data if wf is not None else None, recs.ctypes.data,
               status.ctypes.data, chunk_minibatches)
    return rc, recs, status


@pytest.mark.gpu
@pytest.mark.parametrize("chem,kw", [("rna002", {}), ("rna004", {"short_frac": 0.2}), ("rna004", {"stress": True})])
def test_compressed_ingest_equals_plain_ingest(chem, kw):
    """records of the compressed pipelined ingest (H2D of svb16 streams, device decode) == records of the plain int16
    call, byte for byte, incl. a short last minibatch: with every minibatch a chunk and with small chunks at both ends
    (the default context and its twin), and on a context without a twin, in one chunk and in two chunks that alternate
    between its staging slots"""
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads, detect_reads_svb
    from tests.golden_io import load_cnn_weights

    spc = get_chemistry_specific_config(chem)
    w = load_cnn_weights() if chem == "rna004" else None
    b = make_reads(1130, chem, spc.sig_preload_size, seed=91, **kw)
    want, st_want = detect_reads(b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w, minibatch_size=100,
                                 return_records=True)
    comp, coff, ns = svb16.encode_reads(b.adc, b.offsets)
    for chunk in (1, 3):
        got, st_got = detect_reads_svb(comp, coff, ns, b.full_lens, b.calib_offset, b.calib_scale, spc, model=w, minibatch_size=100,
                                       chunk_minibatches=chunk)
        assert np.array_equal(st_got, st_want), chunk
        assert got.tobytes() == want.tobytes(), chunk
    ctx = _lib.Context(0)
    try:
        for chunk in (64, 8):  # 12 minibatches: one chunk, then chunks of 8 and 4
            rc, got, st_got = _pipelined(ctx, comp, coff, ns, b, spc, w, 100, chunk)
            assert rc == 0, _lib.load().adb_last_error()
            assert np.array_equal(st_got, st_want), chunk
            assert got.tobytes() == want.tobytes(), chunk
    finally:
        ctx.close()


@pytest.mark.gpu
def test_compressed_entry_points_refuse_n_samples_above_m():
    """a C caller's n_samples outside [0, m] is refused by every compressed entry point before anything is decoded"""
    import ctypes as C

    from adapted_b200 import _lib

    spc = get_chemistry_specific_config("rna002")
    m = int(spc.sig_preload_size)
    b = make_reads(30, "rna002", m, seed=4)
    comp, coff, ns = svb16.encode_reads(b.adc, b.offsets)
    frames, foff, _ = svb16.vbz_encode_reads(b.adc, b.offsets)
    ns = ns.copy()
    ns[7] = m + 1
    ctx = _lib.Context(0)
    try:
        for vbz, data, offs in ((False, comp, coff), (True, frames, foff)):
            rc, _, _ = _pipelined(ctx, data, offs, ns, b, spc, None, 10, 1, vbz=vbz)
            assert rc == -2 and _lib.load().adb_last_error() == b"n_samples outside [0, m]", (vbz, rc)
        sb = _lib.AdbSvbBatch(comp=comp.ctypes.data, comp_offsets=coff.ctypes.data, n_samples=ns.ctypes.data, n_reads=ns.size, m=m,
                              batch_size=10, full_lens=b.full_lens.ctypes.data, calib_offset=b.calib_offset.ctypes.data,
                              calib_scale=b.calib_scale.ctypes.data)
        out = np.zeros(int(ns.astype(np.int64).sum()), np.int16)
        assert _lib.load().adb_svb16_decode_host(ctx.handle, C.byref(sb), out.ctypes.data) == -2
        assert _lib.load().adb_last_error() == b"n_samples outside [0, m]"
    finally:
        ctx.close()


@pytest.mark.parametrize("zstd", [False, True])
def test_container_v2_round_trip(tmp_path, zstd):
    """ADBSIG02 (the native pipeline's input): streams come back bit-exact through the numpy decoder, with and without
    the zstd stage (pod5's VBZ = zstd over svb16); reads longer than the preload window are cut when written"""
    from adapted_b200.ingest import F_SVB16, F_ZSTD, _zstd, read_container_v2, write_container_v2

    b = make_reads(12, "rna004", 30000, seed=5, short_frac=0.3)
    ids = [f"read-{i:04d}" for i in range(b.n)]
    p = write_container_v2(str(tmp_path / "c"), b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, ids, zstd=zstd,
                           preload_size=17500)
    c = read_container_v2(p)
    assert c["flags"] == (F_SVB16 | (F_ZSTD if zstd else 0))
    assert [x.decode() for x in c["read_ids"]] == ids and np.array_equal(c["full_lens"], b.full_lens)
    comp, coff = np.asarray(c["comp"]), np.asarray(c["comp_offsets"])
    if zstd:
        z = _zstd()
        streams, off = [], [0]
        for i in range(b.n):
            src = np.ascontiguousarray(comp[coff[i]: coff[i + 1]])
            dst = np.zeros(80000, np.uint8)
            got = z.ZSTD_decompress(dst.ctypes.data, dst.size, src.ctypes.data, src.size)
            assert not z.ZSTD_isError(got)
            streams.append(dst[: (got + 15) // 16 * 16])
            off.append(off[-1] + streams[-1].size)
        comp, coff = np.concatenate(streams + [np.zeros(16, np.uint8)]), np.asarray(off, np.int64)
    dec, doff = svb16.decode_reads(comp, coff, np.asarray(c["n_samples"]))
    want = np.concatenate([b.adc[b.offsets[i]: b.offsets[i] + min(17500, b.offsets[i + 1] - b.offsets[i])] for i in range(b.n)])
    assert np.array_equal(dec, want)
