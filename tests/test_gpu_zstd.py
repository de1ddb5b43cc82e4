"""The zstd stage of VBZ on the GPU (zstd_decode_kernel, adb_zstd.cuh): byte parity with libzstd over a corpus that
uses every part of the compressed-block format (tests/zstd_corpus.py; the walker there asserts the coverage on the
CPU, tests/test_zstd_host.py), a fixed set of malformed frames that must be refused without a write outside their slot,
and the VBZ pipelines against the svb16 ones."""
import numpy as np
import pytest

from adapted_b200 import svb16
from adapted_b200.config import get_chemistry_specific_config
from adapted_b200.synth import make_reads
from tests import zstd_corpus as zc
from tests.golden_io import load_cnn_weights

pytestmark = pytest.mark.gpu
GUARD = 64


def _decode(frames, caps):
    """every frame followed by a guard slot (an empty frame: refused before any write) -> [(status, slot bytes)]"""
    from adapted_b200.detect import zstd_decompress

    blob, offs, cap = [], [0], []
    for f, c in zip(frames, caps):
        blob += [f, b""]
        offs += [offs[-1] + len(f)] * 2
        cap += [c, GUARD]
    out, st = zstd_decompress(np.frombuffer(b"".join(blob) or b"\0", np.uint8), np.asarray(offs), np.asarray(cap))
    o = np.concatenate([[0], np.cumsum(cap)])
    slots = [out[o[k]: o[k + 1]].tobytes() for k in range(len(cap))]
    for k in range(1, len(cap), 2):
        assert st[k] == -1 and slots[k] == b"\0" * GUARD, "a guard slot was written"
    return [(int(st[k]), slots[k]) for k in range(0, len(cap), 2)]


def test_zstd_parity_with_libzstd():
    corpus = zc.corpus()
    got = _decode([f for _, f, _ in corpus], [len(d) for _, _, d in corpus])
    bad = [name for (name, _, d), (s, b) in zip(corpus, got) if s != len(d) or b != d]
    assert not bad, bad[:10]


def test_hand_built_frames():
    """known answers: RLE-mode sequence tables, a new offset, a repeat offset, RLE literals (which libzstd 1.5.5 did
    not emit for any corpus input), a raw block"""
    frames = [zc.rle_seq_frame(2, 3), zc.rle_seq_frame(1, 0), zc.rle_seq_frame(2, 3, rle_literals=True), zc.raw_frame(b"hello")]
    want = [b"abcdabc", b"abcdabc", b"aaaaaaa", b"hello"]
    assert _decode(frames, [len(w) for w in want]) == [(len(w), w) for w in want]


def test_refusals():
    data = zc.inputs()["text"]
    plain = zc.compress(data, 3)
    cks = zc.compress(data, 3, checksum=True)
    reserved = bytearray(plain)
    reserved[zc.frame_header_size(plain)] |= 6  # first block header: type 3
    cks_bad = bytearray(cks)
    cks_bad[-1] ^= 0x40
    cases = [
        ("truncated", plain[:-5], len(data), -1),
        ("reserved block type", bytes(reserved), len(data), -3),
        ("dictionary id", zc.raw_frame(b"hello", fhd_extra=b"\x07", fhd=0x21), 5, -4),
        ("offset beyond the output", zc.rle_seq_frame(5, 0), 7, -6),
        ("checksum mismatch", bytes(cks_bad), len(data), -8),
        ("content size above the capacity", plain, len(data) - 1, -5),
    ]
    got = _decode([c[1] for c in cases] + [plain], [c[2] for c in cases] + [len(data)])
    for (name, _, _, code), (s, _) in zip(cases, got):
        assert s == code, (name, s)
    assert got[-1] == (len(data), data)  # a good frame behind the refused ones


@pytest.mark.parametrize("chem", ["rna002", "rna004"])
def test_detect_reads_vbz_equals_svb(chem):
    from adapted_b200.detect import detect_reads_svb, detect_reads_vbz

    spc = get_chemistry_specific_config(chem)
    m = int(spc.sig_preload_size)
    b = make_reads(700, chem, m, seed=21, short_frac=0.05)
    w = load_cnn_weights() if chem == "rna004" else None
    comp, coff, ns = svb16.encode_reads(b.adc, b.offsets)
    frames, foff, ns2 = svb16.vbz_encode_reads(b.adc, b.offsets)
    assert foff[-1] < coff[-1]
    args = (b.full_lens, b.calib_offset, b.calib_scale, spc, w)
    r1, s1 = detect_reads_svb(comp, coff, ns, *args, minibatch_size=100, chunk_minibatches=2)
    r2, s2 = detect_reads_vbz(frames, foff, ns2, *args, minibatch_size=100, chunk_minibatches=2)
    assert np.array_equal(s1, s2)
    assert r1.tobytes() == r2.tobytes()


def test_detect_reads_vbz_refuses_a_corrupt_frame():
    from adapted_b200 import _lib
    from adapted_b200.detect import detect_reads_vbz

    spc = get_chemistry_specific_config("rna002")
    b = make_reads(50, "rna002", int(spc.sig_preload_size), seed=22)
    frames, foff, ns = svb16.vbz_encode_reads(b.adc, b.offsets)
    frames = frames.copy()
    h = int(foff[10])
    assert frames[h + 4] == 0x60  # single segment, 2-byte content size (value - 256)
    frames[h + 6] += 1  # read 10 claims 256 bytes more than it decodes to
    with pytest.raises(_lib.AdbError):
        detect_reads_vbz(frames, foff, ns, b.full_lens, b.calib_offset, b.calib_scale, spc, minibatch_size=25)


def _native(paths, out, spc, w, host_zstd=False):
    from adapted_b200 import _lib
    from adapted_b200.ingest import detect_files_native

    ctx = _lib.default_context(0)
    ctx.set_option("host_zstd", int(host_zstd))
    try:
        s = detect_files_native(paths, out, spc, model=w, minibatch_size=100, batch_size_output=64, chunk_minibatches=3)
    finally:
        ctx.set_option("host_zstd", 0)
    return s, ctx.query("zstd_host_frames")


@pytest.mark.parametrize("chem", ["rna002", "rna004"])
def test_native_pipeline_vbz_device_decode(tmp_path, chem):
    """zstd containers decoded on the device give the tables of the same reads as svb16 containers and of the host
    decompression, with minibatches running across files and the open-pore overflow read included"""
    from tests.test_gpu_native_pipeline import _tables, _write_job

    (tmp_path / "z").mkdir()
    (tmp_path / "s").mkdir()
    spc, _, vz = _write_job(tmp_path / "z", chem, (530, 260, 415), 300, "zstd")
    _, _, vs = _write_job(tmp_path / "s", chem, (530, 260, 415), 300, "svb16")
    w = load_cnn_weights() if chem == "rna004" else None
    ss, _ = _native(vs, str(tmp_path / "o_svb"), spc, w)
    sd, nd = _native(vz, str(tmp_path / "o_dev"), spc, w)
    sh, nh = _native(vz, str(tmp_path / "o_host"), spc, w, host_zstd=True)
    assert nd == 0 and nh == 1205
    keys = ("reads", "pass", "fail", "lost", "files")
    assert {k: sd[k] for k in keys} == {k: ss[k] for k in keys} == {k: sh[k] for k in keys}
    t_svb, t_dev, t_host = _tables(str(tmp_path / "o_svb")), _tables(str(tmp_path / "o_dev")), _tables(str(tmp_path / "o_host"))
    assert len(t_svb) == ss["files"] and t_dev == t_svb and t_host == t_svb
    assert sd["h2d_bytes"] < ss["h2d_bytes"]


def test_native_pipeline_vbz_long_window(tmp_path):
    """a 131 072-sample preload window: frames of several blocks go through the device path"""
    from adapted_b200.ingest import write_container_v2
    from tests.test_gpu_long_window import long_config, long_reads
    from tests.test_gpu_native_pipeline import _tables

    m = 131072
    spc = long_config("rna004", m)
    b = long_reads("rna004", m, 60, seed=7701)
    ids = [f"long-{i}" for i in range(60)]
    p = {form: write_container_v2(str(tmp_path / form), b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, ids,
                                  zstd=form == "zstd") for form in ("svb16", "zstd")}
    w = load_cnn_weights()
    ss, _ = _native([p["svb16"]], str(tmp_path / "o_svb"), spc, w)
    sd, nd = _native([p["zstd"]], str(tmp_path / "o_dev"), spc, w)
    assert nd == 0 and sd["reads"] == ss["reads"] == 60
    assert _tables(str(tmp_path / "o_dev")) == _tables(str(tmp_path / "o_svb"))


def test_native_pipeline_vbz_dictionary_frame(tmp_path):
    """a frame that names a dictionary stays on the host path and fails the job as under host_zstd"""
    from adapted_b200 import _lib
    from adapted_b200.ingest import read_container_v2, write_container_v2

    spc = get_chemistry_specific_config("rna002")
    b = make_reads(120, "rna002", int(spc.sig_preload_size), seed=41)
    ids = [f"r{i}" for i in range(120)]
    path = write_container_v2(str(tmp_path / "c"), b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, ids, zstd=True)
    c = read_container_v2(path)
    raw = bytearray(open(path, "rb").read())
    hdr = np.frombuffer(bytes(raw[:128]), dtype=[("m", "S8"), ("v", "<u4"), ("f", "<u4"), ("n", "<u8"), ("w", "<u4"), ("r", "<u4"),
                                                 ("o", "<u8", (8,)), ("x", "u1", (32,))])
    off_blob = int(hdr["o"][0][6])
    f0 = off_blob + int(np.asarray(c["comp_offsets"])[60])
    assert raw[f0 + 4] == 0x60
    raw[f0 + 4] = 0x60 | 1  # dictionary ID flag 1: the first content-size byte now reads as the dictionary ID
    open(path, "wb").write(bytes(raw))
    msgs = []
    for host in (False, True):
        with pytest.raises(_lib.AdbError) as e:
            _native([path], str(tmp_path / f"o{int(host)}"), spc, None, host_zstd=host)
        msgs.append((e.value.status, str(e.value)))
    assert msgs[0] == msgs[1]
