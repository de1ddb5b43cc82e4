"""VBZ on the host side: pod5's signal form (one zstd frame per read over its svb16 stream) from
adapted_b200.svb16.vbz_encode_reads, checked against libzstd; the container writer's bytes; the test corpus of the
device decoder (tests/test_gpu_zstd.py) and its hand-built frames checked against libzstd."""
import numpy as np

from adapted_b200 import svb16
from adapted_b200.synth import make_reads
from tests import zstd_corpus as zc


def test_vbz_encode_reads_decompresses_to_svb16_streams():
    b = make_reads(30, "rna004", 17500, seed=5, short_frac=0.2)
    comp, coff, ns = svb16.encode_reads(b.adc, b.offsets)
    frames, foff, ns2 = svb16.vbz_encode_reads(b.adc, b.offsets, level=1)
    assert np.array_equal(ns, ns2) and foff.size == ns.size + 1 and foff[0] == 0
    for i in range(ns.size):
        want = comp[coff[i]: coff[i + 1]].tobytes()
        assert zc.decompress(frames[foff[i]: foff[i + 1]].tobytes(), len(want)) == want
    assert frames[foff[-1]:].tolist() == [0] * 16
    wire = foff[-1] / (b.offsets[-1] - b.offsets[0])
    assert wire < (coff[-1] / (b.offsets[-1] - b.offsets[0]))  # the zstd stage shrinks svb16 streams of synthetic signal


def test_container_v2_zstd_bytes_unchanged(tmp_path):
    """write_container_v2(zstd=True) writes what the per-read ZSTD_compress(level 1) loop wrote"""
    from adapted_b200.ingest import read_container_v2, write_container_v2

    b = make_reads(25, "rna002", 30000, seed=9)
    ids = [f"r{i}" for i in range(25)]
    p = write_container_v2(str(tmp_path / "c"), b.adc, b.offsets, b.full_lens, b.calib_offset, b.calib_scale, ids, zstd=True)
    c = read_container_v2(p)
    comp, coff, _ = svb16.encode_reads(b.adc, b.offsets)
    frames = [zc.compress(comp[coff[i]: coff[i + 1]].tobytes(), 1, simple=True) for i in range(25)]
    want = b"".join(frames) + b"\0" * 16
    zoff = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    assert np.array_equal(np.asarray(c["comp_offsets"]), zoff)
    blob = np.asarray(c["comp"]).tobytes()
    assert blob[: len(want)] == want


def test_hand_built_frames_against_libzstd():
    assert zc.decompress(zc.rle_seq_frame(2, 3), 7) == b"abcdabc"  # offset 4
    assert zc.decompress(zc.rle_seq_frame(1, 0), 7) == b"abcdabc"  # offset value 2: the 2nd initial repeat offset (4)
    assert zc.decompress(zc.rle_seq_frame(2, 3, rle_literals=True), 7) == b"aaaaaaa"
    assert zc.decompress(zc.raw_frame(b"hello"), 5) == b"hello"


def test_corpus_covers_the_block_format():
    """every block type, literal section type and sequence table mode of RFC 8878 appears in the corpus, except RLE
    literals: libzstd 1.5.5 emits them only for a block whose literals are one repeated byte and that still has
    sequences, which none of these inputs produce reliably, so the hand-built frames of test_gpu_zstd.py add one"""
    seen = set()
    for name, frame, data in zc.corpus():
        seen |= zc.features(frame)
    for want in [("block", "raw"), ("block", "rle"), ("block", "compressed"), ("literals", "raw"), ("literals", "huffman-1"),
                 ("literals", "huffman-4"), ("literals", "treeless"), ("seq", "predefined"), ("seq", "fse"), ("seq", "repeat"),
                 ("seq", "rle")]:
        assert want in seen, want
