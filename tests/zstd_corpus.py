"""zstd frames for the device decoder's tests: a corpus compressed by libzstd (the reference implementation, through
ctypes), hand-built frames with known answers and faults, and a block-header walker that reports which parts of the
compressed-block format a frame uses."""
import ctypes

import numpy as np

from adapted_b200 import svb16
from adapted_b200.synth import make_reads

MAGIC = b"\x28\xb5\x2f\xfd"
# ZSTD_cParameter values of the stable advanced API (zstd.h)
C_LEVEL, C_WINDOWLOG, C_CONTENTSIZE, C_CHECKSUM = 100, 101, 200, 201
LEVELS = (-5, 1, 3, 9, 19)


def lib():
    z = ctypes.CDLL("libzstd.so.1")
    sz, vp = ctypes.c_size_t, ctypes.c_void_p
    z.ZSTD_compressBound.restype = sz
    z.ZSTD_compressBound.argtypes = [sz]
    z.ZSTD_createCCtx.restype = vp
    z.ZSTD_freeCCtx.argtypes = [vp]
    z.ZSTD_CCtx_setParameter.restype = sz
    z.ZSTD_CCtx_setParameter.argtypes = [vp, ctypes.c_int, ctypes.c_int]
    z.ZSTD_compress2.restype = sz
    z.ZSTD_compress2.argtypes = [vp, vp, sz, vp, sz]
    z.ZSTD_compress.restype = sz
    z.ZSTD_compress.argtypes = [vp, sz, vp, sz, ctypes.c_int]
    z.ZSTD_decompress.restype = sz
    z.ZSTD_decompress.argtypes = [vp, sz, vp, sz]
    z.ZSTD_isError.restype = ctypes.c_uint
    z.ZSTD_isError.argtypes = [sz]
    return z


def compress(data: bytes, level: int, checksum: bool = False, content_size: bool = True, window_log: int = 0,
             simple: bool = False) -> bytes:
    z = lib()
    src = np.frombuffer(data, np.uint8)
    dst = np.empty(int(z.ZSTD_compressBound(src.size)) + 64, np.uint8)
    if simple:
        got = z.ZSTD_compress(dst.ctypes.data, dst.size, src.ctypes.data, src.size, level)
    else:
        cc = z.ZSTD_createCCtx()
        try:
            for k, v in ((C_LEVEL, level), (C_CHECKSUM, int(checksum)), (C_CONTENTSIZE, int(content_size)), (C_WINDOWLOG, window_log)):
                assert not z.ZSTD_isError(z.ZSTD_CCtx_setParameter(cc, k, v))
            got = z.ZSTD_compress2(cc, dst.ctypes.data, dst.size, src.ctypes.data, src.size)
        finally:
            z.ZSTD_freeCCtx(cc)
    assert not z.ZSTD_isError(got)
    return dst[:got].tobytes()


def decompress(frame: bytes, cap: int) -> bytes:
    z = lib()
    src = np.frombuffer(frame, np.uint8)
    dst = np.empty(max(cap, 1), np.uint8)
    got = z.ZSTD_decompress(dst.ctypes.data, dst.size, src.ctypes.data, src.size)
    assert not z.ZSTD_isError(got)
    return dst[:got].tobytes()


def inputs():
    """name -> bytes: the input classes the decoder must cover"""
    rng = np.random.default_rng(7)
    out = {}
    for chem, m in (("rna004", 17500), ("rna002", 30000)):
        b = make_reads(3, chem, m, seed=11)
        comp, coff, _ = svb16.encode_reads(b.adc, b.offsets)
        for i in range(3):
            out[f"svb16-{chem}-{i}"] = comp[coff[i]: coff[i + 1]].tobytes()
    # a 131 072-sample window: synthetic reads back to back (frames of several blocks)
    b = make_reads(12, "rna004", 17500, seed=12)
    adc = b.adc[b.offsets[0]:][:131072]
    comp, coff, _ = svb16.encode_reads(adc, np.array([0, adc.size], np.int64))
    out["svb16-rna004-131072"] = comp[: coff[1]].tobytes()
    out["random-1k"] = rng.integers(0, 256, 1000, dtype=np.uint8).tobytes()
    out["random-200k"] = rng.integers(0, 256, 200_000, dtype=np.uint8).tobytes()
    out["const-5k"] = b"\0" * 5000
    out["const-300k"] = b"A" * 300_000
    words = [b"poly", b"adapter", b"boundary", b"signal", b"read", b"the", b"of", b"nanopore", b"tail", b"pore"]
    text = b" ".join(words[int(k)] for k in rng.integers(0, len(words), 12000))
    out["text"] = text
    out["text-tiny"] = text[:100]
    out["tiny-200"] = rng.integers(97, 110, 200, dtype=np.uint8).tobytes()
    out["tiny-17"] = b"abcabcabcabcabcab"
    out["repeat-1"] = b"x" + b"ab" * 3000
    out["repeat-3"] = b"".join(bytes([97 + int(k) % 3]) * 1 for k in range(9000)) + rng.integers(0, 256, 500, dtype=np.uint8).tobytes()
    short = bytearray()
    for _ in range(600):
        piece = rng.integers(0, 256, int(rng.integers(1, 5)), dtype=np.uint8).tobytes()
        short += piece * int(rng.integers(2, 12))
    out["short-offsets"] = bytes(short)
    big = bytearray()
    while len(big) < 400_000:
        big += text[int(rng.integers(0, 1000)): int(rng.integers(1000, 9000))] + rng.integers(0, 256, 300, dtype=np.uint8).tobytes()
    out["big-400k"] = bytes(big)
    return out


def corpus():
    """[(name, frame, decoded)] over every input and level, with and without the frame options"""
    out = []
    for name, data in inputs().items():
        for lv in LEVELS:
            if lv == 19 and len(data) > 250_000:
                continue
            out.append((f"{name}@{lv}", compress(data, lv, simple=True), data))
        out.append((f"{name}@3+checksum", compress(data, 3, checksum=True), data))
        out.append((f"{name}@3-contentsize", compress(data, 3, content_size=False), data))
        out.append((f"{name}@9+window10", compress(data, 9, checksum=True, window_log=10), data))
    return out


# ---- block-header walker --------------------------------------------------------------------------------------------

def frame_header_size(f: bytes) -> int:
    fhd = f[4]
    single, did, fcs = (fhd >> 5) & 1, fhd & 3, fhd >> 6
    return 5 + (0 if single else 1) + (0, 1, 2, 4)[did] + ((1 if single else 0) if fcs == 0 else (1 << fcs))


def features(f: bytes) -> set:
    """which block types, literal section types and sequence table modes a frame uses"""
    feats = set()
    ip = frame_header_size(f)
    while True:
        bh = f[ip] | (f[ip + 1] << 8) | (f[ip + 2] << 16)
        ip += 3
        last, btype, size = bh & 1, (bh >> 1) & 3, bh >> 3
        feats.add(("block", ("raw", "rle", "compressed")[btype]))
        if btype == 2:
            blk = f[ip: ip + size]
            lt, lf = blk[0] & 3, (blk[0] >> 2) & 3
            if lt < 2:
                feats.add(("literals", ("raw", "rle")[lt]))
                hs = 1 if (lf & 1) == 0 else (2 if lf == 1 else 3)
                n = (blk[0] >> 3) if hs == 1 else ((blk[0] >> 4) | (blk[1] << 4) if hs == 2 else (blk[0] >> 4) | (blk[1] << 4) | (blk[2] << 12))
                q = hs + (n if lt == 0 else 1)
            else:
                feats.add(("literals", ("huffman-1" if lf == 0 else "huffman-4") if lt == 2 else "treeless"))
                hs, nb = (3, 10) if lf <= 1 else (lf + 2, 14 if lf == 2 else 18)
                h = int.from_bytes(blk[:hs], "little")
                q = hs + ((h >> (4 + nb)) & ((1 << nb) - 1))
            nseq = blk[q]
            q += 1
            if nseq >= 128:
                q += 1 if nseq < 255 else 2
            if nseq:
                modes = blk[q]
                for k, tab in ((6, "ll"), (4, "of"), (2, "ml")):
                    feats.add(("seq", ("predefined", "rle", "fse", "repeat")[(modes >> k) & 3]))
            ip += size
        else:
            ip += 1 if btype == 1 else size
        if last:
            return feats


# ---- hand-built frames -------------------------------------------------------------------------------------------

def raw_frame(content: bytes, fhd_extra: bytes = b"", fhd: int = 0x20) -> bytes:
    """single-segment frame, 1-byte content size (< 256 bytes), one raw last block"""
    return MAGIC + bytes([fhd]) + fhd_extra + bytes([len(content)]) + (len(content) << 3 | 1).to_bytes(3, "little") + content


def rle_seq_frame(of_code: int, of_extra: int, rle_literals: bool = False) -> bytes:
    """literals "abcd" (raw; "aaaa" as an RLE literals section) and one sequence with RLE-mode tables: literal length
    4, match length 3 and offset code `of_code` with `of_extra` extra bits, i.e. offset value (1 << of_code) + of_extra
    (offset = value - 3 above 3, a repeat offset below)"""
    lits = bytes([4 << 3 | 1]) + b"a" if rle_literals else bytes([4 << 3]) + b"abcd"
    bits = (1 << of_code) | of_extra  # the end marker above the offset's extra bits
    seqs = bytes([1, 0x54, 4, of_code, 0]) + bits.to_bytes(max(1, (of_code + 8) // 8), "little")
    blk = lits + seqs
    return MAGIC + bytes([0x20, 7]) + (len(blk) << 3 | 2 << 1 | 1).to_bytes(3, "little") + blk
