"""VBZ-style signal compression without the zstd stage: svb16(zigzag(delta(int16 samples))).

The wire format of the compressed ingest (SURVEY.md row f1) and of the compressed signal container.  It restates the
signal compression of pod5 (`c++/pod5_format/svb16`: one key BIT per value -- 0: one data byte, 1: two data bytes,
little endian, key bits LSB first, all keys in front of the data) from its published sources; pod5 itself is absent
from the image, so the layout is PARITY UNPINNED against real files.  Decoding happens on the GPU
(adapted_b200/csrc/adb_svb16.cuh); the encoders here build inputs (tests, synthetic benchmarks, container writer).

Per read: ``ceil(n / 8)`` key bytes, zero padded to a multiple of 4, then the data bytes.  Streams start 16-byte aligned
in the blob; the blob carries 16 bytes of slack behind its last stream.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

ALIGN = 16
SLACK = 16


def _stream_layout(n_samples: np.ndarray, n_two: np.ndarray):
    key_bytes = ((n_samples.astype(np.int64) + 7) // 8 + 3) // 4 * 4
    size = key_bytes + n_samples + n_two
    padded = (size + ALIGN - 1) // ALIGN * ALIGN
    off = np.zeros(n_samples.size + 1, dtype=np.int64)
    np.cumsum(padded, out=off[1:])
    return key_bytes, size, off


def encode_reads(adc: np.ndarray, offsets: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Ragged int16 reads -> (comp uint8 blob, comp_offsets int64 [n + 1], n_samples int32 [n])."""
    adc = np.ascontiguousarray(adc, dtype=np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = offsets.size - 1
    ns = np.diff(offsets).astype(np.int32)
    total = int(offsets[-1] - offsets[0]) if n > 0 else 0
    x = adc[offsets[0]: offsets[0] + total].astype(np.int32)
    prev = np.empty_like(x)
    prev[1:] = x[:-1]
    starts = (offsets[:-1] - offsets[0])[ns > 0]
    if total:
        prev[0] = 0
        prev[starts] = 0
    d = ((x - prev) & 0xFFFF).astype(np.uint16).view(np.int16).astype(np.int32)   # wrap-around int16 difference
    zz = (((d << 1) ^ (d >> 15)) & 0xFFFF).astype(np.uint32)
    two = zz > 0xFF
    read_of = np.repeat(np.arange(n), ns)
    n_two = np.bincount(read_of, weights=two, minlength=n).astype(np.int64) if total else np.zeros(n, np.int64)
    key_bytes, size, coff = _stream_layout(ns, n_two)
    comp = np.zeros(int(coff[-1]) + SLACK, dtype=np.uint8)
    if total:
        local = np.arange(total, dtype=np.int64) - np.repeat(offsets[:-1] - offsets[0], ns)
        # key bits: bit (j % 8) of byte j / 8, LSB first
        kpos = np.repeat(coff[:-1], ns) + local // 8
        np.add.at(comp, kpos[two], (1 << (local[two] % 8)).astype(np.uint8))
        # data bytes: value j of a read sits behind the bytes of the values before it
        nbytes = 1 + two.astype(np.int64)
        cum = np.cumsum(nbytes) - nbytes
        cum -= np.repeat(cum[np.minimum(offsets[:-1] - offsets[0], total - 1)], ns)
        dpos = np.repeat(coff[:-1] + key_bytes, ns) + cum
        comp[dpos] = (zz & 0xFF).astype(np.uint8)
        comp[dpos[two] + 1] = (zz[two] >> 8).astype(np.uint8)
    return comp, coff, ns


def zstd_frames(blob: np.ndarray, offsets: np.ndarray, level: int = 1) -> Tuple[np.ndarray, np.ndarray]:
    """One zstd frame (libzstd ``ZSTD_compress``) per slice ``blob[offsets[i]: offsets[i + 1]]`` -> (frames uint8 blob
    with 16 zero bytes behind the last frame, frame_offsets int64 [n + 1])."""
    from .ingest import _zstd

    z = _zstd()
    offsets = np.asarray(offsets, np.int64)
    frames, zoff = [], [0]
    for i in range(offsets.size - 1):
        src = np.ascontiguousarray(blob[offsets[i]: offsets[i + 1]])
        dst = np.empty(int(z.ZSTD_compressBound(src.size)), np.uint8)
        got = z.ZSTD_compress(dst.ctypes.data, dst.size, src.ctypes.data, src.size, int(level))
        if z.ZSTD_isError(got):
            raise RuntimeError("ZSTD_compress failed")
        frames.append(dst[:got])
        zoff.append(zoff[-1] + int(got))
    out = np.concatenate(frames + [np.zeros(SLACK, np.uint8)])
    return out, np.asarray(zoff, np.int64)


def vbz_encode_reads(adc: np.ndarray, offsets: np.ndarray, level: int = 1) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """pod5's VBZ, one zstd frame per read: ragged int16 reads -> (frames uint8 blob, frame_offsets int64 [n + 1],
    n_samples int32 [n]).  Frame i decompresses to read i's svb16 stream as ``encode_reads`` lays it out (zero padded
    to a multiple of 16 bytes), so its content size is a multiple of 16."""
    comp, coff, ns = encode_reads(adc, offsets)
    frames, foff = zstd_frames(comp, coff, level)
    return frames, foff, ns


def decode_reads(comp: np.ndarray, comp_offsets: np.ndarray, n_samples: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Plain numpy decoder (the restated pod5 svb16 scalar decoder) -> (adc int16, offsets int64 [n + 1])."""
    n = n_samples.size
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(n_samples, out=off[1:])
    out = np.zeros(int(off[-1]), dtype=np.int16)
    for r in range(n):
        k = int(n_samples[r])
        if k == 0:
            continue
        base = int(comp_offsets[r])
        kb = ((k + 7) // 8 + 3) // 4 * 4
        bits = np.unpackbits(comp[base: base + (k + 7) // 8], bitorder="little")[:k].astype(np.int64)
        pos = base + kb + np.arange(k) + np.cumsum(bits) - bits
        u = comp[pos].astype(np.uint32) | np.where(bits == 1, comp[pos + bits].astype(np.uint32) << 8, 0).astype(np.uint32)
        d = (u >> 1).astype(np.int64) ^ -(u & 1).astype(np.int64)
        out[off[r]: off[r + 1]] = (np.cumsum(d) & 0xFFFF).astype(np.uint16).view(np.int16)
    return out, off


def encode_reads_torch(adc, offsets, m: int, chunk: int = 4000):
    """Same encoder on a torch device (bench.py builds its compressed inputs in HBM): ragged int16 reads of at most
    `m` samples -> (comp uint8, comp_offsets int64 [n + 1], n_samples int32 [n])."""
    import torch

    dev = adc.device
    n = offsets.numel() - 1
    ns = (offsets[1:] - offsets[:-1]).to(torch.int64)
    t = torch.arange(m, device=dev)[None, :]
    comps, sizes = [], []
    for s in range(0, n, chunk):
        e = min(s + chunk, n)
        c = e - s
        k = ns[s:e]
        mask = t < k[:, None]
        x = torch.zeros((c, m), dtype=torch.int32, device=dev)
        x[mask] = adc[offsets[s]: offsets[e]].to(torch.int32)
        d = x.clone()
        d[:, 1:] -= x[:, :-1]
        d = ((d + 32768) & 0xFFFF) - 32768                       # wrap-around int16 difference
        zz = ((d << 1) ^ (d >> 15)) & 0xFFFF
        two = (zz > 0xFF) & mask
        n_two = two.sum(1)
        key_bytes = ((k + 7) // 8 + 3) // 4 * 4
        size = key_bytes + k + n_two
        padded = (size + ALIGN - 1) // ALIGN * ALIGN
        coff = torch.zeros(c + 1, dtype=torch.int64, device=dev)
        coff[1:] = torch.cumsum(padded, 0)
        comp = torch.zeros(int(coff[-1].item()), dtype=torch.uint8, device=dev)
        # keys: pack 8 flags per byte
        mp = (m + 7) // 8 * 8
        flags = torch.zeros((c, mp), dtype=torch.uint8, device=dev)
        flags[:, :m] = two.to(torch.uint8)
        weights = (1 << torch.arange(8, device=dev)).to(torch.uint8)
        kb = (flags.view(c, mp // 8, 8) * weights).sum(2).to(torch.uint8)
        tk = torch.arange(mp // 8, device=dev)[None, :]
        kmask = tk < ((k + 7) // 8)[:, None]
        comp[(coff[:-1, None] + tk)[kmask]] = kb[kmask]
        nbytes = (1 + two.to(torch.int64)) * mask
        pos = torch.cumsum(nbytes, 1) - nbytes + (coff[:-1] + key_bytes)[:, None]
        comp[pos[mask]] = (zz & 0xFF).to(torch.uint8)[mask]
        comp[pos[two] + 1] = (zz >> 8).to(torch.uint8)[two]
        comps.append(comp)
        sizes.append(padded)
        del x, d, zz, two, flags, kb, pos, nbytes, mask
    padded = torch.cat(sizes) if sizes else torch.zeros(0, dtype=torch.int64, device=dev)
    coff = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    coff[1:] = torch.cumsum(padded, 0)
    comp = torch.cat(comps + [torch.zeros(SLACK, dtype=torch.uint8, device=dev)])
    return comp, coff, ns.to(torch.int32)
