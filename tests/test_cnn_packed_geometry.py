"""Geometry of the packed row stream of the tensor-core convolutions (adapted_b200/csrc/adb_cnn_tc.cuh), without a GPU.

The reads of a chunk lie end to end in one row stream, S = L1 + 3 rows apart; the tiles of layer 2 (128 rows) and layer 3
(126-row stride, two rows overlap) walk that stream across read boundaries.  The arithmetic is mirrored here with the
tile constants read from the header, and checked for what the kernels rely on: every position of every read is
produced by exactly one tile of each layer, every row maps to the right (read, position), the rows around a read that
its 7-tap halo and the transposed convolution's neighbours reach are zero padding, the layer-1 input window of a tile
lines up with the x rows the prep kernels write, and the A0T buffer holds every row the tiles write or read.  The
per-read tiling (option cnn_tc_per_read_tiles) is checked the same way."""
import os
import re

import numpy as np
import pytest

HEADER = os.path.join(os.path.dirname(__file__), "..", "adapted_b200", "csrc", "adb_cnn_tc.cuh")


def _defines():
    src = open(HEADER).read()
    raw = dict(re.findall(r"^#define (TC_ROWS|TC_NQ|TC_A0T_PAD|TC_L3_STRIDE|TC_GAP)\s+([^/\n]+)", src, re.M))
    vals = {}
    while len(vals) < len(raw):
        for k, e in raw.items():
            if k not in vals:
                try:
                    vals[k] = int(eval(e, {}, dict(vals)))
                except NameError:
                    pass
    return vals


D = _defines()
ROWS, NQ, PAD, L3S, GAP = D["TC_ROWS"], D["TC_NQ"], D["TC_A0T_PAD"], D["TC_L3_STRIDE"], D["TC_GAP"]


def read_rows(L1, per_read):
    if not per_read:
        return L1 + GAP
    j2, j3 = -(-L1 // ROWS), -(-L1 // L3S)
    return (max(ROWS * j2 + PAD, L3S * (j3 - 1) + NQ) + 7) & ~7


def tiles(layer, n, L1, per_read):
    S, stride = read_rows(L1, per_read), (L3S if layer == 3 else ROWS)
    if per_read:
        jpr = -(-L1 // stride)
        return S, stride, jpr, n * jpr
    nj = -(-(n * S) // stride)
    return S, stride, nj, nj


def row0(job, S, stride, jpr):
    return (job // jpr) * S + (job % jpr) * stride


def a0t_rows(n, L1, per_read):
    S, s2, j2, n2 = tiles(2, n, L1, per_read)
    _, s3, j3, n3 = tiles(3, n, L1, per_read)
    w = row0(n2 - 1, S, s2, j2) + ROWS + PAD
    rd = row0(n3 - 1, S, s3, j3) + NQ
    return (max(w, rd) + 7) & ~7


def row_read(g, S, L1, n):
    """tc_row_read: C division truncates towards zero (rows in front of the stream: read 0, negative position)"""
    g = np.asarray(g)
    r = np.where(g >= 0, g // S, 0)
    p = g - r * S
    return r, p, (p >= 0) & (p < L1) & (r < n)


# multiples of 128 and one off, the shipped window (L1 = 550), and long preload windows
L1S = [1 * 128 - 1, 128, 129, 2 * 126, 3 * 128 - 1, 3 * 128, 3 * 128 + 1, 550, 4000, 14545]


def test_constants():
    assert (ROWS, NQ, PAD, L3S, GAP) == (128, 134, 4, 126, 3)


@pytest.mark.parametrize("per_read", [0, 1])
@pytest.mark.parametrize("L1", L1S)
@pytest.mark.parametrize("n", [1, 2, 5])
def test_packed_stream_geometry(L1, n, per_read):
    S = read_rows(L1, per_read)
    rows = a0t_rows(n, L1, per_read)
    live = np.zeros(n * S + 2 * NQ + ROWS, dtype=bool)  # indexed by g + PAD
    for layer in (2, 3):
        S_, stride, jpr, nj = tiles(layer, n, L1, per_read)
        assert S_ == S
        if per_read:
            assert nj == n * -(-L1 // stride)
        else:
            assert nj == -(-(n * S) // stride)
        owner = np.zeros((n, L1), dtype=np.int64)
        for job in range(nj):
            t0 = row0(job, S, stride, jpr) - (1 if layer == 3 else 0)
            q = np.arange(ROWS)
            g = t0 + q
            r, p, ok = row_read(g, S, L1, n)
            assert (r[ok] * S + p[ok] == g[ok]).all()
            own = ok if layer == 2 else ok & (q >= 1) & (q <= L3S)  # layer 3: rows q in [1, 126] write the output
            np.add.at(owner, (r[own], p[own]), 1)
            # operand rows (rho = g + PAD) inside the buffer
            lo, hi = t0 - 3 + PAD, t0 + ROWS + 3 + PAD
            assert lo >= 0 and hi <= rows, (layer, job, lo, hi, rows)
            if layer == 2:
                live[g + PAD] |= ok
                # layer-1 window: x index of build row q' tap k is x0 + 3 q' + k; it must be read r's sample 3 p - 3 + k
                XS = 3 * (L1 + GAP)
                x0 = (job // jpr) * XS + 3 * ((job % jpr) * ROWS) - 12
                qq = np.arange(NQ)
                rb, pb, okb = row_read(t0 - 3 + qq, S, L1, n)
                assert (x0 + 3 * qq[okb] == rb[okb] * XS + 3 * pb[okb] - 3).all()
        assert (owner == 1).all(), f"layer {layer}: positions produced {owner.min()}..{owner.max()} times"
    # every live row's 7-tap halo (+-3 rows) and transposed-convolution neighbours (+-1 row): rows of the same read at
    # the neighbouring positions, or rows that are no position of any read (zero padding)
    for g in np.flatnonzero(live) - PAD:
        r, p, _ = row_read(g, S, L1, n)
        for d in (-3, -2, -1, 1, 2, 3):
            r2, p2, ok2 = row_read(g + d, S, L1, n)
            assert (not ok2) or (r2 == r and p2 == p + d), (g, d)


@pytest.mark.parametrize("L1", L1S)
def test_x_rows_leave_the_halo_zero(L1):
    """x rows are 3 (L1 + 3) samples long: the samples a read's first and last positions reach outside [0, Lx) lie in
    the zeros behind a read"""
    XS = 3 * (L1 + GAP)
    for Lx in range(3 * L1 - 2, 3 * L1 + 1):  # every Lx with (Lx - 1) // 3 + 1 == L1
        assert (Lx - 1) // 3 + 1 == L1
        assert 3 * (L1 - 1) + 3 < XS and XS - Lx >= 9  # last position's taps; the zeros also cover the next read's x[-3..-1]


def test_shipped_window_tile_counts():
    """RNA004 window, a chunk of 7 598 reads: 4.32 / 4.39 tiles per read instead of 5"""
    n = 7598
    assert tiles(2, n, 550, 1)[3] == 5 * n and tiles(3, n, 550, 1)[3] == 5 * n
    assert tiles(2, n, 550, 0)[3] == 32826 and tiles(3, n, 550, 0)[3] == 33347
    assert a0t_rows(n, 550, 0) < a0t_rows(n, 550, 1)
