"""The column butterflies of the symmetric forward epilogues (csrc/dsoft_kernels.cuh: warp_colsum32 for the 32x32b
TMEM load shape of the one-pass CLIP forward, dsoft_fwd_kernel<MODE_CLIP_SYM>; warp_colsum8 for the 16x256b one of the
symmetric soft forward, dsoft_fwd_kernel<MODE_SOFT_SYM16>), restated lane by lane in numpy: which column's total a lane
ends up with, and that the total is the sum over all 32 rows of the warp.  The CUDA kernels are checked end to end by the GPU
parity tests; this pins the index algebra the kernel comments state (DESIGN section 3)."""
import numpy as np


def shfl_xor(vals, mask):
    """vals[lane] -> value received from lane ^ mask."""
    return np.array([vals[lane ^ mask] for lane in range(32)])


def colsum32(x):
    """x[lane, k]: lane = row, k = column of a 32-column chunk.  Five stages, 31 shuffles; lane l returns column l."""
    x = x.copy()
    for off in (16, 8, 4, 2, 1):
        up = (np.arange(32) & off) != 0
        for i in range(off):
            send = np.where(up, x[:, i], x[:, i + off])
            keep = np.where(up, x[:, i + off], x[:, i])
            x[:, i] = keep + shfl_xor(send, off)
    return x[:, 0]


def fragment_16x256b(tile):
    """tile[row, col] (32 x 32) -> per lane the 4 x 8 values tcgen05.ld.16x256b.x4 (two loads: lanes +0 / +16) delivers:
    lane (g = lane // 4, c2 = lane % 4) holds rows g + 8 i (i = 0..3) and columns 8 j + 2 c2 + e (j = 0..3, e = 0..1)."""
    frag = np.zeros((32, 4, 4, 2))
    for lane in range(32):
        g, c2 = lane // 4, lane % 4
        for i in range(4):
            for j in range(4):
                for e in range(2):
                    frag[lane, i, j, e] = tile[g + 8 * i, 8 * j + 2 * c2 + e]
    return frag


def colsum8(frag):
    """In-register sum over the thread's four rows, then three butterfly stages over the eight row groups (7 shuffles).
    Returns per lane (value, column)."""
    v = frag.sum(axis=1).reshape(32, 8)  # [lane, 2 j + e]
    for off, n in ((16, 4), (8, 2), (4, 1)):
        up = (np.arange(32) & off) != 0
        for k in range(n):
            send = np.where(up, v[:, k], v[:, k + n])
            keep = np.where(up, v[:, k + n], v[:, k])
            v[:, k] = keep + shfl_xor(send, off)
    lanes = np.arange(32)
    g, c2 = lanes // 4, lanes % 4
    return v[:, 0], 8 * (g // 2) + 2 * c2 + (g % 2)


def test_colsum32_returns_column_of_lane():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((32, 32))
    np.testing.assert_allclose(colsum32(x), x.sum(axis=0), rtol=1e-12, atol=1e-12)


def test_colsum8_fragment_mapping():
    rng = np.random.default_rng(1)
    tile = rng.standard_normal((32, 32))
    total, col = colsum8(fragment_16x256b(tile))
    assert sorted(col.tolist()) == list(range(32))  # every column of the chunk lands in exactly one lane
    np.testing.assert_allclose(total, tile.sum(axis=0)[col], rtol=1e-12, atol=1e-12)


def test_row_owner_after_group_reduction():
    """Row sums: xor 1 and xor 2 combine the four lanes of a row group; lane c2 keeps row g + 8 c2 - 32 distinct rows."""
    lanes = np.arange(32)
    rows = lanes // 4 + 8 * (lanes % 4)
    assert sorted(rows.tolist()) == list(range(32))
    rng = np.random.default_rng(2)
    tile = rng.standard_normal((32, 32))
    frag = fragment_16x256b(tile)
    part = frag.sum(axis=(2, 3))  # [lane, i]: the thread's share of its four rows
    for off in (1, 2):
        part = part + np.stack([shfl_xor(part[:, i], off) for i in range(4)], axis=1)
    got = part[lanes, lanes % 4]
    np.testing.assert_allclose(got, tile.sum(axis=1)[rows], rtol=1e-12, atol=1e-12)
