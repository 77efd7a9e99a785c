"""Expected tiles of the halo exchanges when every interior cell holds its GLOBAL linear index y * nx + x (plus an
offset that changes between exchanges): a ghost cell must then hold exactly the index of the cell across its edge --
wrapped when the exchange is periodic in that direction -- or stay untouched (corners, non-periodic domain edges).
Unlike the part ids of halo_check.py this checks WHICH cell arrived, not only from which part.  Everything is
vectorised over the ghost cells (per-part work is numpy slices), so it is fast enough for thousands of parts."""
import numpy as np

UNTOUCHED = -7.0


def tile_offsets(boxes):
    """offsets[P + 1] of the framed tiles, the ddc_halo_tile_offsets layout"""
    b = np.asarray(boxes, dtype=np.int64)
    sizes = (b[:, 2] + 2) * (b[:, 3] + 2)
    return np.concatenate([[0], np.cumsum(sizes)])


def initial_tiles(boxes, offsets, nx, add=0.0):
    """interiors = global index + add, frames UNTOUCHED"""
    buf = np.full(int(offsets[-1]), UNTOUCHED, dtype=np.float64)
    for p, (x0, y0, ex, ey) in enumerate(np.asarray(boxes, dtype=np.int64)):
        t = buf[offsets[p]:offsets[p + 1]].reshape(ey + 2, ex + 2)
        t[1:-1, 1:-1] = (y0 + np.arange(ey))[:, None] * nx + (x0 + np.arange(ex))[None, :] + add
    return buf


def _runs(lengths):
    """for ranges of the given lengths laid end to end: (range index, position in the range) of every element"""
    lengths = np.asarray(lengths, dtype=np.int64)
    g = np.repeat(np.arange(len(lengths)), lengths)
    start = np.cumsum(lengths) - lengths
    return g, np.arange(int(lengths.sum())) - start[g]


def ghost_cells(boxes, offsets):
    """(buffer index, x, y of the cell across the edge) of every ghost cell that is not a corner, all parts"""
    b = np.asarray(boxes, dtype=np.int64)
    x0, y0, ex, ey = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    off = np.asarray(offsets, dtype=np.int64)[:-1]
    idx, xs, ys = [], [], []
    g, j = _runs(ey)  # left and right ghosts, rows j of the box
    for right in (False, True):
        idx.append(off[g] + (j + 1) * (ex[g] + 2) + (ex[g] + 1 if right else 0))
        xs.append(x0[g] + ex[g] if right else x0[g] - 1)
        ys.append(y0[g] + j)
    g, i = _runs(ex)  # bottom and top ghosts, columns i of the box
    for top in (False, True):
        idx.append(off[g] + (ey[g] + 1 if top else 0) * (ex[g] + 2) + i + 1)
        xs.append(x0[g] + i)
        ys.append(y0[g] + ey[g] if top else y0[g] - 1)
    return np.concatenate(idx), np.concatenate(xs), np.concatenate(ys)


def expected_tiles(boxes, offsets, nx, ny, px, py, periodic, add=0.0):
    """initial_tiles(add) after one exchange (interior lists; periodic: the periodic ones too)"""
    buf = initial_tiles(boxes, offsets, nx, add)
    if len(boxes) < 2:
        return buf  # one part: no neighbour tables, nothing is exchanged
    idx, x, y = ghost_cells(boxes, offsets)
    ok = np.ones(len(idx), dtype=bool)
    if not (periodic and px):
        ok &= (x >= 0) & (x < nx)
    if not (periodic and py):
        ok &= (y >= 0) & (y < ny)
    buf[idx[ok]] = ((y % ny) * nx + (x % nx))[ok] + add
    return buf


def shard_ranges(P, G):
    """[(p_begin, p_count)] of every rank: ddc_shard_parts"""
    return [(r * P // G, (r + 1) * P // G - r * P // G) for r in range(G)]


def max_shard_total(boxes, G):
    """the largest rank's tile total: what every rank's halo buffer must hold"""
    off = tile_offsets(boxes)
    return max(int(off[b + c] - off[b]) for b, c in shard_ranges(len(boxes), G))
