"""Expectations of the halo calls with ghost frames of width w (ddc_halo_set_width).

Tile p is (ey + 2 w) x (ex + 2 w), interior cell (i, j) at row j + w, column i + w.  A frame cell at (x, y) gets the
cell's value when the cell -- wrapped in the directions in which it lies outside the domain, all of which must be
periodic (and the exchange periodic) -- lies in a positive-area box; an edge exchange fills only the cells beside the
box's edges, a full exchange the corner blocks too.  The sources come from halo_frame.owner_map, painted over the whole
domain, so these expectations share only the rule with the library's bucket search and rectangle items."""
import numpy as np

import halo_frame as hf
import halo_global as hg


def tile_offsets(boxes, w):
    """offsets[P + 1] of the tiles with frames of width w (ddc_halo_tile_offsets after ddc_halo_set_width(w))"""
    b = np.asarray(boxes, dtype=np.int64)
    sizes = (np.maximum(b[:, 2], 0) + 2 * w) * (np.maximum(b[:, 3], 0) + 2 * w)
    return np.concatenate([[0], np.cumsum(sizes)])


def max_shard_total(boxes, G, w):
    off = tile_offsets(boxes, w)
    return max(int(off[b + c] - off[b]) for b, c in hg.shard_ranges(len(boxes), G))


def scattered(boxes, off, field, tiles, w):
    """tiles with every interior replaced by the field (any dtype of the field's)"""
    out = tiles.copy()
    for p, (x0, y0, ex, ey) in enumerate(np.asarray(boxes, dtype=np.int64)):
        if ex > 0 and ey > 0:
            out[off[p]:off[p + 1]].reshape(ey + 2 * w, ex + 2 * w)[w:w + ey, w:w + ex] = field[y0:y0 + ey, x0:x0 + ex]
    return out


def initial_tiles(boxes, off, nx, ny, w, add=0.0):
    """interiors = global index + add, frames UNTOUCHED"""
    field = np.arange(nx * ny, dtype=np.float64).reshape(ny, nx) + add
    return scattered(boxes, off, field, np.full(int(off[-1]), hg.UNTOUCHED, dtype=np.float64), w)


def frame_cells(boxes, off, w):
    """(buffer index, x, y, corner) of every frame cell of every tile: the bottom and top bands (full tile width) and
    the left and right bands beside the box"""
    b = np.asarray(boxes, dtype=np.int64)
    x0, y0, ex, ey = b[:, 0], b[:, 1], np.maximum(b[:, 2], 0), np.maximum(b[:, 3], 0)
    tw = ex + 2 * w
    o = np.asarray(off, dtype=np.int64)[:-1]
    P = len(b)
    bands = [  # (first row, rows, first column, columns) per part
        (np.zeros(P, np.int64), np.full(P, w), np.zeros(P, np.int64), tw),
        (ey + w, np.full(P, w), np.zeros(P, np.int64), tw),
        (np.full(P, w), ey, np.zeros(P, np.int64), np.full(P, w)),
        (np.full(P, w), ey, ex + w, np.full(P, w)),
    ]
    idx, xs, ys, cs = [], [], [], []
    for r0, nr, c0, nc in bands:
        g, k = hg._runs(nr * nc)
        r, c = r0[g] + k // nc[g], c0[g] + k % nc[g]
        idx.append(o[g] + r * tw[g] + c)
        xs.append(x0[g] + c - w)
        ys.append(y0[g] + r - w)
        cs.append(((c < w) | (c >= w + ex[g])) & ((r < w) | (r >= w + ey[g])))
    return np.concatenate(idx), np.concatenate(xs), np.concatenate(ys), np.concatenate(cs)


def exchanged(boxes, off, nx, ny, px, py, periodic, full, field, tiles, w, tables=None):
    """tiles after an edge (full: full-frame) exchange of width w when every interior holds the field [ny, nx]: every
    frame cell with a source holds the field value of its wrapped cell, the others keep what they held.  tables:
    whether the handle has neighbour tables (default: more than one part, as after ddc_partition)"""
    out = tiles.copy()
    if not (len(boxes) > 1 if tables is None else tables):
        return out
    idx, x, y, corner = frame_cells(boxes, off, w)
    own = hf.owner_map(boxes, nx, ny)
    ok = own[y % ny, x % nx] >= 0
    if not (periodic and px):
        ok &= (x >= 0) & (x < nx)
    if not (periodic and py):
        ok &= (y >= 0) & (y < ny)
    if not full:
        ok &= ~corner
    out[idx[ok]] = field[(y % ny)[ok], (x % nx)[ok]]
    return out


def expected(boxes, off, nx, ny, px, py, periodic, full, w, add=0.0, tables=None):
    """initial_tiles(add) after one exchange of width w"""
    field = np.arange(nx * ny, dtype=np.float64).reshape(ny, nx) + add
    return exchanged(boxes, off, nx, ny, px, py, periodic, full, field, initial_tiles(boxes, off, nx, ny, w, add), w,
                     tables)


def tiny_periodic_cases(oracle):
    """domains narrower and lower than the widest frame: the strips wrap several times; every periodic combination"""
    for k, (nx, ny, P) in enumerate([(2, 3, 2), (3, 2, 3), (4, 4, 3), (1, 5, 2), (5, 1, 2)]):
        for px, py in ((True, True), (True, False), (False, True)):
            d = oracle.partition(np.ones((ny, nx), dtype=np.int32), P, px, py, use_hist=True)
            yield d.boxes, d.nbr, nx, ny, px, py, "tiny%d%d%d" % (k, px, py)
