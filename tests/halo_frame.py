"""Expectations of the full-frame halo exchange (ddc_halo_exchange_full_f64 and its sharded form): the corner table by
brute force and the corner ghosts it fills, beside halo_global's edge ghosts.

The corner table here is built from an owner map painted over the whole domain -- every cell gets the lowest-id box of
positive area that contains it -- so it shares nothing with the library's bucket search but the rule itself."""
import numpy as np

import halo_global as hg


def owner_map(boxes, nx, ny):
    """int32 [ny, nx]: the lowest-id positive-area box that contains each cell, -1 where none does"""
    own = np.full((ny, nx), -1, dtype=np.int32)
    b = np.asarray(boxes, dtype=np.int64)
    for q in range(len(b) - 1, -1, -1):  # the lowest id is painted last
        x0, y0, ex, ey = b[q]
        if ex > 0 and ey > 0:
            own[max(y0, 0):max(min(y0 + ey, ny), 0), max(x0, 0):max(min(x0 + ex, nx), 0)] = q
    return own


def corner_xy(boxes):
    """x [4, P], y [4, P]: the cell of every corner (BOTTOM_LEFT, BOTTOM_RIGHT, TOP_LEFT, TOP_RIGHT) of every part"""
    b = np.asarray(boxes, dtype=np.int64)
    x0, y0, ex, ey = b[:, 0], b[:, 1], np.maximum(b[:, 2], 0), np.maximum(b[:, 3], 0)
    xs = np.stack([x0 - 1, x0 + ex, x0 - 1, x0 + ex])
    ys = np.stack([y0 - 1, y0 - 1, y0 + ey, y0 + ey])
    return xs, ys


def corner_table(boxes, nx, ny, px, py):
    """(ids, starts), int32 [2, 4, P] each: [set (0 interior, 1 periodic)][corner][part] -> source part (-1: none) and
    the cell's index in the source's flattened box (0 where there is no source), the ddc_get_corner_neighbours rule"""
    b = np.asarray(boxes, dtype=np.int64)
    own = owner_map(boxes, nx, ny)
    x, y = corner_xy(boxes)
    out_x, out_y = (x < 0) | (x >= nx), (y < 0) | (y >= ny)
    ok = (~out_x | bool(px)) & (~out_y | bool(py))
    xw, yw = x % nx, y % ny
    q = np.where(ok, own[yw, xw], -1)
    qq = np.maximum(q, 0)
    start = np.where(q >= 0, (yw - b[qq, 1]) * b[qq, 2] + (xw - b[qq, 0]), 0)
    periodic_set = out_x | out_y
    ids = np.stack([np.where(periodic_set, -1, q), np.where(periodic_set, q, -1)]).astype(np.int32)
    starts = np.stack([np.where(periodic_set, 0, start), np.where(periodic_set, start, 0)]).astype(np.int32)
    return ids, starts


def corner_cells(boxes, offsets):
    """buffer index [4, P] of every corner ghost of every tile (the ddc_halo_tile_offsets layout)"""
    b = np.asarray(boxes, dtype=np.int64)
    w, h = np.maximum(b[:, 2], 0) + 2, np.maximum(b[:, 3], 0) + 2
    off = np.asarray(offsets, dtype=np.int64)[:-1]
    return np.stack([off, off + w - 1, off + (h - 1) * w, off + h * w - 1])


def with_corners(boxes, offsets, nx, ny, px, py, periodic, field, tiles, tables=None):
    """tiles with every corner ghost that has a source (interior set; periodic: both) set to the field value of its
    (wrapped) cell; the others keep what they held.  field [ny, nx]: what the interiors hold.  tables: whether the
    handle has neighbour tables -- by default as after ddc_partition, which builds none for one part (and then the
    full-frame exchange does nothing); ddc_neighbours_from_boxes builds them for one part too."""
    out = tiles.copy()
    if not (len(boxes) > 1 if tables is None else tables):
        return out
    ids, _ = corner_table(boxes, nx, ny, px, py)
    x, y = corner_xy(boxes)
    src = ids[0] if not periodic else np.maximum(ids[0], ids[1])
    idx = corner_cells(boxes, offsets)
    ok = src >= 0
    out[idx[ok]] = field[(y % ny)[ok], (x % nx)[ok]]
    return out


def expected_full_tiles(boxes, offsets, nx, ny, px, py, periodic, add=0.0, tables=None):
    """halo_global.initial_tiles(add) after one full-frame exchange: the edge ghosts of halo_global.expected_tiles and
    every corner ghost with a source holding the global index of its wrapped cell (+ add); the rest UNTOUCHED"""
    buf = hg.expected_tiles(boxes, offsets, nx, ny, px, py, periodic, add, tables)
    field = np.arange(nx * ny, dtype=np.float64).reshape(ny, nx) + add
    return with_corners(boxes, offsets, nx, ny, px, py, periodic, field, buf, tables)


def strip_tiling(rng, nx, ny):
    """boxes [P, 4] that tile [0, nx) x [0, ny) as vertical strips cut into parts, some strips of width 0 and some parts
    of height 0 (the degenerate tilings RCB can leave on tiny grids)"""
    def cuts(n, k):
        return np.concatenate([[0], np.sort(rng.integers(0, n + 1, size=k - 1)), [n]])
    xs = cuts(nx, int(rng.integers(1, 5)))
    boxes = []
    for i in range(len(xs) - 1):
        ys = cuts(ny, int(rng.integers(1, 5)))
        for j in range(len(ys) - 1):
            boxes.append((xs[i], ys[j], xs[i + 1] - xs[i], ys[j + 1] - ys[j]))
    return np.array(boxes, dtype=np.int32)


def degenerate_cases(oracle):
    """strip tilings with zero-height parts and zero-width strips, every periodic combination; their neighbour lists
    are what ddc_neighbours_from_boxes computes for them (the oracle's restatement of discover_neighbours).  The lists
    name the zero-area parts too; the exchanges never read one (a part of zero area is never a source)."""
    for seed in range(12):
        rng = np.random.default_rng(500 + seed)
        nx, ny = int(rng.integers(3, 30)), int(rng.integers(3, 30))
        boxes = strip_tiling(rng, nx, ny)
        px, py = bool(seed & 1), bool(seed & 2)
        yield boxes, oracle.neighbours(boxes, nx, ny, px, py), nx, ny, px, py, seed
