"""Expected tiles of the halo exchanges when every interior cell holds its GLOBAL linear index y * nx + x (plus an
offset that changes between exchanges): a ghost cell must then hold exactly the index of the cell across its edge --
wrapped when the exchange is periodic in that direction -- or stay untouched (corners, non-periodic domain edges).
Unlike the part ids of halo_check.py this checks WHICH cell arrived, not only from which part.  Everything is
vectorised over the ghost cells (per-part work is numpy slices), so it is fast enough for thousands of parts.
Beside them: the fields, decompositions and GPU set-up the halo tests share."""
import itertools

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


def expected_tiles(boxes, offsets, nx, ny, px, py, periodic, add=0.0, tables=None):
    """initial_tiles(add) after one exchange (interior lists; periodic: the periodic ones too).  tables: whether the
    handle has neighbour tables -- by default as after ddc_partition, which builds none for one part (and then the
    exchange does nothing); ddc_neighbours_from_boxes builds them for one part too."""
    buf = initial_tiles(boxes, offsets, nx, add)
    if not (len(boxes) > 1 if tables is None else tables):
        return buf
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


# ---- fields as 64-bit patterns, and the tiles they give ---------------------------------------------------------------
SENTINEL = np.uint64(0x7FF4DEADBEEF0001)  # a signalling NaN with a payload: frames keep it bit for bit
SPECIAL = np.array([0x8000000000000000, 0x0000000000000001, 0x800FFFFFFFFFFFFF, 0x7FF0000000000001,
                    0xFFF8DEADBEEFCAFE, 0x7FF0000000000000], dtype=np.uint64)  # -0.0, subnormals, NaNs, inf


def random_bits(rng, n):
    """random 64-bit patterns, with the special values planted at random places"""
    a = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    if n >= len(SPECIAL):
        a[rng.choice(n, size=len(SPECIAL), replace=False)] = SPECIAL
    return a


def scattered(boxes, off, field, tiles):
    """tiles with every interior replaced by the field (uint64 bits)"""
    out = tiles.copy()
    for p, (x0, y0, ex, ey) in enumerate(np.asarray(boxes, dtype=np.int64)):
        if ex > 0 and ey > 0:
            out[off[p]:off[p + 1]].reshape(ey + 2, ex + 2)[1:-1, 1:-1] = field[y0:y0 + ey, x0:x0 + ex]
    return out


def exchanged(boxes, off, nx, ny, px, py, periodic, field, tiles):
    """tiles after an exchange when every interior holds the field: the expected_tiles rule with field values -- a
    ghost cell holds the field cell across its edge (wrapped where periodic) or keeps what it held"""
    out = tiles.copy()
    if len(boxes) < 2:
        return out  # one part: no neighbour tables, nothing is exchanged
    idx, x, y = ghost_cells(boxes, off)
    ok = np.ones(len(idx), dtype=bool)
    if not (periodic and px):
        ok &= (x >= 0) & (x < nx)
    if not (periodic and py):
        ok &= (y >= 0) & (y < ny)
    out[idx[ok]] = field[(y % ny)[ok], (x % nx)[ok]]
    return out


def shard_rows(ny, G):
    """[(y_begin, y_count)] of every rank: ddc_shard_rows"""
    from domain_decomp_b200 import capi
    return [capi.shard_rows(ny, G, r) for r in range(G)]


# ---- the decompositions of the CPU tests (oracle: the conftest fixture) ----------------------------------------------
def decomposition(oracle, seed, px, py):
    """widths and heights that are no multiple of 32; every fourth case 3 parts (fewer than the largest rank count);
    every fifth case fewer rows than the largest rank count, so that ddc_shard_rows leaves the last ranks empty"""
    rng = np.random.default_rng(100 + seed)
    nx, ny = int(rng.integers(5, 70)), int(rng.integers(6, 50)) if seed % 5 else int(rng.integers(2, 5))
    nx += nx % 32 == 0
    ny += ny % 32 == 0
    P = int(rng.integers(2, 14)) if seed % 4 else 3
    mask = (rng.random((ny, nx)) > rng.uniform(0.1, 0.6)).astype(np.int32)
    return oracle.partition(mask, P, px, py, use_hist=True), nx, ny


def empty_part_cases(oracle):
    """RCB output with empty parts: tiny grids cut into more parts than they have ocean columns or rows, which leaves
    zero-height parts and zero-width strips, every periodic combination.  The boxes still tile the domain."""
    out = []
    for case, (px, py) in enumerate(itertools.product((False, True), repeat=2)):
        for k, (nx, ny, P) in enumerate([(11, 11, 36), (6, 5, 19)]):
            seed = 16 + 2 * case + k
            rng = np.random.default_rng(900 + seed)
            mask = (rng.random((ny, nx)) >= 0.6 + 0.3 * rng.random()).astype(np.int32)
            out.append((oracle.partition(mask, P, px, py, use_hist=True), nx, ny, px, py, seed))
    zero_width, zero_height = (any((d.boxes[:, i] == 0).any() for d, *_ in out) for i in (2, 3))
    assert zero_width and zero_height, "the empty-part cases lost their zero-width strips or zero-height parts"
    return out


def cases(oracle):
    for case, (px, py) in enumerate(itertools.product((False, True), repeat=2)):
        for seed in (case, case + 4, case + 8, case + 12):
            d, nx, ny = decomposition(oracle, seed, px, py)
            yield d, nx, ny, px, py, seed
    yield from empty_part_cases(oracle)


# ---- the GPU tests (torch is passed in: this module imports without it) ----------------------------------------------
GPU_CASES = [  # nx, ny, P, px, py
    (528, 522, 64, True, True),
    (2048, 1536, 1000, True, False),
    (8192, 8192, 4096, False, False),
]
GPU_EMPTY_CASES = [  # nx, ny, P, px, py on empty_part_mask: more parts than ocean columns
    (11, 11, 36, True, True),
    (1024, 1024, 1024, True, False),
]
SENT = int(SENTINEL.view(np.int64))


def empty_part_mask(nx, ny):
    """ocean in a band of three rows across the middle and in one column: RCB cuts it into zero-width strips and
    zero-height parts when there are more parts than ocean columns"""
    mask = np.zeros((ny, nx), dtype=np.int32)
    mask[ny // 2 - 1:ny // 2 + 2, :] = 1
    mask[:, nx // 3] = 1
    return mask


class _Dev:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 2,
                                         "strides": None}


def dev_view(torch, ptr, n):
    """float64[n] over raw device memory (a halo buffer of the library)"""
    return torch.as_tensor(_Dev(ptr, n), device="cuda") if n else torch.empty(0, dtype=torch.float64, device="cuda")


def decompose(capi, torch, nx, ny, P, px, py, seed=3, land=0.45):
    """a handle on device 0 with the decomposition of a generated mask; for a GPU_EMPTY_CASES case of empty_part_mask,
    checked to have zero-width strips and zero-height parts"""
    h = capi.Handle(0)
    d_mask = torch.empty((ny, nx), dtype=torch.int32, device="cuda")
    if (nx, ny, P, px, py) in GPU_EMPTY_CASES:
        d_mask.copy_(torch.from_numpy(empty_part_mask(nx, ny)))
        torch.cuda.synchronize()  # (the library works on its own stream)
    else:
        h.generate_mask_device(d_mask.data_ptr(), nx, ny, seed, land)
    h.set_mask_device(d_mask.data_ptr(), nx, ny)
    h.partition(P, px, py)
    h._mask = d_mask
    if (nx, ny, P, px, py) in GPU_EMPTY_CASES:
        b = h.boxes()
        assert (b[:, 2] == 0).any() and (b[:, 3] == 0).any(), "no zero-width strip or no zero-height part"
    return h


def connect(capi, boxes, nx, ny, px, py, G):
    """G handles on device 0 with the boxes, joined by ddc_halo_connect, their shard offsets taken"""
    handles = [capi.Handle(0, q, G, None) for q in range(G)]
    for h in handles:
        h.neighbours_from_boxes(boxes, nx, ny, px, py)
    ptrs = capi.halo_connect(handles, max_shard_total(boxes, G))
    for h in handles:
        h.halo_shard_offsets()
    return handles, ptrs


def random_field(torch, nx, ny, seed):
    """int64 [ny, nx] of random bit patterns on the device, the special values planted; view it as float64 to pass it"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = torch.randint(-2 ** 63, 2 ** 63 - 1, (ny, nx), dtype=torch.int64, device="cuda", generator=g)
    pos = torch.randint(0, nx * ny, (len(SPECIAL),), device="cuda", generator=g)
    f.view(-1)[pos] = torch.from_numpy(SPECIAL.view(np.int64)).cuda()
    return f


def u64(t):
    return t.cpu().numpy().view(np.uint64)
