"""The full-frame halo exchange (corner ghosts: ddc_get_corner_neighbours, ddc_halo_exchange_full_f64 and
ddc_halo_exchange_full_shards_f64) on a machine without a GPU.

1. The kernels on emulated ranks: tests/emu_halo.cpp (built by tests/halo_emu.py) runs the product's own halo plan
   (halo_plan: the corner table and items) and kernels (k_halo_exchange + k_halo_corners on one buffer,
   k_halo_push_full between k_halo_open and k_halo_close on G ranks, mixed with k_halo_push, k_halo_field and
   k_halo_field_shards), under index-order and random schedules.
2. The C ABI itself on oracle/libddc_cuda_emu.so (domain_decomp_b200/csrc/ddc_api.cu over a host stand-in of the CUDA
   runtime): the getter, the single-buffer call, the status codes, and the sharded call with one rank.
The corner table is checked against halo_frame.corner_table, a brute-force owner map.  Says nothing about speed."""
import ctypes as C

import numpy as np
import pytest

import halo_emu
import halo_frame as hf
import halo_global as hg
from halo_frame import degenerate_cases
from halo_global import SENTINEL, cases, exchanged, random_bits, scattered

RANKS = (1, 2, 3, 5)
SEEDS = ("0", "11", "4242")  # DDC_EMU_SCHED_SEED: "0" index order, otherwise random block / thread schedules


def as_bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


# ---- 1. the kernels on emulated ranks --------------------------------------------------------------------------------
def test_corner_table_matches_brute_force(oracle):
    """RCB output, degenerate tilings and overlapping boxes: the product's table equals the owner-map table, self-sourced
    periodic corners included"""
    self_sourced = 0
    boxes_sets = [(d.boxes, d.nbr, nx, ny, px, py) for d, nx, ny, px, py, _ in cases(oracle)]
    boxes_sets += [(b, nb, nx, ny, px, py) for b, nb, nx, ny, px, py, _ in degenerate_cases(oracle)]
    rng = np.random.default_rng(9)
    for k in range(8):  # overlapping boxes; the table does not need neighbour lists
        nx, ny, P = int(rng.integers(4, 25)), int(rng.integers(4, 25)), int(rng.integers(1, 12))
        x0, y0 = rng.integers(0, nx, P), rng.integers(0, ny, P)
        b = np.stack([x0, y0, rng.integers(0, nx - x0 + 1), rng.integers(0, ny - y0 + 1)], axis=1).astype(np.int32)
        boxes_sets.append((b, oracle.neighbours(b, nx, ny, k & 1, k & 2), nx, ny, bool(k & 1), bool(k & 2)))
    # one part spanning a periodic domain: all four corners come from itself
    one = oracle.partition(np.ones((5, 7), dtype=np.int32), 1)
    boxes_sets.append((one.boxes, one.nbr, 7, 5, True, True))
    for boxes, nbr, nx, ny, px, py in boxes_sets:
        off = hg.tile_offsets(np.maximum(boxes, 0))
        run = halo_emu.run(boxes, nbr, nx, ny, px, py, 1, 0, "", np.zeros(int(off[-1]), np.uint64))
        ids, starts = hf.corner_table(boxes, nx, ny, px, py)
        assert np.array_equal(run.ids, ids), (nx, ny, px, py, boxes.tolist())
        assert np.array_equal(run.starts, starts), (nx, ny, px, py, boxes.tolist())
        self_sourced += int((ids[1] == np.arange(len(boxes))[None, :]).sum())
    assert self_sourced > 0


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_full_exchange_fills_the_whole_frame(oracle, monkeypatch, G, sched):
    """interiors hold the global index: after a full exchange every frame cell holds the wrapped global index of its cell
    or stays UNTOUCHED; edges equal ddc_halo_exchange_f64's; sharded equals the single buffer"""
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        off = hg.tile_offsets(d.boxes)
        tiles_in = as_bits(hg.initial_tiles(d.boxes, off, nx))
        for periodic in (0, 1):
            ctx = (G, sched, seed, nx, ny, d.P, periodic)
            full = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, periodic, "f", tiles_in)
            edge = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, periodic, "x", tiles_in)
            assert full.err.tolist() == [0] * G, ctx
            want = as_bits(hf.expected_full_tiles(d.boxes, off, nx, ny, px, py, periodic))
            assert np.array_equal(full.single[0], want), ctx + ("single buffer",)
            assert full.tiles[0].tobytes() == want.tobytes(), ctx + ("sharded",)
            corners = hf.corner_cells(d.boxes, off).reshape(-1)
            other = np.setdiff1d(np.arange(int(off[-1])), corners)
            assert np.array_equal(full.single[0][other], edge.single[0][other]), ctx + ("edges",)
            assert (edge.single[0][corners] == as_bits(hg.UNTOUCHED)).all(), ctx


@pytest.mark.parametrize("G", RANKS)
def test_degenerate_tilings(oracle, G):
    """zero-width strips and zero-height parts (ddc_neighbours_from_boxes input): every ghost of the edge and the
    full exchange holds the cell across it, zero-area receivers included, on one buffer and sharded"""
    for boxes, nbr, nx, ny, px, py, seed in degenerate_cases(oracle):
        off = hg.tile_offsets(boxes)
        tiles_in = as_bits(hg.initial_tiles(boxes, off, nx))
        for periodic in (0, 1):
            ctx = (G, seed, nx, ny, len(boxes), periodic)
            full = halo_emu.run(boxes, nbr, nx, ny, px, py, G, periodic, "f", tiles_in)
            edge = halo_emu.run(boxes, nbr, nx, ny, px, py, G, periodic, "x", tiles_in)
            assert full.err.tolist() == [0] * G and edge.err.tolist() == [0] * G, ctx
            want = as_bits(hg.expected_tiles(boxes, off, nx, ny, px, py, periodic))
            assert np.array_equal(edge.single[0], want), ctx + ("edge, single buffer",)
            assert np.array_equal(edge.tiles[0], want), ctx + ("edge, sharded",)
            want = as_bits(hf.expected_full_tiles(boxes, off, nx, ny, px, py, periodic))
            assert np.array_equal(full.single[0], want), ctx + ("full, single buffer",)
            assert np.array_equal(full.tiles[0], want), ctx + ("full, sharded",)


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_mixed_sequence_on_one_step_counter(oracle, monkeypatch, G, sched):
    """scatter, full exchange, edge exchange, full exchange, gather: random 64-bit patterns, frames a sentinel; the
    harness checks after every op that each block counter is back at zero and no rank stored outside its rows"""
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        rng = np.random.default_rng(seed + 300)
        off = hg.tile_offsets(d.boxes)
        periodic = seed & 1
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
        ops = "sfxfg"
        run = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, periodic, ops, tiles_in, [field],
                           random_bits(rng, nx * ny))
        ctx = (G, sched, seed, nx, ny, d.P, periodic)
        assert run.err.tolist() == [0] * G, ctx
        want = scattered(d.boxes, off, field, tiles_in)
        for i, op in enumerate(ops):
            if op in "xf":
                want = exchanged(d.boxes, off, nx, ny, px, py, periodic, field, want)
            if op == "f":
                want = hf.with_corners(d.boxes, off, nx, ny, px, py, periodic, field, want)
            assert np.array_equal(run.single[i], want), ctx + (i, "single buffer")
            assert run.tiles[i].tobytes() == want.tobytes(), ctx + (i, "sharded")
        assert run.rows[-1].tobytes() == field.tobytes(), ctx
        assert run.field[-1].tobytes() == field.tobytes(), ctx


def test_a_rank_that_never_arrives(oracle):
    """one rank runs none of the kernels: every other rank reports the timeout and writes nothing"""
    for d, nx, ny, px, py, seed in cases(oracle):
        if px and py and d.P >= 3:
            break
    G = 3
    off = hg.tile_offsets(d.boxes)
    tiles_in = random_bits(np.random.default_rng(7), int(off[-1]))
    for stall in range(G):
        run = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, 1, "f", tiles_in, stall=stall)
        assert run.err.tolist() == [0 if r == stall else 1 for r in range(G)], stall
        assert run.tiles[0].tobytes() == tiles_in.tobytes(), stall


@pytest.mark.parametrize("G", (1, 2, 4))
def test_one_part_exchanges_nothing(oracle, G):
    """P = 1 has no neighbour tables: the full exchange does nothing, although the table has self-sourced corners"""
    nx, ny = 13, 9
    d = oracle.partition(np.ones((ny, nx), dtype=np.int32), 1)
    off = hg.tile_offsets(d.boxes)
    tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
    run = halo_emu.run(d.boxes, d.nbr, nx, ny, True, True, G, 1, "ff", tiles_in)
    assert run.err.tolist() == [0] * G
    assert run.ids[1].tolist() == [[0]] * 4
    for i in range(2):
        assert run.tiles[i].tobytes() == tiles_in.tobytes() and run.single[i].tobytes() == tiles_in.tobytes()


# ---- 2. the C ABI on the emulated runtime ----------------------------------------------------------------------------
DDC_ERR_ARG, DDC_ERR_STATE = -1, -5


@pytest.fixture(scope="module")
def capi(oracle):
    return halo_emu.emu_capi(oracle)


def host_view(ptr, n):
    return np.ctypeslib.as_array((C.c_uint64 * n).from_address(ptr)) if n else np.zeros(0, dtype=np.uint64)


def table_of(h):
    got = [[h.corner_neighbours(c, per) for c in range(4)] for per in range(2)]
    return (np.array([[i for i, _ in g] for g in got]), np.array([[s for _, s in g] for g in got]))


@pytest.mark.parametrize("nx,ny,P,px,py", [(37, 29, 7, True, False), (50, 41, 12, True, True), (23, 70, 9, False, True),
                                           (40, 30, 1, True, True), (6, 5, 25, True, True), (6, 5, 18, False, False)])
def test_c_abi_single_buffer(capi, nx, ny, P, px, py):
    """the last two: more parts than columns, so that ddc_partition leaves zero-width strips and zero-height parts"""
    rng = np.random.default_rng(P)
    mask = (rng.random((ny, nx)) > 0.35).astype(np.int32)
    h = capi.Handle(0)
    try:
        h.set_mask_host(mask)
        h.partition(P, px, py)
        boxes = h.boxes()
        if P > nx:
            assert (boxes[:, 2] == 0).any() and (boxes[:, 3] == 0).any(), boxes.tolist()
        ids, starts = table_of(h)
        want_ids, want_starts = hf.corner_table(boxes, nx, ny, px, py)
        assert np.array_equal(ids, want_ids) and np.array_equal(starts, want_starts)
        off = h.halo_tile_offsets()
        for periodic in (0, 1):
            tiles = hg.initial_tiles(boxes, off, nx)
            h.halo_exchange_full_f64(tiles.ctypes.data, periodic)
            h.synchronize()
            want = hf.expected_full_tiles(boxes, off, nx, ny, px, py, periodic)
            assert tiles.tobytes() == want.tobytes(), periodic
    finally:
        h.close()


def test_c_abi_degenerate_boxes(capi, oracle):
    """ddc_neighbours_from_boxes input: the getter, the edge and the full exchange on zero-width strips and zero-height
    parts"""
    h = capi.Handle(0)
    try:
        for boxes, nbr, nx, ny, px, py, seed in degenerate_cases(oracle):
            h.neighbours_from_boxes(boxes, nx, ny, px, py)
            ids, starts = table_of(h)
            want_ids, want_starts = hf.corner_table(boxes, nx, ny, px, py)
            assert np.array_equal(ids, want_ids) and np.array_equal(starts, want_starts), seed
            off = h.halo_tile_offsets()
            edge, full = hg.initial_tiles(boxes, off, nx), hg.initial_tiles(boxes, off, nx)
            h.halo_exchange_f64(edge.ctypes.data, 1)
            h.halo_exchange_full_f64(full.ctypes.data, 1)
            h.synchronize()
            want = hg.expected_tiles(boxes, off, nx, ny, px, py, 1, tables=True)
            assert edge.tobytes() == want.tobytes(), seed
            want = hf.expected_full_tiles(boxes, off, nx, ny, px, py, 1, tables=True)
            assert full.tobytes() == want.tobytes(), seed
    finally:
        h.close()


def test_c_abi_errors(capi):
    L = capi._lib
    h = capi.Handle(0)
    try:
        t = np.zeros(10000, dtype=np.float64)
        ids = np.zeros(64, dtype=np.int32)
        assert L.ddc_get_corner_neighbours(h.h, 0, 0, ids.ctypes.data, None) == DDC_ERR_STATE  # before ddc_partition
        assert L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 0) == DDC_ERR_STATE
        h.set_mask_host(capi.generate_mask_host(40, 30, 1, 0.4))
        h.partition(6, True, False)
        assert L.ddc_get_corner_neighbours(h.h, 4, 0, ids.ctypes.data, None) == DDC_ERR_ARG
        assert L.ddc_get_corner_neighbours(h.h, -1, 0, ids.ctypes.data, None) == DDC_ERR_ARG
        assert L.ddc_get_corner_neighbours(h.h, 0, 2, ids.ctypes.data, None) == DDC_ERR_ARG
        assert L.ddc_get_corner_neighbours(h.h, 3, 1, None, None) == 0
        assert L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 0) == DDC_ERR_STATE  # before the tile offsets
        assert b"ddc_halo_tile_offsets" in L.ddc_last_error(h.h)
        h.halo_tile_offsets()
        assert L.ddc_halo_exchange_full_f64(h.h, None, 0) == DDC_ERR_ARG
        assert L.ddc_halo_exchange_full_shards_f64(h.h, 0) == DDC_ERR_STATE  # no halo buffers
        assert b"no halo buffers" in L.ddc_last_error(h.h)
        # new boxes invalidate the corner items even when the part count stays the same
        boxes = h.boxes()
        h.neighbours_from_boxes(boxes[::-1].copy(), 40, 30, True, False)
        assert L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 0) == DDC_ERR_STATE
        h.halo_tile_offsets()
        h.set_mask_host(capi.generate_mask_host(40, 30, 1, 0.4))  # (ddc_neighbours_from_boxes dropped the mask)
        h.partition(6, False, False)  # a repartition invalidates them again
        assert L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 0) == DDC_ERR_STATE
    finally:
        h.close()


def test_c_abi_sharded_one_rank(capi):
    """ddc_halo_connect with one rank: the sharded full exchange, its checks, and one step counter shared with the
    edge exchange, scatter and gather"""
    L = capi._lib
    nx, ny, P = 45, 38, 8
    rng = np.random.default_rng(4)
    h = capi.Handle(0, 0, 1, None)
    try:
        h.set_mask_host(capi.generate_mask_host(nx, ny, 2, 0.4))
        h.partition(P, True, True)
        boxes = h.boxes()
        off = hg.tile_offsets(boxes)
        hs, out = (C.c_void_p * 1)(h.h.value), (C.c_void_p * 1)()
        assert L.ddc_halo_connect(hs, 1, int(off[-1]), out) == 0
        assert L.ddc_halo_exchange_full_shards_f64(h.h, 1) == DDC_ERR_STATE  # no shard offsets yet
        h.halo_shard_offsets()
        view = host_view(out[0], int(off[-1]))
        view[:] = SENTINEL
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        h.halo_scatter_shards_f64(field.ctypes.data)
        h.halo_exchange_shards_f64(True)
        h.halo_exchange_full_shards_f64(True)
        h.synchronize()
        want = scattered(boxes, off, field, np.full(int(off[-1]), SENTINEL, dtype=np.uint64))
        want = exchanged(boxes, off, nx, ny, True, True, 1, field, want)
        want = hf.with_corners(boxes, off, nx, ny, True, True, 1, field, want)
        assert view.tobytes() == want.tobytes()
        rows = random_bits(rng, nx * ny)
        h.halo_gather_shards_f64(rows.ctypes.data)
        h.synchronize()
        assert rows.tobytes() == field.tobytes()
        # a decomposition whose tiles do not fit: DDC_ERR_ARG, as for the edge exchange
        h.set_mask_host(capi.generate_mask_host(90, 80, 2, 0.4))
        h.partition(P, True, True)
        h.halo_shard_offsets()
        assert L.ddc_halo_exchange_full_shards_f64(h.h, 1) == DDC_ERR_ARG
        h.halo_close()
    finally:
        h.close()
