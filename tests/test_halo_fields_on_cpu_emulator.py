"""Halo scatter and gather (ddc_halo_scatter_f64 / ddc_halo_gather_f64 and the sharded forms) on a machine without a GPU.

1. The kernels on emulated ranks: tests/emu_halo.cpp (built by tests/halo_emu.py) runs the product's own k_halo_field /
   k_halo_field_shards (between k_halo_open and k_halo_close, mixed with k_halo_push exchanges) for G emulated ranks,
   phase by phase, and the single-buffer kernels beside them.  Fields are random 64-bit patterns viewed as float64 (NaN payloads, -0.0 and
   subnormals included), frames hold a signalling-NaN sentinel, and everything is compared as bits.
2. The C ABI itself: oracle/libddc_cuda_emu.so is domain_decomp_b200/csrc/ddc_api.cu over a host stand-in of the CUDA
   runtime.  That stand-in maps no peer memory between processes but runs ddc_halo_connect for one rank, so the
   sharded calls are covered there with G = 1 (several ranks: part 1).
Says nothing about speed."""
import ctypes as C

import numpy as np
import pytest

import halo_emu
import halo_global as hg
from halo_global import SENTINEL, cases, decomposition, exchanged, random_bits, scattered

RANKS = (1, 2, 3, 5)
SEEDS = ("0", "11", "4242")  # DDC_EMU_SCHED_SEED: "0" index order, otherwise random block / thread schedules


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_sharded_scatter_matches_single_buffer_and_field(oracle, monkeypatch, G, sched):
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        rng = np.random.default_rng(seed)
        off = hg.tile_offsets(d.boxes)
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
        tiles, single, rows, _, err = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, 0, "s", tiles_in, [field],
                                                    random_bits(rng, nx * ny))[:5]
        ctx = (G, sched, seed, nx, ny, d.P)
        assert err.tolist() == [0] * G, ctx
        want = scattered(d.boxes, off, field, tiles_in)
        assert np.array_equal(single[0], want), ctx + ("single buffer",)
        assert tiles[0].tobytes() == want.tobytes(), ctx + ("sharded",)


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_gather_writes_every_cell_from_interiors_only(oracle, monkeypatch, G, sched):
    """frames hold garbage, the rows hold other garbage before: afterwards the rows in rank order are the field"""
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        rng = np.random.default_rng(seed + 50)
        off = hg.tile_offsets(d.boxes)
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        tiles_in = scattered(d.boxes, off, field, random_bits(rng, int(off[-1])))
        tiles, single, rows, single_field, err = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, 0, "g", tiles_in,
                                                              rows_in=random_bits(rng, nx * ny))[:5]
        ctx = (G, sched, seed, nx, ny, d.P)
        assert err.tolist() == [0] * G, ctx
        assert rows[0].tobytes() == field.tobytes(), ctx + ("sharded",)
        assert single_field[0].tobytes() == field.tobytes(), ctx + ("single buffer",)
        assert tiles[0].tobytes() == tiles_in.tobytes() and single[0].tobytes() == tiles_in.tobytes(), ctx


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_scatter_exchange_exchange_gather(oracle, monkeypatch, G, sched):
    """one step counter across scatter, two exchanges and gather; the harness also checks after every op that each
    rank's block counter is back at zero and that no rank stored outside its rows"""
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        rng = np.random.default_rng(seed + 100)
        off = hg.tile_offsets(d.boxes)
        for periodic in (0, 1):
            field = random_bits(rng, nx * ny).reshape(ny, nx)
            tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
            tiles, single, rows, single_field, err = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, periodic, "sxxg",
                                                                  tiles_in, [field], random_bits(rng, nx * ny))[:5]
            ctx = (G, sched, seed, nx, ny, d.P, periodic)
            assert err.tolist() == [0] * G, ctx
            want = scattered(d.boxes, off, field, tiles_in)
            for i in range(4):
                if i in (1, 2):
                    want = exchanged(d.boxes, off, nx, ny, px, py, periodic, field, want)
                assert np.array_equal(single[i], want), ctx + (i, "single buffer")
                assert tiles[i].tobytes() == want.tobytes(), ctx + (i, "sharded")
            assert rows[3].tobytes() == field.tobytes(), ctx
            assert single_field[3].tobytes() == field.tobytes(), ctx


def test_a_rank_that_never_arrives(oracle):
    """emulation only: one rank runs none of the kernels; every other rank reports the timeout and writes nothing --
    a scatter leaves every tile as it was, a gather every row"""
    d, nx, ny = decomposition(oracle, 5, True, False)
    G = 3
    rng = np.random.default_rng(7)
    off = hg.tile_offsets(d.boxes)
    field = random_bits(rng, nx * ny).reshape(ny, nx)
    tiles_in = random_bits(rng, int(off[-1]))
    rows_in = random_bits(rng, nx * ny)
    for stall in range(G):
        for op in "sg":
            tiles, _, rows, _, err = halo_emu.run(d.boxes, d.nbr, nx, ny, True, False, G, 0, op, tiles_in, [field],
                                                  rows_in, stall=stall)[:5]
            assert err.tolist() == [0 if r == stall else 1 for r in range(G)], (stall, op)
            assert tiles[0].tobytes() == tiles_in.tobytes(), (stall, op)
            assert rows[0].tobytes() == rows_in.tobytes(), (stall, op)


@pytest.mark.parametrize("G", (1, 2, 4))
def test_one_part_moves_the_whole_field(oracle, G):
    """P = 1 has no neighbour tables: the exchange does nothing, scatter and gather still move every cell"""
    nx, ny = 13, 9
    mask = np.ones((ny, nx), dtype=np.int32)
    mask[2:5, 3:7] = 0  # land is scattered and gathered like the ocean
    d = oracle.partition(mask, 1)
    rng = np.random.default_rng(3)
    off = hg.tile_offsets(d.boxes)
    field = random_bits(rng, nx * ny).reshape(ny, nx)
    tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
    tiles, single, rows, single_field, err = halo_emu.run(d.boxes, d.nbr, nx, ny, False, False, G, 1, "sxg", tiles_in,
                                                          [field], random_bits(rng, nx * ny))[:5]
    want = scattered(d.boxes, off, field, tiles_in)
    assert err.tolist() == [0] * G
    for i in range(3):
        assert tiles[i].tobytes() == want.tobytes() and single[i].tobytes() == want.tobytes(), i
    assert rows[2].tobytes() == field.tobytes() and single_field[2].tobytes() == field.tobytes()


# ---- 2. the C ABI on the emulated runtime ----------------------------------------------------------------------------
DDC_ERR_ARG, DDC_ERR_STATE = -1, -5


@pytest.fixture(scope="module")
def capi(oracle):
    return halo_emu.emu_capi(oracle)


def host_view(ptr, n):
    """uint64[n] over the "device" memory of the emulated runtime (host memory)"""
    return np.ctypeslib.as_array((C.c_uint64 * n).from_address(ptr)) if n else np.zeros(0, dtype=np.uint64)


@pytest.mark.parametrize("nx,ny,P,flags", [(37, 29, 1, 3), (37, 29, 7, 3), (50, 41, 12, 0), (64, 33, 5, 2),
                                           (23, 70, 9, 1)])
def test_c_abi_single_buffer(capi, oracle, nx, ny, P, flags):
    """flags 0 / 1: no neighbour tables; scatter and gather still move the whole field"""
    rng = np.random.default_rng(P)
    mask = (rng.random((ny, nx)) > 0.35).astype(np.int32)
    h = capi.Handle(0)
    try:
        h.set_mask_host(mask)
        h.partition(P, True, False, flags=flags)
        boxes = h.boxes()
        off = h.halo_tile_offsets()
        assert off.tolist() == hg.tile_offsets(boxes).tolist()
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        tiles = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
        h.halo_scatter_f64(field.ctypes.data, tiles.ctypes.data)
        h.synchronize()
        assert tiles.tobytes() == scattered(boxes, off, field, np.full_like(tiles, SENTINEL)).tobytes()
        tiles[tiles == SENTINEL] = np.uint64(12345)  # frames: garbage that gather must not read
        back = random_bits(rng, nx * ny)
        h.halo_gather_f64(tiles.ctypes.data, back.ctypes.data)
        h.synchronize()
        assert back.tobytes() == field.tobytes()
    finally:
        h.close()


def test_c_abi_errors(capi):
    L = capi._lib
    h = capi.Handle(0)
    try:
        f = np.zeros(40 * 30, dtype=np.float64)
        t = np.zeros(10000, dtype=np.float64)
        assert L.ddc_halo_scatter_f64(h.h, f.ctypes.data, t.ctypes.data) == DDC_ERR_STATE  # before ddc_partition
        h.set_mask_host(capi.generate_mask_host(40, 30, 1, 0.4))
        h.partition(6, True, False)
        assert L.ddc_halo_scatter_f64(h.h, f.ctypes.data, t.ctypes.data) == DDC_ERR_STATE  # before the tile offsets
        assert L.ddc_halo_gather_f64(h.h, t.ctypes.data, f.ctypes.data) == DDC_ERR_STATE
        assert b"ddc_halo_tile_offsets" in L.ddc_last_error(h.h)
        h.halo_tile_offsets()
        assert L.ddc_halo_scatter_f64(h.h, None, t.ctypes.data) == DDC_ERR_ARG
        assert L.ddc_halo_scatter_f64(h.h, f.ctypes.data, None) == DDC_ERR_ARG
        assert L.ddc_halo_gather_f64(h.h, None, f.ctypes.data) == DDC_ERR_ARG
        assert L.ddc_halo_gather_f64(h.h, t.ctypes.data, None) == DDC_ERR_ARG
        # sharded without halo buffers
        assert L.ddc_halo_scatter_shards_f64(h.h, f.ctypes.data) == DDC_ERR_STATE
        assert L.ddc_halo_gather_shards_f64(h.h, f.ctypes.data) == DDC_ERR_STATE
        assert b"no halo buffers" in L.ddc_last_error(h.h)
        # a repartition invalidates the offsets again
        h.partition(5, True, False)
        assert L.ddc_halo_gather_f64(h.h, t.ctypes.data, f.ctypes.data) == DDC_ERR_STATE
        # so do new boxes with the same part count (here with a larger tile total)
        h.partition(6, True, False)
        h.halo_tile_offsets()
        x0 = np.array([0, 7, 14, 21, 28, 34])
        strips = np.stack([x0, 0 * x0, np.diff(np.append(x0, 40)), 0 * x0 + 30], axis=1).astype(np.int32)
        h.neighbours_from_boxes(strips, 40, 30, True, False)
        assert L.ddc_halo_scatter_f64(h.h, f.ctypes.data, t.ctypes.data) == DDC_ERR_STATE
        assert L.ddc_halo_gather_f64(h.h, t.ctypes.data, f.ctypes.data) == DDC_ERR_STATE
        assert L.ddc_halo_exchange_f64(h.h, t.ctypes.data, 1) == DDC_ERR_STATE
        assert h.halo_tile_offsets()[-1] <= t.size
        assert L.ddc_halo_scatter_f64(h.h, f.ctypes.data, t.ctypes.data) == 0
        assert L.ddc_halo_exchange_f64(h.h, t.ctypes.data, 1) == 0
        assert L.ddc_halo_gather_f64(h.h, t.ctypes.data, f.ctypes.data) == 0
        h.synchronize()
    finally:
        h.close()


def test_c_abi_sharded_one_rank(capi, oracle):
    """ddc_halo_connect with one rank runs on the emulated runtime: the sharded scatter and gather, the capacity and
    state checks, and one step counter shared with the exchange"""
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
        ptr = out[0]
        rows = random_bits(rng, nx * ny)
        assert L.ddc_halo_scatter_shards_f64(h.h, rows.ctypes.data) == DDC_ERR_STATE  # no shard offsets yet
        assert h.halo_shard_offsets().tolist() == off.tolist()
        assert L.ddc_halo_scatter_shards_f64(h.h, None) == DDC_ERR_ARG  # this rank holds rows
        view = host_view(ptr, int(off[-1]))
        view[:] = SENTINEL
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        h.halo_scatter_shards_f64(field.ctypes.data)
        h.synchronize()
        want = scattered(boxes, off, field, np.full(int(off[-1]), SENTINEL, dtype=np.uint64))
        assert view.tobytes() == want.tobytes()
        h.halo_exchange_shards_f64(True)
        h.synchronize()
        assert view.tobytes() == exchanged(boxes, off, nx, ny, True, True, 1, field, want).tobytes()
        h.halo_gather_shards_f64(rows.ctypes.data)
        h.synchronize()
        assert rows.tobytes() == field.tobytes()
        # a decomposition whose tiles do not fit: DDC_ERR_ARG, as for the exchange
        h.set_mask_host(capi.generate_mask_host(90, 80, 2, 0.4))
        h.partition(P, True, True)
        h.halo_shard_offsets()
        big = np.zeros(90 * 80, dtype=np.float64)
        assert L.ddc_halo_scatter_shards_f64(h.h, big.ctypes.data) == DDC_ERR_ARG
        assert L.ddc_halo_gather_shards_f64(h.h, big.ctypes.data) == DDC_ERR_ARG
        h.halo_close()
    finally:
        h.close()
