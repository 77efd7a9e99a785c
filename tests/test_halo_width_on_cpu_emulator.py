"""Wide halos (ddc_halo_set_width: ghost frames of width w for scatter, gather and both exchanges) on a machine without a
GPU.

1. The kernels on emulated ranks: tests/emu_halo.cpp (built by tests/halo_emu.py) runs the product's halo plan with the
   width (the rectangle items) and kernels (k_halo_rects on one buffer, k_halo_push_rects between k_halo_open and
   k_halo_close on G ranks, mixed with k_halo_field and k_halo_field_shards at that width), under index-order and random
   schedules, against halo_width's expectation over the whole buffer, untouched cells included.
2. The C ABI on oracle/libddc_cuda_emu.so: w = 1 is the default bit for bit, the width's status codes, and the sharded
   calls with one rank.
3. The same kernels at w = 2 and 3 under AddressSanitizer + UBSan (tests/halo_asan_worker.py).
Says nothing about speed."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import halo_emu
import halo_frame as hf
import halo_global as hg
import halo_width as hw
from conftest import ROOT
from halo_frame import degenerate_cases
from halo_global import SENTINEL, cases, random_bits

WIDTHS = (1, 2, 3, 5)
RANKS = (1, 2, 3, 5)
SEEDS = ("0", "11", "4242")  # DDC_EMU_SCHED_SEED: "0" index order, otherwise random block / thread schedules


def as_bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def all_cases(oracle):
    """RCB output with every periodic combination and with empty parts, degenerate tilings, tiny periodic domains"""
    for d, nx, ny, px, py, seed in cases(oracle):
        yield d.boxes, d.nbr, nx, ny, px, py, seed
    yield from degenerate_cases(oracle)
    yield from hw.tiny_periodic_cases(oracle)


# ---- 1. the kernels on emulated ranks --------------------------------------------------------------------------------
@pytest.mark.parametrize("w", WIDTHS)
def test_exchanges_follow_the_rule(oracle, w):
    """interiors hold the global index: an edge exchange, then a full exchange, on one buffer and on two ranks, equal
    the owner-map expectation over the whole buffer"""
    tiny = 0
    for boxes, nbr, nx, ny, px, py, seed in all_cases(oracle):
        off = hw.tile_offsets(boxes, w)
        tiles_in = as_bits(hw.initial_tiles(boxes, off, nx, ny, w))
        tiny += w > nx or w > ny
        for periodic in (0, 1):
            ctx = (w, seed, nx, ny, len(boxes), px, py, periodic)
            run = halo_emu.run(boxes, nbr, nx, ny, px, py, 2, periodic, "xf", tiles_in, w=w)
            assert run.err.tolist() == [0, 0], ctx
            for i, full in enumerate((False, True)):
                want = as_bits(hw.expected(boxes, off, nx, ny, px, py, periodic, full, w))
                assert np.array_equal(run.single[i], want), ctx + (full, "single buffer")
                assert np.array_equal(run.tiles[i], want), ctx + (full, "sharded")
    assert tiny > 0 or w == 1


def test_wide_frames_wrap_several_times(oracle):
    """a 2 x 3 periodic domain with w = 5: every frame cell is filled, most of them from wrapped pieces of the part
    itself or of its neighbour"""
    nx, ny, w = 2, 3, 5
    d = oracle.partition(np.ones((ny, nx), dtype=np.int32), 2, True, True, use_hist=True)
    off = hw.tile_offsets(d.boxes, w)
    run = halo_emu.run(d.boxes, d.nbr, nx, ny, True, True, 1, 1, "f", as_bits(hw.initial_tiles(d.boxes, off, nx, ny, w)),
                       w=w)
    got = run.single[0].view(np.float64)
    assert not (got == hg.UNTOUCHED).any()
    idx, x, y, _ = hw.frame_cells(d.boxes, off, w)
    assert np.array_equal(got[idx], ((y % ny) * nx + x % nx).astype(np.float64))


@pytest.mark.parametrize("G", RANKS)
@pytest.mark.parametrize("sched", SEEDS)
def test_mixed_sequence_on_one_step_counter(oracle, monkeypatch, G, sched):
    """scatter, edge exchange, full exchange, edge exchange, gather at w = 2 and 3: random 64-bit patterns, frames a
    sentinel; the harness checks after every op that each block counter is back at zero and no rank stored outside its
    rows"""
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", sched)
    for d, nx, ny, px, py, seed in cases(oracle):
        w = 2 + seed % 2
        rng = np.random.default_rng(seed + 700)
        off = hw.tile_offsets(d.boxes, w)
        periodic = seed & 1
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
        ops = "sxfxg"
        run = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, G, periodic, ops, tiles_in, [field], random_bits(rng, nx * ny),
                           w=w)
        ctx = (G, sched, seed, w, nx, ny, d.P, periodic)
        assert run.err.tolist() == [0] * G, ctx
        want = hw.scattered(d.boxes, off, field, tiles_in, w)
        for i, op in enumerate(ops):
            if op in "xf":
                want = hw.exchanged(d.boxes, off, nx, ny, px, py, periodic, op == "f", field, want, w)
            assert np.array_equal(run.single[i], want), ctx + (i, "single buffer")
            assert run.tiles[i].tobytes() == want.tobytes(), ctx + (i, "sharded")
        assert run.rows[-1].tobytes() == field.tobytes(), ctx
        assert run.field[-1].tobytes() == field.tobytes(), ctx


def test_width_one_is_the_one_cell_frame(oracle):
    """w = 1 is the one-cell frame: scatter, edge exchange, full exchange and gather on one buffer and on two ranks give
    the one-cell expectations of halo_global and halo_frame, built from the global field"""
    for d, nx, ny, px, py, seed in cases(oracle):
        rng = np.random.default_rng(seed)
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        off = hg.tile_offsets(d.boxes)
        tiles_in = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
        assert np.array_equal(hw.tile_offsets(d.boxes, 1), off)
        ops = "sxfg"
        run = halo_emu.run(d.boxes, d.nbr, nx, ny, px, py, 2, 1, ops, tiles_in, [field], w=1)
        assert run.err.tolist() == [0, 0], seed
        want = hg.scattered(d.boxes, off, field, tiles_in)
        for i, op in enumerate(ops):
            if op in "xf":
                want = hg.exchanged(d.boxes, off, nx, ny, px, py, 1, field, want)
            if op == "f":
                want = hf.with_corners(d.boxes, off, nx, ny, px, py, 1, field, want)
            assert np.array_equal(run.single[i], want), (seed, i, "single buffer")
            assert run.tiles[i].tobytes() == want.tobytes(), (seed, i, "sharded")
        assert run.rows[-1].tobytes() == field.tobytes() and run.field[-1].tobytes() == field.tobytes(), seed


# ---- 2. the C ABI on the emulated runtime ----------------------------------------------------------------------------
DDC_ERR_ARG, DDC_ERR_STATE = -1, -5
MAX_WIDTH = 1024  # DDC_MAX_HALO_WIDTH


@pytest.fixture(scope="module")
def capi(oracle):
    return halo_emu.emu_capi(oracle)


def host_view(ptr, n):
    return np.ctypeslib.as_array((C.c_uint64 * n).from_address(ptr)) if n else np.zeros(0, dtype=np.uint64)


def test_max_width_is_the_header_bound():
    with open(os.path.join(ROOT, "include", "ddc.h")) as f:
        assert "#define DDC_MAX_HALO_WIDTH %d\n" % MAX_WIDTH in f.read()


def test_c_abi_width_one_is_the_default(capi):
    """scatter + full exchange + gather: a handle that never set the width, one set to 1 and one set to 2 and back to 1
    give the same bytes"""
    nx, ny, P = 37, 29, 9
    mask = (np.random.default_rng(2).random((ny, nx)) > 0.35).astype(np.int32)
    field = random_bits(np.random.default_rng(3), nx * ny).reshape(ny, nx)
    out = []
    for widths in ((), (1,), (2, 1)):
        h = capi.Handle(0)
        try:
            for w in widths:
                h.halo_set_width(w)
            h.set_mask_host(mask)
            h.partition(P, True, False)
            off = h.halo_tile_offsets()
            tiles = np.full(int(off[-1]), SENTINEL, dtype=np.uint64)
            h.halo_scatter_f64(field.ctypes.data, tiles.ctypes.data)
            h.halo_exchange_full_f64(tiles.ctypes.data, True)
            back = np.zeros_like(field)
            h.halo_gather_f64(tiles.ctypes.data, back.ctypes.data)
            h.synchronize()
            assert back.tobytes() == field.tobytes()
            out.append((off.tobytes(), tiles.tobytes()))
        finally:
            h.close()
    assert out[0] == out[1] == out[2]


@pytest.mark.parametrize("w", (2, 3, 5))
def test_c_abi_single_buffer(capi, oracle, w):
    """scatter, edge exchange, full exchange, gather through the C ABI at width w, RCB output with and without empty
    parts, and degenerate tilings through ddc_neighbours_from_boxes"""
    h = capi.Handle(0)
    try:
        h.halo_set_width(w)  # before ddc_partition
        for nx, ny, P, px, py in [(37, 29, 7, True, False), (50, 41, 12, True, True), (6, 5, 25, True, True),
                                  (6, 5, 18, False, False)]:
            mask = (np.random.default_rng(P).random((ny, nx)) > 0.35).astype(np.int32)
            h.set_mask_host(mask)
            h.partition(P, px, py)
            boxes = h.boxes()
            off = h.halo_tile_offsets()
            assert np.array_equal(off, hw.tile_offsets(boxes, w))
            field = np.arange(nx * ny, dtype=np.float64).reshape(ny, nx)
            for periodic in (0, 1):
                for full in (False, True):
                    tiles = np.full(int(off[-1]), hg.UNTOUCHED)
                    h.halo_scatter_f64(field.ctypes.data, tiles.ctypes.data)
                    (h.halo_exchange_full_f64 if full else h.halo_exchange_f64)(tiles.ctypes.data, periodic)
                    back = np.zeros_like(field)
                    h.halo_gather_f64(tiles.ctypes.data, back.ctypes.data)
                    h.synchronize()
                    want = hw.expected(boxes, off, nx, ny, px, py, periodic, full, w)
                    assert tiles.tobytes() == want.tobytes(), (nx, ny, P, periodic, full)
                    assert back.tobytes() == field.tobytes()
        for boxes, nbr, nx, ny, px, py, seed in degenerate_cases(oracle):
            h.neighbours_from_boxes(boxes, nx, ny, px, py)
            off = h.halo_tile_offsets()
            tiles = hw.initial_tiles(boxes, off, nx, ny, w)
            h.halo_exchange_full_f64(tiles.ctypes.data, 1)
            h.synchronize()
            want = hw.expected(boxes, off, nx, ny, px, py, 1, True, w, tables=True)
            assert tiles.tobytes() == want.tobytes(), seed
    finally:
        h.close()


def test_c_abi_errors(capi):
    L = capi._lib
    h = capi.Handle(0)
    try:
        t = np.zeros(100000, dtype=np.float64)
        for bad in (0, -1, -1000, MAX_WIDTH + 1, 1 << 30):
            assert L.ddc_halo_set_width(h.h, bad) == DDC_ERR_ARG, bad
        assert b"ddc_halo_set_width" in L.ddc_last_error(h.h)
        assert L.ddc_halo_set_width(None, 2) == DDC_ERR_ARG
        assert L.ddc_halo_set_width(h.h, MAX_WIDTH) == 0
        assert L.ddc_halo_set_width(h.h, 1) == 0
        h.set_mask_host(capi.generate_mask_host(40, 30, 1, 0.4))
        h.partition(6, True, False)
        h.halo_tile_offsets()
        assert L.ddc_halo_exchange_f64(h.h, t.ctypes.data, 0) == 0
        assert L.ddc_halo_set_width(h.h, 1) == 0  # the same width keeps the offsets
        assert L.ddc_halo_exchange_f64(h.h, t.ctypes.data, 0) == 0
        assert L.ddc_halo_set_width(h.h, 3) == 0  # another width drops them
        for call in (lambda: L.ddc_halo_exchange_f64(h.h, t.ctypes.data, 0),
                     lambda: L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 1),
                     lambda: L.ddc_halo_scatter_f64(h.h, t.ctypes.data, t.ctypes.data),
                     lambda: L.ddc_halo_gather_f64(h.h, t.ctypes.data, t.ctypes.data)):
            assert call() == DDC_ERR_STATE
            assert b"ddc_halo_tile_offsets" in L.ddc_last_error(h.h)
        off = h.halo_tile_offsets()
        assert np.array_equal(off, hw.tile_offsets(h.boxes(), 3))
        assert L.ddc_halo_exchange_full_f64(h.h, t.ctypes.data, 1) == 0
        h.synchronize()
        # the corner table describes the diagonal cell whatever the width
        ids = np.zeros(6, dtype=np.int32)
        assert L.ddc_get_corner_neighbours(h.h, 0, 0, ids.ctypes.data, None) == 0
    finally:
        h.close()


def test_c_abi_sharded_one_rank(capi):
    """ddc_halo_connect with one rank at w = 2: scatter, edge and full exchange and gather on one step counter; a width
    change before the shard offsets are taken again is DDC_ERR_STATE, and buffers too small for the wider layout are
    DDC_ERR_ARG"""
    L = capi._lib
    nx, ny, P, w = 45, 38, 8, 2
    rng = np.random.default_rng(4)
    h = capi.Handle(0, 0, 1, None)
    try:
        h.set_mask_host(capi.generate_mask_host(nx, ny, 2, 0.4))
        h.partition(P, True, True)
        boxes = h.boxes()
        off = hw.tile_offsets(boxes, w)
        hs, out = (C.c_void_p * 1)(h.h.value), (C.c_void_p * 1)()
        assert L.ddc_halo_connect(hs, 1, int(off[-1]), out) == 0
        h.halo_shard_offsets()
        h.halo_set_width(w)
        assert L.ddc_halo_exchange_shards_f64(h.h, 1) == DDC_ERR_STATE
        assert L.ddc_halo_scatter_shards_f64(h.h, None) == DDC_ERR_STATE
        assert np.array_equal(h.halo_shard_offsets(), off)
        view = host_view(out[0], int(off[-1]))
        view[:] = SENTINEL
        field = random_bits(rng, nx * ny).reshape(ny, nx)
        h.halo_scatter_shards_f64(field.ctypes.data)
        h.halo_exchange_shards_f64(True)
        h.halo_exchange_full_shards_f64(False)
        h.synchronize()
        want = hw.scattered(boxes, off, field, np.full(int(off[-1]), SENTINEL, dtype=np.uint64), w)
        want = hw.exchanged(boxes, off, nx, ny, True, True, 1, False, field, want, w)
        want = hw.exchanged(boxes, off, nx, ny, True, True, 0, True, field, want, w)
        assert view.tobytes() == want.tobytes()
        rows = random_bits(rng, nx * ny)
        h.halo_gather_shards_f64(rows.ctypes.data)
        h.synchronize()
        assert rows.tobytes() == field.tobytes()
        # the buffer holds the tiles at w = 2, not at w = 3: every sharded call refuses
        h.halo_set_width(3)
        h.halo_shard_offsets()
        for call in (lambda: L.ddc_halo_exchange_shards_f64(h.h, 1), lambda: L.ddc_halo_exchange_full_shards_f64(h.h, 0),
                     lambda: L.ddc_halo_scatter_shards_f64(h.h, field.ctypes.data),
                     lambda: L.ddc_halo_gather_shards_f64(h.h, rows.ctypes.data)):
            assert call() == DDC_ERR_ARG
        assert view.tobytes() == want.tobytes()
        h.halo_close()
    finally:
        h.close()


# ---- 3. AddressSanitizer + UBSan -------------------------------------------------------------------------------------
def test_wide_halo_kernels_are_clean_under_address_sanitizer(oracle):
    """scatter, edge and full exchange and gather at w = 2 and 3 on tilings with zero-width strips and zero-height parts
    and on RCB output with empty parts: no kernel reads or writes outside an allocation"""
    oracle.build()
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    asan = subprocess.run([cc, "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0:halt_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "halo_asan_worker.py"), "2", "3"],
                         capture_output=True, text=True, timeout=900, env=env)
    assert "ERROR: AddressSanitizer" not in out.stderr and "runtime error:" not in out.stderr, out.stderr[-4000:]
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "HALO ASAN RUN OK" in out.stdout and "widths [2, 3]" in out.stdout
