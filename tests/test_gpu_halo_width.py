"""Wide halos (ddc_halo_set_width) on the GPU.

Single buffer: scatter, edge exchange, full exchange and gather at w = 2, 3, 4, bit for bit against halo_width's
expectation up to C4 (interiors hold the global cell index), both periodic settings.  At C5, w = 2: every cell of the
buffer -- interiors and the whole frame -- checked on the device after a scatter and a full exchange.  Sharded on one
B200: G = 2, 3, 4 handles on device 0 (ddc_halo_connect, one host thread) against the single buffer, in a sequence that
mixes scatter, full and edge exchanges and gather on one step counter.  Two user-level checks: two sweeps of a 5-point
Laplacian from one w = 2 exchange equal two sweeps each behind a w = 1 exchange, and a 5 x 5 box sum after a w = 2 full
exchange equals the box sum of the global field.  With two or more GPUs, tests/halo_width_worker.py runs the sharded
calls over CUDA IPC, one process per GPU, under torchrun.
The library runs on its handles' own streams: torch's work is synchronised before every call that reads or writes it."""
import os
import subprocess
import sys

import numpy as np
import pytest

import halo_global as hg
import halo_width as hw
from conftest import ROOT
from halo_global import (GPU_CASES as CASES, GPU_EMPTY_CASES as EMPTY_CASES, SENT, SENTINEL, decompose, dev_view,
                         random_field, u64)

pytestmark = pytest.mark.gpu
WIDTHS = (2, 3, 4)


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from domain_decomp_b200 import capi
    return capi, torch


def case_id(c):
    return "%dx%d_p%d" % c[:3]


@pytest.mark.parametrize("w", WIDTHS)
@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=case_id)
def test_single_buffer(env, case, w):
    capi, torch = env
    nx, ny, P, px, py = case
    h = decompose(capi, torch, nx, ny, P, px, py)
    h.halo_set_width(w)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    assert np.array_equal(off, hw.tile_offsets(boxes, w))
    init = hw.initial_tiles(boxes, off, nx, ny, w)
    field = torch.arange(nx * ny, dtype=torch.float64, device="cuda").view(ny, nx)
    tiles = torch.full((int(off[-1]),), hg.UNTOUCHED, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    h.halo_scatter_f64(field.data_ptr(), tiles.data_ptr())
    h.synchronize()
    assert tiles.cpu().numpy().tobytes() == init.tobytes()
    d_init = tiles.clone()
    for periodic in (0, 1):
        for full in (False, True):
            tiles.copy_(d_init)
            torch.cuda.synchronize()
            (h.halo_exchange_full_f64 if full else h.halo_exchange_f64)(tiles.data_ptr(), bool(periodic))
            h.synchronize()
            want = hw.exchanged(boxes, off, nx, ny, px, py, periodic, full, np.arange(nx * ny, dtype=np.float64)
                                .reshape(ny, nx), init, w)
            assert tiles.cpu().numpy().tobytes() == want.tobytes(), (periodic, full)
    back = torch.zeros_like(field)
    torch.cuda.synchronize()
    h.halo_gather_f64(tiles.data_ptr(), back.data_ptr())
    h.synchronize()
    assert torch.equal(back, field)
    h.close()


def test_c5_width_two(env):
    """C5 (32768^2, 16384 parts, periodic in x) at w = 2: after scatter and a periodic full exchange every interior cell
    holds its global index and every frame cell its wrapped cell, or UNTOUCHED across the non-periodic bottom and top
    (about 9 GB of tiles, checked on the device)"""
    capi, torch = env
    nx = ny = 32768
    w = 2
    h = decompose(capi, torch, nx, ny, 16384, True, False, seed=32)
    del h._mask
    h.halo_set_width(w)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = torch.arange(nx * ny, dtype=torch.float64, device="cuda").view(ny, nx)
    tiles = torch.full((int(off[-1]),), hg.UNTOUCHED, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    h.halo_scatter_f64(field.data_ptr(), tiles.data_ptr())
    h.halo_exchange_full_f64(tiles.data_ptr(), True)
    h.synchronize()
    del field
    b = torch.from_numpy(np.asarray(boxes, dtype=np.int64)).cuda()
    o = torch.from_numpy(np.asarray(off, dtype=np.int64)).cuda()
    filled = 0
    for k0 in range(0, int(off[-1]), 1 << 27):
        k = torch.arange(k0, min(k0 + (1 << 27), int(off[-1])), device="cuda")
        p = torch.searchsorted(o, k, right=True) - 1
        x0, y0, ex, ey = b[p].unbind(1)
        r, c = (k - o[p]) // (ex + 2 * w), (k - o[p]) % (ex + 2 * w)
        x, y = x0 + c - w, y0 + r - w
        inside = (r >= w) & (r < ey + w) & (c >= w) & (c < ex + w)
        has = (y >= 0) & (y < ny)  # periodic in x only; the boxes tile the domain
        want = torch.where(inside | has, ((y % ny) * nx + x % nx).double(), hg.UNTOUCHED)
        assert torch.equal(tiles[k0:k0 + len(k)], want), k0
        filled += int((has & ~inside).sum())
        del k, p, x0, y0, ex, ey, r, c, x, y, inside, has, want
    assert filled > 4 * 2 * 200 * 16384  # four strips of two rows of ~256 cells per part
    h.close()
    del tiles
    torch.cuda.empty_cache()


def connect(capi, boxes, nx, ny, px, py, G, w):
    """G handles on device 0 with the boxes at width w, joined by ddc_halo_connect, their shard offsets taken"""
    handles = [capi.Handle(0, q, G, None) for q in range(G)]
    for h in handles:
        h.neighbours_from_boxes(boxes, nx, ny, px, py)
        h.halo_set_width(w)
    ptrs = capi.halo_connect(handles, hw.max_shard_total(boxes, G, w))
    for h in handles:
        h.halo_shard_offsets()
    return handles, ptrs


@pytest.mark.parametrize("w", WIDTHS)
@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=case_id)
def test_one_gpu_shards(env, case, w):
    """scatter, full exchange, edge exchange, full exchange, gather on G handles sharing the B200, against the single
    buffer and the expectation after every call"""
    capi, torch = env
    nx, ny, P, px, py = case
    single_h = decompose(capi, torch, nx, ny, P, px, py)
    single_h.halo_set_width(w)
    boxes = single_h.boxes()
    off = single_h.halo_tile_offsets()
    total = int(off[-1])
    for G in (2, 3, 4):
        handles, ptrs = connect(capi, boxes, nx, ny, px, py, G, w)
        ranges = hg.shard_ranges(P, G)
        views = [dev_view(torch, ptrs[q], int(off[b + c] - off[b])).view(torch.int64) for q, (b, c) in enumerate(ranges)]
        rows = [capi.shard_rows(ny, G, q) for q in range(G)]
        single = torch.empty(total, dtype=torch.int64, device="cuda")
        periodic = G & 1
        ctx = (nx, ny, P, G, w, periodic)
        field = random_field(torch, nx, ny, 30 * G + w)
        for v in views:
            v.fill_(SENT)
        single.fill_(SENT)
        torch.cuda.synchronize()
        for q, h in enumerate(handles):  # one thread: each call only enqueues
            b, c = rows[q]
            h.halo_scatter_shards_f64(field[b:b + c].data_ptr() if c else 0)
        single_h.halo_scatter_f64(field.data_ptr(), single.data_ptr())
        for h in handles + [single_h]:
            h.synchronize()
        f = u64(field)
        want = hw.scattered(boxes, off, f, np.full(total, SENTINEL, dtype=np.uint64), w)
        assert u64(single).tobytes() == want.tobytes(), ctx
        for op in "fxf":
            for h in handles:
                (h.halo_exchange_full_shards_f64 if op == "f" else h.halo_exchange_shards_f64)(bool(periodic))
            (single_h.halo_exchange_full_f64 if op == "f" else single_h.halo_exchange_f64)(single.data_ptr(),
                                                                                           bool(periodic))
            for h in handles + [single_h]:
                h.synchronize()
            want = hw.exchanged(boxes, off, nx, ny, px, py, periodic, op == "f", f, want, w)
            assert torch.equal(torch.cat(views), single), ctx + (op,)
            assert u64(single).tobytes() == want.tobytes(), ctx + (op,)
        out = [torch.full((c, nx), 7, dtype=torch.int64, device="cuda") for _, c in rows]
        torch.cuda.synchronize()
        for h, o in zip(handles, out):
            h.halo_gather_shards_f64(o.data_ptr() if o.numel() else 0)
        for h in handles:
            h.synchronize()
        assert torch.equal(torch.cat(out), field), ctx + ("gather",)
        for h in handles:
            h.halo_close()
        for h in handles:
            h.close()
    single_h.close()


def tile_views(boxes, off, tiles, w):
    b = np.asarray(boxes, dtype=np.int64)
    return [tiles[off[p]:off[p + 1]].reshape(ey + 2 * w, ex + 2 * w) for p, (_, _, ex, ey) in enumerate(b)]


def laplace(t, m):
    """the 5-point Laplacian of tile t on its cells at least m + 1 from the tile's edge, written in place (the order of
    the operations is fixed, so equal inputs give equal bits)"""
    h, w = t.shape
    if h < 2 * m + 3 or w < 2 * m + 3:
        return
    c = t[m + 1:h - m - 1, m + 1:w - m - 1]
    lap = (((t[m:h - m - 2, m + 1:w - m - 1] + t[m + 2:h - m, m + 1:w - m - 1]) + t[m + 1:h - m - 1, m:w - m - 2])
           + t[m + 1:h - m - 1, m + 2:w - m]) - 4.0 * c
    t[m + 1:h - m - 1, m + 1:w - m - 1] = lap


@pytest.mark.parametrize("case", CASES[:2] + EMPTY_CASES, ids=case_id)
def test_two_sweeps_per_wide_exchange(env, case):
    """two sweeps of a 5-point Laplacian from ONE w = 2 exchange (full: the ring cells beside the box's corners read
    the diagonal cells) equal, bit for bit, two sweeps each behind a w = 1 edge exchange.  The first sweep runs over the
    interior and the one-cell ring around it; ring cells outside a non-periodic domain edge are reset to 0, the boundary
    value the one-cell frames keep there"""
    capi, torch = env
    nx, ny, P, px, py = case
    h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = h.boxes()
    field = np.random.default_rng(P + 1).standard_normal((ny, nx))
    d_field = torch.from_numpy(field).cuda()
    results = []
    for w in (2, 1):
        h.halo_set_width(w)
        off = h.halo_tile_offsets()
        tiles = torch.zeros(int(off[-1]), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        h.halo_scatter_f64(d_field.data_ptr(), tiles.data_ptr())
        for sweep in range(2):
            if w == 1:
                h.halo_exchange_f64(tiles.data_ptr(), True)
            elif sweep == 0:  # (a ring cell beside a corner of the box reads the diagonal cell)
                h.halo_exchange_full_f64(tiles.data_ptr(), True)
            h.synchronize()
            host = tiles.cpu().numpy()
            for p, t in enumerate(tile_views(boxes, off, host, w)):
                m = sweep if w == 2 else 0  # w = 2: the first sweep covers the ring too, the second the interior
                laplace(t, m)
                if w == 2 and sweep == 0:  # the ring outside a non-periodic domain edge is boundary, not field
                    x0, y0, ex, ey = (int(v) for v in boxes[p])
                    if not py and y0 == 0:
                        t[w - 1, :] = 0.0
                    if not py and y0 + ey == ny:
                        t[w + ey, :] = 0.0
                    if not px and x0 == 0:
                        t[:, w - 1] = 0.0
                    if not px and x0 + ex == nx:
                        t[:, w + ex] = 0.0
            tiles.copy_(torch.from_numpy(host))
            torch.cuda.synchronize()
        back = torch.zeros_like(d_field)
        h.halo_gather_f64(tiles.data_ptr(), back.data_ptr())
        h.synchronize()
        results.append(back.cpu().numpy())
    assert results[0].tobytes() == results[1].tobytes()
    assert not np.array_equal(results[0], field)
    h.close()


@pytest.mark.parametrize("case", CASES[:2] + EMPTY_CASES, ids=case_id)
def test_five_by_five_box_sum(env, case):
    """scatter -> w = 2 full exchange -> 5 x 5 box sum per tile -> gather == the box sum of the global field, zero-padded
    in non-periodic directions and wrapped in periodic ones (integer-valued doubles: the sums are exact)"""
    capi, torch = env
    nx, ny, P, px, py = case
    w = 2
    h = decompose(capi, torch, nx, ny, P, px, py)
    h.halo_set_width(w)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = np.random.default_rng(P).integers(-1000, 1000, size=(ny, nx)).astype(np.float64)
    d_field = torch.from_numpy(field).cuda()
    tiles = torch.zeros(int(off[-1]), dtype=torch.float64, device="cuda")  # frames preset to 0
    torch.cuda.synchronize()
    h.halo_scatter_f64(d_field.data_ptr(), tiles.data_ptr())
    h.halo_exchange_full_f64(tiles.data_ptr(), True)
    h.synchronize()
    host = tiles.cpu().numpy()
    summed = np.zeros_like(host)
    for t, s in zip(tile_views(boxes, off, host, w), tile_views(boxes, off, summed, w)):
        eh, ew = t.shape
        s[w:eh - w, w:ew - w] = sum(t[w + dy:eh - w + dy, w + dx:ew - w + dx] for dy in range(-2, 3) for dx in range(-2, 3))
    d_summed = torch.from_numpy(summed).cuda()
    back = torch.zeros_like(d_field)
    torch.cuda.synchronize()
    h.halo_gather_f64(d_summed.data_ptr(), back.data_ptr())
    h.synchronize()
    padded = np.pad(field, 2, mode="wrap")
    if not px:
        padded[:, :2], padded[:, -2:] = 0, 0
    if not py:
        padded[:2, :], padded[-2:, :] = 0, 0
    want = sum(padded[2 + dy:ny + 2 + dy, 2 + dx:nx + 2 + dx] for dy in range(-2, 3) for dx in range(-2, 3))
    assert np.array_equal(back.cpu().numpy(), want)
    h.close()


def test_multi_gpu_worker(env):
    capi, torch = env
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (have %d)" % n)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29549", os.path.join(ROOT, "tests", "halo_width_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    assert out.returncode == 0 and ("HALO WIDTH OK world=%d" % n) in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
