"""The full-frame halo exchange (corner ghosts) on the GPU.

Single buffer: bit for bit against halo_frame's expectation up to C4 (interiors hold the global cell index), both
periodic settings; at C5 the edges against ddc_halo_exchange_f64 and all 4 P corners against the corner table.  Sharded
on one B200: G = 2, 3, 4 handles on device 0 (ddc_halo_connect, one host thread) against the single buffer, in a
sequence that mixes scatter, full and edge exchanges and gather on one step counter.  A user-level check: a 3 x 3 box sum
per tile from its full frame, gathered, equals the box sum of the global field.  With two or more GPUs,
tests/halo_frame_worker.py runs the sharded calls over CUDA IPC, one process per GPU, under torchrun.
The library runs on its handles' own streams: torch's work is synchronised before every call that reads or writes it."""
import os
import subprocess
import sys

import numpy as np
import pytest

import halo_frame as hf
import halo_global as hg
from conftest import ROOT
from halo_global import (GPU_CASES as CASES, GPU_EMPTY_CASES as EMPTY_CASES, SENT, SENTINEL, connect, decompose,
                         dev_view, exchanged, random_field, scattered, u64)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from domain_decomp_b200 import capi
    return capi, torch


@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_single_buffer(env, case):
    capi, torch = env
    nx, ny, P, px, py = case
    h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    ids = np.array([[h.corner_neighbours(c, per)[0] for c in range(4)] for per in range(2)])
    assert np.array_equal(ids, hf.corner_table(boxes, nx, ny, px, py)[0])
    init = torch.from_numpy(hg.initial_tiles(boxes, off, nx)).cuda()
    for periodic in (0, 1):
        tiles = init.clone()
        torch.cuda.synchronize()
        h.halo_exchange_full_f64(tiles.data_ptr(), bool(periodic))
        h.synchronize()
        want = hf.expected_full_tiles(boxes, off, nx, ny, px, py, periodic)
        assert tiles.cpu().numpy().tobytes() == want.tobytes(), periodic
    h.close()


def check_scattered_index(torch, boxes, off, tiles, nx, chunk=1 << 27):
    """every interior cell of the tiles holds its global index y * nx + x, every frame cell UNTOUCHED: on the tiles'
    device, `chunk` buffer cells at a time"""
    b = torch.from_numpy(np.asarray(boxes, dtype=np.int64)).to(tiles.device)
    o = torch.from_numpy(np.asarray(off, dtype=np.int64)).to(tiles.device)
    for k0 in range(0, int(off[-1]), chunk):
        k = torch.arange(k0, min(k0 + chunk, int(off[-1])), device=tiles.device)
        p = torch.searchsorted(o, k, right=True) - 1
        x0, y0, ex, ey = b[p].unbind(1)
        r, c = (k - o[p]) // (ex + 2), (k - o[p]) % (ex + 2)
        inside = (r >= 1) & (r <= ey) & (c >= 1) & (c <= ex)
        want = torch.where(inside, ((y0 + r - 1) * nx + x0 + c - 1).double(), hg.UNTOUCHED)
        assert torch.equal(tiles[k0:k0 + len(k)], want), k0
        del k, p, x0, y0, ex, ey, r, c, inside, want


def test_c5_edges_and_corners(env):
    """C5 (32768^2, 16384 parts, periodic in x), interiors the global index: the scatter puts every cell where it
    belongs, the edge exchange gives every edge ghost its wrapped cell (16.7 M), the full exchange leaves every non-corner
    cell as the edge exchange does, and every one of the 4 P corners as the corner table says (about 35 GB)"""
    capi, torch = env
    nx = ny = 32768
    px, py = True, False
    h = decompose(capi, torch, nx, ny, 16384, px, py, seed=32)
    del h._mask
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = torch.arange(nx * ny, dtype=torch.float64, device="cuda").view(ny, nx)
    edge = torch.full((int(off[-1]),), hg.UNTOUCHED, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    h.halo_scatter_f64(field.data_ptr(), edge.data_ptr())
    h.synchronize()
    del field
    check_scattered_index(torch, boxes, off, edge, nx)
    full = edge.clone()
    torch.cuda.synchronize()
    h.halo_exchange_f64(edge.data_ptr(), True)
    h.halo_exchange_full_f64(full.data_ptr(), True)
    h.synchronize()
    gi, gx, gy = (torch.from_numpy(a).cuda() for a in hg.ghost_cells(boxes, off))
    want = torch.where((gy >= 0) & (gy < ny), ((gy % ny) * nx + gx % nx).double(), hg.UNTOUCHED)  # px, not py
    assert len(gi) > 16_000_000 and torch.equal(edge[gi], want)
    del gi, gx, gy, want
    idx = torch.from_numpy(hf.corner_cells(boxes, off).reshape(-1)).cuda()
    got = full[idx].cpu().numpy()
    assert bool((edge[idx] == hg.UNTOUCHED).all())
    full[idx] = edge[idx]
    assert torch.equal(full, edge)
    ids, _ = hf.corner_table(boxes, nx, ny, px, py)
    x, y = hf.corner_xy(boxes)
    src = np.maximum(ids[0], ids[1]).reshape(-1)
    want = np.where(src >= 0, ((y % ny) * nx + (x % nx)).reshape(-1).astype(np.float64), hg.UNTOUCHED)
    assert np.array_equal(got, want)
    assert (src >= 0).sum() > 3 * 16384  # (all but the corners on the non-periodic bottom and top)
    h.close()
    del edge, full, idx
    torch.cuda.empty_cache()


@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_one_gpu_shards(env, case):
    """scatter, full exchange, edge exchange, full exchange, gather on G handles sharing the B200, against the single
    buffer after every call"""
    capi, torch = env
    nx, ny, P, px, py = case
    single_h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = single_h.boxes()
    off = single_h.halo_tile_offsets()
    total = int(off[-1])
    for G in (2, 3, 4):
        handles, ptrs = connect(capi, boxes, nx, ny, px, py, G)
        ranges = hg.shard_ranges(P, G)
        views = [dev_view(torch, ptrs[q], int(off[b + c] - off[b])).view(torch.int64) for q, (b, c) in enumerate(ranges)]
        rows = [capi.shard_rows(ny, G, q) for q in range(G)]
        single = torch.empty(total, dtype=torch.int64, device="cuda")
        for rep, periodic in enumerate((0, 1)):
            ctx = (nx, ny, P, G, periodic)
            field = random_field(torch, nx, ny, 20 * G + rep)
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
            want = scattered(boxes, off, f, np.full(total, SENTINEL, dtype=np.uint64))
            for op in "fxf":
                for h in handles:
                    (h.halo_exchange_full_shards_f64 if op == "f" else h.halo_exchange_shards_f64)(bool(periodic))
                (single_h.halo_exchange_full_f64 if op == "f" else single_h.halo_exchange_f64)(single.data_ptr(),
                                                                                               bool(periodic))
                for h in handles + [single_h]:
                    h.synchronize()
                want = exchanged(boxes, off, nx, ny, px, py, periodic, f, want)
                if op == "f":
                    want = hf.with_corners(boxes, off, nx, ny, px, py, periodic, f, want)
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


def box_sum_tiles(boxes, off, tiles):
    """every tile's interior <- the 3 x 3 sum of its cells read from the tile itself, frame included"""
    out = np.zeros_like(tiles)
    for p, (x0, y0, ex, ey) in enumerate(np.asarray(boxes, dtype=np.int64)):
        t = tiles[off[p]:off[p + 1]].reshape(ey + 2, ex + 2)
        o = out[off[p]:off[p + 1]].reshape(ey + 2, ex + 2)
        o[1:-1, 1:-1] = sum(t[1 + dy:ey + 1 + dy, 1 + dx:ex + 1 + dx] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    return out


@pytest.mark.parametrize("case", CASES[:2] + EMPTY_CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_nine_point_stencil(env, case):
    """scatter -> full exchange -> 3 x 3 box sum per tile -> gather == the box sum of the global field, zero-padded in
    non-periodic directions and wrapped in periodic ones (integer-valued doubles: the sums are exact)"""
    capi, torch = env
    nx, ny, P, px, py = case
    h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = np.random.default_rng(P).integers(-1000, 1000, size=(ny, nx)).astype(np.float64)
    d_field = torch.from_numpy(field).cuda()
    tiles = torch.zeros(int(off[-1]), dtype=torch.float64, device="cuda")  # frames preset to 0
    torch.cuda.synchronize()
    h.halo_scatter_f64(d_field.data_ptr(), tiles.data_ptr())
    h.halo_exchange_full_f64(tiles.data_ptr(), True)
    h.synchronize()
    summed = torch.from_numpy(box_sum_tiles(boxes, off, tiles.cpu().numpy())).cuda()
    back = torch.zeros_like(d_field)
    torch.cuda.synchronize()
    h.halo_gather_f64(summed.data_ptr(), back.data_ptr())
    h.synchronize()
    padded = np.pad(field, 1)
    if px:
        padded[:, 0], padded[:, -1] = padded[:, -2], padded[:, 1]
    if py:
        padded[0, :], padded[-1, :] = padded[-2, :], padded[1, :]
    want = sum(padded[1 + dy:ny + 1 + dy, 1 + dx:nx + 1 + dx] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    if px and py:
        assert np.array_equal(want, sum(np.roll(field, (dy, dx), axis=(0, 1)) for dy in (-1, 0, 1) for dx in (-1, 0, 1)))
    assert np.array_equal(back.cpu().numpy(), want)
    h.close()


def test_multi_gpu_worker(env):
    capi, torch = env
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (have %d)" % n)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "halo_frame_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and ("HALO FRAME OK world=%d" % n) in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
