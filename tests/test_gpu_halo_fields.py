"""Halo scatter and gather (ddc_halo_scatter_f64 / ddc_halo_gather_f64 and the sharded forms) on the GPU.

Single buffer: scatter and gather against the numpy expectation, bit for bit, up to C4; C5 as a round trip on the
device.  Sharded on one B200: G = 2, 3, 4 handles on device 0 (ddc_halo_connect, one host thread) against the single
buffer, and scatter -> exchange -> exchange -> gather twice on one step counter.  With two or more GPUs,
tests/halo_fields_worker.py runs the sharded calls over CUDA IPC, one process per GPU, under torchrun.
Fields are random 64-bit patterns viewed as float64 (NaN payloads, -0.0, subnormals); frames hold a sentinel.
The library runs on its handles' own streams: torch's work is synchronised before every call that reads or writes it."""
import os
import subprocess
import sys

import numpy as np
import pytest

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


def frame_cells(boxes, off):
    """buffer index of every frame cell of every tile"""
    b = np.asarray(boxes, dtype=np.int64)
    ex, ey, off = b[:, 2], b[:, 3], np.asarray(off, dtype=np.int64)[:-1]
    w = ex + 2
    g, i = hg._runs(w)
    rows = [off[g] + i, off[g] + (ey[g] + 1) * w[g] + i]
    g, j = hg._runs(ey)
    rows += [off[g] + (j + 1) * w[g], off[g] + (j + 1) * w[g] + ex[g] + 1]
    return np.concatenate(rows)


@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_single_buffer(env, case):
    capi, torch = env
    nx, ny, P, px, py = case
    h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = random_field(torch, nx, ny, P)
    tiles = torch.full((int(off[-1]),), SENT, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    h.halo_scatter_f64(field.data_ptr(), tiles.data_ptr())
    h.synchronize()
    want = scattered(boxes, off, u64(field), np.full(int(off[-1]), SENTINEL, dtype=np.uint64))
    assert u64(tiles).tobytes() == want.tobytes()
    fr = torch.from_numpy(frame_cells(boxes, off)).cuda()
    tiles[fr] = torch.randint(-2 ** 63, 2 ** 63 - 1, (len(fr),), dtype=torch.int64, device="cuda")  # frames: garbage
    back = torch.full_like(field, 7)
    torch.cuda.synchronize()
    h.halo_gather_f64(tiles.data_ptr(), back.data_ptr())
    h.synchronize()
    assert torch.equal(back, field)
    h.close()


def test_c5_round_trip(env):
    """C5 (32768^2, 16384 parts): gather(scatter(f)) == f on the device, frames untouched (about 26 GB)"""
    capi, torch = env
    nx = ny = 32768
    h = decompose(capi, torch, nx, ny, 16384, True, False, seed=32)
    del h._mask
    boxes = h.boxes()
    off = h.halo_tile_offsets()
    field = random_field(torch, nx, ny, 5)
    tiles = torch.full((int(off[-1]),), SENT, dtype=torch.int64, device="cuda")
    back = torch.zeros_like(field)
    torch.cuda.synchronize()
    h.halo_scatter_f64(field.data_ptr(), tiles.data_ptr())
    h.halo_gather_f64(tiles.data_ptr(), back.data_ptr())
    h.synchronize()
    assert torch.equal(back, field)
    fr = torch.from_numpy(frame_cells(boxes, off)).cuda()
    assert bool((tiles[fr] == SENT).all())
    h.close()
    del field, tiles, back, fr
    torch.cuda.empty_cache()


@pytest.mark.parametrize("case", CASES + EMPTY_CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_one_gpu_shards(env, case):
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
        for rep, periodic in enumerate((0, 1)):  # twice: the step counter carries across the calls
            ctx = (nx, ny, P, G, periodic)
            field = random_field(torch, nx, ny, 10 * G + rep)
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
            assert torch.equal(torch.cat(views), single), ctx + ("scatter",)
            want = scattered(boxes, off, u64(field), np.full(total, SENTINEL, dtype=np.uint64))
            assert u64(single).tobytes() == want.tobytes(), ctx + ("scatter",)
            for k in range(2):
                for h in handles:
                    h.halo_exchange_shards_f64(bool(periodic))
                single_h.halo_exchange_f64(single.data_ptr(), bool(periodic))
                for h in handles + [single_h]:
                    h.synchronize()
                want = exchanged(boxes, off, nx, ny, px, py, periodic, u64(field), want)
                assert torch.equal(torch.cat(views), single), ctx + ("exchange", k)
                assert u64(single).tobytes() == want.tobytes(), ctx + ("exchange", k)
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


def test_multi_gpu_worker(env):
    capi, torch = env
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (have %d)" % n)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tests", "halo_fields_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and ("HALO FIELDS OK world=%d" % n) in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
