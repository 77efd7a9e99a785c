"""The sharded halo exchange (ddc_halo_exchange_shards_f64) on the GPU.

One B200: G = 2, 3, 4 handles on device 0 hold the parts' tiles in G library-owned buffers, joined by
ddc_halo_connect and driven by one host thread.  The buffers concatenated in rank order must equal, bit for bit,
ddc_halo_exchange_f64 on one buffer and the expected tiles (interiors = global cell index, tests/halo_global.py).
With two or more GPUs, tests/halo_shards_worker.py runs the same over CUDA IPC, one process per GPU, under torchrun."""
import os
import subprocess
import sys

import numpy as np
import pytest

import halo_global as hg
from conftest import ROOT

pytestmark = pytest.mark.gpu

CASES = [  # nx, ny, P, px, py
    (528, 522, 64, True, True),
    (2048, 1536, 1000, True, False),
    (8192, 8192, 4096, False, False),
]


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from domain_decomp_b200 import capi
    return capi, torch


class _Dev:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 2,
                                         "strides": None}


def dev_view(torch, ptr, n):
    """float64[n] over raw device memory (a halo buffer of the library)"""
    return torch.as_tensor(_Dev(ptr, n), device="cuda") if n else torch.empty(0, dtype=torch.float64, device="cuda")


def decompose(capi, torch, nx, ny, P, px, py, seed=3, land=0.45):
    h = capi.Handle(0)
    d_mask = torch.empty((ny, nx), dtype=torch.int32, device="cuda")
    h.generate_mask_device(d_mask.data_ptr(), nx, ny, seed, land)
    h.set_mask_device(d_mask.data_ptr(), nx, ny)
    h.partition(P, px, py)
    h._mask = d_mask
    return h


def check_exchanges(capi, torch, single_h, handles, ptrs, nx, ny, px, py, steps=2):
    """exchanges on the shards and on one buffer (single_h), interiors changed in between: bit-identical + expected"""
    boxes = single_h.boxes()
    P, G = len(boxes), len(handles)
    off = hg.tile_offsets(boxes)
    assert single_h.halo_tile_offsets().tolist() == off.tolist()
    ranges = hg.shard_ranges(P, G)
    for q, h in enumerate(handles):
        b, c = ranges[q]
        assert h.halo_shard_offsets().tolist() == (off[b:b + c + 1] - off[b]).tolist()
    views = [dev_view(torch, ptrs[q], int(off[b + c] - off[b])) for q, (b, c) in enumerate(ranges)]
    for periodic in (0, 1):
        single = None
        for k in range(steps):
            fresh = torch.from_numpy(hg.initial_tiles(boxes, off, nx, 1000.0 * (periodic * steps + k))).cuda()
            if single is None:  # whole tiles first, then interiors only: a ghost nobody writes keeps its old value
                single = fresh.clone()
                interior = fresh != hg.UNTOUCHED
            else:
                single = torch.where(interior, fresh, single)
            for q, (b, c) in enumerate(ranges):
                if k == 0:
                    views[q].copy_(fresh[int(off[b]):int(off[b + c])])
                else:
                    sl = slice(int(off[b]), int(off[b + c]))
                    views[q].copy_(torch.where(interior[sl], fresh[sl], views[q]))
            torch.cuda.synchronize()
            for h in handles:  # one thread: each call only enqueues
                h.halo_exchange_shards_f64(bool(periodic))
            for h in handles:
                h.synchronize()
            single_h.halo_exchange_f64(single.data_ptr(), bool(periodic))
            single_h.synchronize()
            cat = torch.cat(views)
            ctx = (nx, ny, P, G, periodic, k)
            assert torch.equal(cat.view(torch.int64), single.view(torch.int64)), ctx
            want = hg.expected_tiles(boxes, off, nx, ny, px, py, periodic, 1000.0 * (periodic * steps + k))
            assert np.array_equal(cat.cpu().numpy(), want), ctx


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%dx%d_p%d" % c[:3])
def test_one_gpu_shards(env, case):
    capi, torch = env
    nx, ny, P, px, py = case
    single_h = decompose(capi, torch, nx, ny, P, px, py)
    boxes = single_h.boxes()
    for G in (2, 3, 4):
        handles = [capi.Handle(0, q, G, None) for q in range(G)]
        for h in handles:
            h.neighbours_from_boxes(boxes, nx, ny, px, py)
        ptrs = capi.halo_connect(handles, hg.max_shard_total(boxes, G))
        check_exchanges(capi, torch, single_h, handles, ptrs, nx, ny, px, py)
        for h in handles:
            h.halo_close()
        for h in handles:
            h.close()


def test_repartition_reuses_or_refuses(env):
    """a decomposition into other parts reuses the buffers when its tiles fit; otherwise every rank refuses with
    DDC_ERR_ARG before anything is enqueued, and the next one that fits runs"""
    capi, torch = env
    G = 3
    first = decompose(capi, torch, 528, 522, 64, True, True)
    fits = decompose(capi, torch, 528, 522, 40, True, False)
    elems = max(hg.max_shard_total(first.boxes(), G), hg.max_shard_total(fits.boxes(), G))
    handles = [capi.Handle(0, q, G, None) for q in range(G)]
    for h in handles:
        h.neighbours_from_boxes(first.boxes(), 528, 522, True, True)
    ptrs = capi.halo_connect(handles, elems)
    check_exchanges(capi, torch, first, handles, ptrs, 528, 522, True, True, steps=1)
    too_big = decompose(capi, torch, 700, 600, 96, False, True)
    assert hg.max_shard_total(too_big.boxes(), G) > elems
    for h in handles:
        h.neighbours_from_boxes(too_big.boxes(), 700, 600, False, True)
        # no ddc_halo_shard_offsets for this decomposition yet: DDC_ERR_STATE
        assert h.L.ddc_halo_exchange_shards_f64(h.h, 0) == -5
        h.halo_shard_offsets()
        assert h.L.ddc_halo_exchange_shards_f64(h.h, 1) == -1  # DDC_ERR_ARG on every rank
    for h in handles:
        h.neighbours_from_boxes(fits.boxes(), 528, 522, True, False)
    check_exchanges(capi, torch, fits, handles, ptrs, 528, 522, True, False, steps=1)
    for h in handles:
        h.halo_close()
        h.close()


def test_decomposition_launches_unchanged(env):
    """the halo buffers add nothing to the decomposition path: same kernel launches with and without them"""
    capi, torch = env
    nx, ny, P = 2048, 1536, 1000
    plain = decompose(capi, torch, nx, ny, P, True, False)
    plain.partition(P, True, False)
    want = plain.stats()["gpu_launches"]
    h = capi.Handle(0)
    h.set_mask_device(plain._mask.data_ptr(), nx, ny)
    (ptr,) = capi.halo_connect([h], hg.max_shard_total(plain.boxes(), 1))
    h.partition(P, True, False)
    h.partition(P, True, False)
    assert h.stats()["gpu_launches"] == want
    h.halo_shard_offsets()
    h.halo_exchange_shards_f64(True)
    h.synchronize()
    h.partition(P, True, False)
    assert h.stats()["gpu_launches"] == want
    assert h.boxes().tolist() == plain.boxes().tolist()
    h.halo_close()
    h.close()


def test_multi_gpu_worker(env):
    capi, torch = env
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (have %d)" % n)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "halo_shards_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0 and ("HALO SHARDS OK world=%d" % n) in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
