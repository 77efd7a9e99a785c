"""Byte masks on one B200 (ddc_set_mask_u8_*, k_scan_mask_u8), bit for bit against the int32 path on the same cells
and the same handle: boxes, pid, changes, median iterations, part loads, n_ocean, load min / max, edge cut, launch
counts and all eight neighbour lists.  C4 and C5 also against the CPU oracle's digests (tests/golden/bench_digests.json)."""
import json
import os

import numpy as np
import pytest

import mask_bytes as MB
import many_leaves as ML
from conftest import ROOT

pytestmark = pytest.mark.gpu

WORKLOADS = {k: v for k, v in json.load(open(os.path.join(ROOT, "tests", "golden", "bench_digests.json"))).items()}


@pytest.fixture(scope="module")
def capi():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests need one (the product has no CPU fallback)")
    from domain_decomp_b200 import capi
    capi.load()
    return capi


@pytest.fixture(scope="module")
def handle(capi):
    h = capi.Handle(0)
    yield h
    h.close()


def device_pair(h, d_mask, P, px, py, u8):
    """the int32 device mask (twice, so that both compared runs start settled), then the byte tensor u8"""
    ny, nx = d_mask.shape
    h.set_mask_device(d_mask.data_ptr(), nx, ny)
    h.partition(P, px, py)
    h.partition(P, px, py)
    a = MB.snapshot(h, "device")
    h.set_mask_u8_device(u8.data_ptr(), nx, ny)
    h.partition(P, px, py)
    return a, MB.snapshot(h, "device")


def generated(h, nx, ny, seed, land):
    import torch
    d = torch.empty((ny, nx), dtype=torch.int32, device="cuda")
    h.generate_mask_device(d.data_ptr(), nx, ny, seed, land)
    torch.cuda.synchronize()  # (the handle's stream is not torch's: the tensors derived from d must see the mask)
    return d


def workload(name):
    w = WORKLOADS[name]
    return w["nx"], w["ny"], w["parts"], w["seed"], w["land_frac"], bool(w["periodic_x"]), bool(w["periodic_y"])


@pytest.mark.parametrize("name", ["C2_528x522_p64", "C3_4096x4096_p1024", "C4_8192x8192_p4096"])
def test_workloads_every_periodicity(handle, name):
    import torch
    nx, ny, P, seed, land, _, _ = workload(name)
    d = generated(handle, nx, ny, seed, land)
    u8 = (d > 0).to(torch.uint8) * 0xFF
    torch.cuda.synchronize()
    for px in (False, True):
        for py in (False, True):
            a, u = device_pair(handle, d, P, px, py, u8)
            MB.assert_same(a, u, (name, px, py))


@pytest.mark.parametrize("name", ["C4_8192x8192_p4096", "C5_32768x32768_p16384"])
def test_workloads_match_the_oracle_digest(handle, name):
    import torch
    from domain_decomp_b200 import verify
    nx, ny, P, seed, land, px, py = workload(name)
    d = generated(handle, nx, ny, seed, land)
    b = d > 0  # torch.bool
    torch.cuda.synchronize()
    if name.startswith("C5"):
        a, u = device_pair(handle, d, P, px, py, b)
        MB.assert_same(a, u, name)
        del a, u
    del d
    torch.cuda.empty_cache()
    handle.set_mask_u8_device(b.data_ptr(), nx, ny)
    handle.partition(P, px, py)
    assert verify.handle_digest(handle) == WORKLOADS[name]["digest"], name
    assert handle.stats()["n_ocean"] == WORKLOADS[name]["n_ocean"]


def test_bool_uint8_and_unaligned_slices(handle):
    """torch.bool and torch.uint8 tensors, and uint8 views 1..15 bytes past an aligned address (the byte-by-byte path
    unless the view is 4-byte aligned), at widths that are and are not multiples of 4 and 16"""
    import torch
    for nx, ny, P in ((2048, 1500, 256), (1000, 1000, 100), (1001, 777, 97), (4100, 300, 64)):
        d = generated(handle, nx, ny, nx, 0.45)
        ocean = (d > 0).to(torch.uint8)
        first = True
        for off in (0, 1, 2, 4, 7, 15):
            buf = torch.zeros(off + nx * ny, dtype=torch.uint8, device="cuda")
            view = buf[off:].view(ny, nx)
            view.copy_(ocean * 0x80 if off & 1 else ocean)
            torch.cuda.synchronize()
            if first:
                a, u = device_pair(handle, d, P, True, False, view)
                first = False
            else:
                handle.set_mask_u8_device(view.data_ptr(), nx, ny)
                handle.partition(P, True, False)
                u = MB.snapshot(handle, "device")
            MB.assert_same(a, u, (nx, ny, off))
        b = d > 0
        torch.cuda.synchronize()
        handle.set_mask_u8_device(b.data_ptr(), nx, ny)
        handle.partition(P, True, False)
        MB.assert_same(a, MB.snapshot(handle, "device"), (nx, ny, "bool"))


def test_host_pinned_and_pageable(handle, capi):
    import torch
    nx, ny, P = 1001, 777, 97
    m = capi.generate_mask_host(nx, ny, 11, 0.45)
    rng = np.random.default_rng(1)
    b = MB.byte_mask(m, rng)
    pinned = torch.from_numpy(b).pin_memory()
    for set_ in (lambda h: h.set_mask_u8_host(b), lambda h: h.set_mask_u8_host(pinned.numpy()),
                 lambda h: h.set_mask_u8_host(np.ascontiguousarray(m > 0))):
        a, u = MB.run_pair(handle, m, set_, P, True, True)
        MB.assert_same(a, u)


@pytest.mark.parametrize("case", [ML.GPU_CASES[6], ML.GPU_CASES[11], ML.GPU_CASES[4]], ids=ML.case_id)
def test_many_strips(handle, capi, oracle, case):
    """many strips and parts per strip (tests/many_leaves.py): the scan's outputs feed the walking cut kernels"""
    mask, o, loads = ML.expected(oracle, case)
    rng = np.random.default_rng(case.P)
    a, u = MB.run_pair(handle, mask, lambda h: h.set_mask_u8_host(MB.byte_mask(mask, rng)), case.P, case.px, case.py)
    MB.assert_same(a, u, ML.case_id(case))
    assert u["boxes"].tolist() == o.boxes.tolist() and np.array_equal(u["pid"], o.pid)
