"""The product's own C-ABI implementation on a machine without a GPU.

oracle/libddc_cuda_emu.so is domain_decomp_b200/csrc/ddc_api.cu itself -- its `<<< >>>` launches rewritten by
oracle/emu/make_api_emu.py, nothing else -- compiled over a host stand-in of the CUDA runtime
(oracle/emu/cuda_runtime_fake.h) and the fiber emulation of the execution model.  The GPU parity tests of
tests/test_gpu_parity.py that fit a CPU (small masks) are run against it unchanged, through the same ctypes
front-end: besides the kernels this exercises the HOST logic of the library -- the assumed plan and the
re-run on a mismatch, DDC_ASYNC, the capacity re-run of the neighbour fill pass, reduced flag sets, caller-
supplied boxes (the all-pairs warp kernel), the error paths.  One rank; several ranks: test_kernels_on_cpu_emulator.
The product never loads this library: only this test module binds it."""
import ctypes as C
import os

import numpy as np
import pytest

import test_gpu_parity as T
from conftest import ROOT


class EmuCapi:
    """the parts of domain_decomp_b200.capi the tests use, bound to the emulation library"""

    def __init__(self, real, lib):
        self._real, self._lib = real, lib
        for name in ("WANT_PID", "WANT_NEIGHBOURS", "PROFILE", "ASYNC", "DdcError", "generate_mask_host", "LEFT", "RIGHT",
                     "BOTTOM", "TOP"):
            setattr(self, name, getattr(real, name))
        outer = self

        class Handle(real.Handle):
            def __init__(self, device=0, rank=0, nranks=1, nccl_id=None):
                self.L = outer._lib
                self.h = C.c_void_p()
                rc = self.L.ddc_create(C.byref(self.h), device, rank, nranks, nccl_id)
                if rc:
                    raise real.DdcError("ddc_create: %s" % self.L.ddc_last_error(None).decode())
                self.rank, self.nranks, self.nparts, self.shape, self._keep = rank, nranks, 0, None, None

        self.Handle = Handle


@pytest.fixture(scope="module")
def capi(oracle):
    from domain_decomp_b200 import capi as real
    oracle.build()
    path = os.path.join(ROOT, "oracle", "libddc_cuda_emu.so")
    assert os.path.exists(path)
    lib = C.CDLL(path)
    ref = real.load()
    for name in real.SYMBOLS:  # same prototypes as the CUDA library's
        getattr(lib, name).argtypes = getattr(ref, name).argtypes
        getattr(lib, name).restype = getattr(ref, name).restype
    return EmuCapi(real, lib)


@pytest.fixture()
def handle(capi):
    h = capi.Handle(0)
    yield h
    h.close()


def test_box_known_answers(goldens, handle):
    T.test_box_known_answers(goldens, handle)


@pytest.mark.parametrize("case", ["test_1", "test_2", "test_1_px", "test_1_py", "test_1_px_py"])
def test_integration_goldens(goldens, handle, case):
    T.test_integration_goldens(goldens, handle, case)


def test_rect3030(goldens, handle, oracle):
    T.test_rect3030(goldens, handle, oracle)


def test_random_small_masks(handle, oracle):
    """as tests/test_gpu_parity.py::test_random_small_masks, fewer iterations; ONE handle across changing extents"""
    rng = np.random.default_rng(11)
    for it in range(25):
        NX, NY = int(rng.integers(1, 50)), int(rng.integers(1, 50))
        dens = rng.choice([0.0, 0.02, 0.1, 0.3, 0.6, 0.9, 1.0])
        m = (rng.random((NY, NX)) < dens).astype(np.int32) * int(rng.integers(1, 5))
        if rng.random() < 0.3:
            m[:, rng.integers(0, NX)] = 0
        if rng.random() < 0.2:
            m[m == 0] = -int(rng.integers(0, 3))  # land is "<= 0"
        P = int(rng.integers(1, 24))
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        g = T.run_gpu(handle, m, P, px, py)
        o = oracle.partition(m, P, px, py, use_hist=bool(it & 1))
        T.assert_same(g, o, "it=%d NX=%d NY=%d P=%d dens=%s" % (it, NX, NY, P, dens))
        assert g["loads"].tolist() == oracle.part_loads(o.pid, P).tolist()
        assert g["stats"]["load_max"] == int(g["loads"].max()) and g["stats"]["load_min"] == int(g["loads"].min())


def test_neighbours_from_boxes_random(handle, oracle):
    T.test_neighbours_from_boxes_random(handle, oracle)


def test_flags_and_errors(capi, handle, oracle):
    m = capi.generate_mask_host(160, 120, seed=9, land_frac=0.4)
    a = T.run_gpu(handle, m, 12, True, True)
    handle.set_mask_host(m)
    handle.partition(12, True, True, flags=0)  # boxes only: no pid, no neighbours
    assert handle.boxes().tolist() == a["boxes"].tolist()
    assert handle.stats()["changes"] == a["stats"]["changes"]
    with pytest.raises(capi.DdcError):
        handle.pid_host()
    assert handle.neighbour_counts(0, 0).sum() == 0
    h2 = capi.Handle(0)
    with pytest.raises(capi.DdcError, match="no mask set"):
        h2.partition(4)
    with pytest.raises(capi.DdcError):
        h2.boxes()
    h2.close()


def test_async_steps_and_plan_mismatch(capi, handle, oracle):
    T.test_async_steps_and_plan_mismatch(capi, handle, oracle)


@pytest.mark.parametrize("n,P", [(64, 4), (60, 6)])
def test_nothing_moved_reports_naive_blocks(handle, oracle, n, P):
    T.test_nothing_moved_reports_naive_blocks(handle, oracle, n, P)


@pytest.mark.parametrize("case", [(260, 100, 24, 0.45, 4, "K2"), (8, 19000, 6, 0.45, 4, "K4"), (4096, 8, 1025, 0.4, 7, "K1"),
                                  (4096, 8, 2049, 0.4, 7, "k_strip_rows")],
                         ids=lambda c: "%dx%d-P%d-%s" % (c[0], c[1], c[2], c[5]))
def test_strip_row_kernel_variants(capi, oracle, case):
    """test_gpu_parity.test_strip_row_kernel_variants with shapes the emulation runs in seconds: the same four kernels,
    the K = 1 and k_strip_rows ones through 1024 and 2048 strips of few columns"""
    nx, ny, P, land, seed, kernel = case
    h = capi.Handle(0)
    try:
        m = capi.generate_mask_host(nx, ny, seed, land)
        g = T.run_gpu(h, m, P, True, False)
        T.assert_same(g, oracle.partition(m, P, True, False, use_hist=True), case)
        assert T.strip_row_kernel(nx, ny, P, g["stats"]) == kernel, (case, g["stats"])
    finally:
        h.close()


def test_neighbour_list_capacity_rerun(handle, oracle):
    """lists longer than the 3 P + 64 entries reserved per list: ddc_get_neighbours runs the fill pass again"""
    rng = np.random.default_rng(9)
    for (nx, ny, P, px, py) in [(11, 11, 36, False, False), (5, 6, 23, True, False)]:
        land = 0.5 + 0.4 * rng.random()
        m = (rng.random((ny, nx)) >= land).astype(np.int32)
        o = oracle.partition(m, P, px, py, use_hist=True)
        T.assert_same(T.run_gpu(handle, m, P, px, py), o, (nx, ny, P))
    assert max(len(x) for per in range(2) for x in o.nbr.ids[per]) > 3 * 23 + 64


def test_repeated_and_alternating_geometries_on_one_handle(capi, handle, oracle):
    """the host launches k_init only when the buffers or the geometry differ from what the previous steps left
    clean: the same mask five times, then two geometries in turn (same buffers, other widths), then P changes"""
    a = capi.generate_mask_host(96, 64, 3, 0.45)
    b = capi.generate_mask_host(50, 40, 5, 0.3)
    oa, ob = oracle.partition(a, 12, True, False, use_hist=True), oracle.partition(b, 7, False, True, use_hist=True)
    launches = []
    for _ in range(5):
        g = T.run_gpu(handle, a, 12, True, False)
        T.assert_same(g, oa, "repeat")
        launches.append(g["stats"]["gpu_launches"])
    assert launches[0] == launches[-1] + 1, launches  # only the first step needed k_init
    for _ in range(3):
        T.assert_same(T.run_gpu(handle, b, 7, False, True), ob, "alternating b")
        T.assert_same(T.run_gpu(handle, a, 12, True, False), oa, "alternating a")
    for P in (5, 12, 3):
        T.assert_same(T.run_gpu(handle, a, P, True, False), oracle.partition(a, P, True, False, use_hist=True), P)


def test_argument_and_state_errors(capi, oracle):
    """every entry point answers misuse with a status and a message (Utils.hpp / Grid.hpp conventions of the
    reference: nothing aborts, nothing is silently ignored)"""
    L = capi._lib
    h = capi.Handle(0)
    m = capi.generate_mask_host(40, 30, 1, 0.5)
    try:
        # create: rank outside the communicator, ranks > 1 without a NCCL id
        hh = C.c_void_p()
        assert L.ddc_create(C.byref(hh), 0, 3, 2, None) < 0 and b"bad arguments" in L.ddc_last_error(None)
        # ranks > 1 without a NCCL id: allowed (peer-memory exchange only), but a step without any exchange path fails
        assert L.ddc_create(C.byref(hh), 0, 0, 2, None) == 0
        half = np.ascontiguousarray(m[:15])
        assert L.ddc_set_mask_host(hh, half.ctypes.data, 40, 30, 0, 15) == 0
        assert L.ddc_partition(hh, 4, 0, 0, 3) < 0 and b"no exchange path" in L.ddc_last_error(hh)
        assert L.ddc_destroy(hh) == 0
        assert L.ddc_create(C.byref(hh), 7, 0, 1, None) < 0 and b"out of range" in L.ddc_last_error(None)
        # masks: extents, shard bounds, null pointers
        assert L.ddc_set_mask_host(h.h, m.ctypes.data, 0, 30, 0, 30) < 0
        assert L.ddc_set_mask_host(h.h, m.ctypes.data, 40, 30, 0, 29) < 0 and b"must hold rows" in L.ddc_last_error(h.h)
        assert L.ddc_set_mask_host(h.h, None, 40, 30, 0, 30) < 0
        assert L.ddc_set_mask_host(h.h, m.ctypes.data, 65536, 65536, 0, 65536) < 0  # more cells than an int can index
        # partition: before a mask, bad part count
        with pytest.raises(capi.DdcError, match="no mask set"):
            h.partition(4)
        h.set_mask_host(m)
        with pytest.raises(capi.DdcError, match="nparts"):
            h.partition(0)
        # getters before a partition, bad edge
        with pytest.raises(capi.DdcError, match="ddc_partition"):
            h.boxes()
        h.partition(6, True, False)
        out = np.zeros(6, dtype=np.int32)
        assert L.ddc_get_neighbour_counts(h.h, 4, 0, out.ctypes.data) < 0 and b"edge" in L.ddc_last_error(h.h)
        assert L.ddc_get_neighbour_counts(h.h, 0, 2, out.ctypes.data) < 0
        # a new mask invalidates the old results
        h.set_mask_host(m)
        with pytest.raises(capi.DdcError):
            h.boxes()
        # P == 1: the reference returns before neighbour discovery (quirk Q4): empty lists, no error
        h.partition(1, True, True)
        assert h.boxes().tolist() == [[0, 0, 40, 30]]
        assert all(len(h.neighbours(e, per)[0]) == 0 for e in range(4) for per in range(2))
        assert np.array_equal(h.pid_host(), np.where(m > 0, 0, -1))
        # more parts than cells
        h.partition(40 * 30 + 5)
        o = oracle.partition(m, 40 * 30 + 5, use_hist=True)
        assert h.boxes().tolist() == o.boxes.tolist() and np.array_equal(h.pid_host(), o.pid)
    finally:
        h.close()
    assert L.ddc_destroy(None) == 0 and L.ddc_partition(None, 4, 0, 0, 3) < 0


def test_random_call_sequences_on_one_handle(capi, handle, oracle):
    """the state a handle carries between calls (buffers, the cached plan, which accumulators are clean): a random
    sequence of decompositions over a pool of masks of different extents -- synchronous, DDC_ASYNC twice in a row,
    boxes-only followed by a full step on the same mask, caller-supplied boxes in between"""
    rng = np.random.default_rng(3)
    pool = []
    for i in range(5):
        nx, ny = int(rng.integers(1, 100)), int(rng.integers(1, 100))
        m = (rng.random((ny, nx)) >= rng.random()).astype(np.int32)
        if i == 0:
            m[:] = 1
        if i == 1:
            m[:] = 0
        pool.append(m)
    for it in range(25):
        m = pool[int(rng.integers(0, len(pool)))]
        P = int(rng.integers(1, 30))
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        mode = int(rng.integers(0, 4))
        o = oracle.partition(m, P, px, py, use_hist=True)
        ctx = (it, m.shape, P, mode)
        if mode == 0:
            T.assert_same(T.run_gpu(handle, m, P, px, py), o, ctx)
        elif mode == 1:
            handle.set_mask_host(m)
            for _ in range(2):
                handle.partition(P, px, py, flags=capi.WANT_PID | capi.WANT_NEIGHBOURS | capi.ASYNC)
            assert handle.boxes().tolist() == o.boxes.tolist() and np.array_equal(handle.pid_host(), o.pid), ctx
        elif mode == 2:
            handle.set_mask_host(m)
            handle.partition(P, px, py, flags=0)
            assert handle.boxes().tolist() == o.boxes.tolist(), ctx
            handle.partition(P, px, py)
            assert np.array_equal(handle.pid_host(), o.pid) and handle.stats()["median_iters"] == o.median_iters, ctx
        else:
            handle.neighbours_from_boxes(o.boxes, m.shape[1], m.shape[0], px, py)
            if P > 1:
                assert handle.neighbours(0, 0)[0].tolist() == o.nbr.ids[0][0].tolist(), ctx
            T.assert_same(T.run_gpu(handle, m, P, px, py), o, ctx)


def test_device_mask_generator_and_device_resident_path(capi, handle, oracle):
    """ddc_generate_mask_device == ddc_generate_mask_host (the benchmark's masks are synthesised on the device), and
    the device-pointer entry points (borrowed mask in, pid pointer out) -- "device memory" is host memory here"""
    nx, ny, P = 150, 70, 10
    d = np.full((ny, nx), -7, dtype=np.int32)
    handle.generate_mask_device(d.ctypes.data, nx, ny, 25, 0.45)
    assert np.array_equal(d, capi.generate_mask_host(nx, ny, 25, 0.45))
    half = np.full((30, nx), -7, dtype=np.int32)  # a row block of the same global mask
    handle.generate_mask_device(half.ctypes.data, nx, ny, 25, 0.45, y_begin=20, y_count=30)
    assert np.array_equal(half, d[20:50])
    handle.set_mask_device(d.ctypes.data, nx, ny)
    handle.partition(P, True, False)
    o = oracle.partition(d, P, True, False, use_hist=True)
    ptr = handle.pid_device()
    pid = np.ctypeslib.as_array((C.c_int32 * (nx * ny)).from_address(ptr)).reshape(ny, nx)
    assert np.array_equal(pid, o.pid) and handle.boxes().tolist() == o.boxes.tolist()


def test_halo_exchange_consumes_the_neighbour_tables(capi, handle):
    """ddc_halo_exchange_f64 (the GPU analogue of examples/zoltan_comm.cpp:84-246 of the reference) on the emulation:
    after the exchange every ghost cell that faces a neighbour holds that neighbour's id, derived independently from
    the boxes (tests/halo_check.py) -- interior and periodic lists, ragged coastlines, part counts that are not
    powers of two"""
    import halo_check
    rng = np.random.default_rng(21)
    done = 0
    while done < 12:
        nx, ny, P = int(rng.integers(6, 60)), int(rng.integers(6, 60)), int(rng.integers(2, 14))
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        mask = (rng.random((ny, nx)) < 0.8).astype(np.int32)
        handle.set_mask_host(mask)
        handle.partition(P, px, py)
        boxes = handle.boxes()
        if (boxes[:, 2:] <= 0).any():
            continue  # an empty part has no tile to exchange with
        off = handle.halo_tile_offsets()
        for periodic in (False, True):
            tiles = halo_check.initial_tiles(boxes, off)
            handle.halo_exchange_f64(tiles.ctypes.data, periodic)  # (emulation: "device" memory is host memory)
            handle.L.ddc_synchronize(handle.h)
            want = halo_check.expected_tiles(boxes, off, nx, ny, px, py, periodic)
            assert np.array_equal(tiles, want), (nx, ny, P, px, py, periodic)
        done += 1
