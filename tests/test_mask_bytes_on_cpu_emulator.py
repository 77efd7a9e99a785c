"""Byte masks (ddc_set_mask_u8_*, k_scan_mask_u8) on a machine without a GPU, bit for bit against the int32 path on
the same cells:
  * one rank through the library's own C ABI on the emulated runtime (oracle/libddc_cuda_emu.so): widths around 16k
    and below 16, both scan paths, every kind of ocean byte, unaligned pointers, a type switch on one handle, DDC_ASYNC,
    the plan-mismatch re-run and the status codes;
  * 2, 3 and 5 row-sharded ranks through the multi-rank pipeline with byte shards (tests/emu_mask_bytes.cpp): empty
    row blocks, int32 and byte ranks mixed, both exchange layouts and random block / thread schedules."""
import ctypes as C

import numpy as np
import pytest

import halo_emu
import mask_bytes as MB
import mask_bytes_emu as E
from domain_decomp_b200 import capi as real

WIDE = 16384
WIDTHS = [WIDE, WIDE - 1, WIDE + 1, WIDE - 4, WIDE + 4, WIDE + 15, WIDE - 15, 1, 3, 4, 7, 12, 15]


@pytest.fixture(scope="module")
def capi(oracle):
    return halo_emu.emu_capi(oracle)


@pytest.fixture(scope="module")
def handle(capi):
    h = capi.Handle(0)
    yield h
    h.close()


def set_u8_host(b):
    return lambda h: h.set_mask_u8_host(b)


def set_u8_device(b, offset):
    """b's rows at `offset` bytes into an allocation that ends exactly at the last row ("device" memory of the
    emulated runtime is host memory)"""
    buf = np.zeros(offset + b.size, dtype=np.uint8)
    buf[offset:] = b.reshape(-1)

    def set_(h):
        h._keep = buf
        ny, nx = b.shape
        h.set_mask_u8_device(buf.ctypes.data + offset, nx, ny)
    return set_


@pytest.mark.parametrize("nx", WIDTHS)
def test_widths_and_byte_values(handle, capi, nx):
    """NX at 16k and 16k +- 1..15 (both scan paths, the clamped re-read of the last group) and below 16; row counts
    with and without a tail of fewer than 32 rows; ocean bytes 1 / 2 / 0x7F / 0x80 / 0xFF"""
    rng = np.random.default_rng(nx)
    for ny in ((9, 40) if nx >= WIDE - 15 else (5, 33, 100)):
        m = capi.generate_mask_host(nx, ny, nx + ny, 0.45)
        b = MB.byte_mask(m, rng)
        P = int(rng.integers(2, 12)) if nx * ny > 1 else 1
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        a, u = MB.run_pair(handle, m, set_u8_host(b), P, px, py)
        MB.assert_same(a, u, (nx, ny, P))


@pytest.mark.parametrize("rpc", [8, 16, 64])
def test_row_chunks_and_tail(capi, oracle, rpc):
    """chunks of 8 rows (no 32-row iteration), 16, and 64 rows with the fine-grained tail of smaller chunks (rows >= 4
    chunks); row counts that end on and off a 32-row boundary.  One rank through the multi-rank harness, which takes
    the rows per CTA as an argument (the C ABI picks them by occupancy: 8 on the emulated runtime)."""
    rng = np.random.default_rng(rpc)
    for nx, ny in ((256, 300), (260, 257), (1024, 96), (99, 130)):
        m = capi.generate_mask_host(nx, ny, ny, 0.5)
        _same_as_int32(oracle, MB.byte_mask(m, rng), 16, True, False, 1, scan_rpc=rpc)


@pytest.mark.parametrize("offset", [1, 2, 3, 5, 8, 15])
def test_unaligned_device_pointer(handle, capi, offset):
    """a borrowed pointer 1..15 bytes past an aligned address: the byte-by-byte path unless it is 4-byte aligned, and
    nothing read past the last row"""
    rng = np.random.default_rng(offset)
    for nx, ny in ((128, 70), (333, 41)):
        m = capi.generate_mask_host(nx, ny, offset, 0.4)
        b = MB.byte_mask(m, rng)
        a, u = MB.run_pair(handle, m, set_u8_device(b, offset), 10, False, True)
        MB.assert_same(a, u, (offset, nx, ny))


def test_bool_array_and_type_switch(handle, capi):
    """int32 -> u8 -> int32 -> bool on one handle: each decomposition equals the int32 one"""
    m = capi.generate_mask_host(300, 200, 4, 0.45)
    handle.set_mask_host(m)
    handle.partition(24, True, True)
    handle.partition(24, True, True)  # (the first call on a new shape also clears the buffers: one launch more)
    ref = MB.snapshot(handle)
    for set_ in (lambda h: h.set_mask_u8_host((m > 0).astype(np.uint8) * np.uint8(0xFF)), lambda h: h.set_mask_host(m),
                 lambda h: h.set_mask_u8_host(np.ascontiguousarray(m > 0))):
        set_(handle)
        handle.partition(24, True, True)
        MB.assert_same(ref, MB.snapshot(handle))


def test_byte_rule_is_unsigned(handle, capi):
    """0x80 and 0xFF are ocean under the byte rule (as int32 -128 / -1 they would be land): the decomposition is the
    one of the int32 mask (bytes != 0)"""
    rng = np.random.default_rng(5)
    b = rng.choice(np.array([0, 0x80, 0xFF], np.uint8), size=(60, 80), p=[0.5, 0.25, 0.25])
    a, u = MB.run_pair(handle, (b != 0).astype(np.int32), set_u8_host(b), 9, True, True)
    MB.assert_same(a, u)
    assert u["stats"]["n_ocean"] == int((b != 0).sum())


def test_async_and_plan_mismatch(capi, oracle):
    """a fresh handle per mask: the u8 scan runs the guessed plan, notices the mismatch of a band mask and runs
    again, also when DDC_ASYNC only enqueues; everything equals a fresh int32 handle's run"""
    for shape, band in (((96, 200), (slice(None), slice(90, 101))), ((200, 96), (slice(90, 101), slice(None)))):
        m = np.zeros(shape, dtype=np.int32)
        m[band] = 1
        for P in (8, 13):
            for flags in (real.WANT_PID | real.WANT_NEIGHBOURS, real.WANT_PID | real.WANT_NEIGHBOURS | real.ASYNC):
                got = []
                for u8 in (False, True):
                    h = capi.Handle(0)
                    try:
                        if u8:
                            h.set_mask_u8_host((m * 0xFF).astype(np.uint8))
                        else:
                            h.set_mask_host(m)
                        for _ in range(3):
                            h.partition(P, True, True, flags=flags)
                        got.append(MB.snapshot(h))
                    finally:
                        h.close()
                MB.assert_same(got[0], got[1], (shape, P, flags))
                o = oracle.partition(m, P, True, True)
                assert got[1]["boxes"].tolist() == o.boxes.tolist() and np.array_equal(got[1]["pid"], o.pid)


def test_status_codes(handle, capi):
    L = handle.L
    b = np.ones((30, 40), dtype=np.uint8)
    for fn in (L.ddc_set_mask_u8_host, L.ddc_set_mask_u8_device):
        assert fn(handle.h, None, 40, 30, 0, 30) == -1 and b"null mask" in L.ddc_last_error(handle.h)
        assert fn(handle.h, b.ctypes.data, 40, 30, 0, 29) == -1 and b"must hold rows" in L.ddc_last_error(handle.h)
        assert fn(handle.h, b.ctypes.data, 0, 30, 0, 30) == -1
        assert fn(handle.h, b.ctypes.data, 65536, 65536, 0, 65536) == -1  # more cells than an int can index
        assert fn(None, b.ctypes.data, 40, 30, 0, 30) == -1
    # a rank with a zero-row block may pass NULL
    h2 = capi.Handle(0, 1, 2)
    try:
        assert L.ddc_set_mask_u8_host(h2.h, None, 40, 1, 1, 0) == 0
        assert L.ddc_set_mask_u8_device(h2.h, None, 40, 1, 1, 0) == 0
        assert L.ddc_set_mask_u8_host(h2.h, None, 40, 1, 0, 1) == -1
    finally:
        h2.close()
    with pytest.raises(real.DdcError):
        handle.set_mask_u8_host(np.ones((3, 4), dtype=np.uint8), ny=5)


# ---- several emulated ranks ---------------------------------------------------------------------------------------

def _same_as_int32(oracle, b, P, px, py, ranks, **kw):
    d, info = E.partition(oracle, b, P, px, py, ranks=ranks, **kw)
    o, o_info = oracle.emu_partition((b != 0).astype(np.int32), P, px, py, ranks=ranks,
                                **{k: v for k, v in kw.items() if k not in ("u8_ranks", "offset")})
    ctx = (b.shape, P, ranks, kw)
    assert d.boxes.tolist() == o.boxes.tolist(), ctx
    assert np.array_equal(d.pid, o.pid), ctx
    assert (d.changes, d.median_iters) == (o.changes, o.median_iters), ctx
    assert info == o_info, ctx  # n_ocean, strips, x / y levels, load min / max
    for per in range(2):
        for e in range(4):
            for x, y in ((d.nbr.counts, o.nbr.counts), (d.nbr.ids, o.nbr.ids), (d.nbr.halos, o.nbr.halos),
                         (d.nbr.starts, o.nbr.starts)):
                assert x[per][e].tolist() == y[per][e].tolist(), (ctx, per, e)
    h = oracle.partition((b != 0).astype(np.int32), P, px, py, use_hist=True)
    assert d.boxes.tolist() == h.boxes.tolist() and np.array_equal(d.pid, h.pid), ctx
    return d


@pytest.mark.parametrize("ranks", [2, 3, 5])
def test_ranks(oracle, capi, ranks):
    rng = np.random.default_rng(ranks)
    cases = [(130, 47, 10, True, False), (64, 90, 12, False, True), (67, 31, 7, True, True),
             (200, 3, 6, False, False)]  # ny < ranks: empty row blocks
    for nx, ny, P, px, py in cases:
        b = MB.byte_mask(capi.generate_mask_host(nx, ny, nx * ny, 0.45), rng)
        _same_as_int32(oracle, b, P, px, py, ranks, scan_rpc=int(rng.choice([8, 16, 64])))
        # mixed: every other rank scans int32, and the byte shards start off alignment
        _same_as_int32(oracle, b, P, px, py, ranks, u8_ranks=range(0, ranks, 2), offset=int(rng.integers(1, 16)))


@pytest.mark.parametrize("ranks", [2, 3])
def test_ranks_collectives_and_random_schedules(oracle, capi, ranks, monkeypatch):
    """the NCCL exchange layout (DDC_EMU_COLLECTIVES) and random block / thread schedules (DDC_EMU_SCHED_SEED)"""
    rng = np.random.default_rng(10 + ranks)
    b = MB.byte_mask(capi.generate_mask_host(150, 61, 3, 0.45), rng)
    monkeypatch.setenv("DDC_EMU_SCHED_SEED", str(ranks))
    _same_as_int32(oracle, b, 12, True, False, ranks, scan_rpc=16)
    monkeypatch.setenv("DDC_EMU_COLLECTIVES", "1")
    _same_as_int32(oracle, b, 12, True, False, ranks, u8_ranks=[1], scan_rpc=16)


def test_harness_scans_the_byte_mask(oracle):
    """the byte shards are what the byte ranks scan: a byte mask that differs from the int32 mask gives the byte
    mask's decomposition"""
    b = np.zeros((40, 64), np.uint8)
    b[:, :20] = 7
    L = E.lib()
    assert L.emu_set_byte_mask(b.reshape(-1), 64, 40, 2, 3, 0) == 0
    try:
        with E._harness(oracle):
            d, _ = oracle.emu_partition(np.ones((40, 64), np.int32), 4, ranks=2)
    finally:
        L.emu_set_byte_mask(b.reshape(-1), 64, 40, 1, 0, 0)
    o = oracle.partition((b != 0).astype(np.int32), 4, use_hist=True)
    assert d.boxes.tolist() == o.boxes.tolist() and np.array_equal(d.pid, o.pid)


def test_byte_scan_is_clean_under_address_sanitizer(oracle):
    """the byte shards end exactly at their last row: no load reaches past a row's nx bytes, at widths that are not
    multiples of 16, aligned and not"""
    import test_kernels_asan as A
    oracle.build()
    out = A.run_worker(worker="mask_bytes_asan_worker.py")
    assert "ERROR: AddressSanitizer" not in out.stderr and "runtime error:" not in out.stderr, out.stderr[-4000:]
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "MASK BYTES ASAN RUN OK" in out.stdout
