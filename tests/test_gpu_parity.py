"""GPU parity: the CUDA path, called through the C ABI, against the CPU oracle and the goldens.

Bit-exact everywhere (integer / index work): boxes, pid, neighbour ids, halo sizes, halo starts.
"""
import numpy as np
import pytest

from conftest import golden_mask

pytestmark = pytest.mark.gpu

EDGES = ("left", "right", "bottom", "top")


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


def run_gpu(handle, mask, P, px=False, py=False):
    handle.set_mask_host(np.ascontiguousarray(mask, dtype=np.int32))
    handle.partition(P, px, py)
    out = {
        "boxes": handle.boxes(),
        "pid": handle.pid_host(),
        "stats": handle.stats(),
        "loads": handle.part_loads(),
        "counts": [[handle.neighbour_counts(e, per) for e in range(4)] for per in range(2)],
        "nbr": [[handle.neighbours(e, per) for e in range(4)] for per in range(2)],
    }
    return out


def assert_same(gpu, orc, ctx=""):
    assert gpu["boxes"].tolist() == orc.boxes.tolist(), ctx
    assert np.array_equal(gpu["pid"], orc.pid), ctx
    assert gpu["stats"]["changes"] == orc.changes, ctx
    assert gpu["stats"]["median_iters"] == orc.median_iters, ctx
    for per in range(2):
        for e in range(4):
            assert gpu["counts"][per][e].tolist() == orc.nbr.counts[per][e].tolist(), (ctx, per, e)
            ids, halos, starts = gpu["nbr"][per][e]
            assert ids.tolist() == orc.nbr.ids[per][e].tolist(), (ctx, per, e)
            assert halos.tolist() == orc.nbr.halos[per][e].tolist(), (ctx, per, e)
            assert starts.tolist() == orc.nbr.starts[per][e].tolist(), (ctx, per, e)


def test_box_known_answers(goldens, handle):
    """test/test_zoltan_partitioner_{0,1,2}.cpp through the C ABI."""
    for kat in goldens["box_kats"]:
        mask = golden_mask(goldens, kat["input"])
        g = run_gpu(handle, mask, kat["P"])
        assert g["boxes"].tolist() == kat["boxes"], kat["cite"]


@pytest.mark.parametrize("case", ["test_1", "test_2", "test_1_px", "test_1_py", "test_1_px_py"])
def test_integration_goldens(goldens, handle, case):
    """test/integration-test.sh: pid, boxes and every neighbour table, 3 parts."""
    G = goldens["integration"][case]
    mask = golden_mask(goldens, G["input"])
    g = run_gpu(handle, mask, G["P"], bool(G["px"]), bool(G["py"]))
    md = G["metadata"]
    assert g["pid"].reshape(-1).tolist() == G["pid"]
    assert g["boxes"][:, 0].tolist() == md["domain_x"]
    assert g["boxes"][:, 1].tolist() == md["domain_y"]
    assert g["boxes"][:, 2].tolist() == md["domain_extent_x"]
    assert g["boxes"][:, 3].tolist() == md["domain_extent_y"]
    for per, sfx in ((0, ""), (1, "_periodic")):
        for e, name in enumerate(EDGES):
            assert g["counts"][per][e].tolist() == md["%s_neighbours%s" % (name, sfx)]
            ids, halos, starts = g["nbr"][per][e]
            dim = G["dims"][name[0].upper() + sfx]
            assert len(ids) == dim
            if dim:
                assert ids.tolist() == md["%s_neighbour_ids%s" % (name, sfx)]
                assert halos.tolist() == md["%s_neighbour_halos%s" % (name, sfx)]
                assert starts.tolist() == md["%s_neighbour_halo_starts%s" % (name, sfx)]


def test_rect3030(goldens, handle, oracle):
    mask = golden_mask(goldens, "rect3030")
    for P in (2, 4):
        assert_same(run_gpu(handle, mask, P), oracle.partition(mask, P), "rect3030 P=%d" % P)


@pytest.mark.parametrize("P", [2, 4])
def test_rect3030_equals_the_reference_pictures(goldens, handle, P):
    """the GPU's pid map against the part map read off the reference's own img/partition_{2,4}.png (not via the
    oracle): see tests/test_oracle_golden.py::test_rect3030_equals_the_reference_pictures"""
    from test_oracle_golden import png_part_map
    want = png_part_map(P)
    pid = run_gpu(handle, golden_mask(goldens, "rect3030"), P)["pid"]
    trusted = want > -2
    assert int(trusted.sum()) >= 820 and np.array_equal(pid[trusted], want[trusted])


def test_readme_sample_balance(goldens, handle):
    """README.md:165-192 of the reference: test_2 on 2 ranks -> 6 / 6 dots, imbalance 1.0"""
    g = run_gpu(handle, golden_mask(goldens, "test_2"), 2)
    loads = np.bincount(g["pid"][g["pid"] >= 0].ravel(), minlength=2)
    assert loads.tolist() == [6, 6]


def test_random_small_masks(handle, oracle):
    """ragged extents, empty rows/columns, all-land, all-ocean, P not a power of two, P > columns"""
    rng = np.random.default_rng(11)
    for it in range(400):
        NX = int(rng.integers(1, 70))
        NY = int(rng.integers(1, 70))
        dens = rng.choice([0.0, 0.02, 0.1, 0.3, 0.6, 0.9, 1.0])
        m = (rng.random((NY, NX)) < dens).astype(np.int32) * int(rng.integers(1, 5))
        if rng.random() < 0.3:
            m[:, rng.integers(0, NX)] = 0
        if rng.random() < 0.3:
            m[rng.integers(0, NY), :] = 0
        if rng.random() < 0.2:
            m[m == 0] = -int(rng.integers(0, 3))  # land is "<= 0"
        P = int(rng.integers(1, 24))
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        g = run_gpu(handle, m, P, px, py)
        o = oracle.partition(m, P, px, py, use_hist=bool(it & 1))
        assert_same(g, o, "it=%d NX=%d NY=%d P=%d dens=%s px=%d py=%d" % (it, NX, NY, P, dens, px, py))
        assert int(g["loads"].sum()) == int((m > 0).sum())
        assert g["loads"].tolist() == oracle.part_loads(o.pid, P).tolist()


@pytest.mark.parametrize("px,py", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_arctic25km_64_parts(capi, handle, oracle, px, py):
    """BASELINE config 2: 528 x 522 synthetic mask, 64 parts, periodic combinations."""
    m = capi.generate_mask_host(528, 522, seed=25, land_frac=0.45)
    assert_same(run_gpu(handle, m, 64, bool(px), bool(py)), oracle.partition(m, 64, bool(px), bool(py)),
                "C2 px=%d py=%d" % (px, py))


@pytest.mark.parametrize("nx,ny,P,land", [(1024, 768, 96, 0.45), (777, 1033, 37, 0.6), (2048, 2048, 256, 0.45),
                                          (4096, 128, 64, 0.3), (100, 3000, 50, 0.5),
                                          # 512 strips: the gather variant of the strip row counts
                                          (16384, 64, 2048, 0.3)])
def test_medium_masks(capi, handle, oracle, nx, ny, P, land):
    m = capi.generate_mask_host(nx, ny, seed=3, land_frac=land)
    assert_same(run_gpu(handle, m, P, True, False), oracle.partition(m, P, True, False, use_hist=True),
                "%dx%d P=%d" % (nx, ny, P))


def test_arctic3km_1024_parts(capi, handle, oracle):
    """BASELINE config 3: 4096 x 4096, 1024 parts (oracle: histogram formulation)."""
    m = capi.generate_mask_host(4096, 4096, seed=3, land_frac=0.45)
    assert_same(run_gpu(handle, m, 1024), oracle.partition(m, 1024, use_hist=True), "C3")


def test_device_generator_matches_host(capi, handle):
    import torch
    nx, ny = 528, 522
    d = torch.empty((ny, nx), dtype=torch.int32, device="cuda:0")
    handle.generate_mask_device(d.data_ptr(), nx, ny, seed=25, land_frac=0.45)
    handle.synchronize()
    torch.cuda.synchronize()
    assert np.array_equal(d.cpu().numpy(), capi.generate_mask_host(nx, ny, 25, 0.45))


def test_device_resident_mask_and_pid(capi, handle, oracle):
    """borrowed device pointers in, device pointer out (what the benchmark's `value` times)"""
    import torch
    nx, ny, P = 1024, 1024, 64
    m = capi.generate_mask_host(nx, ny, seed=5, land_frac=0.5)
    d = torch.from_numpy(m).to("cuda:0")
    handle.set_mask_device(d.data_ptr(), nx, ny)
    handle.partition(P, False, False)
    handle.synchronize()
    o = oracle.partition(m, P, use_hist=True)
    assert handle.boxes().tolist() == o.boxes.tolist()
    assert np.array_equal(handle.pid_host(), o.pid)


def test_neighbours_from_boxes_random(handle, oracle):
    """the K7 kernel on caller-supplied boxes (brute-force mode) vs the literal O(P^2) oracle"""
    rng = np.random.default_rng(5)
    for it in range(60):
        NX, NY = int(rng.integers(4, 60)), int(rng.integers(4, 60))
        # a random rectilinear tiling: random x cuts, then random y cuts per strip
        xs = sorted(set([0, NX] + rng.integers(0, NX + 1, size=rng.integers(0, 5)).tolist()))
        boxes = []
        for a, b in zip(xs[:-1], xs[1:]):
            ys = sorted(set([0, NY] + rng.integers(0, NY + 1, size=rng.integers(0, 5)).tolist()))
            for c, d in zip(ys[:-1], ys[1:]):
                boxes.append([a, c, b - a, d - c])
        boxes = np.asarray(boxes, dtype=np.int32)
        rng.shuffle(boxes)  # arbitrary order: no strip structure
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        handle.neighbours_from_boxes(boxes, NX, NY, px, py)
        o = oracle.neighbours(boxes, NX, NY, px, py)
        for per in range(2):
            for e in range(4):
                assert handle.neighbour_counts(e, per).tolist() == o.counts[per][e].tolist()
                ids, halos, starts = handle.neighbours(e, per)
                assert ids.tolist() == o.ids[per][e].tolist()
                assert halos.tolist() == o.halos[per][e].tolist()
                assert starts.tolist() == o.starts[per][e].tolist()


def test_repeatability_and_flags(capi, handle, oracle):
    """idempotence: same handle, same mask, repeated calls and reduced flag sets agree"""
    m = capi.generate_mask_host(640, 480, seed=9, land_frac=0.4)
    a = run_gpu(handle, m, 48, True, True)
    b = run_gpu(handle, m, 48, True, True)
    assert a["boxes"].tolist() == b["boxes"].tolist() and np.array_equal(a["pid"], b["pid"])
    handle.set_mask_host(m)
    handle.partition(48, True, True, flags=0)  # boxes only: no pid, no neighbours
    assert handle.boxes().tolist() == a["boxes"].tolist()
    assert handle.stats()["changes"] == a["stats"]["changes"]
    with pytest.raises(capi.DdcError):
        handle.pid_host()
    assert handle.neighbour_counts(0, 0).sum() == 0


def test_async_steps_and_plan_mismatch(capi, handle, oracle):
    """DDC_ASYNC only enqueues; the getters settle the step.  A mask whose dots sit in a narrow
    band has other x / y level counts than the full-extent guess the launches were sized for:
    the step must notice and run again with the real plan."""
    for shape, band in (((96, 200), (slice(None), slice(90, 101))), ((200, 96), (slice(90, 101), slice(None)))):
        m = np.zeros(shape, dtype=np.int32)
        m[band] = 1
        for P in (8, 13):
            o = oracle.partition(m, P, True, True)
            handle.set_mask_host(m)
            for _ in range(3):  # back-to-back enqueues, nobody looks in between
                handle.partition(P, True, True, flags=capi.WANT_PID | capi.WANT_NEIGHBOURS | capi.ASYNC)
            g = {
                "boxes": handle.boxes(), "pid": handle.pid_host(), "stats": handle.stats(),
                "counts": [[handle.neighbour_counts(e, per) for e in range(4)] for per in range(2)],
                "nbr": [[handle.neighbours(e, per) for e in range(4)] for per in range(2)],
            }
            assert_same(g, o, "band %s P=%d" % (shape, P))
            # and the synchronous call on the now-cached plan
            assert_same(run_gpu(handle, m, P, True, True), o, "band %s P=%d again" % (shape, P))


@pytest.mark.parametrize("n,P", [(64, 4), (96, 16), (60, 6)])
def test_nothing_moved_reports_naive_blocks(handle, oracle, n, P):
    """all ocean, RCB == the naive blocks: `changes == 0`, boxes AND neighbour tables are the
    naive blocks' (the speculative tables of the RCB boxes are rebuilt)"""
    m = np.ones((n, n), dtype=np.int32)
    for px, py in ((False, False), (True, True)):
        o = oracle.partition(m, P, px, py)
        assert_same(run_gpu(handle, m, P, px, py), o, "all ocean n=%d P=%d" % (n, P))


def strip_row_kernel(nx, ny, P, stats, ranks=1):
    """the strip row-count kernel ddc_api.cu launches for a decomposition, from its shape and settled plan: the
    streaming kernel with K rows per warp ("K4", "K2", "K1"), or "k_strip_rows" when even the K = 1 boundary table
    exceeds 48 KiB of shared memory; None without y levels.  K is 4 for shards of at least 32 x 4 x 148 rows, else 2,
    halved while the table of Scap = min(P, 2^x_levels) strips does not fit."""
    if stats["n_ylev"] == 0 or P == 1:
        return None
    ng, scap, rmax = (nx + 127) // 128, min(P, 1 << stats["n_xlev"]), -(-ny // ranks)
    assert stats["nstrips"] <= scap, (stats["nstrips"], scap)
    table = lambda k: 4 * ((ng + 1) + (scap + 1) + 8 * k * ((scap + 1) | 1))  # bytes (strip_scan_smem_words)
    k = 4 if rmax >= 32 * 4 * 148 else 2
    while k > 1 and table(k) > 48 * 1024:
        k //= 2
    return "K%d" % k if table(k) <= 48 * 1024 else "k_strip_rows"


# (nx, ny, P, land, seed, the strip row-count kernel the shape reaches)
STRIP_ROW_CASES = [(1024, 768, 96, 0.45, 4, "K2"), (777, 1033, 37, 0.6, 9, "K2"), (4096, 515, 64, 0.5, 2, "K2"),
                   (1500, 19000, 300, 0.45, 3, "K4"),  # >= 18944 rows
                   (20000, 40, 1200, 0.4, 7, "K1"),  # 1024 strips: the K = 2 table exceeds 48 KiB
                   (40000, 24, 2049, 0.4, 7, "k_strip_rows")]  # 2048 strips: so does the K = 1 table


@pytest.mark.parametrize("case", STRIP_ROW_CASES, ids=lambda c: "%dx%d-P%d-%s" % (c[0], c[1], c[2], c[5]))
def test_strip_row_kernel_variants(capi, oracle, case):
    """every variant of the strip row-count kernel (rows per warp 1 / 2 / 4, and the kernel for boundary tables beyond
    shared memory), reached through the shape of the decomposition"""
    nx, ny, P, land, seed, kernel = case
    h = capi.Handle(0)
    try:
        m = capi.generate_mask_host(nx, ny, seed, land)
        g = run_gpu(h, m, P, True, False)
        assert_same(g, oracle.partition(m, P, True, False, use_hist=True), case)
        assert strip_row_kernel(nx, ny, P, g["stats"]) == kernel, (case, g["stats"])
    finally:
        h.close()


def test_halo_exchange_consumes_the_neighbour_tables(capi, handle):
    """ddc_halo_exchange_f64 (the GPU analogue of examples/zoltan_comm.cpp:84-246 of the reference): every ghost cell
    facing a neighbour ends up with that neighbour's id -- expected values from the boxes alone (tests/halo_check.py);
    528 x 522 into 64 parts with both directions periodic, and a 2048 x 1536 coastline into 1000 parts"""
    import halo_check
    import torch
    for (nx, ny, P, land, seed, px, py) in ((528, 522, 64, 0.45, 25, True, True), (2048, 1536, 1000, 0.4, 5, True, False)):
        mask = capi.generate_mask_host(nx, ny, seed, land)
        handle.set_mask_host(mask)
        handle.partition(P, px, py)
        boxes = handle.boxes()
        assert (boxes[:, 2:] > 0).all()
        off = handle.halo_tile_offsets()
        for periodic in (False, True):
            tiles = torch.from_numpy(halo_check.initial_tiles(boxes, off)).cuda()
            handle.halo_exchange_f64(tiles.data_ptr(), periodic)
            handle.L.ddc_synchronize(handle.h)
            torch.cuda.synchronize()
            want = halo_check.expected_tiles(boxes, off, nx, ny, px, py, periodic)
            assert np.array_equal(tiles.cpu().numpy(), want), (nx, ny, P, periodic)


def test_two_handles_with_different_shared_memory_needs(capi, oracle):
    """the dynamic shared memory a cut kernel is opted in for is a property of the FUNCTION: a second handle with a
    small grid must not lower what a first handle with a large one relies on (round 2: 'invalid argument')"""
    big = capi.generate_mask_host(300, 30000, 9, 0.4)
    small = capi.generate_mask_host(64, 48, 2, 0.3)
    a, b = capi.Handle(0), capi.Handle(0)
    try:
        for h, m, P in ((a, big, 32), (b, small, 6), (a, big, 32), (b, small, 6), (a, big, 24)):
            assert_same(run_gpu(h, m, P), oracle.partition(m, P, use_hist=True), "P=%d" % P)
    finally:
        a.close()
        b.close()
