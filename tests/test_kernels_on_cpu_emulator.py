"""The product's REAL kernels on a machine without a GPU.

oracle/emu/ compiles domain_decomp_b200/csrc/ddc_kernels.cuh as host C++ (-DDDC_HOST_EMU) and runs it on an
emulation of the CUDA execution model: every thread of a block is a fiber, __syncthreads and the warp
collectives are rendezvous between fibers, blocks run one after the other; emu_pipeline.cpp launches the
kernels in the order and with the grids / buffers of ddc_api.cu, for G emulated ranks that exchange their
histograms through each other's slots exactly as over NVLink.  Whole decompositions of small masks are
compared with the oracle, bit for bit: boxes, pid, the eight neighbour tables, `changes`, the median
iteration count.  (The GPU suite checks the same on the device up to 10^9 cells; this suite keeps the kernel
LOGIC under test in every CPU-only run -- every kernel, both exchange layouts, every variant of the strip
row-count kernel, the global-memory prefix paths -- and says nothing about speed.)"""
import numpy as np
import pytest

from conftest import golden_mask


def assert_same(d, o, ctx=""):
    assert d.boxes.tolist() == o.boxes.tolist(), ctx
    assert np.array_equal(d.pid, o.pid), ctx
    assert d.changes == o.changes, ctx
    assert d.median_iters == o.median_iters, ctx
    for per in range(2):
        for e in range(4):
            assert d.nbr.counts[per][e].tolist() == o.nbr.counts[per][e].tolist(), (ctx, per, e)
            assert d.nbr.ids[per][e].tolist() == o.nbr.ids[per][e].tolist(), (ctx, per, e)
            assert d.nbr.halos[per][e].tolist() == o.nbr.halos[per][e].tolist(), (ctx, per, e)
            assert d.nbr.starts[per][e].tolist() == o.nbr.starts[per][e].tolist(), (ctx, per, e)


def test_box_known_answers(goldens, oracle):
    """the reference's bounding-box known-answer tests (test_zoltan_partitioner_{0,1,2}.cpp) through the kernels"""
    for kat in goldens["box_kats"]:
        d, _ = oracle.emu_partition(golden_mask(goldens, kat["input"]), kat["P"])
        assert d.boxes.tolist() == kat["boxes"], kat["cite"]


@pytest.mark.parametrize("case", ["test_1", "test_2", "test_1_px", "test_1_py", "test_1_px_py"])
def test_integration_goldens(goldens, oracle, case):
    G = goldens["integration"][case]
    mask = golden_mask(goldens, G["input"])
    md = G["metadata"]
    for ranks in (1, 2):
        d, _ = oracle.emu_partition(mask, G["P"], bool(G["px"]), bool(G["py"]), ranks=ranks)
        assert d.pid.ravel().tolist() == list(G["pid"])
        assert d.boxes[:, 0].tolist() == md["domain_x"] and d.boxes[:, 2].tolist() == md["domain_extent_x"]
        assert d.boxes[:, 1].tolist() == md["domain_y"] and d.boxes[:, 3].tolist() == md["domain_extent_y"]
        for per, sfx in ((0, ""), (1, "_periodic")):
            for e, name in enumerate(("left", "right", "bottom", "top")):
                assert d.nbr.counts[per][e].tolist() == md[name + "_neighbours" + sfx]
                assert d.nbr.ids[per][e].tolist() == md.get(name + "_neighbour_ids" + sfx, [])
                assert d.nbr.halos[per][e].tolist() == md.get(name + "_neighbour_halos" + sfx, [])
                assert d.nbr.starts[per][e].tolist() == md.get(name + "_neighbour_halo_starts" + sfx, [])


def test_rect3030(goldens, oracle):
    mask = golden_mask(goldens, "rect3030")
    for P in (2, 4):
        d, _ = oracle.emu_partition(mask, P)
        assert_same(d, oracle.partition(mask, P, use_hist=True), "rect3030 P=%d" % P)


def test_random_small_masks_one_rank(oracle):
    """ragged widths (the scalar load / store paths), empty rows and columns, P not a power of two, P > columns"""
    rng = np.random.default_rng(101)
    for i in range(14):
        nx, ny = int(rng.integers(1, 70)), int(rng.integers(1, 50))
        P = int(rng.integers(1, 20))
        mask = (rng.random((ny, nx)) >= rng.random() * 0.9).astype(np.int32) * int(rng.integers(1, 4))
        if i % 5 == 0:
            mask[:, : nx // 2] = 0
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        d, _ = oracle.emu_partition(mask, P, px, py)
        assert_same(d, oracle.partition(mask, P, px, py, use_hist=True), (nx, ny, P, px, py))


def test_nothing_moved_and_all_land(oracle):
    """`changes == 0`: the naive blocks are reported and the neighbour tables are rebuilt from them in K5"""
    for (n, P) in [(64, 4), (60, 6)]:
        m = np.ones((n, n), dtype=np.int32)
        d, _ = oracle.emu_partition(m, P, True, True)
        o = oracle.partition(m, P, True, True, use_hist=True)
        assert o.changes == 0
        assert_same(d, o, (n, P))
    m = np.zeros((12, 18), dtype=np.int32)
    d, _ = oracle.emu_partition(m, 6)
    assert_same(d, oracle.partition(m, 6, use_hist=True), "all land")


@pytest.mark.parametrize("ranks", [2, 3, 5])
def test_row_sharded_ranks_exchange_through_their_slots(oracle, ranks):
    """G emulated ranks: column counts pushed by the last CTA of a column block (16-bit), strip row counts pushed as
    chunks, `changes` in the flag; a rank without rows (5 ranks, 4 rows) still pushes and signals"""
    from domain_decomp_b200 import capi
    cases = [(capi.generate_mask_host(130, 77, 7, 0.5), 12, True, False), (capi.generate_mask_host(64, 4, 2, 0.3), 8, False, False),
             (np.ones((24, 24), dtype=np.int32), 4, False, True)]
    for mask, P, px, py in cases:
        d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks)
        assert_same(d, oracle.partition(mask, P, px, py, use_hist=True), (mask.shape, P, ranks))


@pytest.mark.parametrize("strip_k", [1, 2, 4, 16])
def test_strip_row_count_kernel_variants(oracle, strip_k):
    """rows per warp 1 / 2 / 4, and the kernel for tables beyond shared memory (16)"""
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(300, 90, 11, 0.45)
    for ranks in (1, 2):
        d, _ = oracle.emu_partition(mask, 24, True, False, ranks=ranks, strip_k=strip_k)
        assert_same(d, oracle.partition(mask, 24, True, False, use_hist=True), (strip_k, ranks))


def test_cut_kernels_with_histograms_in_global_memory(oracle):
    """a shared-memory limit of a few KB forces K2 / K4 onto their global-memory prefix path (no bit map of
    non-empty bins: binary searches over the prefix sums), as for grids beyond ~55000 columns or rows"""
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(200, 150, 5, 0.5)
    for ranks in (1, 2):
        d, _ = oracle.emu_partition(mask, 16, False, True, ranks=ranks, smem_limit=2048)
        assert_same(d, oracle.partition(mask, 16, False, True, use_hist=True), ranks)


def test_scan_rows_per_cta(oracle):
    """the mask scan with 8 ... 128 rows per CTA (the host picks by occupancy): several staged flushes per CTA,
    a last CTA with fewer rows, more than one CTA per column block counting down to the push"""
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(140, 203, 9, 0.4)
    o = oracle.partition(mask, 10, use_hist=True)
    for rpc in (8, 24, 128):
        d, _ = oracle.emu_partition(mask, 10, ranks=2, scan_rpc=rpc)
        assert_same(d, o, rpc)


@pytest.mark.parametrize("nx,ny,P,ranks,kw", [(9000, 6, 5, 2, {}), (33000, 3, 4, 2, {}), (33000, 3, 4, 1, {}),
                                              (5000, 9, 6, 3, {"smem_limit": 2048}), (70, 9000, 6, 2, {}),
                                              (40, 33000, 5, 2, {})])
def test_histograms_of_several_sub_tiles_and_tiles(oracle, nx, ny, P, ranks, kw):
    """the prefix scan of the cut kernels: a thread owns 4 bins in each of 8 sub-tiles of 4096, a tile is 32768
    bins -- histograms of 5000 ... 33000 bins reach the later sub-tiles and the second tile, with the slots of
    several ranks summed in the loader"""
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(nx, ny, 5, 0.4)
    d, _ = oracle.emu_partition(mask, P, True, False, ranks=ranks, **kw)
    assert_same(d, oracle.partition(mask, P, True, False, use_hist=True), (nx, ny, P, ranks))


def test_column_counts_travel_as_data_and_flag_words(oracle):
    """exchange step 1 (ll_word): two 16-bit counts per word while every rank holds < 65536 rows, one 32-bit count per
    word beyond that; several column blocks (every one pushes its own words), columns that are not a multiple of 4"""
    from domain_decomp_b200 import capi
    for nx, ny, P, ranks in ((12, 131080, 3, 2), (2501, 40, 6, 3), (1030, 17, 4, 2)):
        mask = capi.generate_mask_host(nx, ny, 5, 0.4)
        d, _ = oracle.emu_partition(mask, P, True, False, ranks=ranks)
        assert_same(d, oracle.partition(mask, P, True, False, use_hist=True), (nx, ny, P, ranks))


def test_row_counts_with_one_flag_per_rank_or_per_block(oracle):
    """exchange step 2: on 2 ranks every block of the row-count kernel raises its own flag and the y-cut kernel polls
    ranks x blocks flags, with more row blocks than one y-cut block has threads to poll them in one go; on 3 ranks
    the kernel's last block raises one flag per rank (block counter)"""
    from domain_decomp_b200 import capi
    for nx, ny, P, ranks in ((70, 9000, 6, 2), (150, 301, 12, 3)):
        mask = capi.generate_mask_host(nx, ny, 11, 0.4)
        o = oracle.partition(mask, P, False, True, use_hist=True)
        for strip_k in (0, 1):
            d, _ = oracle.emu_partition(mask, P, False, True, ranks=ranks, strip_k=strip_k)
            assert_same(d, o, (nx, ny, P, ranks, strip_k))


def test_random_multi_rank_cases(oracle, monkeypatch):
    """random shapes, part counts, periodic flags, 2-8 ranks (ragged and empty shards included), random block / thread
    schedules: boxes, pid, neighbour tables and `changes` equal the oracle's"""
    import random
    from domain_decomp_b200 import capi
    rng = random.Random(20261018)
    for _ in range(40):
        nx, ny = rng.choice([5, 33, 130, 1030, 2500]), rng.choice([7, 40, 203, 900])
        P, ranks = rng.randint(2, 24), rng.choice([2, 3, 4, 5, 8])
        px, py = rng.random() < .5, rng.random() < .5
        monkeypatch.setenv("DDC_EMU_SCHED_SEED", str(rng.randint(1, 2 ** 40)))
        mask = capi.generate_mask_host(nx, ny, rng.randint(1, 99), rng.choice([0.2, 0.5, 0.8]))
        d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks, scan_rpc=rng.choice([8, 16, 64]))
        assert_same(d, oracle.partition(mask, P, px, py, use_hist=True), (nx, ny, P, ranks, px, py))
    monkeypatch.delenv("DDC_EMU_SCHED_SEED")


def test_results_do_not_depend_on_the_schedule(oracle, monkeypatch):
    """the emulation can run the blocks of a grid in a random order and the threads of a block in a new random order
    every scheduling round (DDC_EMU_SCHED_SEED): a missing barrier, an assumption about block order or about
    which CTA of a column block finishes last would make results differ between seeds"""
    from domain_decomp_b200 import capi
    cases = [(capi.generate_mask_host(130, 77, 7, 0.5), 12, True, False, 2), (capi.generate_mask_host(67, 90, 3, 0.4), 9, False, True, 3),
             (np.ones((24, 24), dtype=np.int32), 4, True, True, 1)]
    for mask, P, px, py, ranks in cases:
        o = oracle.partition(mask, P, px, py, use_hist=True)
        for seed in (1, 99991, 2 ** 40 + 7):
            monkeypatch.setenv("DDC_EMU_SCHED_SEED", str(seed))
            d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks, scan_rpc=16)
            assert_same(d, o, (mask.shape, P, ranks, seed))
    monkeypatch.delenv("DDC_EMU_SCHED_SEED")


def test_more_parts_than_cells_per_row(oracle):
    """tiny grids cut into many (mostly empty) parts: zero-width strips, zero-height parts, neighbour lists far
    longer than the 3 P + 64 entries reserved per list, so that the fill pass runs again with the exact capacity"""
    longest = 0
    for seed, ranks in ((9, 3), (41, 1)):
        rng = np.random.default_rng(seed)  # (seeds picked because they do overflow the reserved capacity)
        for (nx, ny, P, px, py) in [(11, 11, 36, False, False), (5, 6, 23, True, False), (4, 4, 16, True, True)]:
            land = 0.5 + 0.4 * rng.random()
            mask = (rng.random((ny, nx)) >= land).astype(np.int32)
            d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks)
            o = oracle.partition(mask, P, px, py, use_hist=True)
            longest = max(longest, max(len(x) - (3 * P + 64) for per in range(2) for x in o.nbr.ids[per]))
            assert_same(d, o, (seed, nx, ny, P, ranks))
    assert longest > 0, "no case overflowed the reserved list capacity: the re-run path was not exercised"


def test_assumed_plan_mismatch_reruns_the_step(oracle):
    """the host sizes the launches after K2 for an ASSUMED number of x / y levels (those of a full-extent bounding
    box); when the ocean occupies a flat band the real plan has more x levels, K2 flags the mismatch, the later
    kernels do nothing and the step runs again with the real plan"""
    mask = np.zeros((64, 64), dtype=np.int32)
    mask[3:9, :] = 1
    mask[5, 10:20] = 0
    for ranks in (1, 2):
        d, info = oracle.emu_partition(mask, 16, False, False, ranks=ranks)
        assert (info["x_levels"], info["y_levels"]) == (4, 0)  # a 64 x 64 bounding box would give 2 and 2
        assert_same(d, oracle.partition(mask, 16, use_hist=True), ranks)


def test_rows_of_65536_cells_or_more(oracle):
    """NX >= 65536 with a y level: 32-bit strip row counts (16-byte stores of 4 counts), three prefix tiles in
    global memory for the column histogram, ragged width (66001: the scalar load / store paths of K1 and K6)"""
    from domain_decomp_b200 import capi
    for (nx, ny, P, kw) in [(66001, 530, 200, {"strip_k": 16}), (65600, 540, 256, {})][:1]:
        mask = capi.generate_mask_host(nx, ny, 5, 0.4)
        d, info = oracle.emu_partition(mask, P, True, False, **kw)
        assert info["x_levels"] == 7 and info["y_levels"] == 1
        assert_same(d, oracle.partition(mask, P, True, False, use_hist=True), (nx, ny, P))


@pytest.mark.parametrize("ranks", [1, 2, 3])
def test_back_to_back_steps_without_k_init(oracle, ranks, monkeypatch):
    """k_init is only launched for buffers that K2 (column counts, y-range pairs, scalars) and the scan's last CTA
    (its counters) have not left clean: four more decompositions are enqueued first, from the third step on
    without k_init, on both parities of the exchange slots"""
    from domain_decomp_b200 import capi
    monkeypatch.setenv("DDC_EMU_REPEAT", "4")
    for mask, P, px, py in [(capi.generate_mask_host(130, 77, 7, 0.5), 12, True, False), (np.ones((24, 24), dtype=np.int32), 4, False, True),
                            (capi.generate_mask_host(64, 64, 3, 0.97), 8, False, False)][:3 if ranks < 3 else 1]:
        d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks)
        assert_same(d, oracle.partition(mask, P, px, py, use_hist=True), (mask.shape, P, ranks))


@pytest.mark.parametrize("P,ranks", [(77, 1), (100, 2), (129, 1), (255, 1)])
def test_part_counts_that_are_not_powers_of_two(oracle, P, ranks):
    """ceil(n/2) | floor(n/2) splits at every level: leaves at different depths, targets that are not W / 2 (the FP64
    target path of the median), strips with different numbers of parts"""
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(600, 500, 13, 0.5)
    d, _ = oracle.emu_partition(mask, P, True, True, ranks=ranks)
    assert_same(d, oracle.partition(mask, P, True, True, use_hist=True), (P, ranks))


@pytest.mark.parametrize("ranks", [2, 3])
def test_row_sharded_ranks_with_collectives(oracle, ranks, monkeypatch):
    """the NCCL fallback of ddc_api.cu (decompositions that exceed the exported peer buffers): an all-reduce of the
    column counts + y-range pairs, an all-gather of the strip row counts ([G][rank block], which K4 indexes by
    rank = y / Rmax) and a MAX of `changes` BETWEEN the kernels, emulated by host loops; the kernels then take
    their single-buffer paths (pc.n == 1, pr.n == 1) with G > 1.  Twice in a row: the second step without k_init"""
    from domain_decomp_b200 import capi
    monkeypatch.setenv("DDC_EMU_COLLECTIVES", "1")
    monkeypatch.setenv("DDC_EMU_REPEAT", "2")
    for mask, P, px, py in [(capi.generate_mask_host(130, 77, 7, 0.5), 12, True, False),
                            (capi.generate_mask_host(64, 4, 2, 0.3), 8, False, False), (np.ones((24, 24), dtype=np.int32), 4, False, True)]:
        d, _ = oracle.emu_partition(mask, P, px, py, ranks=ranks)
        assert_same(d, oracle.partition(mask, P, px, py, use_hist=True), (mask.shape, P, ranks))
