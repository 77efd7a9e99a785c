"""The cut kernels past their level tables on a machine without a GPU (tests/many_leaves.py: the cases and the branches
each one reaches), bit for bit against the histogram oracle:
  * one rank through the library's own C ABI on the emulated runtime (oracle/libddc_cuda_emu.so), one handle for the
    whole module, every case twice in a row;
  * 2 and 3 row-sharded ranks through oracle.emu_partition, one of them with random block and thread schedules.
The emulation runs every thread of a block as a fiber, so K4 costs it milliseconds per strip with y levels and rank.
The band cases with thousands of such strips therefore run here with fewer parts (4500 instead of 8192: the same
4096 strips, K2 walks on its global-memory prefix path, K4 loops over ~14 strips per block) and the
more-strips-than-columns case at 1100 x 2 -> 2200; the GPU suite runs the full part counts."""
import pytest

import halo_emu
import many_leaves as ML
import test_gpu_parity as T
import test_kernels_on_cpu_emulator as K

BAND = ML.Case(65536, 32, 4500, 7, 0.4, True, True, {"k2_walk", "k2_global", "k4_multi", "rows32"})
SPARSE = ML.Case(1100, 2, 2200, 5, 0.3, False, True, {"k2_walk", "zero_width", "zero_height", "k4_multi"})
TALL = ML.GPU_CASES[4]  # 24 x 40000 -> 2049: a walking strip and a strip cut level by level in one K4 launch

# in an order that makes the strip capacity and the buffers sized by it grow and shrink from one case to the next
ONE_RANK = [TALL, BAND, ML.GPU_CASES[9], ML.GPU_CASES[5], ML.GPU_CASES[1], SPARSE, ML.GPU_CASES[0]]


@pytest.fixture(scope="module")
def handle(oracle):
    h = halo_emu.emu_capi(oracle).Handle(0)
    yield h
    h.close()


@pytest.mark.parametrize("case", ONE_RANK, ids=ML.case_id)
def test_one_rank_through_the_c_abi(handle, oracle, case):
    mask, o, loads = ML.expected(oracle, case)
    for k in range(2):  # the guessed plan (and a re-run if it was wrong), then the settled one
        ctx = (ML.case_id(case), k)
        g = T.run_gpu(handle, mask, case.P, case.px, case.py)
        T.assert_same(g, o, ctx)
        assert g["loads"].tolist() == loads.tolist(), ctx
        st = g["stats"]
        assert (st["load_min"], st["load_max"]) == (int(loads.min()), int(loads.max())), ctx
        ML.assert_reaches(case, st["nstrips"], st["n_xlev"], st["n_ylev"], g["boxes"])


@pytest.mark.parametrize("case,ranks,seed", [(BAND, 2, 0), (TALL, 2, 0), (TALL, 3, 20261021), (SPARSE, 3, 0)],
                         ids=lambda v: ML.case_id(v) if isinstance(v, ML.Case) else str(v))
def test_row_sharded_ranks(oracle, monkeypatch, case, ranks, seed):
    """the ranks exchange column and strip row counts through each other's slots; with a seed, blocks and threads run
    in a random order, which checks the barrier between K4's walk writing a strip's boxes and the search over them
    that fills the row -> part table"""
    if seed:
        monkeypatch.setenv("DDC_EMU_SCHED_SEED", str(seed))
    mask, o, loads = ML.expected(oracle, case)
    d, info = oracle.emu_partition(mask, case.P, case.px, case.py, ranks=ranks, nbr_cap=max(1, ML.list_total(o)))
    ctx = (ML.case_id(case), ranks)
    K.assert_same(d, o, ctx)
    assert (info["load_min"], info["load_max"]) == (int(loads.min()), int(loads.max())), ctx
    ML.assert_reaches(case, info["strips"], info["x_levels"], info["y_levels"], d.boxes)
