"""The cut kernels past their level tables on the device: more than 1024 strips (K2 walks), more than 1024 parts in a
strip (K4 walks), more strips than K4 has blocks, and the global-memory prefix paths of both, bit for bit against the
histogram oracle (tests/many_leaves.py lists the cases and the branches each one reaches)."""
import pytest

import many_leaves as ML
import test_gpu_parity as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("no CUDA device: the -m gpu tests need one (the product has no CPU fallback)")
    from domain_decomp_b200 import capi
    capi.load()
    return capi


def check(h, oracle, case, ctx):
    mask, o, loads = ML.expected(oracle, case)
    g = T.run_gpu(h, mask, case.P, case.px, case.py)
    T.assert_same(g, o, ctx)
    assert g["loads"].tolist() == loads.tolist(), ctx
    st = g["stats"]
    assert (st["load_min"], st["load_max"]) == (int(loads.min()), int(loads.max())), ctx
    ML.assert_reaches(case, st["nstrips"], st["n_xlev"], st["n_ylev"], g["boxes"])


@pytest.mark.parametrize("case", ML.GPU_CASES, ids=ML.case_id)
def test_each_case_twice_on_a_fresh_handle(capi, oracle, case):
    """the first call runs with the plan the host guessed from the extents (and again if the real one differs), the
    second with the plan the first one settled"""
    h = capi.Handle(0)
    try:
        for k in range(2):
            check(h, oracle, case, (ML.case_id(case), k))
    finally:
        h.close()


def test_all_cases_on_one_handle(capi, oracle):
    """one handle through every case, forwards and back: the strip capacity, the row -> part table, the row-count
    buffers, the global prefix sums of K4 and the shared-memory variant of each cut kernel grow and shrink between
    calls"""
    h = capi.Handle(0)
    try:
        for k, case in enumerate(ML.GPU_CASES + ML.GPU_CASES[::-1]):
            check(h, oracle, case, (ML.case_id(case), k))
    finally:
        h.close()
