"""Pins the CPU oracle against every golden the reference ships for this path."""
import numpy as np
import pytest

from conftest import golden_mask

EDGES = ("left", "right", "bottom", "top")


def test_box_known_answers(goldens, oracle):
    """test/test_zoltan_partitioner_{0,1,2}.cpp: the box of every rank."""
    assert len(goldens["box_kats"]) == 8
    for kat in goldens["box_kats"]:
        mask = golden_mask(goldens, kat["input"])
        for use_hist in (False, True):
            d = oracle.partition(mask, kat["P"], use_hist=use_hist)
            assert d.boxes.tolist() == kat["boxes"], (kat["cite"], use_hist)


@pytest.mark.parametrize("case", ["test_1", "test_2", "test_1_px", "test_1_py", "test_1_px_py"])
@pytest.mark.parametrize("use_hist", [False, True])
def test_integration_goldens(goldens, oracle, case, use_hist):
    """test/integration-test.sh: pid map, boxes and all neighbour tables on 3 ranks."""
    G = goldens["integration"][case]
    mask = golden_mask(goldens, G["input"])
    d = oracle.partition(mask, G["P"], bool(G["px"]), bool(G["py"]), use_hist=use_hist)
    md = G["metadata"]
    assert d.pid.reshape(-1).tolist() == G["pid"]
    assert d.boxes[:, 0].tolist() == md["domain_x"]
    assert d.boxes[:, 1].tolist() == md["domain_y"]
    assert d.boxes[:, 2].tolist() == md["domain_extent_x"]
    assert d.boxes[:, 3].tolist() == md["domain_extent_y"]
    for per, sfx in ((0, ""), (1, "_periodic")):
        for e, name in enumerate(EDGES):
            assert d.nbr.counts[per][e].tolist() == md["%s_neighbours%s" % (name, sfx)]
            dim = G["dims"][name[0].upper() + sfx]
            assert len(d.nbr.ids[per][e]) == dim
            if dim:
                assert d.nbr.ids[per][e].tolist() == md["%s_neighbour_ids%s" % (name, sfx)]
                assert d.nbr.halos[per][e].tolist() == md["%s_neighbour_halos%s" % (name, sfx)]
                assert d.nbr.starts[per][e].tolist() == md["%s_neighbour_halo_starts%s" % (name, sfx)]


def test_naive_blocks_match_grid_kats(goldens, oracle):
    """test/test_grid_{0,1,2}.cpp: object counts of the naive decomposition."""
    for kat in goldens["grid_kats"]:
        inp = goldens["inputs"][kat["input"]]
        mask = golden_mask(goldens, kat["input"])
        x0, y0, ex, ey = oracle.naive_block(kat["P"], inp["nx"], inp["ny"], kat["rank"])
        assert ex * ey == kat["num_objects"], kat["cite"]
        assert int((mask[y0:y0 + ey, x0:x0 + ex] > 0).sum()) == kat["num_nonzero_objects"]


def test_find_factors(oracle):
    # Grid.cpp:18-35: largest EVEN i with i*i <= n dividing n, else 1-D
    assert oracle.find_factors(1) == [1, 1]
    assert oracle.find_factors(2) == [2, 1]
    assert oracle.find_factors(3) == [3, 1]
    assert oracle.find_factors(4) == [2, 2]
    assert oracle.find_factors(9) == [9, 1]
    assert oracle.find_factors(12) == [2, 6]
    assert oracle.find_factors(64) == [8, 8]
    assert oracle.find_factors(1024) == [32, 32]
    assert oracle.find_factors(16384) == [128, 128]


def test_domain_overlap_against_reference_build(oracle):
    """oracle/_ref is the reference's own DomainUtils.cpp compiled here; compare exhaustively.  Without it, against
    the stored answers of the same seeded cases (tests/reference_answers.py)."""
    from reference_answers import Answers
    ref = oracle.ref_lib()
    answers = Answers("test_oracle_golden::test_domain_overlap_against_reference_build", ref is not None)
    rng = np.random.default_rng(7)
    L = oracle.lib()
    got = []
    for _ in range(20000):
        a = rng.integers(-3, 12, size=4)
        b = rng.integers(-3, 12, size=4)
        ax1, ax2 = sorted(a[:2]); ay1, ay2 = sorted(a[2:])
        bx1, bx2 = sorted(b[:2]); by1, by2 = sorted(b[2:])
        for e in range(4):
            args = [int(v) for v in (ax1, ay1, ax2, ay2, bx1, by1, bx2, by2, e)]
            got.append(L.orc_domain_overlap(*args))
            if ref is not None:
                assert got[-1] == ref.ref_domain_overlap(*args)
    for i in range(0, len(got), 10000):  # one stored answer per 2500 rectangle pairs
        answers.check(got[i:i + 10000], i // 4)
    answers.finish()


def test_rect3030_two_and_four_parts(goldens, oracle):
    """BASELINE config 1 (no golden exists): dots == hist, cut positions as in img/partition_*.png."""
    mask = golden_mask(goldens, "rect3030")
    assert int((mask > 0).sum()) == 456
    for P in (2, 4):
        a = oracle.partition(mask, P)
        b = oracle.partition(mask, P, use_hist=True)
        assert a.boxes.tolist() == b.boxes.tolist()
        assert np.array_equal(a.pid, b.pid)
        assert a.changes == b.changes
        loads = oracle.part_loads(a.pid, P)
        assert loads.sum() == 456


def png_part_map(P):
    """the part map read off the reference's own picture of rect3030 into P parts (scripts/make_golden_png.py), in
    the decomposer's frame: want[y][x], -2 where the picture cannot be trusted (blended colours, clipped column)"""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rect3030_png_parts.json")) as f:
        G = json.load(f)
    v = np.asarray(G["partition_%d.png" % P]["value"])  # [picture row j][column i]
    part = np.rint(v).astype(int)
    part[np.abs(v - np.rint(v)) > 0.25] = -2
    part[:, 29] = -2  # clipped by the plot frame
    if P == 4 and G["swap_1_2_in_partition_4"]:  # the picture predates REMAP=0 numbering (SURVEY 2)
        one, two = part == 1, part == 2
        part[one], part[two] = 2, 1
    return part.T  # picture (j, i) = decomposer (x, y)


@pytest.mark.parametrize("P", [2, 4])
def test_rect3030_equals_the_reference_pictures(goldens, oracle, P):
    """a4 pinned on an irregular coastline: every cell of img/partition_{2,4}.png whose colour can be read carries the
    part the restatement gives it -- 861 / 825 of 900 cells; the rest are the clipped last column and cells
    whose colour is blended with the land (or the other part) next to them.  In the pictures' frame the cuts are x = 15.5 (2 parts) and
    y = 14.5 then x = 14.5 / 16.5 (4 parts): the direction count of RCB_SET_DIRECTIONS and the "all cuts of the first
    direction, then the second" order of the restatement (DESIGN.md 2)."""
    mask = golden_mask(goldens, "rect3030")
    want = png_part_map(P)
    for use_hist in (False, True):
        pid = oracle.partition(mask, P, use_hist=use_hist).pid
        trusted = want > -2
        assert int(trusted.sum()) >= 820  # 861 (2 parts) and 825 (4 parts) of 900 cells read cleanly
        assert np.array_equal(pid[trusted], want[trusted]), np.argwhere((pid != want) & trusted)[:10]
    boxes = oracle.partition(mask, P).boxes.tolist()
    assert boxes == ([[0, 0, 30, 16], [0, 16, 30, 14]] if P == 2 else
                     [[0, 0, 15, 15], [0, 15, 15, 15], [15, 0, 15, 17], [15, 17, 15, 13]])


def test_readme_sample_balance(goldens, oracle):
    """README.md:165-192 of the reference: test_2 on 2 ranks -- 12 dots, 6 on each part, imbalance 1.0"""
    mask = golden_mask(goldens, "test_2")
    o = oracle.partition(mask, 2)
    loads = oracle.part_loads(o.pid, 2)
    assert int((mask > 0).sum()) == 12 and loads.tolist() == [6, 6]
    assert loads.max() / loads.mean() == 1.0
