"""Decompositions past the level tables of the cut kernels, shared by tests/test_gpu_many_leaves.py and
tests/test_many_leaves_on_cpu_emulator.py.

K2 (x cuts) and K4 (y cuts) split a set level by level, one thread per set, while a histogram has at most LEVEL_NODES
(1024) leaves; with more, every leaf's thread walks its own path down the tree (rcb_walk).  K4 runs
min(strips, 2 * 148) blocks, and each block loops over the strips s = blockIdx.x, blockIdx.x + gridDim.x, ...
Elongated domains reach those paths with ordinary part counts: a zonal band 65536 x 32 into 8192 parts has 4096
strips.  Every case states the branches it is there for, and `reached` derives them from what the library reports
(strip count, x / y levels) and from the boxes, so that a change to the assumed plan or to the mask generator cannot
move a case off its branch without a test failing."""
import collections

LEVEL_NODES = 1024  # ddc_kernels.cuh
YCUT_BLOCKS = 148 * 2  # the y-cut grid: min(strips, 2 x the SMs of a B200) blocks (ddc_api.cu)
SMEM_OPTIN = 232448  # bytes of dynamic shared memory a B200 block may opt in to
CUT_STATIC = 1056 + 64  # what the cut kernels hold statically, plus the library's margin

Case = collections.namedtuple("Case", "nx ny P seed land px py reaches")


def case_id(c):
    return "%dx%d-P%d" % (c.nx, c.ny, c.P)


# Branch names (see `reached`):
#   k2_levels_full  1024 strips: K2's level table at its limit      k2_walk   more than 1024 strips: K2 walks
#   k2_global       the column histogram does not fit shared memory: K2's prefix sums and medians in global memory
#   no_y_levels     K2 cuts every part: k_paint_strips paints the column -> strip table, K4 does not run
#   k4_levels_full  a strip of exactly 1024 leaves: K4's level table at its limit
#   k4_walk         a strip of more than 1024 leaves: K4 walks and reads its boxes back for the row -> part table
#   k4_both         one K4 launch with a walking strip and a strip cut level by level
#   k4_global       the row histogram does not fit shared memory: K4's prefix sums in global memory (y_smem == 0)
#   k4_multi        more strips with y levels than K4 has blocks: blocks loop over several strips
#   rows16 / rows32 strip row counts of 16 / 32 bits (rows of fewer / at least 65536 cells)
#   zero_width      zero-width strips (more strips than the ocean's columns): their parts have zero width
#   zero_height     parts of zero height
GPU_CASES = [
    Case(40000, 24, 1024, 7, 0.4, False, False, {"k2_levels_full", "no_y_levels"}),
    Case(40000, 24, 1025, 7, 0.4, True, False, {"k2_walk", "no_y_levels"}),
    Case(24, 40000, 1024, 7, 0.4, False, True, {"k4_levels_full"}),
    Case(24, 40000, 1025, 7, 0.4, True, True, {"k4_walk"}),
    Case(24, 40000, 2049, 7, 0.4, False, False, {"k4_walk", "k4_levels_full", "k4_both"}),
    Case(24, 60000, 2048, 7, 0.4, True, False, {"k4_walk", "k4_global"}),
    Case(65536, 32, 8192, 7, 0.4, False, True, {"k2_walk", "k2_global", "k4_multi", "rows32"}),
    Case(60000, 24, 8192, 7, 0.4, True, True, {"k2_walk", "k2_global", "k4_multi", "rows16"}),
    Case(32768, 64, 4096, 7, 0.4, False, False, {"k2_levels_full", "k4_multi", "rows16"}),
    Case(20000, 40, 1200, 7, 0.4, True, False, {"k2_levels_full", "k4_multi", "rows16"}),
    Case(16384, 512, 16384, 7, 0.4, False, True, {"k4_multi", "rows16"}),
    Case(4096, 2, 8192, 5, 0.3, True, True, {"k2_walk", "zero_width", "zero_height", "k4_multi"}),
]


def smem_fits(n):
    """the histogram of n bins (prefix sums + bit map + two levels of sets) fits a cut kernel's shared memory"""
    tiles = (n + 32767) // 32768
    need = 4 * ((((n + 1) + 3) & ~3) + tiles * (1024 + 32 + 1)) + (2 * LEVEL_NODES * 16 + 16)
    return need + CUT_STATIC <= SMEM_OPTIN


def strip_parts(boxes, ny):
    """parts per strip, in strip order.  A strip is a run of parts with the same columns whose rows tile [0, ny) in
    order, so a new strip starts where the columns change or where the previous part ends at ny and this one starts
    at row 0 (zero-width strips side by side share their columns)."""
    out = []
    prev = None
    for x0, y0, ex, ey in boxes.tolist():
        if prev is None or (x0, ex) != (prev[0], prev[2]) or (prev[1] + prev[3] == ny and y0 == 0):
            out.append(0)
        out[-1] += 1
        prev = (x0, y0, ex, ey)
    return out


def reached(nx, ny, nstrips, xlev, ylev, boxes):
    """the branches of K2 / K4 / the host sizing that a decomposition went through"""
    parts = strip_parts(boxes, ny)
    assert len(parts) == nstrips, (len(parts), nstrips)
    leaves = [min(n, 1 << ylev) for n in parts]  # leaves_below(n, ylevels) of every strip
    r = set()
    if xlev > 0:
        r.add("k2_walk" if nstrips > LEVEL_NODES else "k2_levels")
        if nstrips == LEVEL_NODES:
            r.add("k2_levels_full")
        if not smem_fits(nx):
            r.add("k2_global")
    if ylev == 0:
        r.add("no_y_levels")
    else:
        if any(n > LEVEL_NODES for n in leaves):
            r.add("k4_walk")
            if any(1 < n <= LEVEL_NODES for n in leaves):
                r.add("k4_both")
        if LEVEL_NODES in leaves:
            r.add("k4_levels_full")
        if not smem_fits(ny):
            r.add("k4_global")
        if nstrips > YCUT_BLOCKS:
            r.add("k4_multi")
        r.add("rows32" if nx >= 65536 else "rows16")
    if (boxes[:, 2] == 0).any():
        r.add("zero_width")
    if (boxes[:, 3] == 0).any():
        r.add("zero_height")
    return r


def assert_reaches(case, nstrips, xlev, ylev, boxes):
    got = reached(case.nx, case.ny, nstrips, xlev, ylev, boxes)
    assert case.reaches <= got, (case_id(case), sorted(case.reaches - got))


def list_total(o):
    """entries of the eight neighbour lists together"""
    return sum(len(o.nbr.ids[per][e]) for per in range(2) for e in range(4))


_expected = {}


def expected(oracle, case):
    """(mask, the histogram oracle's decomposition with neighbour lists, part loads), computed once per case"""
    key = tuple(case[:7])
    if key not in _expected:
        mask = oracle.generate_mask(case.nx, case.ny, case.seed, case.land)
        o = oracle.partition(mask, case.P, case.px, case.py, use_hist=True)
        _expected[key] = (mask, o, oracle.part_loads(o.pid, case.P))
    return _expected[key]
