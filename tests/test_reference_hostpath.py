"""The oracle (and the host library's Grid) against the REFERENCE's own host code.

oracle/_ref/libref_hostpath.so is the reference's Grid.cpp + Partitioner.cpp + DomainUtils.cpp compiled
where they lie (oracle/Makefile target `ref`) against stand-in MPI / netCDF headers: P ranks are P
threads, files live in memory, and Zoltan's answers (part boxes, owner map, `changes`) are handed in.
Everything of the path that is not Zoltan is therefore checked against real reference code on
arbitrary inputs, not only on the five goldens:
  Grid: find_factors, naive blocks, slab reads, ocean lists          (Grid.cpp:18-35,132-198)
  the code around the Zoltan call: P == 1 shortcut, box clamp, labels (ZoltanPartitioner.cpp:96-121,172-219)
  discover_neighbours / is_neighbour / halo_start / domain_overlap   (Partitioner.cpp:20-80,329-435)
  get_neighbour_info[_periodic], save_mask, save_metadata            (Partitioner.cpp:98-318)
CPU only.  Where the reference checkout (hence oracle/_ref) is absent, the comparisons run against the answers stored
in tests/golden/reference_answers.json (tests/reference_answers.py); the tests whose subject is the reference's
code itself skip."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden_mask
from reference_answers import Answers

EDGES = ("left", "right", "bottom", "top")


@pytest.fixture(scope="module")
def ref(oracle):
    if oracle.ref_host_lib() is None:
        pytest.skip("oracle/_ref/libref_hostpath.so not built (no reference checkout here)")
    return oracle


@pytest.fixture(scope="module")
def live(oracle):
    """True where oracle/_ref is built: the live comparison with the reference's code runs beside the stored answers"""
    return oracle.ref_host_lib() is not None


def boxes_of(md):
    return np.stack([md["domain_x"], md["domain_y"], md["domain_extent_x"], md["domain_extent_y"]], axis=1).astype(np.int32)


@pytest.mark.parametrize("case", ["test_1", "test_2", "test_1_px", "test_1_py", "test_1_px_py"])
def test_reference_code_reproduces_its_goldens(goldens, ref, case):
    """given the golden boxes and owner map, the reference's own neighbour discovery and writers produce the
    golden files (this pins the stand-in MPI / netCDF as much as the reference code)"""
    G = goldens["integration"][case]
    inp = goldens["inputs"][G["input"]]
    mask = golden_mask(goldens, G["input"])
    pid = np.asarray(G["pid"], dtype=np.int32).reshape(mask.shape)
    r = ref.ref_host_run(mask, G["P"], bool(G["px"]), bool(G["py"]), boxes=boxes_of(G["metadata"]), pid=pid,
                         xdim=inp["xdim"], ydim=inp["ydim"], maskname=inp["mask_name"])
    meta, mfile = r["files"]["metadata"], r["files"]["mask"]
    assert dict(meta["dims"]) == G["dims"]
    got = {name: vals for (grp, name), (dims, vals) in meta["vars"].items()}
    # (ncdump prints no data for a variable over a zero-length dimension: the goldens do not list those)
    assert {k: v for k, v in got.items() if v} == G["metadata"]
    assert len(got) == 4 + 2 * 4 * 4
    assert not meta["unwritten"] and not mfile["unwritten"]
    assert mfile["dims"] == [("y", inp["ny"]), ("x", inp["nx"])] and mfile["atts"] == {"num_processes": G["P"]}
    assert mfile["vars"][("/", "pid")] == ("(y,x)", list(G["pid"]))
    groups = {name: grp for (grp, name) in meta["vars"]}
    assert groups["domain_x"] == "bounding_boxes" and groups["left_neighbour_ids_periodic"] == "connectivity"


def sane_blocks(oracle, P, nx, ny):
    """every naive block is non-empty (otherwise the reference resizes a vector to a negative size)"""
    return all(b[2] >= 1 and b[3] >= 1 for b in (oracle.naive_block(P, nx, ny, r) for r in range(P)))


def test_grid_against_reference_grid(oracle, live):
    """Grid::create on P ranks: block, counts, slab, global ids -- the reference vs the oracle's naive
    blocks vs plain numpy"""
    ref = oracle
    answers = Answers("test_reference_hostpath::test_grid_against_reference_grid", live)
    rng = np.random.default_rng(17)
    checked = 0
    while checked < 60:
        nx, ny, P = int(rng.integers(1, 40)), int(rng.integers(1, 40)), int(rng.integers(1, 13))
        if not sane_blocks(ref, P, nx, ny):
            continue
        mask = (rng.random((ny, nx)) < rng.random()).astype(np.int32) * rng.integers(1, 4, size=(ny, nx)).astype(np.int32)
        answers.check([ref.naive_block(P, nx, ny, rank) for rank in range(P)], (nx, ny, P))
        checked += 1
        if not live:
            continue
        r = ref.ref_host_run(mask, P)
        for rank, got in enumerate(r["ranks"]):
            x0, y0, ex, ey = ref.naive_block(P, nx, ny, rank)
            assert got["block"] == [x0, y0, ex, ey], (nx, ny, P, rank)
            slab = mask[y0:y0 + ey, x0:x0 + ex]
            assert got["objects"] == ex * ey and got["nonzero"] == int((slab > 0).sum())
            assert got["mask"] == slab.ravel().tolist()
            yy, xx = np.nonzero(slab > 0)
            assert got["ids"] == ((yy + y0) * nx + xx + x0).tolist()
    answers.finish()


def test_grid_dimension_names_order_and_group(ref):
    mask = (np.arange(35).reshape(5, 7) % 3).astype(np.int32)
    # named dimensions and the nextSIM restart layout (everything in group "data", Grid.cpp:58-62)
    r = ref.ref_host_run(mask, 2, xdim="m", ydim="n", maskname="land_mask", data_group=True)
    assert r["ranks"][0]["block"] == ref.naive_block(2, 7, 5, 0)
    # a variable declared (x, y): with `-o xy` the reference reads it block-wise in file order (quirk Q7)
    sq = (np.arange(36).reshape(6, 6) % 2).astype(np.int32)
    r = ref.ref_host_run(sq, 1, order_xy=True)
    assert r["ranks"][0]["mask"] == sq.ravel().tolist()
    with pytest.raises(RuntimeError, match="Dimension ordering provided does not match"):
        ref.ref_host_run(sq, 1, order_xy=False, file_order_xy=True)
    # --ignore-mask on one rank: every cell is an object (on several ranks the reference's ids lose the
    # block's y offset, quirk Q5 -- documented, not reproduced)
    r = ref.ref_host_run(sq, 1, ignore_mask=True)
    assert r["ranks"][0]["nonzero"] == 36 and r["ranks"][0]["ids"] == list(range(36))


def per_part(nbr, P, per, e):
    """the oracle's flat list of one edge -> a list per part of (id, halo, start)"""
    cnt = nbr.counts[per][e]
    off = np.concatenate([[0], np.cumsum(cnt)])
    ids, halos, starts = nbr.ids[per][e], nbr.halos[per][e], nbr.starts[per][e]
    return [[(int(ids[k]), int(halos[k]), int(starts[k])) for k in range(off[p], off[p + 1])] for p in range(P)]


def check_against_oracle(ref, mask, P, px, py, answers, live):
    """the oracle's decomposition is the stored answer of this case and, where oracle/_ref is built (`live`), what the
    reference's own neighbour discovery and writers give back for its boxes and owners"""
    ny, nx = mask.shape
    o = ref.partition(mask, P, px, py, use_hist=True)
    boxes = o.boxes if o.changes else np.asarray([ref.naive_block(P, nx, ny, r) for r in range(P)], dtype=np.int32)
    assert o.boxes.tolist() == boxes.tolist()  # the oracle already reports the naive blocks when nothing moved
    ctx = (nx, ny, P, px, py)
    answers.check({"boxes": o.boxes, "pid": o.pid, "changes": o.changes, "counts": o.nbr.counts, "ids": o.nbr.ids,
                   "halos": o.nbr.halos, "starts": o.nbr.starts}, ctx)
    if not live:
        return
    r = ref.ref_host_run(mask, P, px, py, boxes=o.boxes, pid=o.pid, changes=o.changes)
    for p in range(P):
        assert r["ranks"][p]["box"] == o.boxes[p].tolist(), ctx
        for per in range(2):
            for e in range(4):
                want = per_part(o.nbr, P, per, e)[p] if P > 1 else []
                assert r["ranks"][p]["nbr"][per][e] == want, (ctx, p, per, e)
    meta = {name: vals for (grp, name), (dims, vals) in r["files"]["metadata"]["vars"].items()}
    dims = dict(r["files"]["metadata"]["dims"])
    assert dims["NX"] == nx and dims["NY"] == ny and dims["P"] == P
    for i, key in enumerate(("domain_x", "domain_y", "domain_extent_x", "domain_extent_y")):
        assert meta[key] == o.boxes[:, i].tolist(), ctx
    for per, sfx in ((0, ""), (1, "_periodic")):
        for e, name in enumerate(EDGES):
            if P == 1:  # the reference returns before neighbour discovery (quirk Q4)
                assert meta[name + "_neighbours" + sfx] == [0]
                continue
            assert meta[name + "_neighbours" + sfx] == o.nbr.counts[per][e].tolist(), (ctx, name, sfx)
            assert meta[name + "_neighbour_ids" + sfx] == o.nbr.ids[per][e].tolist(), (ctx, name, sfx)
            assert meta[name + "_neighbour_halos" + sfx] == o.nbr.halos[per][e].tolist(), (ctx, name, sfx)
            assert meta[name + "_neighbour_halo_starts" + sfx] == o.nbr.starts[per][e].tolist(), (ctx, name, sfx)
            assert dims["LRBT"[e] + sfx] == len(o.nbr.ids[per][e])
    assert not r["files"]["metadata"]["unwritten"]
    # the mask file: every rank writes the owners of its naive block; together they are the whole map
    assert r["files"]["mask"]["vars"][("/", "pid")][1] == o.pid.ravel().tolist(), ctx
    assert not r["files"]["mask"]["unwritten"]


def test_neighbours_and_files_against_reference_code_random(oracle, live):
    """random coastlines, 1 .. 24 parts, all periodic combinations: the oracle's boxes / owners go through the
    reference's own neighbour discovery and writers and must come back as the oracle's tables"""
    ref = oracle
    answers = Answers("test_reference_hostpath::test_neighbours_and_files_against_reference_code_random", live)
    rng = np.random.default_rng(23)
    done = 0
    while done < 120:
        nx, ny, P = int(rng.integers(2, 48)), int(rng.integers(2, 48)), int(rng.integers(1, 25))
        if not sane_blocks(ref, P, nx, ny):
            continue
        land = rng.random() * 0.8
        mask = (rng.random((ny, nx)) >= land).astype(np.int32)
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        check_against_oracle(ref, mask, P, px, py, answers, live)
        done += 1
    answers.finish()


def test_nothing_moved_and_all_land_against_reference_code(oracle, live):
    """`changes == 0`: the reference reports the naive blocks and finds THEIR neighbours"""
    answers = Answers("test_reference_hostpath::test_nothing_moved_and_all_land_against_reference_code", live)
    for (n, P) in [(64, 4), (60, 6), (96, 16)]:
        check_against_oracle(oracle, np.ones((n, n), dtype=np.int32), P, True, True, answers, live)
    check_against_oracle(oracle, np.zeros((12, 18), dtype=np.int32), 6, False, True, answers, live)
    check_against_oracle(oracle, np.zeros((4, 6), dtype=np.int32), 2, False, False, answers, live)  # test_zoltan_partitioner_0.cpp:39-66
    answers.finish()


def test_host_library_grid_matches_reference_grid(oracle, live, tmp_path):
    """this repository's Grid (host library, through nc_tool on a classic netCDF file) == the reference's Grid"""
    ref = oracle
    answers = Answers("test_reference_hostpath::test_host_library_grid_matches_reference_grid", live)
    scipy_io = pytest.importorskip("scipy.io")
    from domain_decomp_b200 import build
    build.build_all()
    tool = os.path.join(ROOT, "domain_decomp_b200", "nc_tool")
    rng = np.random.default_rng(5)
    for (nx, ny, P) in [(6, 4, 2), (30, 30, 4), (17, 9, 3), (33, 20, 6), (21, 34, 8)]:
        assert sane_blocks(ref, P, nx, ny)
        mask = (rng.random((ny, nx)) < 0.6).astype(np.int32)
        path = str(tmp_path / ("g_%d_%d.nc" % (nx, ny)))
        f = scipy_io.netcdf_file(path, "w", version=1)
        f.createDimension("x", nx)
        f.createDimension("y", ny)
        f.createVariable("mask", "i4", ("y", "x"))[:] = mask
        f.close()
        r = ref.ref_host_run(mask, P) if live else None
        for rank in range(P):
            out = subprocess.run([tool, "grid", path, "x", "y", "yx", "mask", "ranks", str(P), str(rank)],
                                 capture_output=True, text=True, timeout=60)
            assert out.returncode == 0, out.stderr
            lines = dict(l.split(" ", 1) for l in out.stdout.strip().splitlines())
            answers.check({k: lines[k] for k in ("block", "objects", "mask")}, (nx, ny, P, rank))
            if not live:
                continue
            got = r["ranks"][rank]
            assert list(map(int, lines["block"].split())) == got["block"]
            assert lines["objects"] == "%d nonzero %d" % (got["objects"], got["nonzero"])
            assert list(map(int, lines["mask"].split())) == got["mask"]
    answers.finish()


@pytest.mark.parametrize("px,py", [(0, 0), (1, 1)])
def test_arctic25km_64_parts_against_reference_code(oracle, live, px, py):
    """BASELINE config 2 (528 x 522 synthetic coastline, 64 parts) on 64 thread-ranks of reference code"""
    answers = Answers("test_reference_hostpath::test_arctic25km_64_parts_against_reference_code[%d-%d]" % (px, py), live)
    from domain_decomp_b200 import capi
    mask = capi.generate_mask_host(528, 522, 25, 0.45)
    assert sane_blocks(oracle, 64, 528, 522)
    check_against_oracle(oracle, mask, 64, bool(px), bool(py), answers, live)
    answers.finish()
