"""The host layer (domain_decomp_b200/host: Grid, Partitioner, CudaRcbPartitioner, the `decomp` CLI) on a machine
WITHOUT a GPU: oracle/Makefile links the very same host sources into test binaries under oracle/_ref/, with, behind
the C ABI, either the CPU oracle (oracle/ddc_oracle_stub.c: *_oracle) or the PRODUCT's own C-ABI implementation and
kernels on the host emulation of CUDA (oracle/libddc_cuda_emu.so: *_emu -- the whole product stack, CLI to
kernels).  (The product binaries link libddc_cuda.so and have no such path; tests/test_host_cpp.py runs them on
the GPU.)  Checked here:
  * the reference's unit tests re-expressed (host_tests.cpp: test_grid_*, test_zoltan_partitioner_*),
  * the reference's integration test: CLI output byte-identical to the golden ncdump text,
  * binary netCDF grids in, partition_mask_<P>.nc out,
  * on random coastlines: what this host layer writes == what the REFERENCE's own Partitioner.cpp writes
    (oracle/_ref/libref_hostpath.so) for the same boxes -- rank views, per-edge offsets, zero-length dims."""
import hashlib
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from reference_answers import Answers
from test_host_cpp import CASES, write_input_cdl
from test_reference_hostpath import sane_blocks

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
DECOMP = os.path.join(REF_DIR, "decomp_oracle")
DECOMP_EMU = os.path.join(REF_DIR, "decomp_emu")
HOST_TESTS = os.path.join(REF_DIR, "host_tests_oracle")
HOST_TESTS_EMU = os.path.join(REF_DIR, "host_tests_emu")


@pytest.fixture(scope="module", autouse=True)
def built(oracle):
    oracle.build()
    if not all(os.path.exists(p) for p in (DECOMP, HOST_TESTS, DECOMP_EMU, HOST_TESTS_EMU)):
        pytest.fail("oracle.build() did not build the host-layer test binaries (oracle/Makefile target hostcpu)")


@pytest.fixture(scope="module")
def fixture_dir(tmp_path_factory, goldens):
    d = tmp_path_factory.mktemp("grids_cpu")
    for name in ("test_0", "test_1", "test_2"):
        write_input_cdl(os.path.join(d, name + ".cdl"), name, goldens["inputs"][name])
    return str(d)


@pytest.mark.parametrize("exe", [HOST_TESTS, HOST_TESTS_EMU], ids=["oracle", "emu"])
def test_reference_unit_tests_on_the_host_layer(fixture_dir, exe):
    out = subprocess.run([exe, fixture_dir], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert " 0 failed" in out.stdout


@pytest.mark.parametrize("exe", [DECOMP, DECOMP_EMU], ids=["oracle", "emu"])
@pytest.mark.parametrize("case", sorted(CASES))
def test_cli_integration_goldens(goldens, fixture_dir, tmp_path, case, exe):
    inp, flags = CASES[case]
    out = subprocess.run([exe, "-g", os.path.join(fixture_dir, inp + ".cdl"), "--parts", "3"] + flags,
                         capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert out.returncode == 0, out.stdout + out.stderr
    G = goldens["integration"][case]
    for fname, key in (("partition_mask_3.cdl", "mask_cdl_sha256"), ("partition_metadata_3.cdl", "metadata_cdl_sha256")):
        text = open(os.path.join(tmp_path, fname)).read()
        assert hashlib.sha256(text.encode()).hexdigest() == G[key], "%s differs from the golden:\n%s" % (fname, text)


def parse_cdl(text):
    dims = {}
    for mm in re.finditer(r"^\t(\w+) = (\w+) ;(?: // \((\d+) currently\))?$", text, re.M):
        dims[mm.group(1)] = (0 if mm.group(2) == "UNLIMITED" else int(mm.group(2)), mm.group(2) == "UNLIMITED")
    data = {}
    for body in re.split(r"\bdata:\n", text)[1:]:
        for mm in re.finditer(r"^\s*(\w+) =\s*([-0-9,\s]+?);", body, re.S | re.M):
            data[mm.group(1)] = [int(v) for v in mm.group(2).replace("\n", " ").split(",")]
    return dims, data


def write_nc(path, mask, version=1):
    scipy_io = pytest.importorskip("scipy.io")
    ny, nx = mask.shape
    f = scipy_io.netcdf_file(path, "w", version=version)
    f.createDimension("x", nx)
    f.createDimension("y", ny)
    f.createVariable("mask", "i4", ("y", "x"))[:] = mask
    f.close()


@pytest.mark.parametrize("exe", [DECOMP, DECOMP_EMU], ids=["oracle", "emu"])
def test_cli_on_binary_netcdf_and_stats(goldens, tmp_path, exe):
    scipy_io = pytest.importorskip("scipy.io")
    inp = goldens["inputs"]["test_1"]
    write_nc(str(tmp_path / "test_1.nc"), np.asarray(inp["mask"], dtype=np.int32).reshape(inp["ny"], inp["nx"]))
    out = subprocess.run([exe, "-g", "test_1.nc", "--parts", "3", "--px", "--stats"], capture_output=True, text=True,
                         timeout=300, cwd=tmp_path)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "Total weight of dots = 24" in out.stdout
    G = goldens["integration"]["test_1_px"]
    text = open(tmp_path / "partition_metadata_3.cdl").read()
    assert hashlib.sha256(text.encode()).hexdigest() == G["metadata_cdl_sha256"]
    m = scipy_io.netcdf_file(str(tmp_path / "partition_mask_3.nc"), "r", mmap=False)
    assert m.num_processes == 3 and m.variables["pid"].data.ravel().tolist() == list(G["pid"])
    m.close()


def test_cli_errors(fixture_dir, tmp_path):
    r = subprocess.run([DECOMP], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1 and "'--grid' is required" in r.stderr
    r = subprocess.run([DECOMP, "-g", os.path.join(fixture_dir, "test_1.cdl"), "-o", "zz"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1 and "must be either 'xy' or 'yx'" in r.stderr
    r = subprocess.run([DECOMP, "-g", os.path.join(fixture_dir, "test_2.cdl"), "--parts", "2"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1  # default names x / y / mask do not exist in test_2
    r = subprocess.run([DECOMP, "-g", "/nonexistent/grid.nc"], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1 and "ERROR" in r.stderr


def test_files_written_by_the_host_layer_equal_the_reference_writers(oracle, tmp_path):
    """random coastlines through the CLI; the same boxes / owners through the reference's own save_mask and
    save_metadata (Partitioner.cpp:128-318): dimension lengths (0 => UNLIMITED), every variable, every value.
    Without oracle/_ref, against the stored answers of the same seeded cases (tests/reference_answers.py)."""
    live = oracle.ref_host_lib() is not None
    answers = Answers("test_host_layer_cpu::test_files_written_by_the_host_layer_equal_the_reference_writers", live)
    rng = np.random.default_rng(77)
    done = 0
    while done < 25:
        exe = DECOMP_EMU if done % 5 == 4 else DECOMP  # every fifth case through the whole product stack
        nx, ny, P = int(rng.integers(3, 40)), int(rng.integers(3, 40)), int(rng.integers(2, 17))
        if not sane_blocks(oracle, P, nx, ny):
            continue
        mask = (rng.random((ny, nx)) >= rng.random() * 0.7).astype(np.int32)
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        d = tmp_path / ("case%d" % done)
        d.mkdir()
        write_nc(str(d / "g.nc"), mask, version=1 + done % 2)
        cmd = [exe, "-g", "g.nc", "--parts", str(P)] + (["--px"] if px else []) + (["--py"] if py else [])
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=d)
        assert out.returncode == 0, out.stdout + out.stderr
        dims, data = parse_cdl(open(d / ("partition_metadata_%d.cdl" % P)).read())
        mdims, mdata = parse_cdl(open(d / ("partition_mask_%d.cdl" % P)).read())
        answers.check({"dims": dims, "data": data, "mask_dims": mdims, "pid": mdata["pid"]}, (nx, ny, P, px, py))
        done += 1
        if not live:
            continue
        o = oracle.partition(mask, P, px, py, use_hist=True)
        ref = oracle.ref_host_run(mask, P, px, py, boxes=o.boxes, pid=o.pid, changes=o.changes)
        # metadata
        rdims = dict(ref["files"]["metadata"]["dims"])
        assert {k: v[0] for k, v in dims.items()} == rdims, (nx, ny, P)
        for k, (length, unlimited) in dims.items():
            assert unlimited == (rdims[k] == 0), (k, "nc_def_dim(len = 0) makes the dimension UNLIMITED")
        rvars = {name: vals for (grp, name), (vd, vals) in ref["files"]["metadata"]["vars"].items()}
        assert data == {k: v for k, v in rvars.items() if v}, (nx, ny, P, px, py)
        # mask
        assert {k: v[0] for k, v in mdims.items()} == dict(ref["files"]["mask"]["dims"])
        assert mdata["pid"] == ref["files"]["mask"]["vars"][("/", "pid")][1]
    answers.finish()


@pytest.mark.parametrize("exe", [DECOMP, DECOMP_EMU], ids=["oracle", "emu"])
def test_cli_ignore_mask_and_rect3030(goldens, oracle, fixture_dir, tmp_path, exe):
    """--ignore-mask (every cell is an object) and the nextSIM restart layout of grids/rect3030.res.cdl: group
    `data`, a double mask declared (x, y), read with -o xy (BASELINE config 1)"""
    out = subprocess.run([exe, "-g", os.path.join(fixture_dir, "test_0.cdl"), "--parts", "4", "-i"], capture_output=True,
                         text=True, timeout=300, cwd=tmp_path)
    assert out.returncode == 0, out.stderr
    _, data = parse_cdl(open(tmp_path / "partition_mask_4.cdl").read())
    o = oracle.partition(np.ones((4, 6), dtype=np.int32), 4, use_hist=True)  # test_0 is all land: ignored
    assert data["pid"] == o.pid.ravel().tolist()
    # rect3030: rebuilt from the golden JSON in the reference's layout
    inp = goldens["inputs"]["rect3030"]
    vals = np.asarray(inp["mask"], dtype=np.int32)
    rows = ",\n".join("  " + ", ".join("%d" % v for v in vals[i * 30:(i + 1) * 30]) for i in range(30))
    cdl = ("netcdf rect3030 {\n\ngroup: data {\n  dimensions:\n  \tx = 30 ;\n  \ty = 30 ;\n  variables:\n  \tdouble mask(x, y) ;\n"
           "  data:\n\n   mask =\n%s ;\n  } // group data\n}\n" % rows)
    (tmp_path / "rect3030.cdl").write_text(cdl)
    for P in (2, 4):
        out = subprocess.run([exe, "-g", "rect3030.cdl", "-o", "xy", "--parts", str(P)], capture_output=True, text=True,
                             timeout=300, cwd=tmp_path)
        assert out.returncode == 0, out.stderr
        _, data = parse_cdl(open(tmp_path / ("partition_mask_%d.cdl" % P)).read())
        o = oracle.partition(vals.reshape(30, 30), P, use_hist=True)
        assert data["pid"] == o.pid.ravel().tolist()
        _, meta = parse_cdl(open(tmp_path / ("partition_metadata_%d.cdl" % P)).read())
        assert meta["domain_x"] == o.boxes[:, 0].tolist() and meta["domain_extent_y"] == o.boxes[:, 3].tolist()


# ---- the netCDF-C backend of the host layer (HAVE_NETCDF) ---------------------------------------------------------------
def _host_nc_run(oracle, mask, P, px=False, py=False, xdim="x", ydim="y", maskname="mask", order_xy=False,
                 file_order_xy=None, data_group=False, ignore_mask=False):
    import ctypes as C
    path = os.path.join(REF_DIR, "libhost_netcdf.so")
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/libhost_netcdf.so not built")
    L = C.CDLL(path)
    i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
    L.host_nc_run.argtypes = [C.c_int, C.c_int, C.c_int, i32p, C.c_char_p, C.c_char_p, C.c_char_p] + [C.c_int] * 6
    L.host_nc_run.restype = C.c_char_p
    L.host_nc_error.restype = C.c_char_p
    m = np.ascontiguousarray(mask, dtype=np.int32)
    ny, nx = m.shape
    out = L.host_nc_run(P, nx, ny, m, xdim.encode(), ydim.encode(), maskname.encode(), int(order_xy),
                        int(order_xy if file_order_xy is None else file_order_xy), int(data_group), int(ignore_mask),
                        int(px), int(py))
    if out is None:
        raise RuntimeError(L.host_nc_error().decode())
    text = out.decode()
    head = dict(l.split(" ", 1) for l in text.splitlines()[:2])
    files = oracle._parse_report("\n".join(text.splitlines()[2:]).encode(), P)["files"]
    return head, files


def test_netcdf4_outputs_through_netcdf_c_equal_the_reference_writers(oracle):
    """The host layer built with -DHAVE_NETCDF writes partition_mask_<P>.nc and the GROUPED partition_metadata_<P>.nc
    (groups bounding_boxes / connectivity) through netCDF-C calls (host/NcLibrary.cpp); the reference's own
    Partitioner.cpp (Partitioner.cpp:128-318, compiled where it lies) writes them for the same decomposition through
    the same in-memory netCDF.  Both files must be equal in everything a reader can see: dimension names, order and
    lengths (a zero length -- no neighbour on an edge -- is an UNLIMITED dimension in both), the global attribute,
    groups, variables, their dimensions and every value.  Without oracle/_ref, against the stored answers of the same
    seeded cases (tests/reference_answers.py)."""
    live = oracle.ref_host_lib() is not None
    answers = Answers("test_host_layer_cpu::test_netcdf4_outputs_through_netcdf_c_equal_the_reference_writers", live)
    rng = np.random.default_rng(5)
    cases = 0
    for it in range(40):
        nx, ny = int(rng.integers(4, 40)), int(rng.integers(4, 40))
        P = int(rng.integers(1, 13))
        px, py = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
        mask = (rng.random((ny, nx)) < rng.choice([0.0, 0.3, 0.7, 1.0])).astype(np.int32)
        if not sane_blocks(oracle, P, nx, ny):
            continue
        head, got = _host_nc_run(oracle, mask, P, px, py)
        assert head["grid"] == "%d %d" % (nx, ny) and head["gridmask"].split() == [str(v) for v in mask.ravel()]
        answers.check(got, (nx, ny, P, px, py))
        if live:
            o = oracle.partition(mask, P, px, py)
            want = oracle.ref_host_run(mask, P, px, py, boxes=o.boxes, pid=o.pid, changes=o.changes)["files"]
            assert got == want, (nx, ny, P, px, py)
        cases += 1
    assert cases >= 25
    answers.finish()


def test_grid_input_through_netcdf_c(oracle):
    """Grid::create over nc_open / nc_inq_* / nc_get_vara_int (Grid.cpp:51-130): other dimension and variable names,
    group `data` of the nextSIM restart layout, (x, y)-declared masks with -o xy, --ignore-mask, and the reference's
    error for a wrong dimension order"""
    rng = np.random.default_rng(9)
    mask = (rng.random((7, 5)) < 0.6).astype(np.int32)
    head, _ = _host_nc_run(oracle, mask, 2, xdim="m", ydim="n", maskname="land_mask", data_group=True)
    assert head["grid"] == "5 7" and head["gridmask"].split() == [str(v) for v in mask.ravel()]
    sq = (rng.random((6, 6)) < 0.6).astype(np.int32)
    head, _ = _host_nc_run(oracle, sq, 2, order_xy=True, file_order_xy=True)
    assert head["gridmask"].split() == [str(v) for v in sq.ravel()]  # raw reinterpretation (DESIGN.md Q7)
    head, _ = _host_nc_run(oracle, mask, 3, ignore_mask=True)
    assert set(head["gridmask"].split()) == {"1"}
    with pytest.raises(RuntimeError, match="Dimension ordering provided does not match"):
        _host_nc_run(oracle, sq, 2, order_xy=False, file_order_xy=True)
