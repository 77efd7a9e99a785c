"""ctypes front-end of the CPU oracle (oracle/ddc_oracle.c).

TEST INFRASTRUCTURE ONLY -- imported by tests/, by __graft_entry__.smoke() and
by bench.py's cpu_baseline / ``--impl reference`` leg, never by the product
package ``domain_decomp_b200``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libddc_oracle.so")
_REF_LIB = os.path.join(_HERE, "_ref", "libref_domainutils.so")
_REF_HOST_LIB = os.path.join(_HERE, "_ref", "libref_hostpath.so")

EDGES = ("left", "right", "bottom", "top")  # DomainUtils.hpp:15 enum order L,R,B,T


def build(force: bool = False) -> str:
    """Compile the C restatement, the emulation libraries and the host-layer test binaries; with
    DDC_REFERENCE_DIR naming a checkout of the reference, also its own sources into oracle/_ref."""
    src = os.path.join(_HERE, "ddc_oracle.c")
    if force or not os.path.exists(_LIB) or os.path.getmtime(_LIB) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "libddc_oracle.so"])
    # make decides what is stale
    subprocess.check_call(["make", "-s", "-j4", "-C", _HERE, "libddc_median_emu.so", "libddc_emu.so", "libddc_cuda_emu.so", "hostcpu"]
                          + (["-B"] if force else []))
    ref = os.environ.get("DDC_REFERENCE_DIR")
    if ref:
        subprocess.check_call(["make", "-s", "-j4", "-C", _HERE, "ref", "REF=" + os.path.abspath(ref)] + (["-B"] if force else []))
    return _LIB


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        L.orc_find_factors.argtypes = [C.c_int, C.POINTER(C.c_int)]
        L.orc_naive_block.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.orc_partition.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, C.c_void_p,
                                    C.POINTER(C.c_int), C.POINTER(C.c_long)]
        L.orc_partition.restype = C.c_int
        L.orc_neighbours.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, i32p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_domain_overlap.argtypes = [C.c_int] * 9
        L.orc_domain_overlap.restype = C.c_int
        L.orc_set_threads.argtypes = [C.c_int]
        L.orc_max_threads.restype = C.c_int
        L.orc_part_loads.argtypes = [i32p, C.c_size_t, C.c_int,
                                     np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")]
        _lib = L
    return _lib


def ref_lib():
    """The reference's own DomainUtils.cpp compiled in oracle/_ref (None if not built)."""
    if not os.path.exists(_REF_LIB):
        return None
    L = C.CDLL(_REF_LIB)
    L.ref_domain_overlap.argtypes = [C.c_int] * 9
    L.ref_domain_overlap.restype = C.c_int
    return L


def median_emu_lib():
    """The scalar core of the CUDA cut kernels (csrc/ddc_median.cuh) compiled as host code, with the fuzz
    driver of oracle/emu_median_harness.cpp."""
    build()
    L = C.CDLL(os.path.join(_HERE, "libddc_median_emu.so"))
    L.emu_fuzz.argtypes = [C.c_uint64, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                           C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.emu_fuzz.restype = C.c_long
    L.emu_fuzz_neighbours.argtypes = [C.c_uint64, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.emu_fuzz_neighbours.restype = C.c_long
    return L


_emu = None


def emu_partition(mask: np.ndarray, P: int, px: bool = False, py: bool = False, *, ranks: int = 1, strip_k: int = 0,
                  scan_rpc: int = 0, smem_limit: int = 0, nbr_cap: int | None = None):
    """One decomposition through the product's REAL kernels on the host emulation of the CUDA execution model
    (oracle/emu/), on `ranks` emulated row-sharded ranks.  Returns (Decomposition, info dict).
    nbr_cap: entries reserved for the eight neighbour lists together (ids, halos and starts each); by default enough
    for every part to list every other one, 16 P^2, which is gigabytes beyond a few thousand parts.  A capacity below
    the lists' total is an error."""
    global _emu
    if _emu is None:
        build()
        L = C.CDLL(os.path.join(_HERE, "libddc_emu.so"))
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        L.emu_partition.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    i32p, i32p, i32p, i32p, C.c_long, np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")]
        L.emu_partition.restype = C.c_int
        L.emu_last_error.restype = C.c_char_p
        _emu = L
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    ny, nx = mask.shape
    boxes = np.zeros((P, 4), dtype=np.int32)
    pid = np.zeros((ny, nx), dtype=np.int32)
    counts = np.zeros(8 * P, dtype=np.int32)
    cap = 8 * (3 * P + 64) + 16 * P * P if nbr_cap is None else int(nbr_cap)
    flat = np.zeros(3 * cap, dtype=np.int32)
    out = np.zeros(8, dtype=np.int64)
    rc = _emu.emu_partition(mask, nx, ny, P, int(px), int(py), ranks, strip_k, scan_rpc, smem_limit, boxes, pid, counts, flat,
                            cap, out)
    if rc != 0:
        raise RuntimeError("emu_partition: " + _emu.emu_last_error().decode())
    c = counts.reshape(2, 4, P)
    totals = counts.reshape(8, P).sum(axis=1)
    off = np.concatenate([[0], np.cumsum(totals)])
    sl = lambda k, l: flat[k * cap + off[l]:k * cap + off[l + 1]].copy()
    nbr = Neighbours(
        counts=[[c[per, e].copy() for e in range(4)] for per in range(2)],
        ids=[[sl(0, per * 4 + e) for e in range(4)] for per in range(2)],
        halos=[[sl(1, per * 4 + e) for e in range(4)] for per in range(2)],
        starts=[[sl(2, per * 4 + e) for e in range(4)] for per in range(2)],
    )
    d = Decomposition(NX=nx, NY=ny, P=P, boxes=boxes, pid=pid, changes=int(out[0]), median_iters=int(out[1]), nbr=nbr)
    info = dict(n_ocean=int(out[2]), strips=int(out[3]), x_levels=int(out[4]), y_levels=int(out[5]), load_min=int(out[6]),
                load_max=int(out[7]))
    return d, info


_ref_host = None


def ref_host_lib():
    """The reference's own Grid.cpp + Partitioner.cpp + DomainUtils.cpp compiled in oracle/_ref against
    the stand-in MPI / netCDF headers of oracle/ref_shim (None if not built)."""
    global _ref_host
    if _ref_host is None:
        if not os.path.exists(_REF_HOST_LIB):
            return None
        L = C.CDLL(_REF_HOST_LIB)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        L.ref_host_run.argtypes = [C.c_int, C.c_int, C.c_int, i32p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.ref_host_run.restype = C.c_char_p
        L.ref_host_error.restype = C.c_char_p
        _ref_host = L
    return _ref_host


def _parse_report(out: bytes, P: int) -> dict:
    ranks = [dict(nbr=[[None] * 4 for _ in range(2)]) for _ in range(P)]
    files, cur = {}, None
    for line in out.decode().splitlines():
        t = line.split()
        if t[0] == "rank":
            r, what = ranks[int(t[1])], t[2]
            if what == "block":
                r["block"] = list(map(int, t[3:7]))
                r["objects"], r["nonzero"] = int(t[8]), int(t[10])
            elif what in ("mask", "ids"):
                r[what] = list(map(int, t[3:]))
            elif what == "box":
                r["box"] = list(map(int, t[3:7]))
            elif what == "nbr":
                r["nbr"][int(t[4])][int(t[3])] = [tuple(map(int, x.split(":"))) for x in t[5:]]
        elif t[0] == "file":
            cur = files.setdefault(t[1], dict(dims=[], atts={}, vars={}, unwritten={}))
        elif t[0] == "dim":
            cur["dims"].append((t[1], int(t[2])))
        elif t[0] == "att":
            cur["atts"][t[1]] = int(t[2])
        elif t[0] == "var":
            cur["vars"][(t[1], t[2])] = (t[3], list(map(int, t[4:])))
        elif t[0] == "unwritten":
            cur["unwritten"][t[1]] = int(t[2])
    return dict(ranks=ranks, files=files)


_ref_binding = {}


def ref_binding_lib(cpu):
    """The reference's host sources + integration/reference_binding (the CudaRcbPartitioner a maintainer adds
    to the reference tree) -- linked with the CUDA library (cpu=False) or, without a GPU, with the oracle
    answering its ddc_* calls (cpu=True) or with the product's own C ABI and kernels on the host emulation
    (cpu="emu").  None if not built."""
    if cpu not in _ref_binding:
        name = {True: "libref_binding_cpu.so", False: "libref_binding.so", "emu": "libref_binding_emu.so"}[cpu]
        path = os.path.join(_HERE, "_ref", name)
        if not os.path.exists(path):
            return None
        L = C.CDLL(path)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        L.ref_binding_run.argtypes = [C.c_int, C.c_int, C.c_int, i32p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int,
                                      C.c_int, C.c_int, C.c_int]
        L.ref_binding_run.restype = C.c_char_p
        L.ref_host_error.restype = C.c_char_p
        _ref_binding[cpu] = L
    return _ref_binding[cpu]


def ref_binding_run(mask: np.ndarray, P: int, px: bool = False, py: bool = False, *, cpu, xdim: str = "x",
                    ydim: str = "y", maskname: str = "mask", ignore_mask: bool = False, device: int = 0) -> dict:
    """Grid::create (reference) -> CudaRcbPartitioner::partition (the binding over the C ABI) -> the
    reference's discover_neighbours, getters, save_mask, save_metadata, on P thread-ranks.  Same report as
    ref_host_run."""
    L = ref_binding_lib(cpu)
    if L is None:
        raise RuntimeError("oracle/_ref/libref_binding (%s) is not built" % cpu)
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    ny, nx = mask.shape
    out = L.ref_binding_run(P, nx, ny, mask, xdim.encode(), ydim.encode(), maskname.encode(), int(ignore_mask),
                            int(px), int(py), device)
    if out is None:
        raise RuntimeError(L.ref_host_error().decode())
    return _parse_report(out, P)


def ref_host_run(mask: np.ndarray, P: int, px: bool = False, py: bool = False, *, boxes=None, pid=None,
                 changes: int = 1, xdim: str = "x", ydim: str = "y", maskname: str = "mask", order_xy: bool = False,
                 file_order_xy=None, data_group: bool = False, ignore_mask: bool = False) -> dict:
    """Run the REFERENCE's host path (Grid::create, the code around the Zoltan call, discover_neighbours,
    the getters, save_mask, save_metadata) on P thread-ranks; boxes [P,4] / pid [NY,NX] stand in for
    Zoltan's answers (None: only Grid is exercised).  Returns the parsed report:
      ranks[r] = {block, objects, nonzero, mask, ids, box, nbr[periodic][edge] = [(id, halo, start), ...]}
      files[name] = {dims: [(name, len)], atts: {..}, vars: {(group, name): (dims, values)}, unwritten: {..}}"""
    L = ref_host_lib()
    if L is None:
        raise RuntimeError("oracle/_ref/libref_hostpath.so is not built (needs DDC_REFERENCE_DIR)")
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    ny, nx = mask.shape
    b = None if boxes is None else np.ascontiguousarray(boxes, dtype=np.int32)
    q = None if pid is None else np.ascontiguousarray(pid, dtype=np.int32)
    out = L.ref_host_run(P, nx, ny, mask, xdim.encode(), ydim.encode(), maskname.encode(), int(order_xy),
                         int(order_xy if file_order_xy is None else file_order_xy), int(data_group), int(ignore_mask), int(px), int(py), int(changes),
                         None if b is None else b.ctypes.data, None if q is None else q.ctypes.data)
    if out is None:
        raise RuntimeError(L.ref_host_error().decode())
    return _parse_report(out, P)


def set_threads(t: int) -> None:
    """threads for the dot-based RCB (OpenMP tasks over the independent halves); default 1"""
    lib().orc_set_threads(int(t))


def max_threads() -> int:
    return int(lib().orc_max_threads())


def find_factors(P: int):
    out = (C.c_int * 2)()
    lib().orc_find_factors(P, out)
    return [out[0], out[1]]


def naive_block(P: int, NX: int, NY: int, r: int):
    out = (C.c_int * 4)()
    lib().orc_naive_block(P, NX, NY, r, out)
    return [out[0], out[1], out[2], out[3]]


@dataclass
class Neighbours:
    """counts[periodic][edge] -> int32[P]; ids/halos/starts[periodic][edge] -> flat int32 list
    (concatenation over parts 0..P-1 of each part's id-ascending list)."""
    counts: list
    ids: list
    halos: list
    starts: list


@dataclass
class Decomposition:
    NX: int
    NY: int
    P: int
    boxes: np.ndarray  # int32 [P,4] = x0, y0, ext_x, ext_y
    pid: np.ndarray | None  # int32 [NY,NX], -1 on land
    changes: int
    median_iters: int
    nbr: Neighbours | None = None


def neighbours(boxes: np.ndarray, NX: int, NY: int, px: bool, py: bool) -> Neighbours:
    boxes = np.ascontiguousarray(boxes, dtype=np.int32)
    P = boxes.shape[0]
    counts = np.zeros(8 * P, dtype=np.int32)
    lib().orc_neighbours(boxes, P, NX, NY, int(px), int(py), counts, None, None, None, None)
    totals = counts.reshape(8, P).sum(axis=1).astype(np.int64)
    offsets = np.zeros(8, dtype=np.int64)
    offsets[1:] = np.cumsum(totals)[:-1]
    n = int(totals.sum())
    ids = np.zeros(max(n, 1), dtype=np.int32)
    halos = np.zeros(max(n, 1), dtype=np.int32)
    starts = np.zeros(max(n, 1), dtype=np.int32)
    lib().orc_neighbours(boxes, P, NX, NY, int(px), int(py), counts,
                         offsets.ctypes.data, ids.ctypes.data, halos.ctypes.data, starts.ctypes.data)
    c = counts.reshape(2, 4, P)
    sl = lambda a, l: a[int(offsets[l]):int(offsets[l] + totals[l])].copy()
    return Neighbours(
        counts=[[c[per, e].copy() for e in range(4)] for per in range(2)],
        ids=[[sl(ids, per * 4 + e) for e in range(4)] for per in range(2)],
        halos=[[sl(halos, per * 4 + e) for e in range(4)] for per in range(2)],
        starts=[[sl(starts, per * 4 + e) for e in range(4)] for per in range(2)],
    )


def partition(mask: np.ndarray, P: int, px: bool = False, py: bool = False, *, use_hist: bool = False,
              want_pid: bool = True, want_neighbours: bool = True) -> Decomposition:
    """The whole reference path on the CPU: mask[NY,NX] int32 -> boxes, pid, neighbours.

    P == 1 follows ZoltanPartitioner.cpp:102-121 (returns before discover_neighbours,
    so no neighbour lists at all, quirk Q4)."""
    mask = np.ascontiguousarray(mask, dtype=np.int32)
    NY, NX = mask.shape
    boxes = np.zeros((P, 4), dtype=np.int32)
    pid = np.empty((NY, NX), dtype=np.int32) if want_pid else None
    changes = C.c_int(0)
    iters = C.c_long(0)
    rc = lib().orc_partition(mask, NX, NY, P, int(use_hist), boxes.reshape(-1),
                             pid.ctypes.data if want_pid else None, C.byref(changes), C.byref(iters))
    if rc != 0:
        raise MemoryError("oracle allocation failed")
    d = Decomposition(NX, NY, P, boxes, pid, changes.value, iters.value)
    if want_neighbours:
        if P == 1:
            z = lambda: [[np.zeros(0, np.int32) for _ in range(4)] for _ in range(2)]
            d.nbr = Neighbours([[np.zeros(1, np.int32) for _ in range(4)] for _ in range(2)], z(), z(), z())
        else:
            d.nbr = neighbours(boxes, NX, NY, px, py)
    return d


def generate_mask(nx: int, ny: int, seed: int, land_frac: float, y_begin: int = 0, y_count: int | None = None) -> np.ndarray:
    """bench.py's synthetic land-sea mask (SURVEY 8d) without the CUDA library: rows [y_begin, y_begin + y_count)"""
    y_count = ny - y_begin if y_count is None else y_count
    out = np.empty((y_count, nx), dtype=np.int32)
    L = lib()
    L.orc_generate_mask.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_double]
    if L.orc_generate_mask(out.ctypes.data, nx, ny, y_begin, y_count, seed, float(land_frac)) != 0:
        raise ValueError("orc_generate_mask: bad arguments")
    return out


def part_loads(pid: np.ndarray, P: int) -> np.ndarray:
    loads = np.zeros(P, dtype=np.int64)
    flat = np.ascontiguousarray(pid, dtype=np.int32).reshape(-1)
    lib().orc_part_loads(flat, flat.size, P, loads)
    return loads
