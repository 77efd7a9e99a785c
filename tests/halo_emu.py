"""The halo calls' kernels and host code on emulated ranks (tests/emu_halo.cpp), and the C ABI on the emulated runtime,
for the CPU suite.

The harness is compiled on first use, like the emulation libraries of oracle/emu it builds on: the product's
ddc_kernels.cuh as host C++ (-DDDC_HOST_EMU) plus the fiber emulation of the CUDA execution model
(oracle/emu/cuda_emu.cpp).  The library goes to a temporary directory, so the tree stays as it is."""
import atexit
import collections
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import halo_global as hg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None

# what run() returns: per op, the sharded tiles (concatenated in rank order), the single buffer, the gathered rows and
# the single-buffer field, all as uint64; the error word of every rank; the corner table [2, 4, P]
Run = collections.namedtuple("Run", "tiles single rows field err ids starts")


def _compiler():
    for cand in ("/usr/bin/g++", shutil.which("g++"), shutil.which("c++")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("no C++ compiler for the emulation harness")


def lib(sanitize=False) -> C.CDLL:
    """the harness, compiled on the first call; later calls return it whatever they ask.  sanitize: built with
    AddressSanitizer + UBSan, for a process that has libasan preloaded (tests/halo_asan_worker.py)."""
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="ddc_emu_halo_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libddc_emu_halo.so")
        emu = os.path.join(ROOT, "oracle", "emu")
        flags = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"] if sanitize else ["-O2"]
        env = {k: v for k, v in os.environ.items() if k != "LD_PRELOAD"}  # (the compiler runs without libasan)
        subprocess.check_call([_compiler()] + flags + ["-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
                               "-ffp-contract=off", "-U_FORTIFY_SOURCE", "-DDDC_HOST_EMU",
                               "-I" + os.path.join(ROOT, "domain_decomp_b200", "csrc"), "-I" + os.path.join(ROOT, "include"),
                               "-I" + emu, "-o", so, os.path.join(ROOT, "tests", "emu_halo.cpp"),
                               os.path.join(emu, "cuda_emu.cpp")], env=env)
        L = C.CDLL(so)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
        L.emu_halo.argtypes = [C.c_int, i32p, i32p, i32p, i32p, i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               i32p, i32p, C.c_int, C.c_char_p, C.c_int, C.c_int, f64p, f64p, f64p, f64p, f64p, f64p, f64p,
                               i32p, i32p, i32p, C.c_int]
        L.emu_halo.restype = C.c_int
        L.emu_halo_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def run(boxes, nbr, nx, ny, px, py, G, periodic, ops, tiles_in, fields=(), rows_in=None, stall=-1, grid_cap=4, w=1):
    """run `ops` ('s' scatter, 'x' edge exchange, 'f' full-frame exchange, 'g' gather) with frames of width w on G
    emulated ranks and on one buffer.  boxes / nbr: a decomposition (oracle.partition's boxes and nbr); tiles_in: the
    tiles before the first op, in the layout of width w; fields: one field [ny, nx] per 's', in order (more are ignored);
    rows_in: what the rows hold before the first op (zeros by default).  Arrays are passed as their 64-bit patterns.
    stall: a rank that runs none of the kernels.  grid_cap: at most that many blocks for the grid-stride kernels, 0 the
    library's grids."""
    L = lib()
    boxes = np.ascontiguousarray(boxes, dtype=np.int32)
    P = len(boxes)
    lists = [(per, e) for per in range(2) for e in range(4)]
    cat = lambda a: np.ascontiguousarray(np.concatenate([a[per][e] for per, e in lists] + [np.zeros(1, np.int32)]),
                                         dtype=np.int32)
    counts = np.ascontiguousarray(np.concatenate([nbr.counts[per][e] for per, e in lists]), dtype=np.int32)
    rows = hg.shard_rows(ny, G)
    bits = lambda a: np.ascontiguousarray(a).reshape(-1).view(np.uint64)
    as_f64 = lambda a: np.ascontiguousarray(a).reshape(-1).view(np.float64)
    if ops.count("s") > len(fields):
        raise ValueError("one field per scatter")
    fields = np.concatenate([bits(f) for f in fields] + [np.zeros(0, np.uint64)])
    tiles_in = bits(tiles_in)
    rows_in = np.zeros(nx * ny, np.uint64) if rows_in is None else bits(rows_in)
    total, n = int(tiles_in.size), len(ops)
    tiles, single = np.zeros(n * total), np.zeros(n * total)
    out_rows, out_field = np.zeros(n * nx * ny), np.zeros(n * nx * ny)
    err = np.zeros(G, dtype=np.int32)
    ids, starts = np.zeros(8 * P, dtype=np.int32), np.zeros(8 * P, dtype=np.int32)
    rc = L.emu_halo(P, boxes.reshape(-1), counts, cat(nbr.ids), cat(nbr.halos), cat(nbr.starts), nx, ny, int(px), int(py),
                    G, np.array([b for b, _ in rows], dtype=np.int32), np.array([c for _, c in rows], dtype=np.int32),
                    int(periodic), ops.encode(), stall, grid_cap, as_f64(fields), as_f64(tiles_in), as_f64(rows_in),
                    tiles, single, out_rows, out_field, err, ids, starts, int(w))
    if rc != 0:
        raise RuntimeError("emu_halo: " + L.emu_halo_last_error().decode())
    u = lambda a, m: a.view(np.uint64).reshape(n, m)
    return Run(u(tiles, total), u(single, total), u(out_rows, nx * ny), u(out_field, nx * ny), err,
               ids.reshape(2, 4, P), starts.reshape(2, 4, P))


def emu_capi(oracle):
    """domain_decomp_b200.capi bound to oracle/libddc_cuda_emu.so (as in test_c_abi_on_cpu_emulator)"""
    import test_c_abi_on_cpu_emulator as A
    from domain_decomp_b200 import capi as real
    oracle.build()
    lib = C.CDLL(os.path.join(ROOT, "oracle", "libddc_cuda_emu.so"))
    ref = real.load()
    for name in real.SYMBOLS:
        getattr(lib, name).argtypes = getattr(ref, name).argtypes
        getattr(lib, name).restype = getattr(ref, name).restype
    return A.EmuCapi(real, lib)
