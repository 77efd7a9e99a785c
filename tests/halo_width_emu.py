"""The halo calls with frames of width w (tests/emu_halo_width.cpp) on emulated ranks, for the CPU suite.

The harness is compiled on first use into a temporary directory, as tests/halo_emu.py compiles tests/emu_halo.cpp: the
product's ddc_kernels.cuh as host C++ (-DDDC_HOST_EMU) plus the fiber emulation of the CUDA execution model
(oracle/emu/cuda_emu.cpp).  run() takes and returns what halo_emu.run() does, plus the width."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import halo_emu
import halo_global as hg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def lib(sanitize=False) -> C.CDLL:
    """the harness, compiled on the first call; later calls return it whatever they ask.  sanitize: built with
    AddressSanitizer + UBSan, for a process that has libasan preloaded (tests/halo_width_asan_worker.py)."""
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="ddc_emu_halo_width_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libddc_emu_halo_width.so")
        emu = os.path.join(ROOT, "oracle", "emu")
        flags = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"] if sanitize else ["-O2"]
        env = {k: v for k, v in os.environ.items() if k != "LD_PRELOAD"}  # (the compiler runs without libasan)
        subprocess.check_call([halo_emu._compiler()] + flags + ["-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
                               "-ffp-contract=off", "-U_FORTIFY_SOURCE", "-DDDC_HOST_EMU",
                               "-I" + os.path.join(ROOT, "domain_decomp_b200", "csrc"), "-I" + os.path.join(ROOT, "include"),
                               "-I" + emu, "-o", so, os.path.join(ROOT, "tests", "emu_halo_width.cpp"),
                               os.path.join(emu, "cuda_emu.cpp")], env=env)
        L = C.CDLL(so)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
        L.emu_halo_width.argtypes = [C.c_int, i32p, i32p, i32p, i32p, i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     i32p, i32p, C.c_int, C.c_char_p, C.c_int, C.c_int, f64p, f64p, f64p, f64p, f64p,
                                     f64p, f64p, i32p, i32p, i32p, C.c_int]
        L.emu_halo_width.restype = C.c_int
        L.emu_halo_width_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def run(boxes, nbr, nx, ny, px, py, G, periodic, ops, tiles_in, fields=(), rows_in=None, stall=-1, grid_cap=4, w=1):
    """run `ops` ('s' scatter, 'x' edge exchange, 'f' full-frame exchange, 'g' gather) with frames of width w on G
    emulated ranks and on one buffer; the arguments and the result are those of halo_emu.run, and tiles_in is in the
    layout of width w"""
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
    rc = L.emu_halo_width(P, boxes.reshape(-1), counts, cat(nbr.ids), cat(nbr.halos), cat(nbr.starts), nx, ny, int(px),
                          int(py), G, np.array([b for b, _ in rows], dtype=np.int32),
                          np.array([c for _, c in rows], dtype=np.int32), int(periodic), ops.encode(), stall, grid_cap,
                          as_f64(fields), as_f64(tiles_in), as_f64(rows_in), tiles, single, out_rows, out_field, err, ids,
                          starts, int(w))
    if rc != 0:
        raise RuntimeError("emu_halo_width: " + L.emu_halo_width_last_error().decode())
    u = lambda a, m: a.view(np.uint64).reshape(n, m)
    return halo_emu.Run(u(tiles, total), u(single, total), u(out_rows, nx * ny), u(out_field, nx * ny), err,
                        ids.reshape(2, 4, P), starts.reshape(2, 4, P))
