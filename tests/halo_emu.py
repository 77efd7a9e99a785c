"""The sharded halo exchange's kernels on emulated ranks (tests/emu_halo_shards.cpp), for the CPU suite.

The harness is compiled on first use, like the emulation libraries of oracle/emu it builds on: the product's
ddc_kernels.cuh as host C++ (-DDDC_HOST_EMU) plus the fiber emulation of the CUDA execution model
(oracle/emu/cuda_emu.cpp).  The library goes to a temporary directory, so the tree stays as it is."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def _compiler():
    for cand in ("/usr/bin/g++", shutil.which("g++"), shutil.which("c++")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("no C++ compiler for the emulation harness")


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="ddc_emu_halo_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libddc_emu_halo.so")
        emu = os.path.join(ROOT, "oracle", "emu")
        subprocess.check_call([_compiler(), "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
                               "-ffp-contract=off", "-U_FORTIFY_SOURCE", "-DDDC_HOST_EMU",
                               "-I" + os.path.join(ROOT, "domain_decomp_b200", "csrc"), "-I" + os.path.join(ROOT, "include"),
                               "-I" + emu, "-o", so, os.path.join(ROOT, "tests", "emu_halo_shards.cpp"),
                               os.path.join(emu, "cuda_emu.cpp")])
        L = C.CDLL(so)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
        L.emu_halo_shards.argtypes = [C.c_int, i32p, i32p, i32p, i32p, i32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      f64p, f64p, f64p, i32p]
        L.emu_halo_shards.restype = C.c_int
        L.emu_halo_last_error.restype = C.c_char_p
        _lib = L
    return _lib


def emu_halo_shards(d, ranks: int, periodic: bool, tiles_in: np.ndarray, stall: int = -1):
    """The sharded halo exchange (k_halo_open / k_halo_push / k_halo_close) of decomposition `d` (oracle.partition)
    on `ranks` emulated ranks, one exchange per row of tiles_in [nsteps, total] (interiors copied in before each; whole
    tiles before the first), with k_halo_exchange on one buffer beside it.  stall: a rank that runs none of the kernels.
    Returns (sharded [nsteps, total], single [nsteps, total], error word per rank)."""
    L = lib()
    tiles_in = np.ascontiguousarray(tiles_in, dtype=np.float64)
    lists = [(per, e) for per in range(2) for e in range(4)]
    cat = lambda a: np.ascontiguousarray(np.concatenate([a[per][e] for per, e in lists] + [np.zeros(1, np.int32)]),
                                         dtype=np.int32)
    counts = np.ascontiguousarray(np.concatenate([d.nbr.counts[per][e] for per, e in lists]), dtype=np.int32)
    out = np.zeros_like(tiles_in)
    single = np.zeros_like(tiles_in)
    err = np.zeros(ranks, dtype=np.int32)
    rc = L.emu_halo_shards(d.P, np.ascontiguousarray(d.boxes, dtype=np.int32).reshape(-1), counts, cat(d.nbr.ids),
                           cat(d.nbr.halos), cat(d.nbr.starts), ranks, int(periodic), tiles_in.shape[0], stall, tiles_in,
                           out, single, err)
    if rc != 0:
        raise RuntimeError("emu_halo_shards: " + L.emu_halo_last_error().decode())
    return out, single, err
