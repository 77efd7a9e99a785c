"""Byte masks on emulated ranks (tests/emu_mask_bytes.cpp) and through the C ABI on the emulated runtime, for the CPU
suite.

The harness is compiled on first use into a temporary directory, like tests/halo_emu.py: the product's ddc_kernels.cuh as
host C++ (-DDDC_HOST_EMU), the multi-rank pipeline of oracle/emu/emu_pipeline.cpp and the fiber emulation of the CUDA
execution model.  `partition` runs through oracle.emu_partition, with this library in place of oracle/libddc_emu.so for
the duration of the call."""
import atexit
import contextlib
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


def lib(sanitize=False) -> C.CDLL:
    """the harness, compiled on the first call; later calls return it whatever they ask.  sanitize: built with
    AddressSanitizer + UBSan, for a process that has libasan preloaded (tests/mask_bytes_asan_worker.py)."""
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="ddc_emu_u8_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libddc_emu_u8.so")
        emu = os.path.join(ROOT, "oracle", "emu")
        flags = ["-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"] if sanitize else ["-O2"]
        env = {k: v for k, v in os.environ.items() if k != "LD_PRELOAD"}  # (the compiler runs without libasan)
        subprocess.check_call([_compiler()] + flags + ["-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
                               "-ffp-contract=off", "-U_FORTIFY_SOURCE", "-DDDC_HOST_EMU",
                               "-I" + os.path.join(ROOT, "domain_decomp_b200", "csrc"), "-I" + os.path.join(ROOT, "include"),
                               "-I" + emu, "-o", so, os.path.join(ROOT, "tests", "emu_mask_bytes.cpp"),
                               os.path.join(emu, "cuda_emu.cpp")], env=env)
        L = C.CDLL(so)
        i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
        L.emu_partition.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    i32p, i32p, i32p, i32p, C.c_long, np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")]
        L.emu_partition.restype = C.c_int
        L.emu_last_error.restype = C.c_char_p
        L.emu_set_byte_mask.argtypes = [np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS"), C.c_int, C.c_int, C.c_int,
                                        C.c_uint, C.c_int]
        L.emu_set_byte_mask.restype = C.c_int
        _lib = L
    return _lib


@contextlib.contextmanager
def _harness(orc):
    saved = orc._emu
    orc._emu = lib()
    try:
        yield
    finally:
        orc._emu = saved


def partition(orc, m, P, px=False, py=False, *, ranks=1, u8_ranks=None, offset=0, **kw):
    """oracle.emu_partition on `ranks` emulated ranks; the ranks in u8_ranks (default: all) scan the byte mask
    m.view(uint8) at `offset` bytes into their shard's allocation, the others scan (m != 0) as int32."""
    m = np.ascontiguousarray(m)
    b = m.view(np.uint8) if m.dtype == np.bool_ else np.ascontiguousarray(m, dtype=np.uint8)
    ny, nx = b.shape
    sel = sum(1 << g for g in (range(ranks) if u8_ranks is None else u8_ranks))
    L = lib()
    assert L.emu_set_byte_mask(b.reshape(-1), nx, ny, ranks, sel, offset) == 0
    try:
        with _harness(orc):
            return orc.emu_partition((b != 0).astype(np.int32), P, px, py, ranks=ranks, **kw)
    finally:
        L.emu_set_byte_mask(b.reshape(-1), nx, ny, 1, 0, 0)  # free the shards
