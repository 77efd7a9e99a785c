"""Memory check of the kernels without a GPU: the host emulation (oracle/emu) built with AddressSanitizer and
UBSan.  Device "global memory" are heap arrays of the emulated driver and `__shared__` variables are statics, so
an out-of-bounds access of a kernel is an ASan report.  (compute-sanitizer, the GPU-side tool for this, is closed
on this GPU pool.)  The decomposition kernels run through oracle/libddc_emu_asan.so (tests/asan_worker.py), the halo
kernels through the halo harness built with the same sanitizers (tests/halo_asan_worker.py)."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def run_worker(extra_env=None, worker="asan_worker.py"):
    # the runtime of the compiler oracle/Makefile and tests/halo_emu.py build with (the distribution gcc when there is one)
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    asan = subprocess.run([cc, "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    if worker == "asan_worker.py":  # (the halo worker builds its harness itself)
        r = subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "libddc_emu_asan.so"], capture_output=True,
                           text=True)
        assert r.returncode == 0, r.stderr
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0:halt_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1")
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "tests", worker)], capture_output=True, text=True,
                          timeout=900, env=env)


def test_kernels_are_clean_under_address_sanitizer(oracle):
    oracle.build()
    out = run_worker()
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "ASAN RUN OK" in out.stdout
    assert "ERROR: AddressSanitizer" not in out.stderr and "runtime error:" not in out.stderr, out.stderr[-4000:]


def test_halo_kernels_are_clean_under_address_sanitizer(oracle):
    """scatter, edge and full exchange and gather on tilings with zero-width strips and zero-height parts: no kernel
    divides by a zero width or reads outside an allocation"""
    oracle.build()
    out = run_worker(worker="halo_asan_worker.py")
    assert "ERROR: AddressSanitizer" not in out.stderr and "runtime error:" not in out.stderr, out.stderr[-4000:]
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "HALO ASAN RUN OK" in out.stdout


def test_the_sanitizer_build_is_live(oracle):
    """a deliberate one-element overrun inside the library must be reported"""
    oracle.build()
    out = run_worker({"DDC_EMU_OOB_SELFTEST": "1"})
    assert out.returncode != 0 and "AddressSanitizer" in out.stderr
