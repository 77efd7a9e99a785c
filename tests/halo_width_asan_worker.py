"""The halo kernels with frames of width 2 and 3 under AddressSanitizer + UBSan: scatter, edge exchange, full exchange,
edge exchange and gather ('sxfxg') on one step counter, through the harness tests/emu_halo_width.cpp built with the
sanitizers (halo_width_emu.lib(True)), on the degenerate tilings and on RCB output with empty parts, for 1, 2 and 3
emulated ranks.  Started by test_halo_width_on_cpu_emulator.py with libasan preloaded; what ASan can and cannot see in the
harness's layout is said in tests/halo_asan_worker.py.  Every rank's buffer is sized for the wide layout, so a
rectangle item that addresses a tile of the wrong width is reported."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle.oracle as orc  # noqa: E402

import halo_frame as hf  # noqa: E402
import halo_global as hg  # noqa: E402
import halo_width as hw  # noqa: E402
import halo_width_emu  # noqa: E402

halo_width_emu.lib(sanitize=True)
todo = [(b, nbr, nx, ny, px, py, seed) for b, nbr, nx, ny, px, py, seed in hf.degenerate_cases(orc)]
todo += [(d.boxes, d.nbr, nx, ny, px, py, seed) for d, nx, ny, px, py, seed in hg.empty_part_cases(orc)]
runs = 0
for w in (2, 3):
    for G in (1, 2, 3):
        for boxes, nbr, nx, ny, px, py, seed in todo:
            rng = np.random.default_rng(seed)
            off = hw.tile_offsets(boxes, w)
            field = hg.random_bits(rng, nx * ny).reshape(ny, nx)
            run = halo_width_emu.run(boxes, nbr, nx, ny, px, py, G, 1, "sxfxg",
                                     np.full(int(off[-1]), hg.SENTINEL, np.uint64), [field], hg.random_bits(rng, nx * ny),
                                     w=w)
            assert run.err.tolist() == [0] * G, (w, G, seed)
            assert run.rows[-1].tobytes() == field.tobytes(), (w, G, seed)
            runs += 1
print("HALO WIDTH ASAN RUN OK: %d runs" % runs)
