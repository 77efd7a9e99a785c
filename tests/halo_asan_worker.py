"""The halo kernels under AddressSanitizer + UBSan: scatter, edge exchange, full exchange, edge exchange and gather
('sxfxg') on one step counter, through the harness tests/emu_halo.cpp built with the sanitizers (halo_emu.lib(True)),
on the degenerate tilings and on RCB output with empty parts, for 1, 2 and 3 emulated ranks, at every frame width given
on the command line (default: 1).  Started by test_kernels_asan.py (w = 1) and test_halo_width_on_cpu_emulator.py
(w = 2 and 3) with libasan preloaded.

What the harness's layout lets ASan see: the boxes, the neighbour lists and the halo plan are allocations of their own,
and so is every rank's halo buffer ([head][the rank's tiles], then at most 32 doubles of alignment slack), so an access
past a table or past a rank's buffer is reported.  Every rank's buffer is sized for the width, so a rectangle item that
addresses a tile of the wrong width is reported too.  What it does not see: the single buffer holds every tile in one
allocation, so a read past a tile that stays inside that buffer lands in another tile and is not seen; the same holds
between the tiles of one rank's buffer and for the head in front of its first tile.  Wrong values there are for the
emulator tests, which compare every cell, to find.  UBSan reports integer division by zero and overflow, and shifts out
of range."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle.oracle as orc  # noqa: E402

import halo_emu  # noqa: E402
import halo_frame as hf  # noqa: E402
import halo_global as hg  # noqa: E402
import halo_width as hw  # noqa: E402

widths = [int(a) for a in sys.argv[1:]] or [1]
halo_emu.lib(sanitize=True)
todo = [(b, nbr, nx, ny, px, py, seed) for b, nbr, nx, ny, px, py, seed in hf.degenerate_cases(orc)]
todo += [(d.boxes, d.nbr, nx, ny, px, py, seed) for d, nx, ny, px, py, seed in hg.empty_part_cases(orc)]
runs = 0
for w in widths:
    for G in (1, 2, 3):
        for boxes, nbr, nx, ny, px, py, seed in todo:
            rng = np.random.default_rng(seed)
            off = hw.tile_offsets(boxes, w)
            field = hg.random_bits(rng, nx * ny).reshape(ny, nx)
            run = halo_emu.run(boxes, nbr, nx, ny, px, py, G, 1, "sxfxg", np.full(int(off[-1]), hg.SENTINEL, np.uint64),
                               [field], hg.random_bits(rng, nx * ny), w=w)
            assert run.err.tolist() == [0] * G, (w, G, seed)
            assert run.rows[-1].tobytes() == field.tobytes(), (w, G, seed)
            runs += 1
print("HALO ASAN RUN OK: %d runs at widths %s" % (runs, widths))
