"""The byte-mask scan under AddressSanitizer + UBSan: decompositions on 1, 2 and 3 emulated ranks through the harness
tests/emu_mask_bytes.cpp built with the sanitizers (mask_bytes_emu.lib(True)).  Every rank's byte shard is an
allocation of exactly offset + rows * nx bytes, so a load past the last row's nx bytes is reported; the widths are not
multiples of 16, and cover both scan paths (nx % 4 == 0 with an aligned shard: 4-byte loads with the last group's lanes
re-reading the row's last 4 bytes; otherwise byte loads).  Started by test_mask_bytes_on_cpu_emulator.py with libasan
preloaded."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle.oracle as orc  # noqa: E402

import mask_bytes as MB  # noqa: E402
import mask_bytes_emu as E  # noqa: E402
from domain_decomp_b200 import capi  # noqa: E402

E.lib(sanitize=True)
rng = np.random.default_rng(7)
runs = 0
for nx, ny, P, ranks, offset in [(20, 37, 6, 1, 0), (100, 40, 12, 2, 0), (132, 33, 9, 3, 0), (67, 31, 7, 1, 0),
                                 (1001, 13, 10, 2, 0), (36, 50, 8, 2, 1), (44, 29, 5, 3, 2), (13, 7, 4, 2, 3),
                                 (4, 70, 3, 1, 0), (7, 2, 4, 3, 0)]:
    b = MB.byte_mask(capi.generate_mask_host(nx, ny, nx + ny, 0.45), rng)
    for rpc in (8, 64):
        d, _ = E.partition(orc, b, P, True, False, ranks=ranks, offset=offset, scan_rpc=rpc)
        o = orc.partition((b != 0).astype(np.int32), P, True, False, use_hist=True)
        assert d.boxes.tolist() == o.boxes.tolist() and np.array_equal(d.pid, o.pid), (nx, ny, P, ranks, offset)
        runs += 1
print("MASK BYTES ASAN RUN OK: %d decompositions" % runs)
