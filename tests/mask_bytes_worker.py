"""Byte masks across GPUs: run under torchrun, one rank per GPU.

    torchrun --nproc-per-node 2 tests/mask_bytes_worker.py

The cases of tests/mgpu_worker.py (empty shards and an all-land mask included), over NCCL and over peer memory.  Every
rank first decomposes with its int32 shard, then with its shard as bytes, in two passes: all ranks on bytes, and
mixed (ranks of one parity on bytes, the others on int32, the parity alternating by case).  Every rank compares
everything it holds (boxes, its pid rows, stats, part loads, the eight neighbour lists) with its int32 run, bit for
bit.  --big adds C4 and C5 over peer memory, against the CPU oracle's digests."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from domain_decomp_b200 import capi, verify  # noqa: E402
import mask_bytes as MB  # noqa: E402
from mgpu_worker import CASES  # noqa: E402


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ids = [capi.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    h = capi.Handle(local, rank, world, ids[0])
    failures = 0
    rng = np.random.default_rng(rank)
    for mode in ("nccl", "peer"):
        if mode == "peer":
            handles = [None] * world
            dist.all_gather_object(handles, h.peer_export(4096, 4096, 1024))
            h.peer_import(handles)
        for ci, (nx, ny, P, land, seed, px, py) in enumerate(CASES):
            mask = capi.generate_mask_host(nx, ny, seed, land)
            yb, yc = capi.shard_rows(ny, world, rank)
            shard = np.ascontiguousarray(mask[yb:yb + yc]).reshape(yc, nx)
            b = MB.byte_mask(shard, rng)
            for mixed in (False, True):
                h.set_mask_host(shard, ny=ny, y_begin=yb)
                for rep in range(2):  # both parities of the double-buffered exchange
                    h.partition(P, bool(px), bool(py))
                a = MB.snapshot(h)
                if not mixed or (rank + ci) % 2 == 0:
                    h.set_mask_u8_host(b, ny=ny, y_begin=yb)
                for rep in range(2):
                    h.partition(P, bool(px), bool(py))
                u = MB.snapshot(h)
                try:
                    MB.assert_same(a, u)
                    ok = world == 1 or u["stats"]["exchange"] == (1 if mode == "nccl" else 2)
                except AssertionError:
                    ok = False
                print("rank %d/%d %s %s case %dx%d P=%d: %s" % (rank, world, mode, "mixed" if mixed else "u8", nx, ny, P,
                                                               "ok" if ok else "MISMATCH"), flush=True)
                failures += 0 if ok else 1
    if "--big" in sys.argv:
        with open(os.path.join(ROOT, "tests", "golden", "bench_digests.json")) as f:
            golden = json.load(f)
        dev = torch.device("cuda", local)
        for name in ("C4_8192x8192_p4096", "C5_32768x32768_p16384"):
            g = golden[name]
            nx, ny, P, px, py = g["nx"], g["ny"], g["parts"], bool(g["periodic_x"]), bool(g["periodic_y"])
            yb, yc = capi.shard_rows(ny, world, rank)
            d_mask = torch.empty((max(yc, 1), nx), dtype=torch.int32, device=dev)
            hh = capi.Handle(local, rank, world, None)
            handles = [None] * world
            dist.all_gather_object(handles, hh.peer_export(nx, ny, P))
            hh.peer_import(handles)
            hh.generate_mask_device(d_mask.data_ptr(), nx, ny, g["seed"], g["land_frac"], yb, yc)
            torch.cuda.synchronize()  # (the handle's stream is not torch's)
            hh.set_mask_device(d_mask.data_ptr(), nx, ny, yb, yc)
            hh.partition(P, px, py)
            hh.partition(P, px, py)
            a = MB.snapshot(hh, "device")
            d_u8 = d_mask[:yc] > 0
            torch.cuda.synchronize()
            hh.set_mask_u8_device(d_u8.data_ptr(), nx, ny, yb, yc)
            hh.partition(P, px, py)
            u = MB.snapshot(hh, "device")
            try:
                MB.assert_same(a, u)
                ok = verify.handle_digest(hh) == g["digest"] and (world == 1 or u["stats"]["exchange"] == 2)
            except AssertionError:
                ok = False
            print("rank %d/%d peer u8 case %s: %s" % (rank, world, name, "ok" if ok else "MISMATCH"), flush=True)
            failures += 0 if ok else 1
            del a, u
            hh.peer_close()
            dist.barrier()
            hh.close()
            del d_mask, d_u8
    t = torch.tensor([failures], device="cuda")
    dist.all_reduce(t)
    h.peer_close()
    dist.barrier()  # nobody frees its exchange buffer while a peer still has it mapped
    h.close()
    dist.destroy_process_group()
    if int(t.item()):
        sys.exit(1)
    if rank == 0:
        print("MASK BYTES MGPU OK world=%d" % world, flush=True)


if __name__ == "__main__":
    main()
