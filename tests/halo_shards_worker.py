"""Sharded halo exchange across GPUs: run under torchrun, one rank per GPU.

    torchrun --nproc-per-node G tests/halo_shards_worker.py

Every rank decomposes the same synthetic masks with its row shard (ddc_partition; the histograms exchanged through
NCCL, then through peer memory), holds the tiles of its parts [r P / G, (r + 1) P / G) in its own halo buffer
(ddc_halo_export, the IPC handles gathered through torch.distributed, ddc_halo_import) and runs
ddc_halo_exchange_shards_f64.  Interiors hold the global cell index; each rank checks its own buffer against the
expected tiles (tests/halo_global.py) after every exchange.  Prints "HALO SHARDS OK world=G" on success.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import halo_global as hg  # noqa: E402
from domain_decomp_b200 import capi  # noqa: E402

CASES = [  # nx, ny, P, px, py, seed
    (528, 522, 64, 1, 1, 25),
    (2048, 1536, 1000, 1, 0, 7),
    (8192, 8192, 4096, 0, 0, 3),
]


class _Dev:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (int(ptr), False), "version": 2,
                                         "strides": None}


def decompose(h, dev, world, rank, nx, ny, P, px, py, seed):
    yb, yc = capi.shard_rows(ny, world, rank)
    d_mask = torch.empty((max(yc, 1), nx), dtype=torch.int32, device=dev)
    h.generate_mask_device(d_mask.data_ptr(), nx, ny, seed, 0.45, yb, yc)
    h.set_mask_device(d_mask.data_ptr(), nx, ny, yb, yc)
    h.partition(P, bool(px), bool(py))
    h.synchronize()
    return d_mask


def main():
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ids = [capi.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    h = capi.Handle(local, rank, world, ids[0])
    # the buffers must hold the largest rank's tiles of every case (the boxes are replicated: every rank knows them)
    elems = 0
    for (nx, ny, P, px, py, seed) in CASES:
        m = decompose(h, dev, world, rank, nx, ny, P, px, py, seed)
        elems = max(elems, hg.max_shard_total(h.boxes(), world))
        del m
    ptr, mine = h.halo_export(elems)
    handles = [None] * world
    dist.all_gather_object(handles, mine)
    h.halo_import(handles)
    failures = 0
    for mode in ("nccl", "peer"):
        if mode == "peer":
            handles = [None] * world
            dist.all_gather_object(handles, h.peer_export(8192, 8192, 4096))
            h.peer_import(handles)
        for (nx, ny, P, px, py, seed) in CASES:
            d_mask = decompose(h, dev, world, rank, nx, ny, P, px, py, seed)
            boxes = h.boxes()
            off = hg.tile_offsets(boxes)
            b, c = capi.shard_parts(P, world, rank)
            ok = h.halo_shard_offsets().tolist() == (off[b:b + c + 1] - off[b]).tolist()
            ok &= h.stats()["exchange"] == (1 if mode == "nccl" else 2)
            sl = slice(int(off[b]), int(off[b + c]))
            n = sl.stop - sl.start
            view = torch.as_tensor(_Dev(ptr, n), device=dev) if n else None
            step = 0
            for periodic in (0, 1):
                for k in range(2):
                    add = 1000.0 * step
                    step += 1
                    fresh = torch.from_numpy(hg.initial_tiles(boxes, off, nx, add)[sl]).to(dev)
                    if view is not None:
                        view.copy_(fresh if k == 0 else torch.where(fresh != hg.UNTOUCHED, fresh, view))
                    torch.cuda.synchronize()  # (no barrier between the ranks: k_halo_open is one)
                    h.halo_exchange_shards_f64(bool(periodic))
                    h.synchronize()
                    want = hg.expected_tiles(boxes, off, nx, ny, px, py, periodic, add)[sl]
                    got = view.cpu().numpy() if view is not None else np.zeros(0)
                    ok &= bool(np.array_equal(got, want))
            print("rank %d/%d %s case %dx%d P=%d: %s" % (rank, world, mode, nx, ny, P, "ok" if ok else "MISMATCH"),
                  flush=True)
            failures += 0 if ok else 1
            del view, d_mask
    t = torch.tensor([failures], device=dev)
    dist.all_reduce(t)
    h.halo_close()
    h.peer_close()
    dist.barrier()  # nobody frees a buffer while a peer still has it mapped
    h.close()
    dist.destroy_process_group()
    if int(t.item()):
        sys.exit(1)
    if rank == 0:
        print("HALO SHARDS OK world=%d" % world, flush=True)


if __name__ == "__main__":
    main()
