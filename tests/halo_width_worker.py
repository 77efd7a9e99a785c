"""The sharded halo calls with frames of width 2 and 3 (ddc_halo_set_width) across GPUs: run under torchrun, one rank
per GPU.

    torchrun --nproc-per-node G tests/halo_width_worker.py

Every rank decomposes the same synthetic masks with its row shard, holds the tiles of its parts in its own halo buffer
(ddc_halo_export, the IPC handles gathered through torch.distributed, ddc_halo_import) and runs, on one step counter,
ddc_halo_scatter_shards_f64 from its rows of a field, ddc_halo_exchange_full_shards_f64, ddc_halo_exchange_shards_f64,
ddc_halo_exchange_full_shards_f64 and ddc_halo_gather_shards_f64, at every width.  Every rank builds the same field from
a seed (random 64-bit patterns) and checks its own buffer after each call against halo_width's expectation and its
gathered rows at the end.  Prints "HALO WIDTH OK world=G" on success.
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import halo_width as hw  # noqa: E402
from domain_decomp_b200 import capi  # noqa: E402
from halo_shards_worker import CASES, _Dev, decompose  # noqa: E402
from halo_global import SENTINEL, random_bits  # noqa: E402

WIDTHS = (2, 3)


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
    elems = 0
    for (nx, ny, P, px, py, seed) in CASES:
        m = decompose(h, dev, world, rank, nx, ny, P, px, py, seed)
        elems = max(elems, hw.max_shard_total(h.boxes(), world, max(WIDTHS)))
        del m
    ptr, mine = h.halo_export(elems)
    handles = [None] * world
    dist.all_gather_object(handles, mine)
    h.halo_import(handles)
    failures = 0
    for (nx, ny, P, px, py, seed), w in [(c, w) for c in CASES for w in WIDTHS]:
        d_mask = decompose(h, dev, world, rank, nx, ny, P, px, py, seed)
        h.halo_set_width(w)
        boxes = h.boxes()
        off = hw.tile_offsets(boxes, w)
        h.halo_shard_offsets()
        b, c = capi.shard_parts(P, world, rank)
        sl = slice(int(off[b]), int(off[b + c]))
        n = sl.stop - sl.start
        view = torch.as_tensor(_Dev(ptr, n), device=dev).view(torch.int64) if n else None
        got = lambda: view.cpu().numpy().view(np.uint64) if view is not None else np.zeros(0, np.uint64)
        yb, yc = capi.shard_rows(ny, world, rank)
        ok = True
        for periodic in (0, 1):
            field = random_bits(np.random.default_rng(seed + 10 + periodic), nx * ny).reshape(ny, nx)
            rows = torch.from_numpy(field[yb:yb + yc].view(np.int64)).to(dev)
            if view is not None:
                view.fill_(int(SENTINEL.view(np.int64)))
            torch.cuda.synchronize()  # (no barrier between the ranks: k_halo_open is one)
            h.halo_scatter_shards_f64(rows.data_ptr() if yc else 0)
            h.synchronize()
            want = hw.scattered(boxes, off, field, np.full(int(off[-1]), SENTINEL, dtype=np.uint64), w)
            ok &= bool(np.array_equal(got(), want[sl]))
            for op in "fxf":
                (h.halo_exchange_full_shards_f64 if op == "f" else h.halo_exchange_shards_f64)(bool(periodic))
                h.synchronize()
                want = hw.exchanged(boxes, off, nx, ny, px, py, periodic, op == "f", field, want, w)
                ok &= bool(np.array_equal(got(), want[sl]))
            out = torch.full((yc, nx), 7, dtype=torch.int64, device=dev)
            torch.cuda.synchronize()
            h.halo_gather_shards_f64(out.data_ptr() if yc else 0)
            h.synchronize()
            ok &= bool(torch.equal(out, rows))
        print("rank %d/%d case %dx%d P=%d w=%d: %s" % (rank, world, nx, ny, P, w, "ok" if ok else "MISMATCH"), flush=True)
        failures += 0 if ok else 1
        del view, d_mask
    t = torch.tensor([failures], device=dev)
    dist.all_reduce(t)
    h.halo_close()
    dist.barrier()  # nobody frees a buffer while a peer still has it mapped
    h.close()
    dist.destroy_process_group()
    if int(t.item()):
        sys.exit(1)
    if rank == 0:
        print("HALO WIDTH OK world=%d" % world, flush=True)


if __name__ == "__main__":
    main()
