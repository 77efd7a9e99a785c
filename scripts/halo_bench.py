#!/usr/bin/env python
"""Time the halo exchanges on the BASELINE decompositions C4 (8192^2 -> 4096 parts) and C5 (32768^2 -> 16384, px).

    python scripts/halo_bench.py --out result.json                   # one GPU
    torchrun --nproc-per-node G scripts/halo_bench.py --out r.json    # G GPUs, one process each

One GPU: ddc_halo_exchange_f64 on one buffer against ddc_halo_exchange_shards_f64 with one rank (the same ghost
cells, plus the open / close barriers of the sharded protocol), alternated in rounds.  G GPUs: the sharded exchange
over CUDA IPC, time per exchange = the slowest rank's.  Times are CUDA events around `--iters` back-to-back
exchanges after `--warmup` (enqueue included: it is what a caller pays).  Exchanges are periodic (the periodic lists
are used where the decomposition has them).  Ghost cells moved come from the neighbour tables: a cell is read once
(8 B) and written once (8 B); "cross-rank" cells are written into another rank's buffer.  The GPU name and power
limit are read in the same run.  Writes JSON to --out (and prints it); nothing in the tree."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from domain_decomp_b200 import capi  # noqa: E402

CONFIGS = {  # tests/golden/bench_digests.json
    "C4": dict(nx=8192, ny=8192, parts=4096, seed=1, land_frac=0.6, px=0, py=0),
    "C5": dict(nx=32768, ny=32768, parts=16384, seed=32, land_frac=0.45, px=1, py=0),
}


def gpu_info(dev):
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(dev)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:  # (a missing nvidia-smi does not stop the measurement)
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def ghost_counts(h, P, G, periodic):
    """ghost cells one exchange writes: (all, written into another rank's buffer)"""
    owner = lambda p: ((p + 1) * G - 1) // P
    total = cross = 0
    for per in range(2 if periodic else 1):
        for e in range(4):
            counts = h.neighbour_counts(e, per)
            ids, halos, _ = h.neighbours(e, per)
            recv = np.repeat(np.arange(P, dtype=np.int64), counts)  # the part whose ghosts the entry fills
            total += int(halos.sum())
            cross += int(halos[owner(recv) != owner(ids.astype(np.int64))].sum())
    return total, cross


def timed(fn, stream, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(iters):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / iters


def decompose(h, dev, cfg, world, rank):
    nx, ny = cfg["nx"], cfg["ny"]
    yb, yc = capi.shard_rows(ny, world, rank)
    d_mask = torch.empty((max(yc, 1), nx), dtype=torch.int32, device=dev)
    h.generate_mask_device(d_mask.data_ptr(), nx, ny, cfg["seed"], cfg["land_frac"], yb, yc)
    h.set_mask_device(d_mask.data_ptr(), nx, ny, yb, yc)
    h.partition(cfg["parts"], bool(cfg["px"]), bool(cfg["py"]))
    h.synchronize()
    return d_mask


def row(name, cfg, G, ms, cells, cross):
    bytes_moved = 16 * cells  # 8 B read + 8 B written per ghost cell
    return dict(config=name, nx=cfg["nx"], ny=cfg["ny"], parts=cfg["parts"], ranks=G, ms_per_exchange=round(ms, 5),
                ghost_cells=cells, ghost_cells_local=cells - cross, ghost_cells_cross_rank=cross,
                bytes_read=8 * cells, bytes_written=8 * cells,
                achieved_GBps=round(bytes_moved / (ms * 1e-3) / 1e9, 1))


def one_gpu(args):
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)  # (a stream of its own: 0 would hand the handle back its internal stream)
    results = []
    for name in args.configs:
        cfg = CONFIGS[name]
        h = capi.Handle(0)
        h.set_stream(stream.cuda_stream)
        d_mask = decompose(h, dev, cfg, 1, 0)
        del d_mask
        P = cfg["parts"]
        off = h.halo_tile_offsets()
        single = torch.zeros(int(off[-1]), dtype=torch.float64, device=dev)
        (ptr,) = capi.halo_connect([h], int(off[-1]))
        h.halo_shard_offsets()
        cells, cross = ghost_counts(h, P, 1, True)
        variants = {"single_buffer": lambda: h.halo_exchange_f64(single.data_ptr(), True),
                    "sharded_G1": lambda: h.halo_exchange_shards_f64(True)}
        for fn in variants.values():
            timed(fn, stream, args.warmup)
        samples = {k: [] for k in variants}
        for _ in range(args.rounds):  # alternated: the two share whatever else the machine does
            for k, fn in variants.items():
                samples[k].append(timed(fn, stream, args.iters))
        h.synchronize()
        for k in variants:
            r = row(name, cfg, 1, float(np.median(samples[k])), cells, cross)
            r.update(variant=k, samples_ms=[round(s, 5) for s in samples[k]], iters=args.iters)
            results.append(r)
            print(json.dumps(r), flush=True)
        h.halo_close()
        h.close()
        del single
        torch.cuda.empty_cache()
    return results


def multi_gpu(args):
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(dev)
    results = []
    for name in args.configs:
        cfg = CONFIGS[name]
        h = capi.Handle(local, rank, world, None)
        handles = [None] * world
        dist.all_gather_object(handles, h.peer_export(cfg["nx"], cfg["ny"], cfg["parts"]))
        h.peer_import(handles)
        h.set_stream(stream.cuda_stream)
        d_mask = decompose(h, dev, cfg, world, rank)
        del d_mask
        P = cfg["parts"]
        off = h.halo_tile_offsets()
        elems = max(int(off[(r + 1) * P // world] - off[r * P // world]) for r in range(world))
        ptr, mine = h.halo_export(elems)
        handles = [None] * world
        dist.all_gather_object(handles, mine)
        h.halo_import(handles)
        h.halo_shard_offsets()
        cells, cross = ghost_counts(h, P, world, True)
        fn = lambda: h.halo_exchange_shards_f64(True)
        timed(fn, stream, args.warmup)
        samples = []
        for _ in range(args.rounds):
            dist.barrier()
            samples.append(timed(fn, stream, args.iters))
        t = torch.tensor(samples, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # per round: the slowest rank
        r = row(name, cfg, world, float(np.median(t.cpu().numpy())), cells, cross)
        r.update(variant="sharded", samples_ms=[round(float(s), 5) for s in t.cpu()], iters=args.iters)
        results.append(r)
        if rank == 0:
            print(json.dumps(r), flush=True)
        h.halo_close()
        h.peer_close()
        dist.barrier()
        h.close()
        torch.cuda.empty_cache()
    dist.destroy_process_group()
    return results if rank == 0 else None


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", nargs="+", default=["C4", "C5"], choices=sorted(CONFIGS))
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("halo_bench: no CUDA device (there is nothing to measure without one)")
    t0 = time.time()
    results = multi_gpu(args) if "WORLD_SIZE" in os.environ else one_gpu(args)
    if results is None:
        return
    doc = dict(gpu_info(0), ranks=int(os.environ.get("WORLD_SIZE", "1")), results=results,
               wall_s=round(time.time() - t0, 1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
