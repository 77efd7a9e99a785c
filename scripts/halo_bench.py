#!/usr/bin/env python
"""Time the halo exchanges, scatters and gathers on the BASELINE decompositions C4 (8192^2 -> 4096 parts) and C5
(32768^2 -> 16384, px).

    python scripts/halo_bench.py --out result.json                   # one GPU
    torchrun --nproc-per-node G scripts/halo_bench.py --out r.json    # G GPUs, one process each
    python scripts/halo_bench.py --widths 1 2 4 --out result.json    # frames of width 1, 2 and 4 (ddc_halo_set_width)

One GPU: ddc_halo_exchange_f64 on one buffer against ddc_halo_exchange_shards_f64 with one rank (the same ghost
cells, plus the open / close barriers of the sharded protocol), the full-frame exchanges (ddc_halo_exchange_full_f64 /
_full_shards_f64: the same plus the corner ghosts), and ddc_halo_scatter_f64 / ddc_halo_gather_f64 against their
sharded forms with one rank, all alternated in rounds.  The host time of ddc_halo_tile_offsets (which also builds the
corner items) and of one ddc_get_corner_neighbours (the corner table alone) is reported per configuration.  G GPUs: the sharded calls over CUDA IPC, time per call =
the slowest rank's.  Times are CUDA events around `--iters` back-to-back calls after `--warmup` (enqueue included: it
is what a caller pays).  Exchanges are periodic (the periodic lists are used where the decomposition has them).  Ghost
cells moved come from the neighbour tables: a cell is read once (8 B) and written once (8 B); "cross-rank" cells are
written into another rank's buffer.  Scatter and gather move every cell of the field (nx ny cells, 8 B read + 8 B
written each); their "cross-rank" cells are those whose row (ddc_shard_rows) and part (ddc_shard_parts) belong to
different ranks.  Rates are compared with the 6546.9 GB/s of a read+write copy measured on a B200 (DESIGN.md 4).  The
GPU name and power limit are read in the same run.  --widths: every call and the host time of ddc_halo_tile_offsets
are measured at each frame width (default 1), every row says its width; one halo buffer, sized for the widest frame,
serves all widths.  Ghost cells at w >= 2 are counted from the boxes by the source rule of ddc.h (the decompositions
tile the domain, so a frame cell has a source unless it lies across a non-periodic edge), cross-rank ones only with one
rank (0).  Writes JSON to --out (and prints it); nothing in the tree."""
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

COPY_GBPS = 6546.9  # a read+write device copy on a B200 (MEASURED_PEAKS.json:hbm_gbs, DESIGN.md 4)
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


def corner_counts(h, P, G, periodic):
    """corner ghosts one full-frame exchange writes: (all, written into another rank's buffer)"""
    owner = lambda p: ((p + 1) * G - 1) // P
    total = cross = 0
    for per in range(2 if periodic else 1):
        for c in range(4):
            ids, _ = h.corner_neighbours(c, per)
            has = ids >= 0
            total += int(has.sum())
            cross += int((owner(ids[has].astype(np.int64)) != owner(np.nonzero(has)[0])).sum())
    return total, cross


def wide_counts(boxes, nx, ny, px, py, w):
    """(edge-strip ghosts, corner-block ghosts) one periodic exchange of width w fills: a frame cell of a tiling has a
    source unless it lies across a non-periodic domain edge"""
    b = np.asarray(boxes, dtype=np.int64)
    x0, y0, ex, ey = b[:, 0], b[:, 1], np.maximum(b[:, 2], 0), np.maximum(b[:, 3], 0)
    cx = np.where(px, w, np.minimum(w, x0)) + np.where(px, w, np.minimum(w, nx - x0 - ex))  # columns left + right
    cy = np.where(py, w, np.minimum(w, y0)) + np.where(py, w, np.minimum(w, ny - y0 - ey))  # rows below + above
    return int((cx * ey + cy * ex).sum()), int((cx * cy).sum())


def host_ms(fn, reps=5):
    """median host time of fn() in ms"""
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return round(float(np.median(t)), 4)


def field_counts(boxes, ny, P, G):
    """cells a scatter / gather moves: (all, those whose row block and part belong to different ranks)"""
    b = np.asarray(boxes, dtype=np.int64)
    y0, ex, ey = b[:, 1], np.maximum(b[:, 2], 0), np.maximum(b[:, 3], 0)
    owner = ((np.arange(P, dtype=np.int64) + 1) * G - 1) // P
    local = np.zeros(P, dtype=np.int64)  # rows of each part inside its owner's row block
    for r in range(G):
        yb, yc = capi.shard_rows(ny, G, r)
        mine = owner == r
        local[mine] = np.clip(np.minimum(y0 + ey, yb + yc) - np.maximum(y0, yb), 0, None)[mine]
    return int((ex * ey).sum()), int((ex * (ey - local)).sum())


def field_row(name, cfg, G, variant, ms, cells, cross):
    bytes_moved = 16 * cells  # 8 B read + 8 B written per cell
    gbps = bytes_moved / (ms * 1e-3) / 1e9
    return dict(config=name, nx=cfg["nx"], ny=cfg["ny"], parts=cfg["parts"], ranks=G, variant=variant,
                ms_per_call=round(ms, 5), cells=cells, cells_cross_rank=cross, bytes_read=8 * cells,
                bytes_written=8 * cells, bytes_cross_rank=16 * cross, achieved_GBps=round(gbps, 1),
                share_of_copy_rate=round(gbps / COPY_GBPS, 4))


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


def row(name, cfg, G, ms, cells, cross, corners=(0, 0)):
    """an exchange; corners: (corner ghosts, of them cross-rank) -- (0, 0) for the edge exchange"""
    cells, cross = cells + corners[0], cross + corners[1]
    bytes_moved = 16 * cells  # 8 B read + 8 B written per ghost cell
    return dict(config=name, nx=cfg["nx"], ny=cfg["ny"], parts=cfg["parts"], ranks=G, ms_per_exchange=round(ms, 5),
                ghost_cells=cells, ghost_cells_local=cells - cross, ghost_cells_cross_rank=cross,
                corner_cells=corners[0], corner_cells_cross_rank=corners[1],
                bytes_read=8 * cells, bytes_written=8 * cells,
                achieved_GBps=round(bytes_moved / (ms * 1e-3) / 1e9, 1))


def exchange_counts(h, cfg, w):
    """(ghost cells, cross-rank, (corner cells, cross-rank)) of one periodic exchange at width w, one rank"""
    P = cfg["parts"]
    if w == 1:
        return ghost_counts(h, P, 1, True) + (corner_counts(h, P, 1, True),)
    edge, corner = wide_counts(h.boxes(), cfg["nx"], cfg["ny"], cfg["px"], cfg["py"], w)
    return edge, 0, (corner, 0)


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
        h.halo_set_width(max(args.widths))
        elems = int(h.halo_tile_offsets()[-1])
        single = torch.zeros(elems, dtype=torch.float64, device=dev)
        (ptr,) = capi.halo_connect([h], elems)
        fcells, fcross = field_counts(h.boxes(), cfg["ny"], P, 1)
        field = torch.zeros((cfg["ny"], cfg["nx"]), dtype=torch.float64, device=dev)
        back = torch.zeros_like(field)
        for w in args.widths:
            h.halo_set_width(w)
            h.halo_tile_offsets()
            host = dict(config=name, parts=P, width=w, tile_offsets_host_ms=host_ms(h.halo_tile_offsets),
                        corner_table_host_ms=host_ms(lambda: h.corner_neighbours(0, 1)))
            print(json.dumps(host), flush=True)
            h.halo_shard_offsets()
            cells, cross, corners = exchange_counts(h, cfg, w)
            variants = {"single_buffer": lambda: h.halo_exchange_f64(single.data_ptr(), True),
                        "sharded_G1": lambda: h.halo_exchange_shards_f64(True),
                        "full_single_buffer": lambda: h.halo_exchange_full_f64(single.data_ptr(), True),
                        "full_sharded_G1": lambda: h.halo_exchange_full_shards_f64(True),
                        "scatter_single_buffer": lambda: h.halo_scatter_f64(field.data_ptr(), single.data_ptr()),
                        "gather_single_buffer": lambda: h.halo_gather_f64(single.data_ptr(), back.data_ptr()),
                        "scatter_sharded_G1": lambda: h.halo_scatter_shards_f64(field.data_ptr()),
                        "gather_sharded_G1": lambda: h.halo_gather_shards_f64(back.data_ptr())}
            for fn in variants.values():
                timed(fn, stream, args.warmup)
            samples = {k: [] for k in variants}
            for _ in range(args.rounds):  # alternated: the variants share whatever else the machine does
                for k, fn in variants.items():
                    samples[k].append(timed(fn, stream, args.iters))
            h.synchronize()
            for k in variants:
                ms = float(np.median(samples[k]))
                r = row(name, cfg, 1, ms, cells, cross) if k in ("single_buffer", "sharded_G1") else \
                    row(name, cfg, 1, ms, cells, cross, corners) if k.startswith("full") else \
                    field_row(name, cfg, 1, k, ms, fcells, fcross)
                if k.startswith(("single", "sharded", "full")):
                    r["share_of_copy_rate"] = round(r["achieved_GBps"] / COPY_GBPS, 4)
                r.update(variant=k, width=w, samples_ms=[round(s, 5) for s in samples[k]], iters=args.iters)
                results.append(r)
                print(json.dumps(r), flush=True)
            results.append(host)
        h.halo_close()
        h.close()
        del single, field, back
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
        corners = corner_counts(h, P, world, True)
        fcells, fcross = field_counts(h.boxes(), cfg["ny"], P, world)
        yb, yc = capi.shard_rows(cfg["ny"], world, rank)
        rows = torch.zeros((max(yc, 1), cfg["nx"]), dtype=torch.float64, device=dev)
        variants = {"sharded": lambda: h.halo_exchange_shards_f64(True),
                    "full_sharded": lambda: h.halo_exchange_full_shards_f64(True),
                    "scatter_sharded": lambda: h.halo_scatter_shards_f64(rows.data_ptr()),
                    "gather_sharded": lambda: h.halo_gather_shards_f64(rows.data_ptr())}
        for fn in variants.values():
            timed(fn, stream, args.warmup)
        samples = {k: [] for k in variants}
        for _ in range(args.rounds):
            for k, fn in variants.items():
                dist.barrier()
                samples[k].append(timed(fn, stream, args.iters))
        for k in variants:
            t = torch.tensor(samples[k], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # per round: the slowest rank
            ms = float(np.median(t.cpu().numpy()))
            r = row(name, cfg, world, ms, cells, cross) if k == "sharded" else \
                row(name, cfg, world, ms, cells, cross, corners) if k == "full_sharded" else \
                field_row(name, cfg, world, k, ms, fcells, fcross)
            r.update(variant=k, samples_ms=[round(float(s), 5) for s in t.cpu()], iters=args.iters)
            results.append(r)
            if rank == 0:
                print(json.dumps(r), flush=True)
        del rows
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
    ap.add_argument("--widths", nargs="+", type=int, default=[1], help="frame widths (ddc_halo_set_width); one GPU only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if "WORLD_SIZE" in os.environ and args.widths != [1]:
        sys.exit("halo_bench: --widths is measured on one GPU only (the cross-rank ghosts of wide frames are not counted)")
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
