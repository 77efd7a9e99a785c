#!/usr/bin/env python
"""Byte masks against int32 masks: the decomposition step, the mask scan and the C-ABI end to end.

    python scripts/mask_bytes_bench.py --out result.json                   # one GPU, C2 .. C5
    torchrun --nproc-per-node G scripts/mask_bytes_bench.py --out r.json    # G GPUs over peer memory, one process each

Step: ddc_partition with the mask already in HBM (ddc_set_mask_device / ddc_set_mask_u8_device of a device tensor
holding the same cells), int32 and u8 alternated in every round: `--warmup` steps, then `--steps` steps timed one by
one with CUDA events (a 256 MiB buffer is overwritten between steps, outside the events, so that no step starts with
the mask in L2); a round's value is the mean step, the reported value the median of `--rounds` rounds (with G GPUs
the slowest rank's).  Scan: stage_ms[0] of DDC_PROFILE runs (CUDA events around the scan), with the bytes it moves
(the mask read once: 4 or 1 B per cell; the bit map written: NB B per row) over the 6546.9 GB/s of a read+write copy
measured on a B200 (DESIGN.md 4).  End to end (one GPU): ddc_set_mask_*_host from pinned memory + ddc_partition +
ddc_get_pid_host into pinned memory, alternated the same way.  Parity: every u8 line carries the check against the
int32 run of the same round: the digest of the replicated tables (boxes, neighbour lists, part loads, changes) and
the pid rows on the device.  The GPU name and power limit are read in the same run.  Writes JSON to --out (and
prints it); nothing in the tree."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from domain_decomp_b200 import capi, verify  # noqa: E402

COPY_GBS = 6546.9
WORKLOADS = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_digests.json")))
NAMES = {"C2": "C2_528x522_p64", "C3": "C3_4096x4096_p1024", "C4": "C4_8192x8192_p4096", "C5": "C5_32768x32768_p16384"}


class DevI32:
    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i4", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q
    except Exception as e:  # noqa: BLE001
        return ["unknown (%s)" % e]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["C2", "C3", "C4", "C5"])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--e2e", nargs="*", default=["C4", "C5"], help="workloads of the end-to-end C-ABI measurement")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    slowest = lambda v: v if dist is None else _max(dist, v, dev)
    result = {"gpus": world, "gpu": gpu_info() if rank == 0 else None, "copy_gbs": COPY_GBS, "rows": []}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for key in args.workloads:
        w = WORKLOADS[NAMES[key]]
        nx, ny, P, px, py = w["nx"], w["ny"], w["parts"], bool(w["periodic_x"]), bool(w["periodic_y"])
        yb, yc = capi.shard_rows(ny, world, rank)
        h = capi.Handle(local, rank, world, None)
        if world > 1:
            handles = [None] * world
            dist.all_gather_object(handles, h.peer_export(nx, ny, P))
            h.peer_import(handles)
        d32 = torch.empty((max(yc, 1), nx), dtype=torch.int32, device=dev)
        h.generate_mask_device(d32.data_ptr(), nx, ny, w["seed"], w["land_frac"], yb, yc)
        torch.cuda.synchronize()  # (the handle's stream is not torch's)
        d8 = (d32 > 0).to(torch.uint8)
        torch.cuda.synchronize()
        setters = {"int32": lambda: h.set_mask_device(d32.data_ptr(), nx, ny, yb, yc),
                   "u8": lambda: h.set_mask_u8_device(d8.data_ptr(), nx, ny, yb, yc)}
        steps = {"int32": [], "u8": []}
        parity = []
        for _ in range(args.rounds):
            out = {}
            for kind in ("int32", "u8"):
                setters[kind]()
                for _ in range(args.warmup):
                    h.partition(P, px, py)
                torch.cuda.synchronize()
                total = 0.0
                for _ in range(args.steps):
                    flush.fill_(1)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    h.partition(P, px, py)
                    e1.record()
                    torch.cuda.synchronize()
                    total += e0.elapsed_time(e1)
                steps[kind].append(slowest(total / args.steps))
                pid = torch.as_tensor(DevI32(h.pid_device(), (max(yc, 1), nx)), device=dev)[:yc].clone()
                out[kind] = (verify.handle_digest(h), pid, h.stats())
            same_pid = torch.equal(out["int32"][1], out["u8"][1])
            st32, st8 = ({k: v for k, v in s.items() if k != "stage_ms"} for s in (out["int32"][2], out["u8"][2]))
            parity.append(out["int32"][0] == out["u8"][0] and same_pid and st32 == st8)
            del out
        scan = {}
        for kind in ("int32", "u8"):
            setters[kind]()
            v = 0.0
            for _ in range(5):
                flush.fill_(1)
                h.partition(P, px, py, capi.WANT_PID | capi.WANT_NEIGHBOURS | capi.PROFILE)
                v += h.stats()["stage_ms"]["mask_scan"] / 5
            scan[kind] = slowest(v)
        NB = 16 * ((nx + 127) // 128)
        ok = all(parity) and (verify.handle_digest(h) == w["digest"])
        for kind, esize in (("int32", 4), ("u8", 1)):
            byts = yc * (nx * esize + NB)
            row = {"workload": NAMES[key], "mask": kind, "gpus": world, "step_ms_median": float(np.median(steps[kind])),
                   "step_ms_rounds": steps[kind], "scan_ms": scan[kind], "scan_bytes_per_rank": byts,
                   "scan_gbs": byts / (scan[kind] * 1e-3) / 1e9 if scan[kind] > 0 else None,
                   "scan_share_of_copy_rate": byts / (scan[kind] * 1e-3) / 1e9 / COPY_GBS if scan[kind] > 0 else None,
                   "parity_u8_equals_int32_every_round": all(parity), "digest_matches_cpu_oracle": ok or None}
            result["rows"].append(row)
            if rank == 0:
                print(json.dumps(row), flush=True)
        del d32, d8
        if world > 1:
            h.peer_close()
            dist.barrier()
        h.close()
    if world == 1:
        for key in args.e2e:
            result["rows"].append(e2e(key, args, dev))
            print(json.dumps(result["rows"][-1]), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    if rank == 0 and args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


def _max(dist, v, dev):
    t = torch.tensor([v], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def e2e(key, args, dev):
    """pinned host mask -> set_mask_*_host + ddc_partition + ddc_get_pid_host (pinned), host clock around it"""
    import time
    w = WORKLOADS[NAMES[key]]
    nx, ny, P, px, py = w["nx"], w["ny"], w["parts"], bool(w["periodic_x"]), bool(w["periodic_y"])
    h = capi.Handle(dev.index)
    d32 = torch.empty((ny, nx), dtype=torch.int32, device=dev)
    h.generate_mask_device(d32.data_ptr(), nx, ny, w["seed"], w["land_frac"])
    torch.cuda.synchronize()
    m32 = torch.empty((ny, nx), dtype=torch.int32, pin_memory=True)
    m32.copy_(d32)
    m8 = torch.empty((ny, nx), dtype=torch.uint8, pin_memory=True)
    m8.copy_(d32 > 0)
    del d32
    torch.cuda.empty_cache()
    pid = {k: torch.empty((ny, nx), dtype=torch.int32, pin_memory=True) for k in ("int32", "u8")}
    calls = {"int32": lambda: h.set_mask_host_ptr(m32.data_ptr(), nx, ny, 0, ny),
             "u8": lambda: h.set_mask_u8_host(m8.numpy())}
    times = {"int32": [], "u8": []}
    for r in range(args.rounds):
        for kind in ("int32", "u8"):
            calls[kind]()
            h.partition(P, px, py)  # warm: the plan, the buffers
            h.pid_host_into(pid[kind].data_ptr())
            n = 5
            t0 = time.perf_counter()
            for _ in range(n):
                calls[kind]()
                h.partition(P, px, py)
                h.pid_host_into(pid[kind].data_ptr())
            times[kind].append((time.perf_counter() - t0) * 1e3 / n)
    same = torch.equal(pid["int32"], pid["u8"])
    h.close()
    return {"workload": NAMES[key], "end_to_end_ms_median": {k: float(np.median(v)) for k, v in times.items()},
            "end_to_end_ms_rounds": times, "host_mask_bytes": {"int32": 4 * nx * ny, "u8": nx * ny},
            "parity_pid_equal": bool(same),
            "what": "set_mask_*_host (pinned) + ddc_partition + ddc_get_pid_host (pinned), host clock, mean of 5 calls"}


if __name__ == "__main__":
    main()
