#!/usr/bin/env python
"""Benchmark of the hot path: land-sea mask -> RCB boxes + pid labels + neighbours / halos.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one complete decomposition (ddc_partition with pid + neighbour tables) of the
workload's synthetic mask.  With N > 1 (torchrun, one rank per GPU) the SAME mask is row-sharded
over the ranks (strong scaling) and the histograms are combined with NCCL inside the step.
Every timed loop runs K steps.

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (float32 where that is
exact, else float64): boxes [P, 4] (x0, y0, ext_x, ext_y), part_loads [P], neighbour_counts
[2, 4, P] (periodic, edge in the order left, right, bottom, top, part), neighbours [n, 6] with one row
(periodic, edge, part, neighbour id, halo, halo start) per entry of the neighbour tables, in the order of
the metadata file, and the pid map: whole as pid [ny, nx] up to PID_DUMP_CELLS cells, else a fixed
seeded sample pid_sample at the flat indices y * nx + x in pid_sample_index.  (One array for all tables:
the tables of an edge without periodic neighbours are empty.)  The mask comes from the workload's seed,
so two builds run with the same arguments can be compared array for array.

  value       whole-job mask cells partitioned per second, mask already resident in HBM
  e2e         same metric through the C ABI with HOST buffers: pinned-host -> device copy of the
              int32 mask and device -> host read-back of pid, boxes and neighbour tables inside
              the timed region
  roofline    the dominant kernel against the measured HBM copy bandwidth
  cpu_baseline  the CPU oracle (a port of the reference algorithm) on a bounded sample

`--impl reference` times the reference algorithm's CPU port (oracle/, OpenMP tasks over all host
cores) on a bounded sample of the same workload; the reference binary itself needs MPI + Zoltan +
parallel netCDF + Boost, none of which exist in this image (see DESIGN.md).  It runs K steps too, and
one step of the whole default workload takes tens of seconds: pass --steps 1 for a quick number.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name -> nx, ny, parts, land fraction, seed, periodic x, periodic y   (SURVEY 8d / BASELINE.json configs)
WORKLOADS = {
    "C5_32768x32768_p16384": (32768, 32768, 16384, 0.45, 32, 1, 0),
    "C4_8192x8192_p4096": (8192, 8192, 4096, 0.60, 1, 0, 0),
    "C3_4096x4096_p1024": (4096, 4096, 1024, 0.45, 3, 0, 0),
    "C2_528x522_p64": (528, 522, 64, 0.45, 25, 1, 1),
    # not BASELINE configs: one rank's share of C5 on 2 / 8 GPUs as a mask of its own, for tuning the streaming
    # kernels at shard size on one GPU
    "X_shard8_32768x4096_p2048": (32768, 4096, 2048, 0.45, 32, 1, 0),
    "X_shard2_32768x16384_p8192": (32768, 16384, 8192, 0.45, 32, 1, 0),
}
GOLDEN_DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
DEFAULT_WORKLOAD = "C5_32768x32768_p16384"
L2_BYTES = 126 * 1000 * 1000
ALGO_BYTES_PER_CELL = 8  # 4 B int32 mask read + 4 B int32 pid write (SURVEY 8d)
PID_DUMP_CELLS = 1 << 20  # --dump-outputs: pid maps larger than this are sampled (12 B per sampled cell)
DUMP_SEED = 20251020
DUMP_MAX_BYTES = 64 * 1000 * 1000


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str, workload: str):
    """dram bytes per launch of `kernel` from the committed ncu capture, if one exists"""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[workload][kernel]
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """polls SM clock and throttle reasons of one GPU through NVML while the timed region runs"""

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # NVML missing: report it rather than invent numbers
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
            nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM))
                r = get_reasons(self.dev)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": "NVML unavailable" if not self.ok else "no sample fell inside the timed region"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def golden_digest(workload):
    """digest of the decomposition's replicated tables as the CPU oracle computes them (scripts/make_bench_digests.py)"""
    try:
        with open(GOLDEN_DIGESTS) as f:
            return json.load(f)[workload]["digest"]
    except Exception:
        return None


class _DevArray:
    """__cuda_array_interface__ view of an int32 device buffer owned by the library"""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i4", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def _exact_float(a):
    """int array -> float32 when every value is exact in it, else float64"""
    import numpy as np
    a = np.asarray(a)
    return a.astype(np.float32 if a.size == 0 or int(np.abs(a).max()) < (1 << 24) else np.float64)


def dump_outputs(h, out_dir, d_pid, nx, ny, y_begin, y_count, dev, world, rank):
    """--dump-outputs: the results of the handle's last decomposition as DIR/<name>.npy (see the module doc).
    Every rank calls the same getters; the pid rows of all ranks are combined, rank 0 writes."""
    import numpy as np
    import torch
    from domain_decomp_b200 import capi
    out = {"boxes": h.boxes(), "part_loads": h.part_loads()}
    counts, rows = np.zeros((2, 4, h.nparts), dtype=np.int64), []
    for per in range(2):
        for e in range(len(capi.EDGE_NAMES)):
            counts[per, e] = h.neighbour_counts(e, per)
            ids, halos, starts = h.neighbours(e, per)
            part = np.repeat(np.arange(h.nparts), counts[per, e])
            rows.append(np.stack([np.full(ids.size, per), np.full(ids.size, e), part, ids, halos, starts], axis=1))
    out["neighbour_counts"], out["neighbours"] = counts, np.concatenate(rows)
    cells = nx * ny
    whole = cells <= PID_DUMP_CELLS
    idx = (np.arange(cells, dtype=np.int64) if whole else
           np.unique(np.random.default_rng(DUMP_SEED).integers(0, cells, size=PID_DUMP_CELLS)))
    g = torch.from_numpy(idx).to(dev)
    lo = y_begin * nx
    mine = (g >= lo) & (g < lo + y_count * nx)
    vals = torch.zeros(idx.size, dtype=torch.int64, device=dev)
    vals[mine] = d_pid.reshape(-1)[g[mine] - lo].long()
    if world > 1:
        torch.distributed.all_reduce(vals)  # every sampled cell lies in the rows of exactly one rank
    if whole:
        out["pid"] = vals.cpu().numpy().reshape(ny, nx)
    else:
        out["pid_sample"], out["pid_sample_index"] = vals.cpu().numpy(), idx
    if rank != 0:
        return
    # the sample's flat indices exceed float32's exact range: float64, exact below 2**53
    arrays = {k: v.astype(np.float64) if k == "pid_sample_index" else _exact_float(v) for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def plugin_e2e(mask, expect_pid, expect_boxes_soa, nx, ny, P, px, py, gpus, reps):
    """CudaRcbPartitioner::partition through libdomain_decomp.so's ddc_plugin_bench (host/PluginBench.cpp)"""
    import ctypes as C
    import numpy as np
    lib = C.CDLL(os.path.join(ROOT, "domain_decomp_b200", "libdomain_decomp.so"))
    secs = (C.c_double * reps)()
    grid_s, same = C.c_double(0.0), C.c_int(0)
    err = C.create_string_buffer(512)
    vp = C.c_void_p
    lib.ddc_plugin_bench.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.POINTER(C.c_double), C.POINTER(C.c_double), vp, vp, C.POINTER(C.c_int), C.c_char_p, C.c_int]
    rc = lib.ddc_plugin_bench(mask.ctypes.data, nx, ny, P, px, py, 0, gpus, reps, secs, C.byref(grid_s),
                              expect_pid.ctypes.data, np.ascontiguousarray(expect_boxes_soa, dtype=np.int32).ctypes.data,
                              C.byref(same), err, 512)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    t = list(secs)
    return {"seconds": sum(t) / len(t), "best_seconds": min(t), "steps": reps, "same": bool(same.value),
            "grid_seconds": grid_s.value}


def cpu_sample(workload, threads: int, whole: bool = False):
    """the workload for the CPU legs: the whole mask when it is small or `whole` is set, else a bounded sample --
    the top-left 1/8 x 1/8 window of the SAME mask into 1/64 of the parts (same cells per part).  The mask comes
    from the oracle's restatement of the generator: the CPU legs never load the CUDA library."""
    nx, ny, P, land, seed, px, py = WORKLOADS[workload]
    from oracle import oracle as orc
    if nx * ny > 8192 * 8192 and not whole:
        f = 8
        sx, sy, sp = nx // f, ny // f, max(2, P // (f * f))
        desc = ("top-left %dx%d window of the %dx%d mask into %d parts (same cells per part; %d RCB levels "
                "instead of %d, which favours the CPU)" % (sx, sy, nx, ny, sp, (sp - 1).bit_length(), (P - 1).bit_length()))
    else:
        sx, sy, sp, desc = nx, ny, P, "the whole %dx%d mask into %d parts" % (nx, ny, P)
    full = orc.generate_mask(nx, ny, seed, land, 0, sy)  # rows [0, sy) of the global mask
    import numpy as np
    mask = full if sx == nx else np.ascontiguousarray(full[:, :sx])
    return mask, sp, px, py, desc


def run_cpu(mask, P, px, py, threads, steps, warmup):
    from oracle import oracle as orc
    orc.set_threads(threads)
    times = []
    for i in range(warmup + steps):
        t = time.perf_counter()
        orc.partition(mask, P, bool(px), bool(py), use_hist=False, want_pid=True, want_neighbours=True)
        dt = time.perf_counter() - t
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    threads = orc.max_threads()
    nx, ny, P, land, seed, _, _ = WORKLOADS[args.workload]
    # the WHOLE workload when the host has the memory for it: the dot-based restatement keeps Zoltan's dot arrays
    # (24 B per ocean cell) beside the 4 B/cell mask and the 4 B/cell pid
    need = nx * ny * (4 + 4 + 24 * 0.6) * 1.15
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 0
    whole = args.sample == "whole" or (args.sample == "auto" and avail > need)
    t0 = time.perf_counter()
    mask, sp, px, py, desc = cpu_sample(args.workload, threads, whole=whole)
    # a CPU pass over a fresh mask has nothing to warm up: every step counts
    steps, warmup = args.steps, 0
    sec = run_cpu(mask, sp, px, py, threads, steps, warmup)
    value = mask.size / sec
    same_config = mask.shape == (ny, nx) and sp == P
    line = {
        "impl": "reference", "metric": "mask cells partitioned/sec", "value": value, "unit": "cells/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": {"workload": args.workload, "nx": nx, "ny": ny, "parts": P, "land_frac": land, "seed": seed,
                   "periodic_x": px, "periodic_y": py},
        "same_config": same_config,
        "cpu_baseline": {"value": value, "unit": "cells/s", "cores": threads, "kind": "port", "sample": desc,
                         "note": "CPU port of the reference algorithm (oracle/ddc_oracle.c, dot-based Zoltan RCB "
                                 "restatement + labelling + O(P^2) neighbour discovery); the reference binary "
                                 "needs MPI+Zoltan+netCDF+Boost which this image lacks"},
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every timed loop (--impl reference: tens of seconds per step on the default workload)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the result checks (they are outside the timed regions)")
    ap.add_argument("--sample", default="auto", choices=["auto", "whole", "window"],
                    help="--impl reference: the whole workload (when the host memory allows: auto) or the bounded window")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="multi-GPU exchange: stores into the peers' memory from inside the kernels (default) or NCCL collectives")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from domain_decomp_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torchrun --nproc-per-node N)" % (args.gpus, world))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    nccl_id = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        ids = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        nccl_id = ids[0]

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    nx, ny, P, land, seed, px, py = WORKLOADS[args.workload]
    cells = nx * ny
    W, K = max(args.warmup, 3), args.steps
    h = capi.Handle(local_rank, rank, world, nccl_id)
    if world > 1 and args.exchange == "peer":
        handles = [None] * world
        dist.all_gather_object(handles, h.peer_export(nx, ny, P))
        h.peer_import(handles)
    # a real (non-default) stream: the handle launches on it and the timing events are recorded on it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    h.set_stream(stream.cuda_stream)
    assert stream.cuda_stream != 0
    y_begin, y_count = capi.shard_rows(ny, world, rank)
    d_mask = torch.empty((max(y_count, 1), nx), dtype=torch.int32, device=dev)
    h.generate_mask_device(d_mask.data_ptr(), nx, ny, seed, land, y_begin, y_count)
    h.set_mask_device(d_mask.data_ptr(), nx, ny, y_begin, y_count)
    flags = capi.WANT_PID | capi.WANT_NEIGHBOURS
    aflags = flags | capi.ASYNC  # timed loops only enqueue; the events / the final synchronize wait
    shard_bytes = y_count * nx * 4
    need_flush = shard_bytes * 2 < 2 * L2_BYTES  # mask + pid of this rank could sit in the 126 MB L2
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if need_flush else None

    # ---- device-resident timing ---------------------------------------------------------------
    for _ in range(W):
        h.partition(P, px, py, flags)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    torch.cuda.synchronize()
    if not need_flush:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            h.partition(P, px, py, aflags)
        e1.record(stream)
        torch.cuda.synchronize()
        total_ms = e0.elapsed_time(e1)
    else:
        total_ms = 0.0
        for _ in range(K):
            flush_buf.fill_(1)  # evict mask / bit map / pid from L2 (outside the timed events)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            h.partition(P, px, py, aflags)
            e1.record(stream)
            torch.cuda.synchronize()
            total_ms += e0.elapsed_time(e1)
    barrier()
    clocks = sampler.stop()
    ms_per_step = max_over_ranks(total_ms / K)
    value = cells / (ms_per_step * 1e-3)
    st = h.stats()
    if args.dump_outputs:
        d_pid = torch.as_tensor(_DevArray(h.pid_device(), (max(y_count, 1), nx)), device=dev)[:y_count]
        dump_outputs(h, args.dump_outputs, d_pid, nx, ny, y_begin, y_count, dev, world, rank)
        del d_pid

    # ---- per-kernel timing (CUDA events on the launching stream, inside ddc_partition) --------
    stage = {k: 0.0 for k in capi.STAGE_NAMES}
    nprof = 5
    for _ in range(nprof):
        if flush_buf is not None:
            flush_buf.fill_(1)
        h.partition(P, px, py, flags | capi.PROFILE)
        s = h.stats()["stage_ms"]
        for k in stage:
            stage[k] += s[k] / nprof
    peak, peak_src = measured_peak_gbs()
    local_cells = y_count * nx
    kern = {"mask_scan": "k_scan_mask", "label": "k_label"}
    dom = max(kern, key=lambda k: stage[k])
    dom_ms = max_over_ranks(stage[dom])
    achieved = (4.0 * local_cells) / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    roofline = {
        "bound": "hbm", "kernel": kern[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": ncu_traffic(kern[dom], args.workload) if world == 1 else None, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": 4 * local_cells, "kernel_ms": dom_ms,
        "pipeline": {"achieved": ALGO_BYTES_PER_CELL * cells / (ms_per_step * 1e-3) / 1e9,
                     "frac_of_aggregate_peak": ALGO_BYTES_PER_CELL * cells / (ms_per_step * 1e-3) / 1e9 / (peak * world),
                     "algorithmic_bytes_per_cell": ALGO_BYTES_PER_CELL},
        "stage_ms": {k: round(v, 4) for k, v in stage.items()},
    }

    # ---- what was timed is also what is right (outside every timed region) --------------------------
    # every rank: digest of the replicated tables (boxes, 8 neighbour tables, part loads, `changes`) and its own
    # pid rows against the labelling rule restated with torch; rank 0: all ranks agree, the digest is the one the CPU
    # oracle gives for this workload (tests/golden/bench_digests.json), the label counts of all ranks are the loads
    parity = None
    if not args.no_verify:
        from domain_decomp_b200 import verify
        h.partition(P, px, py, flags)
        digest = verify.handle_digest(h)
        d_pid = torch.as_tensor(_DevArray(h.pid_device(), (max(y_count, 1), nx)), device=dev)[:y_count]
        pid_ok, counts = verify.pid_rows_match_boxes(h.boxes(), nx, ny, d_mask[:y_count], d_pid, y_begin)
        if world > 1:
            dist.all_reduce(counts)
            every = [None] * world
            dist.all_gather_object(every, (digest, bool(pid_ok)))
        else:
            every = [(digest, bool(pid_ok))]
        loads_ok = bool(torch.equal(counts.cpu(), torch.from_numpy(h.part_loads().astype(np.int64))))
        golden = golden_digest(args.workload)
        parity = {"checked": True, "digest": digest, "ranks_agree": all(d == digest for d, _ in every),
                  "matches_cpu_oracle": (digest == golden) if golden else None,
                  "pid_rows_are_the_labelling_of_the_boxes": all(ok for _, ok in every),
                  "label_counts_equal_part_loads": loads_ok,
                  "what": "sha256 of boxes + 8 neighbour tables + part loads + changes on every rank; golden = CPU oracle "
                          "(scripts/make_bench_digests.py); pid checked on the device against the labelling rule"}
        parity["passed"] = bool(parity["ranks_agree"] and parity["matches_cpu_oracle"] is not False
                                and parity["pid_rows_are_the_labelling_of_the_boxes"] and loads_ok)
        del d_pid
        if not parity["passed"]:
            if rank == 0:
                print(json.dumps({"parity": parity, "error": "PARITY FAILURE: the timed output is wrong"}), flush=True)
            raise SystemExit(3)

    # ---- end to end through the C ABI with host buffers -----------------------------------------
    e2e = None
    if not args.no_e2e:
        h_mask = torch.empty((max(y_count, 1), nx), dtype=torch.int32, pin_memory=True)
        h_pid = torch.empty((max(y_count, 1), nx), dtype=torch.int32, pin_memory=True)
        h_mask.copy_(d_mask)  # the same synthetic mask, now living in pinned host memory
        torch.cuda.synchronize()

        def e2e_step():
            h.set_mask_host_ptr(h_mask.data_ptr(), nx, ny, y_begin, y_count)  # H2D
            h.partition(P, px, py, flags)
            h.pid_host_into(h_pid.data_ptr())  # D2H, 4 B / cell
            b = h.boxes()
            n = b.nbytes
            for per in range(2):
                for e in range(4):
                    n += h.neighbour_counts(e, per).nbytes
                    n += sum(a.nbytes for a in h.neighbours(e, per))
            return n

        small = e2e_step()
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            e2e_step()
        e1.record(stream)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3 / K
        ev_ms = e0.elapsed_time(e1) / K
        barrier()
        e2e_ms = max_over_ranks(max(wall, ev_ms))
        e2e = {"value": cells / (e2e_ms * 1e-3), "unit": "cells/s", "ms_per_step": e2e_ms, "steps": K,
               "h2d_bytes_per_step": shard_bytes * world if world > 1 else shard_bytes,
               "d2h_bytes_per_step": (shard_bytes + small) * world if world > 1 else shard_bytes + small,
               "path": "C ABI (ddc_set_mask_host, ddc_partition, ddc_get_pid_host, table getters), one process per GPU",
               "note": "pinned host int32 mask -> device, partition, pid + boxes + neighbour tables -> host"}
        boxes_soa = np.ascontiguousarray(h.boxes().T)  # x0[P] y0[P] ex[P] ey[P]
        h.set_mask_device(d_mask.data_ptr(), nx, ny, y_begin, y_count)
        # the same through the reference-facing plugin: Grid + Partitioner::Factory::create + partition(grid)
        # (main.cpp:84-94 of the reference), one process, one host thread per GPU
        plugin = None
        if world > 1:  # rank 0 needs the whole mask / pid on the host: gather the shards through shared memory
            shm = "/dev/shm/ddc_bench_%s" % os.environ.get("MASTER_PORT", "0")
            gathered = {}
            for name, t in (("mask", h_mask), ("pid", h_pid)):
                path = "%s_%s.i32" % (shm, name)
                arr = np.memmap(path, dtype=np.int32, mode="w+", shape=(ny, nx)) if rank == 0 else None  # rank 0 creates
                dist.barrier()
                if rank != 0:
                    arr = np.memmap(path, dtype=np.int32, mode="r+", shape=(ny, nx))
                arr[y_begin:y_begin + y_count] = t.numpy()[:y_count]
                arr.flush()
                dist.barrier()
                gathered[name] = arr
            g_mask, g_pid = gathered["mask"], gathered["pid"]
        else:
            g_mask, g_pid = h_mask.numpy(), h_pid.numpy()
        if rank == 0:
            try:
                plugin = plugin_e2e(np.ascontiguousarray(g_mask), np.ascontiguousarray(g_pid), boxes_soa, nx, ny, P, px, py,
                                    world, K)
            except Exception as exc:  # the C ABI number stands
                plugin = {"error": str(exc)}
        if world > 1:
            dist.barrier()
            if rank == 0:
                for name in ("mask", "pid"):
                    try:
                        os.unlink("%s_%s.i32" % (shm, name))
                    except OSError:
                        pass
        del h_mask, h_pid, g_mask, g_pid
        if plugin and "error" not in plugin:
            e2e = {"value": cells / plugin["seconds"], "unit": "cells/s", "ms_per_step": plugin["seconds"] * 1e3,
                   "steps": plugin["steps"], "h2d_bytes_per_step": cells * 4, "d2h_bytes_per_step": cells * 4 + small,
                   "path": "plugin: Grid (host mask) -> Partitioner::Factory::create(Cuda_RCB, --gpus %d) -> partition(grid): "
                           "boxes, neighbour tables and the pid map back in the Partitioner's host memory; one process, one "
                           "host thread per GPU" % world,
                   "same_result_as_c_abi": plugin["same"], "grid_build_seconds": plugin["grid_seconds"],
                   "c_abi": e2e}
        elif plugin:
            e2e["plugin_error"] = plugin["error"]

    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import oracle as orc
        orc.build()
        mask, sp, spx, spy, desc = cpu_sample(args.workload, 1)
        sec = run_cpu(mask, sp, spx, spy, 1, 1, 0)
        cpu = {"value": mask.size / sec, "unit": "cells/s", "cores": 1, "kind": "port", "sample": desc,
               "seconds": sec, "host_cores": os.cpu_count()}

    if rank == 0:
        line = {
            "metric": "mask cells partitioned/sec", "value": value, "unit": "cells/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "i32", "data": "synthetic",
            "config": {"workload": args.workload, "nx": nx, "ny": ny, "parts": P, "land_frac_target": land,
                       "ocean_frac_measured": st["n_ocean"] / cells, "seed": seed, "periodic_x": px,
                       "periodic_y": py, "sharding": "rows over %d GPU(s)%s" % (world, "" if world == 1 else (
                           ", histograms pushed into the peers' memory over NVLink by the producing kernels, flag barriers in the cut kernels" if st["exchange"] == 2
                           else ", NCCL allreduce + allgather")),
                       "outputs": "boxes + pid + neighbour/halo tables",
                       "knobs": {k: os.environ[k] for k in sorted(os.environ) if k.startswith("DDC_")},
                       "l2": ("L2 flushed between timed iterations (256 MiB write)" if need_flush else
                              "inputs larger than L2 (%.0f MiB int32 mask + %.0f MiB pid per GPU vs 126 MB L2)"
                              % (shard_bytes / 2**20, shard_bytes / 2**20))},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": st["gpu_launches"] * K * world,
            "parity": parity,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "result": {"n_ocean": st["n_ocean"], "strips": st["nstrips"], "x_levels": st["n_xlev"],
                       "y_levels": st["n_ylev"], "changes": st["changes"], "median_iters": st["median_iters"],
                       "imbalance": st["load_max"] / max(st["n_ocean"] / P, 1e-9), "edge_cut": st["edge_cut"],
                       "launches_per_step": st["gpu_launches"]},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        h.peer_close()
        dist.barrier()
    h.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
