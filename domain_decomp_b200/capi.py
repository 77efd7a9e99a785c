"""ctypes bindings of the C ABI in include/ddc.h (libddc_cuda.so).

This is the Python view of the drop-in boundary: the functions below are exactly the `ddc_*`
entry points, with numpy arrays / raw device pointers as arguments.  There is no fallback: if the
CUDA library is missing or no GPU is present, `load()` / `Handle()` raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libddc_cuda.so")

LEFT, RIGHT, BOTTOM, TOP = 0, 1, 2, 3
EDGE_NAMES = ("left", "right", "bottom", "top")
WANT_PID, WANT_NEIGHBOURS, PROFILE, ASYNC = 1, 2, 4, 8
NCCL_ID_BYTES = 128
IPC_HANDLE_BYTES = 64
N_STAGES = 8
STAGE_NAMES = ("mask_scan", "x_cuts", "strip_rows", "y_cuts", "label", "finalize", "neighbours", "total")

# every symbol include/ddc.h declares (tests check the library exports all of them)
SYMBOLS = (
    "ddc_get_nccl_unique_id", "ddc_create", "ddc_destroy", "ddc_last_error", "ddc_set_stream",
    "ddc_set_mask_host", "ddc_set_mask_device", "ddc_shard_rows", "ddc_partition", "ddc_synchronize",
    "ddc_get_boxes", "ddc_get_pid_host", "ddc_get_pid_device", "ddc_get_neighbour_counts",
    "ddc_get_neighbour_total", "ddc_get_neighbours", "ddc_get_part_loads", "ddc_get_stats",
    "ddc_neighbours_from_boxes", "ddc_generate_mask_device", "ddc_generate_mask_host", "ddc_version",
    "ddc_peer_export", "ddc_peer_import", "ddc_peer_close", "ddc_host_alloc", "ddc_host_free", "ddc_peer_connect", "ddc_halo_tile_offsets", "ddc_halo_exchange_f64",
    "ddc_shard_parts", "ddc_halo_shard_offsets", "ddc_halo_export", "ddc_halo_import", "ddc_halo_connect",
    "ddc_halo_exchange_shards_f64", "ddc_halo_close",
    "ddc_halo_scatter_f64", "ddc_halo_gather_f64", "ddc_halo_scatter_shards_f64", "ddc_halo_gather_shards_f64",
)


class Stats(C.Structure):
    _fields_ = [
        ("nx", C.c_int32), ("ny", C.c_int32), ("nparts", C.c_int32),
        ("nlev", C.c_int32), ("n_xlev", C.c_int32), ("n_ylev", C.c_int32),
        ("nstrips", C.c_int32), ("changes", C.c_int32),
        ("n_ocean", C.c_int64), ("load_min", C.c_int64), ("load_max", C.c_int64),
        ("edge_cut", C.c_int64),
        ("median_iters", C.c_int32), ("gpu_launches", C.c_int32),
        ("stage_ms", C.c_float * N_STAGES),
        ("exchange", C.c_int32),
    ]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "stage_ms"}
        d["stage_ms"] = {STAGE_NAMES[i]: float(self.stage_ms[i]) for i in range(N_STAGES)}
        return d


class DdcError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """dlopen libddc_cuda.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DdcError(
            "%s is missing: build it with `python -m domain_decomp_b200.build` "
            "(the product has no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int
    L.ddc_version.restype = C.c_char_p
    L.ddc_last_error.restype = C.c_char_p
    L.ddc_last_error.argtypes = [vp]
    L.ddc_get_nccl_unique_id.argtypes = [vp]
    L.ddc_create.argtypes = [C.POINTER(vp), i32, i32, i32, vp]
    L.ddc_destroy.argtypes = [vp]
    L.ddc_set_stream.argtypes = [vp, vp]
    L.ddc_peer_export.argtypes = [vp, i32, i32, i32, vp]
    L.ddc_peer_import.argtypes = [vp, vp]
    L.ddc_peer_close.argtypes = [vp]
    L.ddc_set_mask_host.argtypes = [vp, vp, i32, i32, i32, i32]
    L.ddc_set_mask_device.argtypes = [vp, vp, i32, i32, i32, i32]
    L.ddc_shard_rows.argtypes = [i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    L.ddc_shard_rows.restype = None
    L.ddc_partition.argtypes = [vp, i32, i32, i32, i32]
    L.ddc_synchronize.argtypes = [vp]
    L.ddc_get_boxes.argtypes = [vp, vp, vp, vp, vp]
    L.ddc_get_pid_host.argtypes = [vp, vp]
    L.ddc_get_pid_device.argtypes = [vp, C.POINTER(vp)]
    L.ddc_get_neighbour_counts.argtypes = [vp, i32, i32, vp]
    L.ddc_get_neighbour_total.argtypes = [vp, i32, i32, C.POINTER(C.c_int64)]
    L.ddc_get_neighbours.argtypes = [vp, i32, i32, vp, vp, vp]
    L.ddc_get_part_loads.argtypes = [vp, vp]
    L.ddc_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.ddc_neighbours_from_boxes.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32]
    L.ddc_halo_tile_offsets.argtypes = [vp, vp]
    L.ddc_halo_exchange_f64.argtypes = [vp, vp, i32]
    L.ddc_shard_parts.argtypes = [i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    L.ddc_shard_parts.restype = None
    L.ddc_halo_shard_offsets.argtypes = [vp, vp]
    L.ddc_halo_export.argtypes = [vp, C.c_int64, C.POINTER(vp), vp]
    L.ddc_halo_import.argtypes = [vp, vp]
    L.ddc_halo_connect.argtypes = [C.POINTER(vp), i32, C.c_int64, C.POINTER(vp)]
    L.ddc_halo_exchange_shards_f64.argtypes = [vp, i32]
    L.ddc_halo_close.argtypes = [vp]
    L.ddc_halo_scatter_f64.argtypes = [vp, vp, vp]
    L.ddc_halo_gather_f64.argtypes = [vp, vp, vp]
    L.ddc_halo_scatter_shards_f64.argtypes = [vp, vp]
    L.ddc_halo_gather_shards_f64.argtypes = [vp, vp]
    L.ddc_generate_mask_device.argtypes = [vp, vp, i32, i32, i32, i32, C.c_uint64, C.c_double]
    L.ddc_generate_mask_host.argtypes = [vp, i32, i32, i32, i32, C.c_uint64, C.c_double]
    _lib = L
    return L


def shard_rows(ny: int, nranks: int, rank: int):
    b, c = C.c_int(), C.c_int()
    load().ddc_shard_rows(ny, nranks, rank, C.byref(b), C.byref(c))
    return b.value, c.value


def shard_parts(nparts: int, nranks: int, rank: int):
    """(p_begin, p_count): the parts whose tiles `rank` holds in the sharded halo exchange"""
    b, c = C.c_int(), C.c_int()
    load().ddc_shard_parts(nparts, nranks, rank, C.byref(b), C.byref(c))
    return b.value, c.value


def halo_connect(handles: list["Handle"], elems: int) -> list[int]:
    """join the halo buffers of handles that live in this process (handles[q] = rank q); returns each rank's tiles
    pointer (device memory for up to `elems` doubles)"""
    n = len(handles)
    hs = (C.c_void_p * n)(*[h.h.value for h in handles])
    out = (C.c_void_p * n)()
    L = load()
    if L.ddc_halo_connect(hs, n, elems, out):
        err = [L.ddc_last_error(h.h).decode() for h in handles]
        raise DdcError("ddc_halo_connect: %s" % (next((e for e in err if e), None) or L.ddc_last_error(None).decode()))
    return [int(p) for p in out]


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(NCCL_ID_BYTES)
    rc = load().ddc_get_nccl_unique_id(buf)
    if rc:
        raise DdcError("ddc_get_nccl_unique_id: %s" % load().ddc_last_error(None).decode())
    return buf.raw


def generate_mask_host(nx: int, ny: int, seed: int, land_frac: float, y_begin: int = 0,
                       y_count: int | None = None, out: np.ndarray | None = None) -> np.ndarray:
    """The synthetic land-sea mask of SURVEY 8d on the host (pure input generation)."""
    y_count = ny - y_begin if y_count is None else y_count
    if out is None:
        out = np.empty((y_count, nx), dtype=np.int32)
    rc = load().ddc_generate_mask_host(out.ctypes.data, nx, ny, y_begin, y_count, seed, land_frac)
    if rc:
        raise DdcError("ddc_generate_mask_host failed (%d)" % rc)
    return out


class Handle:
    """One ddc handle = one GPU (one rank)."""

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: bytes | None = None):
        self.L = load()
        self.h = C.c_void_p()
        rc = self.L.ddc_create(C.byref(self.h), device, rank, nranks, nccl_id)
        if rc:
            raise DdcError("ddc_create: %s" % self.L.ddc_last_error(None).decode())
        self.rank, self.nranks = rank, nranks
        self.nparts = 0
        self.shape = None
        self._keep = None

    def _ck(self, rc, what):
        if rc:
            raise DdcError("%s: %s" % (what, self.L.ddc_last_error(self.h).decode()))

    def close(self):
        if self.h:
            self.L.ddc_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def peer_export(self, nx: int, ny: int, nparts: int) -> bytes:
        """allocate this rank's exchange buffer; returns its CUDA IPC handle (IPC_HANDLE_BYTES bytes)"""
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        self._ck(self.L.ddc_peer_export(self.h, nx, ny, nparts, buf), "ddc_peer_export")
        return buf.raw

    def peer_import(self, handles: list[bytes]):
        """handles: the ddc_peer_export() result of every rank, in rank order"""
        blob = b"".join(handles)
        self._ck(self.L.ddc_peer_import(self.h, blob), "ddc_peer_import")

    def peer_close(self):
        self._ck(self.L.ddc_peer_close(self.h), "ddc_peer_close")

    def set_stream(self, cuda_stream: int | None):
        self._ck(self.L.ddc_set_stream(self.h, cuda_stream), "ddc_set_stream")

    def set_mask_host(self, rows: np.ndarray, ny: int | None = None, y_begin: int = 0):
        """rows: int32 [y_count, nx] host array (this rank's rows)."""
        assert rows.dtype == np.int32 and rows.flags.c_contiguous and rows.ndim == 2
        y_count, nx = rows.shape
        ny = y_count if ny is None else ny
        self._keep = rows
        self.shape = (ny, nx, y_begin, y_count)
        self._ck(self.L.ddc_set_mask_host(self.h, rows.ctypes.data, nx, ny, y_begin, y_count), "ddc_set_mask_host")

    def set_mask_host_ptr(self, ptr: int, nx: int, ny: int, y_begin: int, y_count: int):
        self.shape = (ny, nx, y_begin, y_count)
        self._ck(self.L.ddc_set_mask_host(self.h, ptr, nx, ny, y_begin, y_count), "ddc_set_mask_host")

    def set_mask_device(self, dev_ptr: int, nx: int, ny: int, y_begin: int = 0, y_count: int | None = None):
        y_count = ny if y_count is None else y_count
        self.shape = (ny, nx, y_begin, y_count)
        self._ck(self.L.ddc_set_mask_device(self.h, dev_ptr, nx, ny, y_begin, y_count), "ddc_set_mask_device")

    def generate_mask_device(self, dev_ptr: int, nx: int, ny: int, seed: int, land_frac: float,
                             y_begin: int = 0, y_count: int | None = None):
        y_count = ny if y_count is None else y_count
        self._ck(self.L.ddc_generate_mask_device(self.h, dev_ptr, nx, ny, y_begin, y_count, seed, land_frac),
                 "ddc_generate_mask_device")

    def partition(self, nparts: int, px: bool = False, py: bool = False, flags: int = WANT_PID | WANT_NEIGHBOURS):
        self.nparts = nparts
        self._ck(self.L.ddc_partition(self.h, nparts, int(px), int(py), flags), "ddc_partition")

    def synchronize(self):
        self._ck(self.L.ddc_synchronize(self.h), "ddc_synchronize")

    def boxes(self) -> np.ndarray:
        """int32 [P, 4] = x0, y0, ext_x, ext_y"""
        P = self.nparts
        a = [np.empty(P, dtype=np.int32) for _ in range(4)]
        self._ck(self.L.ddc_get_boxes(self.h, *[v.ctypes.data for v in a]), "ddc_get_boxes")
        return np.stack(a, axis=1)

    def pid_host(self) -> np.ndarray:
        ny, nx, y_begin, y_count = self.shape
        out = np.empty((y_count, nx), dtype=np.int32)
        self._ck(self.L.ddc_get_pid_host(self.h, out.ctypes.data), "ddc_get_pid_host")
        return out

    def pid_host_into(self, ptr: int):
        self._ck(self.L.ddc_get_pid_host(self.h, ptr), "ddc_get_pid_host")

    def pid_device(self) -> int:
        p = C.c_void_p()
        self._ck(self.L.ddc_get_pid_device(self.h, C.byref(p)), "ddc_get_pid_device")
        return p.value

    def halo_tile_offsets(self) -> np.ndarray:
        """element offsets of the framed tiles of all parts in one buffer (ddc_halo_tile_offsets)"""
        out = np.empty(self.nparts + 1, dtype=np.int64)
        self._ck(self.L.ddc_halo_tile_offsets(self.h, out.ctypes.data), "ddc_halo_tile_offsets")
        return out

    def halo_exchange_f64(self, tiles_dev_ptr: int, periodic: bool = False):
        self._ck(self.L.ddc_halo_exchange_f64(self.h, tiles_dev_ptr, int(periodic)), "ddc_halo_exchange_f64")

    def halo_shard_offsets(self) -> np.ndarray:
        """element offsets of this rank's framed tiles in its own halo buffer (ddc_halo_shard_offsets)"""
        _, count = shard_parts(self.nparts, self.nranks, self.rank)
        out = np.empty(count + 1, dtype=np.int64)
        self._ck(self.L.ddc_halo_shard_offsets(self.h, out.ctypes.data), "ddc_halo_shard_offsets")
        return out

    def halo_export(self, elems: int):
        """allocate this rank's halo buffer for up to `elems` doubles; returns (tiles device pointer, CUDA IPC handle)"""
        ptr = C.c_void_p()
        buf = C.create_string_buffer(IPC_HANDLE_BYTES)
        self._ck(self.L.ddc_halo_export(self.h, elems, C.byref(ptr), buf), "ddc_halo_export")
        return int(ptr.value), buf.raw

    def halo_import(self, handles: list[bytes]):
        """handles: the halo_export() IPC handle of every rank, in rank order"""
        self._ck(self.L.ddc_halo_import(self.h, b"".join(handles)), "ddc_halo_import")

    def halo_exchange_shards_f64(self, periodic: bool = False):
        self._ck(self.L.ddc_halo_exchange_shards_f64(self.h, int(periodic)), "ddc_halo_exchange_shards_f64")

    def halo_close(self):
        self._ck(self.L.ddc_halo_close(self.h), "ddc_halo_close")

    def halo_scatter_f64(self, field_ptr: int, tiles_ptr: int):
        """tile interiors <- the field (device double [ny][nx]), one buffer in the halo_tile_offsets() layout"""
        self._ck(self.L.ddc_halo_scatter_f64(self.h, field_ptr, tiles_ptr), "ddc_halo_scatter_f64")

    def halo_gather_f64(self, tiles_ptr: int, field_ptr: int):
        """the field (device double [ny][nx]) <- tile interiors, one buffer in the halo_tile_offsets() layout"""
        self._ck(self.L.ddc_halo_gather_f64(self.h, tiles_ptr, field_ptr), "ddc_halo_gather_f64")

    def halo_scatter_shards_f64(self, rows_ptr: int):
        """every rank's tile interiors <- this rank's rows (device double [y_count][nx] of shard_rows)"""
        self._ck(self.L.ddc_halo_scatter_shards_f64(self.h, rows_ptr), "ddc_halo_scatter_shards_f64")

    def halo_gather_shards_f64(self, rows_ptr: int):
        """this rank's rows (device double [y_count][nx] of shard_rows) <- every rank's tile interiors"""
        self._ck(self.L.ddc_halo_gather_shards_f64(self.h, rows_ptr), "ddc_halo_gather_shards_f64")

    def neighbour_counts(self, edge: int, periodic: int) -> np.ndarray:
        out = np.empty(self.nparts, dtype=np.int32)
        self._ck(self.L.ddc_get_neighbour_counts(self.h, edge, periodic, out.ctypes.data), "ddc_get_neighbour_counts")
        return out

    def neighbours(self, edge: int, periodic: int):
        tot = C.c_int64()
        self._ck(self.L.ddc_get_neighbour_total(self.h, edge, periodic, C.byref(tot)), "ddc_get_neighbour_total")
        n = tot.value
        ids, halos, starts = (np.empty(n, dtype=np.int32) for _ in range(3))
        self._ck(self.L.ddc_get_neighbours(self.h, edge, periodic, ids.ctypes.data, halos.ctypes.data,
                                           starts.ctypes.data), "ddc_get_neighbours")
        return ids, halos, starts

    def part_loads(self) -> np.ndarray:
        out = np.empty(self.nparts, dtype=np.int64)
        self._ck(self.L.ddc_get_part_loads(self.h, out.ctypes.data), "ddc_get_part_loads")
        return out

    def stats(self) -> dict:
        s = Stats()
        self._ck(self.L.ddc_get_stats(self.h, C.byref(s)), "ddc_get_stats")
        return s.as_dict()

    def neighbours_from_boxes(self, boxes: np.ndarray, nx: int, ny: int, px: bool, py: bool):
        b = np.ascontiguousarray(boxes, dtype=np.int32)
        cols = [np.ascontiguousarray(b[:, i]) for i in range(4)]
        self.nparts = b.shape[0]
        self._ck(self.L.ddc_neighbours_from_boxes(self.h, self.nparts, nx, ny, *[c.ctypes.data for c in cols],
                                                  int(px), int(py)), "ddc_neighbours_from_boxes")
