"""Shared by the byte-mask tests: everything a handle holds after ddc_partition, and byte masks with every kind of
ocean byte.  The oracle of every byte-mask run is the int32 run of the same cells."""
import numpy as np

OCEAN_BYTES = np.array([1, 2, 0x7F, 0x80, 0xFF], dtype=np.uint8)  # all ocean under the byte rule


def byte_mask(m, rng):
    """m's ocean cells (m > 0) as random non-zero bytes, its land as 0"""
    return np.where(m > 0, rng.choice(OCEAN_BYTES, size=m.shape), 0).astype(np.uint8)


class DevPid:
    """__cuda_array_interface__ view of the library's int32 pid rows"""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i4", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def snapshot(h, pid="host"):
    """boxes, pid rows, stats (stage times left out), part loads and all eight neighbour lists of handle h.
    pid: "host" (a numpy copy), "device" (a torch copy on the handle's GPU) or None."""
    out = {"boxes": h.boxes(), "loads": h.part_loads()}
    st = dict(h.stats())
    st.pop("stage_ms")
    out["stats"] = st
    out["nbr"] = [[(h.neighbour_counts(e, per),) + tuple(h.neighbours(e, per)) for e in range(4)] for per in range(2)]
    if pid == "host":
        out["pid"] = h.pid_host()
    elif pid == "device":
        import torch
        ny, nx, _, y_count = h.shape
        out["pid"] = torch.as_tensor(DevPid(h.pid_device(), (max(y_count, 1), nx)), device="cuda").clone()[:y_count]
    return out


def assert_same(a, b, ctx=""):
    """bit for bit: boxes, pid, changes, median_iters, n_ocean, load min / max, edge_cut, gpu_launches, part loads and
    the eight neighbour lists (counts, ids, halos, starts)"""
    assert a["boxes"].tolist() == b["boxes"].tolist(), ctx
    assert a["stats"] == b["stats"], (ctx, a["stats"], b["stats"])
    assert a["loads"].tolist() == b["loads"].tolist(), ctx
    for per in range(2):
        for e in range(4):
            for x, y in zip(a["nbr"][per][e], b["nbr"][per][e]):
                assert np.array_equal(x, y), (ctx, per, e)
    if "pid" in a or "pid" in b:
        pa, pb = a["pid"], b["pid"]
        if isinstance(pa, np.ndarray):
            assert np.array_equal(pa, pb), ctx
        else:
            assert bool((pa == pb).all()), ctx


def run_pair(h, m_i32, set_u8, P, px=False, py=False, pid="host", flags=None):
    """a decomposition of the int32 mask and one of the byte mask (set_u8(h) sets it) on the same handle.  The int32
    mask runs twice, so that both compared runs start from a settled plan and clean buffers (same launch counts)."""
    kw = {} if flags is None else {"flags": flags}
    h.set_mask_host(np.ascontiguousarray(m_i32, dtype=np.int32))
    h.partition(P, px, py, **kw)
    h.partition(P, px, py, **kw)
    a = snapshot(h, pid)
    set_u8(h)
    h.partition(P, px, py, **kw)
    return a, snapshot(h, pid)
