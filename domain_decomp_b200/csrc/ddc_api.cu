// ddc_api.cu -- C ABI (include/ddc.h) over the kernels in ddc_kernels.cuh.
//
// There is NO CPU fallback in this file: every result is produced by the kernels above; if CUDA
// is unavailable every entry point fails with DDC_ERR_CUDA.
#include "ddc.h"
#include "ddc_kernels.cuh"

#ifndef DDC_HOST_EMU
#include <nvtx3/nvToolsExt.h> // header-only; ranges show up in Nsight Systems timelines, cost nothing otherwise
#else
inline void nvtxRangePushA(const char*) { }
inline void nvtxRangePop() { }
#endif

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <string>
#include <vector>

using namespace ddc;

// ------------------------------------------------------------------------------------------------
// NCCL, loaded lazily (only when nranks > 1) so that the library itself has no link-time
// dependency on a particular libnccl and loads on machines without one.
// ------------------------------------------------------------------------------------------------
namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct {
    char internal[128];
} ncclUniqueId;
enum { ncclSuccess = 0 };
enum { nccl_Int32 = 2, nccl_Uint32 = 3 }; // ncclDataType_t: ncclInt32 = 2, ncclUint32 = 3
enum { nccl_Sum = 0, nccl_Max = 2 }; // ncclRedOp_t: ncclSum = 0, ncclProd = 1, ncclMax = 2

struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    std::string err;
    bool load()
    {
        if (lib)
            return true;
        const char* names[] = { "libnccl.so.2", "libnccl.so" };
        for (const char* n : names) {
            lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (lib)
                break;
        }
        if (!lib) {
            err = std::string("cannot load libnccl: ") + dlerror();
            return false;
        }
#define DDC_SYM(field, name)                                                                       \
    *(void**)(&field) = dlsym(lib, name);                                                          \
    if (!field) {                                                                                  \
        err = std::string("libnccl lacks ") + name;                                                \
        return false;                                                                              \
    }
        DDC_SYM(GetUniqueId, "ncclGetUniqueId");
        DDC_SYM(CommInitRank, "ncclCommInitRank");
        DDC_SYM(CommDestroy, "ncclCommDestroy");
        DDC_SYM(AllReduce, "ncclAllReduce");
        DDC_SYM(AllGather, "ncclAllGather");
        DDC_SYM(GroupStart, "ncclGroupStart");
        DDC_SYM(GroupEnd, "ncclGroupEnd");
        DDC_SYM(GetErrorString, "ncclGetErrorString");
#undef DDC_SYM
        return true;
    }
};
NcclApi g_nccl;
thread_local std::string g_create_error;

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n)
    {
        if (n <= cap)
            return cudaSuccess;
        if (p)
            cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess)
            cap = n;
        return e;
    }
    void release()
    {
        if (p)
            cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// One way to launch a kernel.  pdl: programmatic dependent launch -- the kernel may become resident while the
// kernel before it in the stream is still running and waits for it in its own pdl_wait() (ddc_kernels.cuh).
// Test builds (DDC_HOST_EMU, oracle/emu) run the kernel on the host emulation instead.
template <typename... KArgs, typename... Args>
cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl,
    Args&&... args)
{
#ifdef DDC_HOST_EMU
    (void)stream;
    (void)pdl;
    DDC_EMU_LAUNCH(grid, block, smem, kernel(static_cast<KArgs>(args)...));
    return cudaSuccess;
#else
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
#endif
}
// Dynamic shared memory a kernel has been opted in for (cudaFuncAttributeMaxDynamicSharedMemorySize), per device.
// The attribute belongs to the FUNCTION, not to a handle: it is only ever raised, and the bookkeeping is shared by
// all handles of the process (a second handle that set a smaller value used to leave the first one launching
// with more than the function allowed: "invalid argument").
constexpr int MAX_DEVICES = 64;
std::mutex g_optin_mutex;
size_t g_optin[MAX_DEVICES][3]; // x cuts, y cuts (16-bit counts), y cuts (32-bit counts)
template <typename K>
cudaError_t opt_in_smem(K kernel, int device, int which, size_t need)
{
    std::lock_guard<std::mutex> lk(g_optin_mutex);
    size_t& have = g_optin[device % MAX_DEVICES][which];
    if (need <= have)
        return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need);
    if (e == cudaSuccess)
        have = need;
    return e;
}
} // namespace

struct ddc_handle_s {
    int device = 0, rank = 0, nranks = 1;
    ncclComm_t comm = nullptr;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::string err;

    // input
    int nx = 0, ny = 0, y_begin = 0, y_count = 0;
    const void* d_mask = nullptr; // borrowed or == mask_own.p
    int mask_esize = 4; // bytes per mask cell: 4 int32 (ddc_set_mask_*), 1 uint8 (ddc_set_mask_u8_*)
    bool mask_set = false;
    DevBuf<uint8_t> mask_own;

    // state of the last partition
    bool partitioned = false, have_pid = false, have_nbr = false;
    int nparts = 0, px = 0, py = 0;
    ddc_stats stats {};

    // device buffers
    DevBuf<uint8_t> bits;
    DevBuf<unsigned> colcount, colsum, colpfx, rowcount, rowcount_all, ypfx, done;
    DevBuf<DevScalars> sc;
    // the halo plan (ddc_halo_tile_offsets) and its tables on the device
    HaloPlan halo;
    DevBuf<unsigned char> halo_dev;
    bool halo_ok = false; // the plan is of the current decomposition
    bool halo_shard_ok = false; // ... and ddc_halo_shard_offsets was called for it
    int halo_w = 1; // the frame width of the halo calls (ddc_halo_set_width)
    DevBuf<unsigned> gate; // words polled in place of a kernel boundary (see ddc_create)
    DevBuf<Plan> plan;
    DevBuf<int> strips; // x0[P+1] x1[P+1] p0[P+2] S always
    DevBuf<int> boxes; // x0 y0 ex ey, P each
    DevBuf<int> strip_of_col, part_at; // part_at: [strips][ceil(NY / 32)] row -> part table K4 leaves for the labelling kernel
    DevBuf<long long> loads, loadmm;
    DevBuf<int32_t> pid;
    DevBuf<int> nbr_counts, nbr_offsets, nbr_totals, nbr_ids, nbr_halos, nbr_starts;
    int nbr_cap = 0;
    // the plan the launches were sized for, and what it was assumed for (see enqueue_partition)
    int plan_nx = 0, plan_ny = 0, plan_P = 0, aix = 0, aiy = 0;
    bool pending = false, profiled = false; // a step is enqueued but not yet validated
    int last_flags = 0;
    bool debug_ts = false; // DDC_DEBUG_TS=1 (read in ddc_create): time stamps of every phase (Plan::ts)
    PeerSync fin_ps {}; // the exchange state of the last step, for a k_finalize launched from validate()
    size_t xcuts_static = 0, ycuts_static = 0; // static shared memory of the cut kernels (0: not yet asked)
    // what K2 (column counts, scalars) and the scan's last CTA (counters) left clean for a later step: k_init is
    // only launched when the buffers or the geometry of the step differ (index: parity of the exchange slots)
    struct CleanSig {
        const void *col = nullptr, *done = nullptr;
        int ncol = 0, yr_off = 0, rank = -1, ndone = 0;
        bool operator==(const CleanSig& o) const
        {
            return col == o.col && done == o.done && ncol == o.ncol && yr_off == o.yr_off && rank == o.rank && ndone == o.ndone;
        }
    } clean[2];
    bool clean_p2p = false;
    cudaStream_t side_stream = nullptr; // speculative neighbour tables run beside the labelling
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // peer exchange (CUDA IPC): one buffer per rank, mapped by all ranks
    //   [flags: PEER_STAGES * MAX_PEERS u32, padded to 256 B][col: 2 parities x G slots][row: 2 parities x G slots]
    //   slot g of a rank's buffer is WRITTEN by rank g (pushed by its producing kernel) and read locally
    unsigned* xbuf = nullptr; // this rank's buffer
    unsigned* xpeer[MAX_PEERS] = {}; // every rank's buffer as mapped here (xpeer[rank] == xbuf)
    size_t x_colcap = 0, x_rowcap = 0; // capacity of one col / row slot, in 32-bit words
    size_t x_flagcap = 0; // per-block flags of the row-count kernel, per rank
    bool p2p = false, peer_local = false; // peer_local: the peers are handles of this process (ddc_peer_connect)
    unsigned step = 0; // decompositions enqueued so far (the flag value of the exchange barriers)
    // halo exchange across ranks (ddc_halo_*): one buffer per rank, [HALO_HEAD_BYTES head][tiles of this rank's parts]
    char* halo_buf = nullptr; // this rank's buffer
    char* halo_peer[MAX_PEERS] = {}; // every rank's buffer as mapped here (halo_peer[rank] == halo_buf)
    int64_t halo_elems = 0; // capacity for tiles, in doubles
    bool halo_mapped = false, halo_local = false; // halo_local: the peers are handles of this process (ddc_halo_connect)
    unsigned halo_step = 0; // exchanges enqueued since the buffers were joined
    int* halo_err = nullptr; // pinned, device-mapped: set by a halo kernel whose wait timed out
    int* halo_err_dev = nullptr;
    int h_totals[8] = { 0 };
    bool totals_valid = false;
    // Page-locked copy of the small results (boxes, neighbour counts, part loads; the neighbour lists on demand): the
    // getters used to issue one device -> host copy and one synchronisation each -- ~45 of them to read a decomposition,
    // 0.5 ms, against 0.07 ms of decomposing a 528 x 522 grid.  Now: one batch of copies per group, then memcpy.
    int32_t* host_tab = nullptr;
    size_t host_tab_cap = 0; // ints
    bool small_cached = false, lists_cached = false;
    int cache_P = 0, cache_cap = 0;
    Plan* pin_plan = nullptr; // pinned, device-mapped: the last kernel of a step writes the plan here
    Plan* pin_plan_dev = nullptr; // the same memory as the device addresses it
    cudaEvent_t ev[DDC_N_STAGES + 2] = {};
    bool ev_ok = false;
};

namespace {
// a new decomposition (ddc_partition, ddc_neighbours_from_boxes): the halo plan and the shard offsets are stale
void halo_invalidate(ddc_handle_t h)
{
    h->halo_ok = false;
    h->halo_shard_ok = false;
}

int fail(ddc_handle_t h, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h)
        h->err = buf;
    else
        g_create_error = buf;
    return code;
}
#define CUDA_TRY(h, call)                                                                          \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(h, DDC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                __FILE__, __LINE__);                                                               \
    } while (0)
#define NCCL_TRY(h, call)                                                                          \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != ncclSuccess)                                                                     \
            return fail(h, DDC_ERR_NCCL, "%s failed: %s (%s:%d)", #call,                           \
                g_nccl.GetErrorString(r_), __FILE__, __LINE__);                                    \
    } while (0)

struct Tables {
    StripTable st;
    BoxTable bx;
};
Tables tables(ddc_handle_t h, int P)
{
    Tables t;
    int* q = h->strips.p;
    t.st.x0 = q;
    t.st.x1 = q + (P + 1);
    t.st.p0 = q + 2 * (P + 1);
    t.st.S = q + 3 * (P + 1) + 1;
    t.st.always = q + 3 * (P + 1) + 2;
    int* b = h->boxes.p;
    t.bx = { b, b + P, b + 2 * P, b + 3 * P };
    return t;
}

size_t max_dyn_smem(int device)
{
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    return (size_t)v;
}

// Rows per CTA of the mask scan.  Measured on B200 (scripts/kernel_probe.cu): many small CTAs beat
// one fat wave (more independent load streams in flight, no tail), and the per-CTA epilogue of 1024
// column atomics is cheap; 128 rows keeps the atomics at 8 per 1024 mask cells.  Smaller shards
// (multi-GPU, small grids) step down so that the grid still covers the SMs a few times.
template <typename K>
int pick_rows_per_cta(K kernel, int rows, int gridx)
{
    int per_sm = 0, sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    // CTAs for two full waves -- but on a narrow grid (few column blocks) all CTAs in flight add into the same few
    // thousand column counters, and chunks small enough for two waves spend their time in those atomics: there,
    // three quarters of ONE wave (everything resident at once) with 4-16 x fewer atomics is faster
    // (measured, profiles/r2r_sweep.jsonl: 4096^2 113 -> 107 us with 32 rows instead of 8, 8192^2 174 -> 170 us
    //  with 64-128 instead of 32; 32768 columns: unchanged)
    const long long want = (gridx <= 8 ? 3LL : 8LL) * per_sm * sms / 4;
    int rpc = 128;
    while (rpc > 8 && (long long)gridx * ((rows + rpc - 1) / rpc) < want)
        rpc >>= 1;
    return rpc;
}

// K7 + scans on whatever boxes / strips are in the tables
int run_neighbours(ddc_handle_t h, int P, int nx, int ny, int px, int py)
{
    Tables t = tables(h, P);
    cudaStream_t s = h->stream;
    const int cap = 3 * P + 64;
    CUDA_TRY(h, h->nbr_counts.ensure((size_t)8 * P));
    CUDA_TRY(h, h->nbr_offsets.ensure((size_t)8 * (P + 1)));
    CUDA_TRY(h, h->nbr_totals.ensure(8));
    if (h->nbr_cap < cap) {
        CUDA_TRY(h, h->nbr_ids.ensure((size_t)8 * cap));
        CUDA_TRY(h, h->nbr_halos.ensure((size_t)8 * cap));
        CUDA_TRY(h, h->nbr_starts.ensure((size_t)8 * cap));
        h->nbr_cap = cap;
    }
    const int warps_per_cta = 8;
    const int grid = (std::max(P, 8) + warps_per_cta - 1) / warps_per_cta; // >= 8 * pad32(P) threads
    CUDA_TRY(h, launch_k(k_neighbours<false>, dim3(grid), dim3(256), 0, s, false, t.bx, P, nx, ny, px, py, t.st,
        h->nbr_counts.p, nullptr, nullptr, h->nbr_cap, nullptr, nullptr, nullptr, h->sc.p, nullptr));
    CUDA_TRY(h, launch_k(k_scan_counts, dim3(8), dim3(1024), 0, s, false, h->nbr_counts.p, P, h->nbr_offsets.p,
        h->nbr_totals.p, nullptr));
    CUDA_TRY(h, launch_k(k_neighbours<true>, dim3(grid), dim3(256), 0, s, false, t.bx, P, nx, ny, px, py, t.st,
        h->nbr_counts.p, h->nbr_offsets.p, h->nbr_totals.p, h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p, h->nbr_starts.p,
        h->sc.p, nullptr));
    h->stats.gpu_launches += 3;
    CUDA_TRY(h, cudaGetLastError());
    h->totals_valid = false;
    h->small_cached = h->lists_cached = false;
    h->have_nbr = true;
    return DDC_OK;
}

// make h_totals valid; re-run the fill pass with exact capacity if the bounded one overflowed
int fetch_totals(ddc_handle_t h)
{
    if (h->totals_valid)
        return DDC_OK;
    DevScalars hs;
    CUDA_TRY(h, cudaMemcpyAsync(h->h_totals, h->nbr_totals.p, sizeof(int) * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&hs, h->sc.p, sizeof hs, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (hs.overflow) {
        int need = 0;
        for (int l = 0; l < 8; l++)
            need = std::max(need, h->h_totals[l]);
        CUDA_TRY(h, h->nbr_ids.ensure((size_t)8 * need));
        CUDA_TRY(h, h->nbr_halos.ensure((size_t)8 * need));
        CUDA_TRY(h, h->nbr_starts.ensure((size_t)8 * need));
        h->nbr_cap = need;
        CUDA_TRY(h, cudaMemsetAsync(&h->sc.p->overflow, 0, sizeof(int), h->stream));
        CUDA_TRY(h, cudaMemsetAsync(&h->sc.p->edge_cut, 0, sizeof(unsigned long long), h->stream));
        Tables t = tables(h, h->nparts);
        const int grid = (std::max(h->nparts, 8) + 7) / 8;
        CUDA_TRY(h, launch_k(k_neighbours<true>, dim3(grid), dim3(256), 0, h->stream, false, t.bx, h->nparts, h->nx, h->ny,
            h->px, h->py, t.st, h->nbr_counts.p, h->nbr_offsets.p, h->nbr_totals.p, h->nbr_cap, h->nbr_ids.p,
            h->nbr_halos.p, h->nbr_starts.p, h->sc.p, nullptr));
        CUDA_TRY(h, cudaGetLastError());
        CUDA_TRY(h, cudaMemcpyAsync(&hs, h->sc.p, sizeof hs, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->stats.edge_cut = (int64_t)hs.edge_cut;
    h->totals_valid = true;
    return DDC_OK;
}

// layout of the page-locked copy (ints): boxes [4 P] | counts [8 P] | loads [2 P] | ids, halos, starts [8 cap] each
struct HostTab {
    int32_t *boxes, *counts, *ids, *halos, *starts;
    int64_t* loads;
};
HostTab host_tab_of(ddc_handle_t h)
{
    const size_t P = (size_t)h->cache_P, cap = (size_t)h->cache_cap;
    HostTab t;
    t.boxes = h->host_tab;
    t.counts = t.boxes + 4 * P;
    t.loads = reinterpret_cast<int64_t*>(t.counts + 8 * P); // (12 P ints: 8-byte aligned)
    t.ids = t.counts + 8 * P + 2 * P;
    t.halos = t.ids + 8 * cap;
    t.starts = t.halos + 8 * cap;
    return t;
}
// boxes, neighbour counts and part loads of the current decomposition in page-locked host memory
int fetch_small(ddc_handle_t h)
{
    if (h->small_cached)
        return DDC_OK;
    if (h->have_nbr) { // (first: an overflowed fill pass is run again and may grow the lists)
        int rc = fetch_totals(h);
        if (rc)
            return rc;
    }
    const size_t P = (size_t)h->nparts, cap = h->have_nbr ? (size_t)h->nbr_cap : 0;
    const size_t need = 14 * P + 24 * cap + 16;
    if (need > h->host_tab_cap) {
        if (h->host_tab)
            cudaFreeHost(h->host_tab);
        h->host_tab = nullptr;
        h->host_tab_cap = 0;
        CUDA_TRY(h, cudaHostAlloc((void**)&h->host_tab, need * sizeof(int32_t), cudaHostAllocDefault));
        h->host_tab_cap = need;
    }
    h->cache_P = (int)P;
    h->cache_cap = (int)cap;
    h->lists_cached = false;
    const HostTab t = host_tab_of(h);
    CUDA_TRY(h, cudaMemcpyAsync(t.boxes, h->boxes.p, 4 * P * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (h->have_nbr)
        CUDA_TRY(h, cudaMemcpyAsync(t.counts, h->nbr_counts.p, 8 * P * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(t.loads, h->loads.p, P * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->small_cached = true;
    return DDC_OK;
}
// + the neighbour lists (whole arrays: their used parts are most of them)
int fetch_lists(ddc_handle_t h)
{
    int rc = fetch_small(h);
    if (rc || h->lists_cached || !h->have_nbr)
        return rc;
    const HostTab t = host_tab_of(h);
    const size_t n = 8 * (size_t)h->cache_cap * sizeof(int32_t);
    CUDA_TRY(h, cudaMemcpyAsync(t.ids, h->nbr_ids.p, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(t.halos, h->nbr_halos.p, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(t.starts, h->nbr_starts.p, n, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->lists_cached = true;
    return DDC_OK;
}

// ---- CUDA IPC and peer access, shared by the histogram exchange (ddc_peer_*) and the halo exchange (ddc_halo_*) ----
// the IPC handle of `buf` (the base of a cudaMalloc allocation) into out[DDC_IPC_HANDLE_BYTES]
int ipc_export(ddc_handle_t h, void* buf, void* out)
{
    cudaIpcMemHandle_t ipc;
    CUDA_TRY(h, cudaIpcGetMemHandle(&ipc, buf));
    static_assert(sizeof(cudaIpcMemHandle_t) == DDC_IPC_HANDLE_BYTES, "IPC handle size");
    memcpy(out, &ipc, sizeof ipc);
    return DDC_OK;
}
// map every other rank's buffer (all_handles: nranks IPC handles in rank order); mapped[rank] = own
template <typename T>
int ipc_import(ddc_handle_t h, const void* all_handles, T* own, T** mapped)
{
    CUDA_TRY(h, cudaSetDevice(h->device));
    for (int q = 0; q < h->nranks; q++) {
        if (q == h->rank) {
            mapped[q] = own;
            continue;
        }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const char*)all_handles + (size_t)q * DDC_IPC_HANDLE_BYTES, sizeof ipc);
        void* p = nullptr;
        CUDA_TRY(h, cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
        mapped[q] = (T*)p;
    }
    return DDC_OK;
}
// unmap what ipc_import mapped (local: the peers are handles of this process, nothing was IPC-mapped); the first error
template <typename T>
cudaError_t ipc_unmap(ddc_handle_t h, T** mapped, bool local)
{
    cudaError_t first = cudaSuccess;
    for (int q = 0; q < h->nranks && q < MAX_PEERS; q++) {
        if (mapped[q] && q != h->rank && !local) {
            const cudaError_t e = cudaIpcCloseMemHandle(mapped[q]);
            if (first == cudaSuccess)
                first = e;
        }
        mapped[q] = nullptr;
    }
    return first;
}
// handles of one process: every device may access the memory of every other one
int enable_peer_access(ddc_handle_t* handles, int n)
{
    for (int q = 0; q < n; q++) {
        ddc_handle_t h = handles[q];
        CUDA_TRY(h, cudaSetDevice(h->device));
        for (int r = 0; r < n; r++) {
            if (handles[r]->device == h->device)
                continue;
            int can = 0;
            CUDA_TRY(h, cudaDeviceCanAccessPeer(&can, h->device, handles[r]->device));
            if (!can)
                return fail(h, DDC_ERR_CUDA, "device %d cannot access the memory of device %d", h->device, handles[r]->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(handles[r]->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled)
                cudaGetLastError(); // not an error
            else if (e != cudaSuccess)
                return fail(h, DDC_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", h->device, handles[r]->device,
                    cudaGetErrorString(e));
        }
    }
    return DDC_OK;
}
} // namespace

// ------------------------------------------------------------------------------------------------
extern "C" {

const char* ddc_version(void) { return "domain_decomp_b200 0.1 (sm_100a)"; }

const char* ddc_last_error(ddc_handle_t h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int ddc_get_nccl_unique_id(void* out)
{
    if (!out)
        return fail(nullptr, DDC_ERR_ARG, "ddc_get_nccl_unique_id: null output");
    if (!g_nccl.load())
        return fail(nullptr, DDC_ERR_NCCL, "%s", g_nccl.err.c_str());
    ncclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != ncclSuccess)
        return fail(nullptr, DDC_ERR_NCCL, "ncclGetUniqueId failed: %s", g_nccl.GetErrorString(r));
    memcpy(out, &id, DDC_NCCL_ID_BYTES);
    return DDC_OK;
}

int ddc_create(ddc_handle_t* out, int device, int rank, int nranks, const void* nccl_id)
{
    if (!out || nranks < 1 || rank < 0 || rank >= nranks)
        return fail(nullptr, DDC_ERR_ARG, "ddc_create: bad arguments");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, DDC_ERR_CUDA, "ddc_create: no CUDA device (%s); this library has no CPU path",
            e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev)
        return fail(nullptr, DDC_ERR_ARG, "ddc_create: device %d out of range (have %d)", device, ndev);
    ddc_handle_t h = new ddc_handle_s();
    h->device = device;
    h->rank = rank;
    h->nranks = nranks;
#define CREATE_TRY(call)                                                                           \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            fail(nullptr, DDC_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));           \
            ddc_destroy(h); /* releases whatever was created so far */                             \
            return DDC_ERR_CUDA;                                                                   \
        }                                                                                          \
    } while (0)
    CREATE_TRY(cudaSetDevice(device));
    CREATE_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    {
        // highest priority: the small neighbour kernels must get SM slots while the labelling
        // kernel still has tens of thousands of CTAs queued (also on several GPUs, where every rank builds ALL
        // neighbour tables beside a labelling kernel that has only 1 / G of the cells: DESIGN.md 5)
        int least = 0, greatest = 0;
        CREATE_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CREATE_TRY(cudaStreamCreateWithPriority(&h->side_stream, cudaStreamNonBlocking, greatest));
    }
    CREATE_TRY(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CREATE_TRY(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    CREATE_TRY(cudaHostAlloc((void**)&h->pin_plan, sizeof(Plan), cudaHostAllocMapped));
    CREATE_TRY(cudaHostGetDevicePointer((void**)&h->pin_plan_dev, h->pin_plan, 0));
    memset(h->pin_plan, 0, sizeof(Plan));
    for (auto& ev : h->ev)
        CREATE_TRY(cudaEventCreate(&ev));
    h->ev_ok = true;
    const char* ts = getenv("DDC_DEBUG_TS");
    h->debug_ts = ts && *ts && atoi(ts) != 0;
    CREATE_TRY(h->gate.ensure(2)); // [0] K4 -> second stream (BoxGate), [1] k_sum_cols -> K2 (ChainWord)
    CREATE_TRY(cudaMemset(h->gate.p, 0, 2 * sizeof(unsigned)));
    CREATE_TRY(h->sc.ensure(1));
    CREATE_TRY(h->plan.ensure(1));
    CREATE_TRY(cudaMemset(h->plan.p, 0, sizeof(Plan)));
#undef CREATE_TRY
    if (nranks > 1 && nccl_id) { // without an id the ranks can only exchange through peer memory (ddc_peer_*)
        if (!g_nccl.load()) {
            ddc_destroy(h);
            return fail(nullptr, DDC_ERR_NCCL, "%s", g_nccl.err.c_str());
        }
        ncclUniqueId id;
        memcpy(&id, nccl_id, DDC_NCCL_ID_BYTES);
        int r = g_nccl.CommInitRank(&h->comm, nranks, id, rank);
        if (r != ncclSuccess) {
            ddc_destroy(h);
            return fail(nullptr, DDC_ERR_NCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString(r));
        }
    }
    *out = h;
    return DDC_OK;
}

int ddc_destroy(ddc_handle_t h)
{
    if (!h)
        return DDC_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->side_stream)
        cudaStreamSynchronize(h->side_stream);
    if (h->comm)
        g_nccl.CommDestroy(h->comm);
    ipc_unmap(h, h->xpeer, h->peer_local);
    if (h->xbuf)
        cudaFree(h->xbuf);
    ipc_unmap(h, h->halo_peer, h->halo_local);
    if (h->halo_buf)
        cudaFree(h->halo_buf);
    if (h->halo_err)
        cudaFreeHost(h->halo_err);
    h->mask_own.release();
    h->bits.release();
    h->colcount.release();
    h->colsum.release();
    h->colpfx.release();
    h->rowcount.release();
    h->rowcount_all.release();
    h->ypfx.release();
    h->done.release();
    h->sc.release();
    h->gate.release();
    h->halo_dev.release();
    h->plan.release();
    h->strips.release();
    h->boxes.release();
    h->strip_of_col.release();
    h->part_at.release();
    h->loads.release();
    h->loadmm.release();
    h->pid.release();
    h->nbr_counts.release();
    h->nbr_offsets.release();
    h->nbr_totals.release();
    h->nbr_ids.release();
    h->nbr_halos.release();
    h->nbr_starts.release();
    if (h->pin_plan)
        cudaFreeHost(h->pin_plan);
    if (h->host_tab)
        cudaFreeHost(h->host_tab);
    if (h->ev_ok)
        for (auto& ev : h->ev)
            cudaEventDestroy(ev);
    if (h->ev_fork)
        cudaEventDestroy(h->ev_fork);
    if (h->ev_join)
        cudaEventDestroy(h->ev_join);
    if (h->side_stream)
        cudaStreamDestroy(h->side_stream);
    if (h->own_stream)
        cudaStreamDestroy(h->own_stream);
    delete h;
    return DDC_OK;
}

static void peer_capacity(int nx, int ny, int nparts, int G, size_t* colcap, size_t* rowcap, size_t* flagcap)
{
    int ix, iy;
    guess_plan(nparts, nx, ny, &ix, &iy);
    const size_t Scap = (size_t)std::min<long long>(nparts, 1LL << std::min(ix, 30));
    const size_t Rmax = ((size_t)ny + G - 1) / G;
    const size_t elems = iy > 0 ? Scap * ((Rmax + 31) & ~(size_t)31) : 0; // whole row blocks (row_count_index)
    // a slot holds either the rank's own 32-bit counts + the G y-range pairs, or a peer's data + flag words
    // (ll_word: at most one 8-byte word per column, two for the y-range)
    const size_t yr_off = ((size_t)nx + 3) & ~(size_t)3;
    *colcap = (std::max(yr_off + 2 * (size_t)G, 2 * (yr_off + 2)) + 4 + 3) & ~(size_t)3;
    *rowcap = ((nx < 65536 ? (elems + 1) / 2 : elems) + 4 + 3) & ~(size_t)3;
    *flagcap = iy > 0 ? ((Rmax + 7) / 8 + 4 + 3) & ~(size_t)3 : 0; // one flag per block of the row-count kernel (>= 8 rows each)
}
// words of one rank's exchange buffer: [flags][col: 2 parities x G slots][row: 2 parities x G slots][row flags: G x flagcap]
static size_t peer_words(int G, size_t colcap, size_t rowcap, size_t flagcap)
{
    return 64 + 2 * (size_t)G * (colcap + rowcap) + (size_t)G * flagcap;
}

int ddc_peer_export(ddc_handle_t h, int nx, int ny, int nparts, void* ipc_handle_out)
{
    if (!h || !ipc_handle_out || nx < 1 || ny < 1 || nparts < 1)
        return fail(h, DDC_ERR_ARG, "ddc_peer_export: bad arguments");
    if (h->nranks > MAX_PEERS)
        return fail(h, DDC_ERR_ARG, "ddc_peer_export: at most %d ranks", MAX_PEERS);
    if (h->xbuf)
        return fail(h, DDC_ERR_STATE, "ddc_peer_export: already exported");
    CUDA_TRY(h, cudaSetDevice(h->device));
    peer_capacity(nx, ny, nparts, h->nranks, &h->x_colcap, &h->x_rowcap, &h->x_flagcap);
    const size_t words = peer_words(h->nranks, h->x_colcap, h->x_rowcap, h->x_flagcap);
    CUDA_TRY(h, cudaMalloc((void**)&h->xbuf, words * sizeof(unsigned)));
    CUDA_TRY(h, cudaMemset(h->xbuf, 0, words * sizeof(unsigned)));
    return ipc_export(h, h->xbuf, ipc_handle_out);
}

int ddc_peer_import(ddc_handle_t h, const void* all_handles)
{
    if (!h || !all_handles)
        return fail(h, DDC_ERR_ARG, "ddc_peer_import: bad arguments");
    if (!h->xbuf)
        return fail(h, DDC_ERR_STATE, "ddc_peer_import: call ddc_peer_export() first");
    if (int rc = ipc_import(h, all_handles, h->xbuf, h->xpeer))
        return rc;
    h->p2p = true;
    return DDC_OK;
}

int ddc_peer_connect(ddc_handle_t* handles, int n, int nx, int ny, int nparts)
{
    if (!handles || n < 1 || n > MAX_PEERS || nx < 1 || ny < 1 || nparts < 1)
        return fail(nullptr, DDC_ERR_ARG, "ddc_peer_connect: bad arguments");
    for (int q = 0; q < n; q++)
        if (!handles[q] || handles[q]->nranks != n || handles[q]->rank != q || handles[q]->xbuf)
            return fail(handles[q], DDC_ERR_ARG, "ddc_peer_connect: handle %d must be rank %d of %d and not yet exported", q, q, n);
    if (int rc = enable_peer_access(handles, n))
        return rc;
    for (int q = 0; q < n; q++) {
        ddc_handle_t h = handles[q];
        CUDA_TRY(h, cudaSetDevice(h->device));
        peer_capacity(nx, ny, nparts, n, &h->x_colcap, &h->x_rowcap, &h->x_flagcap);
        const size_t words = peer_words(n, h->x_colcap, h->x_rowcap, h->x_flagcap);
        CUDA_TRY(h, cudaMalloc((void**)&h->xbuf, words * sizeof(unsigned)));
        CUDA_TRY(h, cudaMemset(h->xbuf, 0, words * sizeof(unsigned)));
    }
    // the words and flags of the exchange carry the step number: the ranks count their steps together from here on
    unsigned step = 0;
    for (int q = 0; q < n; q++)
        step = std::max(step, handles[q]->step);
    for (int q = 0; q < n; q++) {
        for (int r = 0; r < n; r++)
            handles[q]->xpeer[r] = handles[r]->xbuf;
        handles[q]->p2p = true;
        handles[q]->peer_local = true;
        handles[q]->step = step;
    }
    return DDC_OK;
}

int ddc_peer_close(ddc_handle_t h)
{
    if (!h)
        return DDC_ERR_ARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, ipc_unmap(h, h->xpeer, h->peer_local));
    h->p2p = false;
    return DDC_OK;
}

int ddc_host_alloc(void** ptr, size_t bytes)
{
    if (!ptr)
        return DDC_ERR_ARG;
    *ptr = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, DDC_ERR_CUDA, "ddc_host_alloc: no CUDA device");
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess)
        return fail(nullptr, DDC_ERR_NOMEM, "cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    *ptr = p;
    return DDC_OK;
}

int ddc_host_free(void* ptr)
{
    if (ptr && cudaFreeHost(ptr) != cudaSuccess)
        return fail(nullptr, DDC_ERR_CUDA, "cudaFreeHost failed");
    return DDC_OK;
}

int ddc_set_stream(ddc_handle_t h, void* cuda_stream)
{
    if (!h)
        return DDC_ERR_ARG;
    cudaStream_t next = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    if (next != h->stream) // nothing orders the new stream after the old one's last step: start from k_init again
        h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig();
    h->stream = next;
    return DDC_OK;
}

void ddc_shard_rows(int ny, int nranks, int rank, int* y_begin, int* y_count)
{
    const int rpr = (ny + nranks - 1) / nranks;
    int b = std::min(ny, rank * rpr), e = std::min(ny, b + rpr);
    if (y_begin)
        *y_begin = b;
    if (y_count)
        *y_count = e - b;
}

void ddc_shard_parts(int nparts, int nranks, int rank, int* p_begin, int* p_count)
{
    int b = 0, e = 0;
    if (nparts > 0 && nranks > 0 && rank >= 0 && rank < nranks) {
        b = (int)((long long)rank * nparts / nranks);
        e = (int)((long long)(rank + 1) * nparts / nranks);
    }
    if (p_begin)
        *p_begin = b;
    if (p_count)
        *p_count = e - b;
}

static int check_shard(ddc_handle_t h, int nx, int ny, int y_begin, int y_count)
{
    if (nx < 1 || ny < 1 || (long long)nx * ny > (long long)INT_MAX)
        return fail(h, DDC_ERR_ARG, "mask extents %d x %d out of range (the reference ids are int)", nx, ny);
    int b, c;
    ddc_shard_rows(ny, h->nranks, h->rank, &b, &c);
    if (b != y_begin || c != y_count)
        return fail(h, DDC_ERR_ARG, "rank %d/%d must hold rows [%d,%d) of %d, got [%d,%d)", h->rank,
            h->nranks, b, b + c, ny, y_begin, y_begin + y_count);
    return DDC_OK;
}

// the four set_mask calls: esize bytes per cell; host: copied into the handle's buffer, else borrowed
static int set_mask(ddc_handle_t h, const void* rows, int esize, bool host, int nx, int ny, int y_begin, int y_count,
    const char* name)
{
    if (!h)
        return DDC_ERR_ARG;
    int rc = check_shard(h, nx, ny, y_begin, y_count);
    if (rc)
        return rc;
    if (!rows && y_count > 0)
        return fail(h, DDC_ERR_ARG, "%s: null mask", name);
    if (host) {
        CUDA_TRY(h, cudaSetDevice(h->device));
        const size_t n = (size_t)nx * y_count * esize;
        CUDA_TRY(h, h->mask_own.ensure(n));
        if (n)
            CUDA_TRY(h, cudaMemcpyAsync(h->mask_own.p, rows, n, cudaMemcpyHostToDevice, h->stream));
        rows = h->mask_own.p;
    }
    h->d_mask = rows;
    h->mask_esize = esize;
    h->nx = nx;
    h->ny = ny;
    h->y_begin = y_begin;
    h->y_count = y_count;
    h->mask_set = true;
    h->partitioned = false;
    return DDC_OK;
}

int ddc_set_mask_device(ddc_handle_t h, const int32_t* rows, int nx, int ny, int y_begin, int y_count)
{
    return set_mask(h, rows, 4, false, nx, ny, y_begin, y_count, "ddc_set_mask_device");
}

int ddc_set_mask_host(ddc_handle_t h, const int32_t* rows, int nx, int ny, int y_begin, int y_count)
{
    return set_mask(h, rows, 4, true, nx, ny, y_begin, y_count, "ddc_set_mask_host");
}

int ddc_set_mask_u8_device(ddc_handle_t h, const uint8_t* rows, int nx, int ny, int y_begin, int y_count)
{
    return set_mask(h, rows, 1, false, nx, ny, y_begin, y_count, "ddc_set_mask_u8_device");
}

int ddc_set_mask_u8_host(ddc_handle_t h, const uint8_t* rows, int nx, int ny, int y_begin, int y_count)
{
    return set_mask(h, rows, 1, true, nx, ny, y_begin, y_count, "ddc_set_mask_u8_host");
}

namespace {
int validate(ddc_handle_t h);
}

int ddc_synchronize(ddc_handle_t h)
{
    if (!h)
        return DDC_ERR_ARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->partitioned && h->pending) {
        if (int rc = validate(h)) // waits for the step and settles the plan
            return rc;
    } else
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    if (h->halo_err && *(volatile int*)h->halo_err) { // a halo exchange kernel gave up waiting for a rank
        *(volatile int*)h->halo_err = 0;
        return fail(h, DDC_ERR_PEER, "halo exchange timed out: a rank did not reach the exchange within %.1f s",
            (double)PEER_TIMEOUT_NS * 1e-9);
    }
    return DDC_OK;
}

// ------------------------------------------------------------------------------------------------
// the hot path
// ------------------------------------------------------------------------------------------------
namespace {
// K5 (one block): `changes` of all ranks; when nothing moved, the naive blocks and the neighbour tables rebuilt
// from them; the plan into the host's pinned copy.  Uses nparts / px / py / nx / ny of the handle.
int launch_finalize(ddc_handle_t h, const PeerSync& ps, bool want_nbr)
{
    const int P = h->nparts;
    Tables t = tables(h, P);
    const NaiveParams nv = naive_params(P, h->nx, h->ny);
    const NbrTables nb = { h->nbr_counts.p, h->nbr_offsets.p, h->nbr_totals.p, h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p,
        h->nbr_starts.p };
    CUDA_TRY(h, launch_k(k_finalize, dim3(1), dim3(1024), 0, h->stream, false, ps, P, h->nx, h->ny, h->px, h->py, nv, h->sc.p,
        h->plan.p, t.st, t.bx, want_nbr ? 1 : 0, nb, h->pin_plan_dev));
    return DDC_OK;
}

int enqueue_partition(ddc_handle_t h, int nparts, int px, int py, int flags)
{
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int P = nparts, NX = h->nx, NY = h->ny, rows = h->y_count, G = h->nranks;
    const int NG = (NX + 127) / 128;
    const bool profile = flags & DDC_PROFILE;
    const bool want_pid = flags & DDC_WANT_PID;
    const bool want_nbr = (flags & DDC_WANT_NEIGHBOURS) && P > 1; // P == 1 returns early (Q4)
    cudaStream_t s = h->stream;
    h->partitioned = false;
    h->have_pid = false;
    h->have_nbr = false;
    h->totals_valid = false;
    h->small_cached = h->lists_cached = false;
    halo_invalidate(h);
    memset(&h->stats, 0, sizeof h->stats);
    int launches = 0;
    // stage i begins: a CUDA event when profiling, and an NVTX range (the host-side enqueue of the stage; Nsight
    // Systems projects it onto the kernels) -- SURVEY 5 "profiling hooks"; the reference has Zoltan's timers
    static const char* const stage_name[DDC_N_STAGES] = { "ddc:mask_scan", "ddc:x_cuts", "ddc:strip_rows", "ddc:y_cuts",
        "ddc:neighbours+label", "ddc:step_end", "ddc:done", "ddc:done" };
    int open_range = -1;
    auto mark = [&](int i) {
        if (profile)
            cudaEventRecord(h->ev[i], s);
        if (open_range >= 0)
            nvtxRangePop();
        open_range = i < 6 ? i : -1;
        if (open_range >= 0)
            nvtxRangePushA(stage_name[i]);
    };
    struct RangeGuard { // error returns leave no range open
        int* open;
        ~RangeGuard()
        {
            if (*open >= 0)
                nvtxRangePop();
            nvtxRangePop();
        }
    } range_guard { &open_range };
    nvtxRangePushA("ddc_partition");

    // the assumed plan
    if (h->plan_nx != NX || h->plan_ny != NY || h->plan_P != P) {
        guess_plan(P, NX, NY, &h->aix, &h->aiy);
        h->plan_nx = NX;
        h->plan_ny = NY;
        h->plan_P = P;
    }
    const int aix = h->aix, aiy = h->aiy;
    const int Scap = (int)std::min<long long>(P, 1LL << std::min(aix, 30)); // strips after aix levels
    const bool ycuts = aiy > 0 && P > 1;
    const bool narrow = NX < 65536; // a strip row holds < 65536 cells: 16-bit row counts

    // buffers
    const int NB = NG * 16; // bytes per bit-map row
    const int yr_off = (NX + 3) & ~3; // per-rank y-range pairs follow the column counts
    const int ncol = yr_off + 2 * G;
    const int Rmax = (NY + G - 1) / G;
    CUDA_TRY(h, h->bits.ensure((size_t)std::max(rows, 1) * NB));
    CUDA_TRY(h, h->colcount.ensure(ncol));
    if (G > 1)
        CUDA_TRY(h, h->colsum.ensure(ncol));
    CUDA_TRY(h, h->strips.ensure((size_t)3 * (P + 1) + 3));
    CUDA_TRY(h, h->boxes.ensure((size_t)4 * P));
    CUDA_TRY(h, h->strip_of_col.ensure(NX));
    const int nchunk = (NY + 31) / 32;
    if (ycuts)
        CUDA_TRY(h, h->part_at.ensure((size_t)Scap * nchunk));
    CUDA_TRY(h, h->loads.ensure(P));
    CUDA_TRY(h, h->loadmm.ensure(2));
    if (want_pid)
        CUDA_TRY(h, h->pid.ensure((size_t)std::max(rows, 1) * NX));
    const size_t rc_elems = (size_t)Scap * (((size_t)Rmax + 31) & ~(size_t)31); // per rank, whole row blocks
    const size_t rc_words = narrow ? (rc_elems + 1) / 2 : rc_elems; // 32-bit words per rank
    const size_t rank_stride = narrow ? rc_words * 2 : rc_words; // elements between two ranks' blocks
    if (ycuts) {
        CUDA_TRY(h, h->rowcount.ensure(rc_words + 4));
        if (G > 1)
            CUDA_TRY(h, h->rowcount_all.ensure(rc_words * G + 4));
    }
    // prefix sums + the bit map of the non-empty bins (ddc_kernels.cuh: Hist)
    // (+ the sets of two RCB levels, see rcb_levels)
    const size_t xneed = sizeof(unsigned) * ((((size_t)NX + 1 + 3) & ~(size_t)3) + hist_bitmap_words(NX)) + LEVEL_NODES_BYTES;
    const size_t yneed = sizeof(unsigned) * ((((size_t)NY + 1 + 3) & ~(size_t)3) + hist_bitmap_words(NY)) + LEVEL_NODES_BYTES;
    const size_t lim = max_dyn_smem(h->device);
    if (!h->xcuts_static) { // what the cut kernels hold statically counts against the same per-block limit
        cudaFuncAttributes fa;
        CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_xcuts<true>));
        h->xcuts_static = fa.sharedSizeBytes + 64;
        CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_ycuts<uint16_t, true>));
        h->ycuts_static = fa.sharedSizeBytes + 64;
    }
    const int x_smem = xneed + h->xcuts_static <= lim, y_smem = yneed + h->ycuts_static <= lim;
    const int ygrid = std::max(1, std::min(Scap, 148 * 2));
    if (!x_smem)
        CUDA_TRY(h, h->colpfx.ensure((size_t)NX + 1));
    if (ycuts && !y_smem)
        CUDA_TRY(h, h->ypfx.ensure((size_t)ygrid * (((size_t)NY + 1 + 3) & ~(size_t)3)));
    if (want_nbr) {
        const int cap = 3 * P + 64;
        CUDA_TRY(h, h->nbr_counts.ensure((size_t)8 * P));
        CUDA_TRY(h, h->nbr_offsets.ensure((size_t)8 * (P + 1)));
        CUDA_TRY(h, h->nbr_totals.ensure(8));
        if (h->nbr_cap < cap) {
            CUDA_TRY(h, h->nbr_ids.ensure((size_t)8 * cap));
            CUDA_TRY(h, h->nbr_halos.ensure((size_t)8 * cap));
            CUDA_TRY(h, h->nbr_starts.ensure((size_t)8 * cap));
            h->nbr_cap = cap;
        }
    }
    Tables t = tables(h, P);
    const NaiveParams nv = naive_params(P, NX, NY);

    // exchange mode: peer memory when the buffers were exchanged and are large enough, else NCCL
    h->step++;
    const int col_packed = Rmax < 65536 ? 1 : 0; // a rank's column counts fit 16 bits: two per data + flag word
    const size_t col_need = std::max<size_t>(ncol, 2 * (ll_column_words(yr_off, col_packed) + 2));
    const bool p2p = G > 1 && h->p2p && col_need <= h->x_colcap && (!ycuts || rc_words + 4 <= h->x_rowcap);
    if (G > 1 && !p2p && !h->comm)
        return fail(h, DDC_ERR_STATE, "%d ranks but no exchange path: created without a NCCL id and %s", G,
            h->p2p ? "the decomposition exceeds the exported peer buffers" : "no peer buffers imported");
    const int par = (int)(h->step & 1u);
    const bool pdl = !profile; // (event records between the kernels would break the chain anyway)
    unsigned long long* dbg = h->debug_ts
        ? reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(h->plan.p) + offsetof(Plan, ts))
        : nullptr;
    if (dbg)
        CUDA_TRY(h, cudaMemsetAsync(dbg, 0, sizeof(((Plan*)nullptr)->ts), s));
    constexpr size_t XFLAGS = 64; // words reserved for the flags at the head of an exchange buffer
    // slot `slot` (written by rank `slot`) of the buffer of rank q, for this step's parity
    auto xcol = [&](int q, int slot) { return h->xpeer[q] + XFLAGS + ((size_t)par * G + slot) * h->x_colcap; };
    auto xrow = [&](int q, int slot) {
        return h->xpeer[q] + XFLAGS + 2 * (size_t)G * h->x_colcap + ((size_t)par * G + slot) * h->x_rowcap;
    };
    // this rank's counts accumulate in plain device memory (the scan's atomics into the peer-mapped exchange buffer ran
    // the scan ~5 % slower on 8 GPUs); only the peers' slots of the exchange buffer are used
    unsigned* colcount = h->colcount.p;
    unsigned* rowcount = p2p ? xrow(h->rank, h->rank) : h->rowcount.p;
    PeerSync ps {};
    ps.rank = h->rank;
    ps.G = G;
    ps.enabled = p2p ? 1 : 0;
    ps.step = h->step;
    PeerCols pc {};
    PeerRows pr {};
    PeerPush push_col {}, push_row {};
    push_col.rank = push_row.rank = h->rank;
    if (p2p) {
        for (int q = 0; q < G; q++) {
            ps.flags[q] = h->xpeer[q];
            pc.col[q] = q == h->rank ? colcount : xcol(h->rank, q); // what rank q pushed into my buffer
            pr.row[q] = xrow(h->rank, q);
            push_col.dst[q] = xcol(q, h->rank); // my slot in rank q's buffer
            push_row.dst[q] = xrow(q, h->rank);
        }
        pc.n = pr.n = push_col.n = push_row.n = G;
        pc.own = h->rank;
        pc.packed = push_col.packed = col_packed;
    } else {
        pc.col[0] = colcount;
        pc.n = pr.n = 1;
        push_col.dst[0] = colcount;
        push_row.dst[0] = rowcount;
        push_col.n = push_row.n = 1;
    }

    mark(0);
    // ---- K1: mask scan -----------------------------------------------------------------------
    const int gridx = (NG + 7) / 8;
    // counters of the "last block" patterns: [0, gridx] mask scan, [gridx + 1] strip row counts, then the
    // 64-bit counter of the labelling kernel; all zero between steps (their last blocks reset them)
    const int d_rows = gridx + 1, d_label = (gridx + 3) & ~1, d_ycuts = d_label + 2, d_sum = d_ycuts + 1, ndone = d_sum + 1;
    CUDA_TRY(h, h->done.ensure((size_t)ndone));
    ddc_handle_s::CleanSig sig;
    sig.col = colcount;
    sig.done = h->done.p;
    sig.ncol = ncol;
    sig.yr_off = yr_off;
    sig.rank = h->rank;
    sig.ndone = ndone;
    const int ci = p2p ? par : 0;
    if (!(h->clean[ci] == sig) || p2p != h->clean_p2p) { // first use of these buffers with this geometry
        CUDA_TRY(h, launch_k(k_init, dim3((std::max(ncol, ndone) + 255) / 256), dim3(256), 0, s, false, colcount, ncol, yr_off,
            h->rank, h->sc.p, h->loadmm.p, h->done.p, ndone));
        launches++;
        if (p2p != h->clean_p2p)
            h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig();
        h->clean_p2p = p2p;
    }
    h->clean[ci] = sig; // K2 of this step puts the buffer back into k_init's state
    // int32 mask: 16-byte loads of 4 columns; byte mask: 4-byte loads of 4 columns
    const bool u8 = h->mask_esize == 1;
    const bool vec = (NX % 4 == 0) && (((uintptr_t)h->d_mask) % (u8 ? 4 : 16) == 0);
    int* yr = reinterpret_cast<int*>(colcount + yr_off + 2 * h->rank);
    if (rows > 0 || p2p) { // an empty shard still has to push its (empty) counts and raise its flag
        const int rpc = u8 ? (vec ? pick_rows_per_cta(k_scan_mask_u8<true>, std::max(rows, 1), gridx)
                                  : pick_rows_per_cta(k_scan_mask_u8<false>, std::max(rows, 1), gridx))
                           : (vec ? pick_rows_per_cta(k_scan_mask<true>, std::max(rows, 1), gridx)
                                  : pick_rows_per_cta(k_scan_mask<false>, std::max(rows, 1), gridx));
        // the last quarter of the rows go in chunks of a quarter of the size (see the kernel)
        const int small = std::max(8, (rpc / 4) & ~7);
        int nbig = (rows + rpc - 1) / rpc, nsmall = 0;
        if (small < rpc && rows >= 4 * rpc) {
            nbig = (int)((long long)rows * 75 / 100) / rpc;
            nsmall = (rows - nbig * rpc + small - 1) / small;
        }
        dim3 grid(gridx, std::max(1, nbig + nsmall));
        if (u8)
            CUDA_TRY(h, launch_k(vec ? k_scan_mask_u8<true> : k_scan_mask_u8<false>, grid, dim3(256), 0, s, pdl,
                static_cast<const uint8_t*>(h->d_mask), NX, rows, h->y_begin, NB, rpc, h->bits.p, colcount, yr, push_col, ps,
                h->done.p, yr_off, dbg, nbig, small));
        else
            CUDA_TRY(h, launch_k(vec ? k_scan_mask<true> : k_scan_mask<false>, grid, dim3(256), 0, s, pdl,
                static_cast<const int32_t*>(h->d_mask), NX, rows, h->y_begin, NB, rpc, h->bits.p, colcount, yr, push_col, ps,
                h->done.p, yr_off, dbg, nbig, small));
        launches++;
    }
    if (G > 1 && !p2p) // the first exchange step: column histogram and every rank's dot y-range in one sum
        NCCL_TRY(h, g_nccl.AllReduce(colcount, colcount, ncol, nccl_Uint32, nccl_Sum, h->comm, s));
    // several GPUs: a grid of blocks waits for the ranks' flags and sums their column-count slots into ONE buffer,
    // the x-cut block then reads global counts as on one GPU
    const bool presum = p2p;
    // between programmatic launches k_sum_cols polls the scan's local flag, and K2 polls the word k_sum_cols publishes,
    // in place of the kernel boundaries (ChainWord)
    const ChainWord w_sum = pdl && presum ? ChainWord { h->gate.p + 1, h->step } : ChainWord { nullptr, 0u };
    if (presum) {
        CUDA_TRY(h, launch_k(k_sum_cols, dim3(gridx), dim3(256), 0, s, pdl, pc, ps, NX, yr_off, h->colsum.p, h->plan.p,
            pdl ? 1 : 0, h->done.p + d_sum, w_sum, dbg));
        launches++;
        pc = PeerCols {};
        pc.col[0] = h->colsum.p;
        pc.n = 1;
    }
    // who puts this rank's column-count slot back to zero once it is consumed: the labelling kernel when the slot is
    // peer-mapped memory (see k_xcuts), else the x-cut block
    const bool label_runs = rows > 0 && (P > 1 || want_pid);
    const bool reset_in_label = presum && label_runs;
    PeerSync ps_x = ps; // (K2 needs the rank, not the flags)
    if (presum)
        ps_x.enabled = 0;
    mark(1);
    // ---- K2: x cuts ----------------------------------------------------------------------------
    if (x_smem) {
        CUDA_TRY(h, opt_in_smem(k_xcuts<true>, h->device, 0, std::max<size_t>(xneed, 48 * 1024)));
        CUDA_TRY(h, launch_k(k_xcuts<true>, dim3(1), dim3(1024), xneed, s, pdl, pc, ps_x, NX, NY, P, nullptr, yr_off, G, aix,
            aiy, h->plan.p, t.st, t.bx, h->loads.p, h->loadmm.p, h->sc.p, colcount, dbg ? 1 : 0,
            h->pin_plan_dev, presum ? 1 : 0, reset_in_label ? 0 : 1, w_sum));
    } else
        CUDA_TRY(h, launch_k(k_xcuts<false>, dim3(1), dim3(1024), LEVEL_NODES_BYTES, s, pdl, pc, ps_x, NX, NY, P, h->colpfx.p, yr_off, G, aix,
            aiy, h->plan.p, t.st, t.bx, h->loads.p, h->loadmm.p, h->sc.p, colcount, dbg ? 1 : 0,
            h->pin_plan_dev, presum ? 1 : 0, reset_in_label ? 0 : 1, w_sum));
    launches++;
    // the column -> strip table K6 reads: painted by K4's blocks; without y levels there is no K4
    if (!ycuts) {
        CUDA_TRY(h, launch_k(k_paint_strips, dim3(std::max(1, std::min((Scap + 7) / 8, 148 * 4))), dim3(256), 0, s, pdl, t.st,
            h->plan.p, h->strip_of_col.p));
        launches++;
    }
    mark(2);
    // the second stream (neighbour tables beside the labelling kernel) is forked by a device-side gate when K4 runs
    // and nothing else has to sit between K4 and the labelling kernel (no profiling events)
    // (not on tiny shards: there the neighbour kernels end the step, and starting them behind a polling kernel instead of
    //  an event costs more than the programmatic launch of a 9 us labelling kernel saves -- 528 x 522: +3 us with the gate)
    const bool gated = want_nbr && ycuts && !profile && (long long)rows * NX >= (1LL << 21);
    BoxGate gate {};
    if (gated) {
        gate.word = h->gate.p;
        gate.done = h->done.p + d_ycuts;
        gate.step = h->step;
    }
    // ---- K3 + K4: strip row counts, y cuts -----------------------------------------------------
    PeerSync ps_rows = ps; // (+ the per-block flags of exchange step 2, when the streaming row-count kernel runs)
    if (ycuts) {
        int rb_shift = 5; // log2(rows per block) of the kernel that writes the row counts
        {
            // the grid covers the Rmax rows of the largest shard: a short (or empty) shard writes its
            // missing rows as empty, and with the peer exchange every count goes to all ranks
            // rows per warp of the streaming kernel: fewer for small shards, so that the grid fills the SMs
            // (measured at C3 / C4 / one eighth of C5: two rows per warp beat one -- whole row in registers or not --
            //  by 2-4 us: half the blocks, each amortising its boundary table over twice the rows)
            int K = Rmax >= 32 * 4 * 148 ? 4 : 2;
            while (K > 1 && sizeof(int) * strip_scan_smem_words(NG, Scap, K) > 48 * 1024)
                K >>= 1;
            const size_t scan_smem = sizeof(int) * strip_scan_smem_words(NG, Scap, K);
            if (scan_smem <= 48 * 1024) { // the streaming kernel: boundary table in shared memory
                const int grid = (Rmax + 8 * K - 1) / (8 * K);
                // one flag per block (row_flags_raise) on 2 ranks: measured -2.4 us on 2 GPUs, but +4 us on 8, where a
                // block has 8 flags to send
                if (p2p && G <= 2 && (size_t)grid <= h->x_flagcap) {
                    const size_t off = peer_words(G, h->x_colcap, h->x_rowcap, 0);
                    for (int q = 0; q < G; q++)
                        ps_rows.rowflag[q] = h->xpeer[q] + off;
                    ps_rows.flagcap = (int)h->x_flagcap;
                    ps_rows.rowblocks = grid;
                }
                rb_shift = K == 4 ? 5 : (K == 2 ? 4 : 3);
#define LAUNCH_SCAN(CT, KK)                                                                        \
    CUDA_TRY(h, launch_k(k_strip_rows_scan<CT, KK>, dim3(grid), dim3(256), scan_smem, s, pdl, h->bits.p, NB, NX, rows, \
        t.st.x0, t.st.p0, h->plan.p, Scap, push_row, Rmax, ps_rows, h->done.p + d_rows, dbg))
                if (narrow) {
                    if (K == 4)
                        LAUNCH_SCAN(uint16_t, 4);
                    else if (K == 2)
                        LAUNCH_SCAN(uint16_t, 2);
                    else
                        LAUNCH_SCAN(uint16_t, 1);
                } else {
                    if (K == 4)
                        LAUNCH_SCAN(unsigned, 4);
                    else if (K == 2)
                        LAUNCH_SCAN(unsigned, 2);
                    else
                        LAUNCH_SCAN(unsigned, 1);
                }
#undef LAUNCH_SCAN
            } else {
                dim3 grid((Rmax + 31) / 32, (Scap + 7) / 8);
                CUDA_TRY(h, launch_k(narrow ? k_strip_rows<uint16_t> : k_strip_rows<unsigned>, grid, dim3(256), 0, s, pdl,
                    h->bits.p, NB, rows, t.st.x0, t.st.x1, t.st.p0, h->plan.p, Scap, push_row, Rmax, ps, h->done.p + d_rows,
                    dbg));
            }
            launches++;
        }
        if (!p2p) {
            pr.row[0] = rowcount;
            if (G > 1) { // the second exchange step
                NCCL_TRY(h, g_nccl.AllGather(rowcount, h->rowcount_all.p, rc_words, nccl_Uint32, h->comm, s));
                pr.row[0] = h->rowcount_all.p;
            }
        }
        mark(3);
        const RowLayout rl = { rank_stride, Rmax, Scap, rb_shift };

#define LAUNCH_YCUTS(CT, SM, which)                                                                \
    do {                                                                                           \
        if (SM)                                                                                    \
            CUDA_TRY(h, opt_in_smem(k_ycuts<CT, SM>, h->device, which, std::max<size_t>(yneed, 48 * 1024))); \
        CUDA_TRY(h, launch_k(k_ycuts<CT, SM>, dim3(ygrid), dim3(1024), SM ? yneed : LEVEL_NODES_BYTES, s, pdl, pr, ps_rows, rl, NY, t.st, \
            h->ypfx.p, t.bx, h->loads.p, h->loadmm.p, h->plan.p, h->strip_of_col.p, dbg ? 1 : 0, gate, h->part_at.p, nchunk)); \
    } while (0)
        if (narrow) {
            if (y_smem)
                LAUNCH_YCUTS(uint16_t, true, 1);
            else
                LAUNCH_YCUTS(uint16_t, false, 1);
        } else {
            if (y_smem)
                LAUNCH_YCUTS(unsigned, true, 2);
            else
                LAUNCH_YCUTS(unsigned, false, 2);
        }
#undef LAUNCH_YCUTS
        launches++;
        if (gated) { // the second stream waits in a one-warp kernel until K4's last block says the boxes are in place
            // (launched AFTER K4: tools that serialise kernels in launch order -- ncu, CUDA_LAUNCH_BLOCKING -- then run
            //  K4 first and the gate finds itself open)
            CUDA_TRY(h, launch_k(k_gate, dim3(1), dim3(32), 0, h->side_stream, false, h->gate.p, h->step, h->plan.p));
            launches++;
        }
    } else
        mark(3);
    mark(4);
    // ---- K7 (speculative): the neighbour tables of the RCB boxes are built on a second stream while
    //      K6 labels the cells; they are final unless K6 finds `changes == 0` (see the redo below)
    h->nparts = P;
    h->px = px;
    h->py = py;
    // the boxes of a step come in strips (K2 has just cleared `always`): thread = (list, part), 8 * pad32(P) threads --
    // a quarter of the warp-per-part grid that caller-supplied boxes need (run_neighbours)
    const int ngrid = std::max(1, (8 * ((P + 31) & ~31) + 255) / 256);
    // The labelling kernel's last block also ends the step (`changes`, exchange step 3, the plan into the host's
    // pinned copy) unless there is no labelling kernel on this rank or the exchange goes through NCCL.
    const bool fuse = label_runs && (G == 1 || p2p);
    if (want_nbr) {
        cudaStream_t q = h->side_stream;
        if (!gated) {
            CUDA_TRY(h, cudaEventRecord(h->ev_fork, s));
            CUDA_TRY(h, cudaStreamWaitEvent(q, h->ev_fork, 0));
        }
        CUDA_TRY(h, launch_k(k_neighbours<false>, dim3(ngrid), dim3(256), 0, q, false, t.bx, P, NX, NY, px, py, t.st,
            h->nbr_counts.p, nullptr, nullptr, h->nbr_cap, nullptr, nullptr, nullptr, h->sc.p, h->plan.p));
        CUDA_TRY(h, launch_k(k_scan_counts, dim3(8), dim3(1024), 0, q, pdl, h->nbr_counts.p, P, h->nbr_offsets.p,
            h->nbr_totals.p, h->plan.p));
        // (the fill kernel with a plain launch: its P / 8 blocks, resident and waiting on the high-priority stream while the
        //  8 blocks of the scan run, took the SMs from the labelling kernel -- +15 us at C5)
        CUDA_TRY(h, launch_k(k_neighbours<true>, dim3(ngrid), dim3(256), 0, q, false, t.bx, P, NX, NY, px, py, t.st,
            h->nbr_counts.p, h->nbr_offsets.p, h->nbr_totals.p, h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p, h->nbr_starts.p,
            h->sc.p, h->plan.p));
        launches += 3;
        CUDA_TRY(h, cudaEventRecord(h->ev_join, q));
    }
    // ---- K6: labels + `changes` -----------------------------------------------------------------
    h->fin_ps = ps;
    if (label_runs) {
        const bool vecp = want_pid && (NX % 4 == 0) && (((uintptr_t)h->pid.p) % 16 == 0);
        // no heavy per-CTA epilogue: many small CTAs keep more stores in flight
        const int rpc = 32;
        const dim3 grid(gridx, (rows + rpc - 1) / rpc);
        LabelEnd fin {};
        fin.fuse = fuse ? 1 : 0;
        fin.P = P;
        fin.ps = ps;
        fin.counter = reinterpret_cast<unsigned long long*>(h->done.p + d_label);
        fin.host_plan = h->pin_plan_dev;
        fin.dbg = dbg;
        fin.part_at.table = ycuts ? h->part_at.p : nullptr;
        fin.part_at.nchunk = nchunk;
        fin.reset_col = reset_in_label ? colcount : nullptr;
        fin.reset_n = ncol;
        fin.yr_off = yr_off;
        auto kernel = !want_pid ? k_label<false, false> : (vecp ? k_label<true, true> : k_label<false, true>);
        // (behind K4 without a stream operation in between when the second stream is gated: programmatic launch)
        CUDA_TRY(h, launch_k(kernel, grid, dim3(256), 0, s, pdl && (gated || !want_nbr), h->bits.p, NX, rows, h->y_begin, NB, rpc, h->strip_of_col.p,
            t.st.p0, t.bx.y0, t.bx.ey, nv, h->pid.p, h->sc.p, h->plan.p, fin));
        launches++;
    }
    if (G > 1 && !p2p)
        NCCL_TRY(h, g_nccl.AllReduce(&h->sc.p->changes, &h->sc.p->changes, 1, nccl_Int32, nccl_Max, h->comm, s));
    mark(5);
    if (want_nbr)
        CUDA_TRY(h, cudaStreamWaitEvent(s, h->ev_join, 0)); // the step is over when the neighbour tables are, too
    // ---- K5 as a kernel of its own (see above; otherwise only from validate(), when nothing moved) ----
    if (!fuse) {
        int rc = launch_finalize(h, ps, want_nbr);
        if (rc)
            return rc;
        launches++;
    }
    mark(6);
    if (want_nbr)
        h->have_nbr = true;
    mark(7);
    CUDA_TRY(h, cudaGetLastError());

    h->stats.gpu_launches = launches;
    h->stats.exchange = G == 1 ? 0 : (p2p ? 2 : 1);
    h->stats.nx = NX;
    h->stats.ny = NY;
    h->stats.nparts = P;
    h->have_pid = want_pid;
    h->last_flags = flags;
    h->profiled = profile;
    h->partitioned = true;
    h->pending = true;
    return DDC_OK;
}

// wait for the step, check the assumed plan against the real one, run the step again if they differ
int validate(ddc_handle_t h)
{
    if (!h->pending)
        return DDC_OK;
    for (int attempt = 0;; attempt++) {
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        h->pending = false;
        const Plan& pl = *h->pin_plan;
        if (!pl.mismatch)
            break;
        if (pl.mismatch == 3) {
            h->partitioned = false;
            h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig(); // the step did not run to its end: start clean
            cudaMemsetAsync(h->plan.p, 0, sizeof(Plan), h->stream);
            return fail(h, DDC_ERR_PEER, "peer exchange timed out: a rank did not reach the step within %.1f s",
                (double)PEER_TIMEOUT_NS * 1e-9);
        }
        if (attempt >= 2) {
            h->partitioned = false;
            h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig();
            return fail(h, DDC_ERR_STATE, "the RCB plan did not settle (x/y levels %d/%d)", pl.ix, pl.iy);
        }
        h->aix = pl.ix;
        h->aiy = pl.iy;
        const int launches = h->stats.gpu_launches;
        int rc = enqueue_partition(h, h->nparts, h->px, h->py, h->last_flags);
        if (rc) {
            h->partitioned = false;
            return rc;
        }
        h->stats.gpu_launches += launches;
    }
    if (h->pin_plan->fixup) {
        // nothing moved on this rank: k_finalize collects the other ranks' verdicts and, if nothing moved
        // anywhere, reports the naive blocks and rebuilds the neighbour tables from them (rare: all land, or
        // the RCB reproduces the naive block layout)
        int rc = launch_finalize(h, h->fin_ps, (h->last_flags & DDC_WANT_NEIGHBOURS) && h->nparts > 1);
        if (rc)
            return rc;
        h->stats.gpu_launches++;
        h->totals_valid = false;
        h->small_cached = h->lists_cached = false;
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        if (h->pin_plan->mismatch == 3) {
            h->partitioned = false;
            h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig();
            return fail(h, DDC_ERR_PEER, "peer exchange timed out: a rank did not reach the end of the step");
        }
    }
    const Plan& pl = *h->pin_plan;
    if (h->debug_ts) {
        const unsigned long long* t = pl.ts;
        auto us = [&](int a, int b) { return t[a] && t[b] ? ((double)t[b] - (double)t[a]) * 1e-3 : -1.0; };
        fprintf(stderr, "[ddc r%d] scan: loop %.1f, last col push +%.1f, flag +%.1f | -> K2 start %.1f | K2: barrier %.1f prefix %.1f "
                        "plan %.1f walks %.1f end %.1f | -> rows %.1f | rows: %.1f | -> K4 %.1f | K4 b0: barrier %.1f prefix %.1f "
                        "walks %.1f, longest block %.1f | -> label %.1f | label: loop %.1f, end +%.1f | step %.1f us\n",
            h->rank, us(11, 12), us(12, 13), us(12, 14), us(12, 0), us(0, 1), us(1, 2), us(2, 3), us(3, 4), us(4, 5),
            us(5, 15), us(15, 16), us(16, 6), us(6, 7), us(7, 8), us(8, 9), (double)t[10] * 1e-3, us(9, 17), us(17, 18),
            us(18, 19), us(11, 19));
        // when the first block of each kernel was on an SM (before its wait), relative to the end of the scan's row loop
        fprintf(stderr, "[ddc r%d] resident at (us after the scan's loop): sum %.1f (flags seen %.1f, done %.1f) K2 %.1f rows %.1f "
                        "K4 %.1f label %.1f | K2 start %.1f rows start %.1f K4 start %.1f label start %.1f\n",
            h->rank, us(12, TS_RES), us(12, TS_RES + 5), us(12, TS_RES + 6), us(12, TS_RES + 1), us(12, TS_RES + 2),
            us(12, TS_RES + 3), us(12, TS_RES + 4), us(12, 0), us(12, 15), us(12, 6), us(12, 17));
        fprintf(stderr, "[ddc r%d] K2 levels (thread 0, us):", h->rank);
        for (int l = 0; l + 1 < 8 && t[TS_XLEV + l + 1]; l++)
            fprintf(stderr, " %.2f", us(TS_XLEV + l, TS_XLEV + l + 1));
        fprintf(stderr, " | K4 block 0 levels:");
        for (int l = 0; l + 1 < 8 && t[TS_YLEV + l + 1]; l++)
            fprintf(stderr, " %.2f", us(TS_YLEV + l, TS_YLEV + l + 1));
        fprintf(stderr, "\n");
    }
    h->stats.nlev = pl.nlev;
    h->stats.n_xlev = pl.ix;
    h->stats.n_ylev = pl.iy;
    h->stats.nstrips = pl.S;
    h->stats.n_ocean = pl.W;
    if (h->profiled) {
        for (int i = 0; i < 7; i++)
            cudaEventElapsedTime(&h->stats.stage_ms[i], h->ev[i], h->ev[i + 1]);
        cudaEventElapsedTime(&h->stats.stage_ms[7], h->ev[0], h->ev[7]);
    }
    return DDC_OK;
}
} // namespace

int ddc_partition(ddc_handle_t h, int nparts, int px, int py, int flags)
{
    if (!h)
        return DDC_ERR_ARG;
    if (!h->mask_set)
        return fail(h, DDC_ERR_STATE, "ddc_partition: no mask set");
    if (nparts < 1)
        return fail(h, DDC_ERR_ARG, "ddc_partition: nparts must be >= 1");
    // (an earlier DDC_ASYNC step that nobody looked at is simply superseded)
    int rc = enqueue_partition(h, nparts, px, py, flags);
    if (rc) {
        h->clean[0] = h->clean[1] = ddc_handle_s::CleanSig(); // whatever was enqueued may not have run
        return rc;
    }
    if (flags & DDC_ASYNC)
        return DDC_OK;
    return validate(h);
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
#define NEED_PARTITION(h)                                                                          \
    if (!h)                                                                                        \
        return DDC_ERR_ARG;                                                                        \
    if (!h->partitioned)                                                                           \
        return fail(h, DDC_ERR_STATE, "%s: call ddc_partition() first", __func__);                 \
    CUDA_TRY(h, cudaSetDevice(h->device));                                                         \
    if (int vrc_ = validate(h))                                                                    \
        return vrc_

int ddc_get_boxes(ddc_handle_t h, int32_t* x0, int32_t* y0, int32_t* ex, int32_t* ey)
{
    NEED_PARTITION(h);
    const int P = h->nparts;
    if (int rc = fetch_small(h))
        return rc;
    int32_t* dst[4] = { x0, y0, ex, ey };
    for (int i = 0; i < 4; i++)
        if (dst[i])
            memcpy(dst[i], host_tab_of(h).boxes + (size_t)i * P, sizeof(int32_t) * P);
    return DDC_OK;
}

int ddc_get_pid_device(ddc_handle_t h, const int32_t** dev_ptr)
{
    NEED_PARTITION(h);
    if (!h->have_pid)
        return fail(h, DDC_ERR_STATE, "pid was not requested (DDC_WANT_PID)");
    *dev_ptr = h->pid.p;
    return DDC_OK;
}

int ddc_get_pid_host(ddc_handle_t h, int32_t* out)
{
    NEED_PARTITION(h);
    if (!h->have_pid)
        return fail(h, DDC_ERR_STATE, "pid was not requested (DDC_WANT_PID)");
    const size_t n = (size_t)h->nx * h->y_count;
    if (n)
        CUDA_TRY(h, cudaMemcpyAsync(out, h->pid.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return DDC_OK;
}

static int list_index(ddc_handle_t h, int edge, int periodic)
{
    if (edge < 0 || edge >= 4 || periodic < 0 || periodic > 1)
        return fail(h, DDC_ERR_ARG, "edge must be 0..3 and periodic 0/1");
    return periodic * 4 + edge;
}

int ddc_get_neighbour_counts(ddc_handle_t h, int edge, int periodic, int32_t* counts)
{
    NEED_PARTITION(h);
    const int l = list_index(h, edge, periodic);
    if (l < 0)
        return l;
    const int P = h->nparts;
    if (!h->have_nbr) { // P == 1 (Q4) or neighbours not requested: empty lists
        memset(counts, 0, sizeof(int32_t) * P);
        return DDC_OK;
    }
    if (int rc = fetch_small(h))
        return rc;
    memcpy(counts, host_tab_of(h).counts + (size_t)l * P, sizeof(int32_t) * P);
    return DDC_OK;
}

int ddc_get_neighbour_total(ddc_handle_t h, int edge, int periodic, int64_t* total)
{
    NEED_PARTITION(h);
    const int l = list_index(h, edge, periodic);
    if (l < 0)
        return l;
    if (!h->have_nbr) {
        *total = 0;
        return DDC_OK;
    }
    int rc = fetch_totals(h);
    if (rc)
        return rc;
    *total = h->h_totals[l];
    return DDC_OK;
}

int ddc_get_neighbours(ddc_handle_t h, int edge, int periodic, int32_t* ids, int32_t* halos, int32_t* starts)
{
    NEED_PARTITION(h);
    const int l = list_index(h, edge, periodic);
    if (l < 0)
        return l;
    if (!h->have_nbr)
        return DDC_OK;
    int rc = fetch_lists(h);
    if (rc)
        return rc;
    const size_t n = (size_t)h->h_totals[l], off = (size_t)l * h->cache_cap;
    const HostTab t = host_tab_of(h);
    if (n) {
        if (ids)
            memcpy(ids, t.ids + off, n * sizeof(int32_t));
        if (halos)
            memcpy(halos, t.halos + off, n * sizeof(int32_t));
        if (starts)
            memcpy(starts, t.starts + off, n * sizeof(int32_t));
    }
    return DDC_OK;
}

int ddc_get_part_loads(ddc_handle_t h, int64_t* loads)
{
    NEED_PARTITION(h);
    if (int rc = fetch_small(h))
        return rc;
    memcpy(loads, host_tab_of(h).loads, sizeof(int64_t) * h->nparts);
    return DDC_OK;
}

int ddc_get_stats(ddc_handle_t h, ddc_stats* out)
{
    NEED_PARTITION(h);
    DevScalars hs;
    long long mm[2];
    Plan pl;
    CUDA_TRY(h, cudaMemcpyAsync(&hs, h->sc.p, sizeof hs, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(mm, h->loadmm.p, sizeof mm, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(&pl, h->plan.p, sizeof pl, cudaMemcpyDeviceToHost, h->stream)); // iters: K4 adds late
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->stats.changes = h->nparts > 1 ? hs.changes_all : 0;
    h->stats.load_min = mm[0];
    h->stats.load_max = mm[1];
    h->stats.median_iters = pl.iters;
    if (h->have_nbr) {
        int rc = fetch_totals(h);
        if (rc)
            return rc;
    }
    *out = h->stats;
    return DDC_OK;
}

int ddc_neighbours_from_boxes(ddc_handle_t h, int nparts, int nx, int ny, const int32_t* x0, const int32_t* y0,
    const int32_t* ex, const int32_t* ey, int px, int py)
{
    if (!h || nparts < 1 || !x0 || !y0 || !ex || !ey)
        return fail(h, DDC_ERR_ARG, "ddc_neighbours_from_boxes: bad arguments");
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int P = nparts;
    cudaStream_t s = h->stream;
    CUDA_TRY(h, h->strips.ensure((size_t)3 * (P + 1) + 3));
    CUDA_TRY(h, h->boxes.ensure((size_t)4 * P));
    Tables t = tables(h, P);
    const int32_t* src[4] = { x0, y0, ex, ey };
    for (int i = 0; i < 4; i++)
        CUDA_TRY(h, cudaMemcpyAsync(h->boxes.p + (size_t)i * P, src[i], sizeof(int32_t) * P, cudaMemcpyHostToDevice, s));
    // no strip structure is assumed for caller-supplied boxes: one always-relevant strip
    const int zero = 0, one = 1, nx_ = nx;
    CUDA_TRY(h, cudaMemcpyAsync(t.st.x0, &zero, sizeof(int), cudaMemcpyHostToDevice, s));
    CUDA_TRY(h, cudaMemcpyAsync(t.st.x1, &nx_, sizeof(int), cudaMemcpyHostToDevice, s));
    const int p0[2] = { 0, P };
    CUDA_TRY(h, cudaMemcpyAsync(t.st.p0, p0, sizeof p0, cudaMemcpyHostToDevice, s));
    CUDA_TRY(h, cudaMemcpyAsync(t.st.S, &one, sizeof(int), cudaMemcpyHostToDevice, s));
    CUDA_TRY(h, cudaMemcpyAsync(t.st.always, &one, sizeof(int), cudaMemcpyHostToDevice, s));
    DevScalars init;
    init.changes = 1;
    init.changes_all = 1;
    init.overflow = 0;
    init.edge_cut = 0;
    CUDA_TRY(h, cudaMemcpyAsync(h->sc.p, &init, sizeof init, cudaMemcpyHostToDevice, s));
    CUDA_TRY(h, cudaStreamSynchronize(s)); // the staging variables above live on this stack frame
    memset(&h->stats, 0, sizeof h->stats);
    h->nparts = P;
    h->nx = nx; // also what an overflow re-run of the fill pass uses
    h->ny = ny;
    h->px = px;
    h->py = py;
    h->mask_set = false; // the mask (if any) has to be set again before the next ddc_partition
    halo_invalidate(h);
    h->d_mask = nullptr;
    h->pending = false;
    int rc = run_neighbours(h, P, nx, ny, px, py);
    if (rc)
        return rc;
    h->partitioned = true; // results (boxes + neighbour tables) are valid; pid / loads are not
    h->have_pid = false;
    CUDA_TRY(h, h->loads.ensure(P));
    CUDA_TRY(h, h->loadmm.ensure(2));
    CUDA_TRY(h, cudaMemsetAsync(h->loads.p, 0, sizeof(long long) * P, s));
    CUDA_TRY(h, cudaMemsetAsync(h->loadmm.p, 0, sizeof(long long) * 2, s));
    CUDA_TRY(h, cudaMemsetAsync(h->plan.p, 0, sizeof(Plan), s));
    return DDC_OK;
}

// ------------------------------------------------------------------------------------------------
// halo exchange (a consumer of the neighbour tables)
// ------------------------------------------------------------------------------------------------
// the halo plan of the current boxes (host only)
static int build_halo_plan(ddc_handle_t h, HaloPlan& hp)
{
    const int P = h->nparts;
    std::vector<int32_t> box[4];
    for (int i = 0; i < 4; i++)
        box[i].resize(P);
    if (int rc = ddc_get_boxes(h, box[0].data(), box[1].data(), box[2].data(), box[3].data()))
        return rc;
    int yb, yc;
    ddc_shard_rows(h->ny, h->nranks, h->rank, &yb, &yc);
    hp = halo_plan(P, h->nranks, h->rank, h->nx, h->ny, h->px, h->py, box[0].data(), box[1].data(), box[2].data(),
        box[3].data(), yb, yc, h->halo_w);
    return DDC_OK;
}

// the halo plan of the current decomposition, also left on the device for the halo kernels: the tile offsets of all
// parts in one buffer, the (part, row) ranges of scatter and gather and the corner items of the full-frame exchange
// (w = 1) or the rectangle items of both exchanges (w >= 2).
// Everything is built here, where the host may wait for the stream: a sharded call must not wait (one host thread may
// drive several ranks, whose open kernels wait for each other).
static int tile_offsets(ddc_handle_t h)
{
    HaloPlan hp;
    if (int rc = build_halo_plan(h, hp))
        return rc;
    CUDA_TRY(h, h->halo_dev.ensure(hp.block.size()));
    CUDA_TRY(h, cudaMemcpyAsync(h->halo_dev.p, hp.block.data(), hp.block.size(), cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    h->halo = std::move(hp);
    h->halo_ok = true;
    return DDC_OK;
}

int ddc_halo_set_width(ddc_handle_t h, int width)
{
    if (!h)
        return DDC_ERR_ARG;
    if (width < 1 || width > DDC_MAX_HALO_WIDTH)
        return fail(h, DDC_ERR_ARG, "ddc_halo_set_width: width %d is not in 1..%d", width, DDC_MAX_HALO_WIDTH);
    if (width != h->halo_w) {
        h->halo_w = width;
        halo_invalidate(h); // another layout: the tile and shard offsets are to be taken again
    }
    return DDC_OK;
}

int ddc_halo_tile_offsets(ddc_handle_t h, int64_t* offsets)
{
    NEED_PARTITION(h);
    if (!offsets)
        return fail(h, DDC_ERR_ARG, "ddc_halo_tile_offsets: null output");
    if (int rc = tile_offsets(h))
        return rc;
    for (int p = 0; p <= h->nparts; p++)
        offsets[p] = h->halo.off()[p];
    return DDC_OK;
}

// the source part and cell of one corner of every part (computed on the host from the boxes)
int ddc_get_corner_neighbours(ddc_handle_t h, int corner, int periodic, int32_t* ids, int32_t* starts)
{
    NEED_PARTITION(h);
    if (corner < 0 || corner >= DDC_N_CORNER || periodic < 0 || periodic > 1)
        return fail(h, DDC_ERR_ARG, "ddc_get_corner_neighbours: corner must be 0..3 and periodic 0/1");
    HaloPlan built;
    if (!h->halo_ok)
        if (int rc = build_halo_plan(h, built))
            return rc;
    const HaloPlan& hp = h->halo_ok ? h->halo : built;
    const size_t P = h->nparts, at = ((size_t)periodic * 4 + corner) * P;
    if (ids)
        memcpy(ids, hp.corner_ids.data() + at, P * sizeof(int32_t));
    if (starts)
        memcpy(starts, hp.corner_starts.data() + at, P * sizeof(int32_t));
    return DDC_OK;
}

// one buffer: the edge ghosts (k_halo_exchange), and with `full` the corner ghosts after them (k_halo_corners); wide
// frames: the rectangle items of both (k_halo_rects)
static int halo_exchange(ddc_handle_t h, double* tiles_dev, int periodic, bool full, const char* name)
{
    if (!tiles_dev)
        return fail(h, DDC_ERR_ARG, "%s: null tiles", name);
    if (!h->halo_ok)
        return fail(h, DDC_ERR_STATE, "%s: call ddc_halo_tile_offsets() for this decomposition first", name);
    if (!h->have_nbr)
        return DDC_OK; // one part (or no tables asked for): nothing to exchange
    if (h->halo.w > 1) {
        const HaloRects rects = h->halo.rects(h->halo_dev.p, 0, periodic, full);
        if (rects.n > 0)
            CUDA_TRY(h, launch_k(k_halo_rects, dim3(halo_field_grid(rects.n)), dim3(256), 0, h->stream, false, rects,
                tiles_dev));
        CUDA_TRY(h, cudaGetLastError());
        return DDC_OK;
    }
    int rc = fetch_totals(h); // (re-runs the fill pass with the exact capacity if the bounded one overflowed)
    if (rc)
        return rc;
    const int P = h->nparts;
    Tables t = tables(h, P);
    CUDA_TRY(h, launch_k(k_halo_exchange<double>, dim3(halo_exchange_grid(P)), dim3(256), 0, h->stream, false, t.bx, P,
        h->nbr_counts.p, h->nbr_offsets.p, h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p, h->nbr_starts.p,
        h->halo.ptrs(h->halo_dev.p).off, tiles_dev, periodic ? 0xffu : 0x0fu));
    const HaloCorners corners = h->halo.corners(h->halo_dev.p, 0, periodic);
    if (full && corners.n > 0) // (corners read interiors only: no order with the edges is needed)
        CUDA_TRY(h, launch_k(k_halo_corners, dim3(halo_corner_grid(corners.n)), dim3(256), 0, h->stream, false, corners,
            tiles_dev));
    CUDA_TRY(h, cudaGetLastError());
    return DDC_OK;
}

int ddc_halo_exchange_f64(ddc_handle_t h, double* tiles_dev, int periodic)
{
    NEED_PARTITION(h);
    return halo_exchange(h, tiles_dev, periodic, false, "ddc_halo_exchange_f64");
}

int ddc_halo_exchange_full_f64(ddc_handle_t h, double* tiles_dev, int periodic)
{
    NEED_PARTITION(h);
    return halo_exchange(h, tiles_dev, periodic, true, "ddc_halo_exchange_full_f64");
}

// halo scatter / gather: the field rows <-> the tile interiors (k_halo_field, k_halo_field_shards)
static int halo_field(ddc_handle_t h, bool scatter, double* field_dev, double* tiles_dev, const char* name)
{
    if (!field_dev || !tiles_dev)
        return fail(h, DDC_ERR_ARG, "%s: null pointer", name);
    if (!h->halo_ok)
        return fail(h, DDC_ERR_STATE, "%s: call ddc_halo_tile_offsets() for this decomposition first", name);
    Tables t = tables(h, h->nparts);
    CUDA_TRY(h, launch_k(scatter ? k_halo_field<true> : k_halo_field<false>, dim3(halo_field_grid(h->halo.items_total[0])),
        dim3(256), 0, h->stream, false, h->halo.items(h->halo_dev.p, 0), t.bx, tiles_dev, field_dev, h->nx));
    CUDA_TRY(h, cudaGetLastError());
    return DDC_OK;
}

int ddc_halo_scatter_f64(ddc_handle_t h, const double* field_dev, double* tiles_dev)
{
    NEED_PARTITION(h);
    return halo_field(h, true, const_cast<double*>(field_dev), tiles_dev, "ddc_halo_scatter_f64");
}

int ddc_halo_gather_f64(ddc_handle_t h, const double* tiles_dev, double* field_dev)
{
    NEED_PARTITION(h);
    return halo_field(h, false, field_dev, const_cast<double*>(tiles_dev), "ddc_halo_gather_f64");
}

// ------------------------------------------------------------------------------------------------
// halo exchange across ranks (parts sharded over the ranks, ghost cells pushed over peer memory)
// ------------------------------------------------------------------------------------------------
int ddc_halo_shard_offsets(ddc_handle_t h, int64_t* offsets)
{
    NEED_PARTITION(h);
    if (!offsets)
        return fail(h, DDC_ERR_ARG, "ddc_halo_shard_offsets: null output");
    if (int rc = tile_offsets(h))
        return rc;
    int b, c;
    ddc_shard_parts(h->nparts, h->nranks, h->rank, &b, &c);
    const long long* off = h->halo.off();
    for (int i = 0; i <= c; i++)
        offsets[i] = off[(size_t)b + i] - off[b];
    h->halo_shard_ok = true;
    return DDC_OK;
}

// this rank's halo buffer: zeroed head (flags, block counter) + room for `elems` doubles; the error word beside it
static int halo_alloc(ddc_handle_t h, int64_t elems)
{
    CUDA_TRY(h, cudaSetDevice(h->device));
    const size_t bytes = HALO_HEAD_BYTES + (size_t)elems * sizeof(double);
    CUDA_TRY(h, cudaMalloc((void**)&h->halo_buf, bytes));
    CUDA_TRY(h, cudaMemsetAsync(h->halo_buf, 0, bytes, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream)); // zero before any peer can see the buffer
    if (!h->halo_err) {
        CUDA_TRY(h, cudaHostAlloc((void**)&h->halo_err, sizeof(int), cudaHostAllocMapped));
        CUDA_TRY(h, cudaHostGetDevicePointer((void**)&h->halo_err_dev, h->halo_err, 0));
        *h->halo_err = 0;
    }
    // Load the exchange kernels now.  Loaded lazily at its first launch (CUDA_MODULE_LOADING=LAZY, the default), a kernel
    // can wait for the kernels running on the device -- and those can be other ranks' k_halo_open, spinning until this
    // rank's arrives (measured: the first exchange of handles sharing a B200 timed out).
    cudaFuncAttributes fa;
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_open));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_push));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_push_full));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_close));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_field_shards<true>));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_field_shards<false>));
    CUDA_TRY(h, cudaFuncGetAttributes(&fa, k_halo_push_rects));
    h->halo_elems = elems;
    h->halo_step = 0;
    return DDC_OK;
}

int ddc_halo_export(ddc_handle_t h, int64_t elems, double** tiles_dev, void* ipc_handle_out)
{
    if (!h || elems < 0 || !tiles_dev || !ipc_handle_out)
        return fail(h, DDC_ERR_ARG, "ddc_halo_export: bad arguments");
    if (h->nranks > MAX_PEERS)
        return fail(h, DDC_ERR_ARG, "ddc_halo_export: at most %d ranks", MAX_PEERS);
    if (h->halo_buf)
        return fail(h, DDC_ERR_STATE, "ddc_halo_export: already exported");
    if (int rc = halo_alloc(h, elems))
        return rc;
    *tiles_dev = (double*)(h->halo_buf + HALO_HEAD_BYTES);
    return ipc_export(h, h->halo_buf, ipc_handle_out);
}

int ddc_halo_import(ddc_handle_t h, const void* all_handles)
{
    if (!h || !all_handles)
        return fail(h, DDC_ERR_ARG, "ddc_halo_import: bad arguments");
    if (!h->halo_buf || h->halo_local)
        return fail(h, DDC_ERR_STATE, "ddc_halo_import: call ddc_halo_export() first");
    if (h->halo_mapped)
        return fail(h, DDC_ERR_STATE, "ddc_halo_import: already imported (ddc_halo_close() first)");
    if (int rc = ipc_import(h, all_handles, h->halo_buf, h->halo_peer))
        return rc;
    h->halo_mapped = true;
    return DDC_OK;
}

int ddc_halo_connect(ddc_handle_t* handles, int n, int64_t elems, double** tiles_dev)
{
    if (!handles || n < 1 || n > MAX_PEERS || elems < 0 || !tiles_dev)
        return fail(nullptr, DDC_ERR_ARG, "ddc_halo_connect: bad arguments");
    for (int q = 0; q < n; q++)
        if (!handles[q] || handles[q]->nranks != n || handles[q]->rank != q || handles[q]->halo_buf)
            return fail(handles[q], DDC_ERR_ARG, "ddc_halo_connect: handle %d must be rank %d of %d and not yet exported", q, q,
                n);
    if (int rc = enable_peer_access(handles, n))
        return rc;
    for (int q = 0; q < n; q++) {
        if (int rc = halo_alloc(handles[q], elems))
            return rc;
        tiles_dev[q] = (double*)(handles[q]->halo_buf + HALO_HEAD_BYTES);
    }
    for (int q = 0; q < n; q++) {
        for (int r = 0; r < n; r++)
            handles[q]->halo_peer[r] = handles[r]->halo_buf;
        handles[q]->halo_mapped = true;
        handles[q]->halo_local = true;
    }
    return DDC_OK;
}

// the checks of every sharded halo call (exchange, scatter, gather).  Each has the same outcome on every rank
// (replicated tables, the same calls), so no rank is left waiting for one that refused.
static int halo_shards_ready(ddc_handle_t h, const char* name)
{
    if (!h->halo_buf || !h->halo_mapped)
        return fail(h, DDC_ERR_STATE, "%s: no halo buffers (ddc_halo_export + ddc_halo_import, or ddc_halo_connect)", name);
    if (!h->halo_shard_ok)
        return fail(h, DDC_ERR_STATE, "%s: call ddc_halo_shard_offsets() for this decomposition first", name);
    if (h->halo.shard_max > h->halo_elems)
        return fail(h, DDC_ERR_ARG, "%s: a rank's tiles need %lld doubles, the buffers hold %lld", name, h->halo.shard_max,
            (long long)h->halo_elems);
    return DDC_OK;
}

// one sharded halo call with the next step number: k_halo_open, the middle kernel middle(hs) launches, k_halo_close
extern "C++" { // (a template)
template <typename Middle>
static int halo_shards_call(ddc_handle_t h, Middle middle)
{
    const HaloShards hs = halo_shards(h->nparts, h->nranks, h->rank, ++h->halo_step, h->halo_peer, h->halo_err_dev);
    CUDA_TRY(h, launch_k(k_halo_open, dim3(1), dim3(32), 0, h->stream, false, hs, 3));
    CUDA_TRY(h, middle(hs));
    CUDA_TRY(h, launch_k(k_halo_close, dim3(1), dim3(32), 0, h->stream, false, hs));
    CUDA_TRY(h, cudaGetLastError());
    return DDC_OK;
}
}

// the edge ghosts (k_halo_push), and with `full` the corner ghosts beside them (k_halo_push_full); wide frames: the
// rectangle items of both whose source part this rank owns (k_halo_push_rects)
static int halo_exchange_shards(ddc_handle_t h, int periodic, bool full, const char* name)
{
    if (int rc = halo_shards_ready(h, name))
        return rc;
    if (!h->have_nbr)
        return DDC_OK; // one part (or no tables asked for): nothing to exchange, no step taken
    if (h->halo.w > 1) {
        const HaloRects rects = h->halo.rects(h->halo_dev.p, 1, periodic, full);
        return halo_shards_call(h, [&](const HaloShards& hs) {
            return launch_k(k_halo_push_rects, dim3(halo_field_grid(rects.n)), dim3(256), 0, h->stream, false, hs, rects);
        });
    }
    if (int rc = fetch_totals(h)) // (may wait for the stream: before anything of the exchange is enqueued)
        return rc;
    Tables t = tables(h, h->nparts);
    const long long* off = h->halo.ptrs(h->halo_dev.p).off;
    const unsigned lists = periodic ? 0xffu : 0x0fu;
    const HaloCorners corners = h->halo.corners(h->halo_dev.p, 1, periodic);
    return halo_shards_call(h, [&](const HaloShards& hs) {
        const dim3 grid(halo_push_grid(hs.p_count, full ? corners.n : 0));
        if (full)
            return launch_k(k_halo_push_full, grid, dim3(256), 0, h->stream, false, hs, t.bx, h->nbr_counts.p,
                h->nbr_offsets.p, h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p, h->nbr_starts.p, off, lists, corners);
        return launch_k(k_halo_push, grid, dim3(256), 0, h->stream, false, hs, t.bx, h->nbr_counts.p, h->nbr_offsets.p,
            h->nbr_cap, h->nbr_ids.p, h->nbr_halos.p, h->nbr_starts.p, off, lists);
    });
}

int ddc_halo_exchange_shards_f64(ddc_handle_t h, int periodic)
{
    NEED_PARTITION(h);
    return halo_exchange_shards(h, periodic, false, "ddc_halo_exchange_shards_f64");
}

int ddc_halo_exchange_full_shards_f64(ddc_handle_t h, int periodic)
{
    NEED_PARTITION(h);
    return halo_exchange_shards(h, periodic, true, "ddc_halo_exchange_full_shards_f64");
}

static int halo_field_shards(ddc_handle_t h, bool scatter, double* rows_dev, const char* name)
{
    if (int rc = halo_shards_ready(h, name))
        return rc;
    int yb, yc;
    ddc_shard_rows(h->ny, h->nranks, h->rank, &yb, &yc);
    if (!rows_dev && yc > 0) // (this rank only: its peers time out waiting for it and report DDC_ERR_PEER)
        return fail(h, DDC_ERR_ARG, "%s: null rows (this rank holds rows %d..%d)", name, yb, yb + yc - 1);
    Tables t = tables(h, h->nparts);
    return halo_shards_call(h, [&](const HaloShards& hs) {
        return launch_k(scatter ? k_halo_field_shards<true> : k_halo_field_shards<false>,
            dim3(halo_field_grid(h->halo.items_total[1])), dim3(256), 0, h->stream, false, hs,
            h->halo.items(h->halo_dev.p, 1), t.bx, rows_dev, h->nx, yb);
    });
}

int ddc_halo_scatter_shards_f64(ddc_handle_t h, const double* rows_dev)
{
    NEED_PARTITION(h);
    return halo_field_shards(h, true, const_cast<double*>(rows_dev), "ddc_halo_scatter_shards_f64");
}

int ddc_halo_gather_shards_f64(ddc_handle_t h, double* rows_dev)
{
    NEED_PARTITION(h);
    return halo_field_shards(h, false, rows_dev, "ddc_halo_gather_shards_f64");
}

int ddc_halo_close(ddc_handle_t h)
{
    if (!h)
        return DDC_ERR_ARG;
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, ipc_unmap(h, h->halo_peer, h->halo_local));
    h->halo_mapped = false;
    return DDC_OK;
}

// ------------------------------------------------------------------------------------------------
// synthetic masks
// ------------------------------------------------------------------------------------------------
static void synth_params(int nx, int ny, uint64_t seed, double land_frac, uint64_t* L1, uint64_t* L2, uint32_t* thresh)
{
    const uint64_t m = (uint64_t)std::max(nx, ny);
    *L1 = std::max<uint64_t>(1, m / 16);
    *L2 = std::max<uint64_t>(1, m / 64);
    // calibrate the threshold to the requested land fraction on a fixed 128 x 128 sample lattice
    const int K = 128;
    std::vector<uint32_t> v;
    v.reserve((size_t)K * K);
    for (int j = 0; j < K; j++)
        for (int i = 0; i < K; i++) {
            const uint64_t x = (uint64_t)(((2 * i + 1) * (uint64_t)nx) / (2 * K));
            const uint64_t y = (uint64_t)(((2 * j + 1) * (uint64_t)ny) / (2 * K));
            v.push_back(synth_value(seed, *L1, *L2, x, y));
        }
    std::sort(v.begin(), v.end());
    double f = land_frac < 0 ? 0 : (land_frac > 1 ? 1 : land_frac);
    size_t k = (size_t)(f * (double)v.size());
    if (k >= v.size())
        *thresh = 0xffffffffu; // everything land
    else
        *thresh = f <= 0 ? 0u : v[k];
}

int ddc_generate_mask_device(ddc_handle_t h, int32_t* dev_rows, int nx, int ny, int y_begin, int y_count, uint64_t seed, double land_frac)
{
    if (!h || nx < 1 || ny < 1 || y_begin < 0 || y_count < 0 || y_begin + y_count > ny || (!dev_rows && y_count))
        return fail(h, DDC_ERR_ARG, "ddc_generate_mask_device: bad arguments");
    CUDA_TRY(h, cudaSetDevice(h->device));
    uint64_t L1, L2;
    uint32_t thresh;
    synth_params(nx, ny, seed, land_frac, &L1, &L2, &thresh);
    if (y_count) {
        const size_t n = (size_t)nx * y_count;
        const int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 32);
        CUDA_TRY(h, launch_k(k_generate_mask, dim3(grid), dim3(256), 0, h->stream, false, dev_rows, nx, y_count, y_begin,
            seed, L1, L2, thresh));
        CUDA_TRY(h, cudaGetLastError());
    }
    return DDC_OK;
}

int ddc_generate_mask_host(int32_t* rows, int nx, int ny, int y_begin, int y_count, uint64_t seed, double land_frac)
{
    if (nx < 1 || ny < 1 || y_begin < 0 || y_count < 0 || y_begin + y_count > ny || (!rows && y_count))
        return DDC_ERR_ARG;
    uint64_t L1, L2;
    uint32_t thresh;
    synth_params(nx, ny, seed, land_frac, &L1, &L2, &thresh);
    for (int y = 0; y < y_count; y++)
        for (int x = 0; x < nx; x++)
            rows[(size_t)y * nx + x] = synth_value(seed, L1, L2, (uint64_t)x, (uint64_t)(y + y_begin)) >= thresh ? 1 : 0;
    return DDC_OK;
}

} // extern "C"
