// ddc_kernels.cuh -- hand-written sm_100a kernels of the domain-decomposition hot path.
//
// Pipeline (one GPU; with several GPUs every rank runs it on its own block of mask rows, K1 and K3
// push their histograms into the other ranks' memory over NVLink and K2 / K4 / K5 wait for flags,
// see "multi-GPU exchange" below; NCCL collectives between the kernels are the fallback, ddc_api.cu):
//
//   K1 k_scan_mask     int32 mask -> 1-bit ocean map + per-column ocean counts + dot y-range
//                      (replaces Grid.cpp:176-188 and the Zoltan geometry callbacks
//                       ZoltanPartitioner.cpp:19-67; HBM-bound, 4 B/cell read)
//   K2 k_xcuts         prefix sums of the column counts, preset cut directions, all x levels of
//                      the RCB: every strip's path root -> strip walked at once, no level barriers
//   K3 k_strip_rows    per-strip per-row ocean counts from the bit map (1/32 of the mask bytes)
//   K4 k_ycuts         all y levels, one CTA per vertical strip -> integer part boxes
//                      (K2+K4 replace Zoltan::LB_Partition + RCB_Box + the ceil/clamp of
//                       ZoltanPartitioner.cpp:161-195)
//   K6 k_label         pid[y][x] = ocean ? part : -1 and Zoltan's `changes` flag
//                      (ZoltanPartitioner.cpp:201-219; HBM-bound, 4 B/cell written)
//   K7 k_neighbours    interval-intersection kernel: neighbour ids, halo sizes, halo starts,
//                      interior and periodic (Partitioner.cpp:20-80,329-435, DomainUtils.cpp:15-35);
//                      runs beside K6 on a second stream
//   K5 k_finalize      one block ends the step: `changes` of all ranks; `changes == 0` => report the
//                      naive blocks (ZoltanPartitioner.cpp:182-187) and rebuild K7's tables from them
//
// Bit map layout: plain row-major little-endian bit map, bit (x & 7) of byte x >> 3 of a row is
// column x; rows are padded to NB = 16 * ceil(NX / 128) bytes so that every row is 16-byte aligned.
// Columns >= NX read as land.
#pragma once
#ifndef DDC_HOST_EMU
#include <cuda_runtime.h>
#endif
#include <stdint.h>

#include "ddc_median.cuh"
#include "ddc_neighbours.cuh"

// dynamic shared memory of a kernel (test builds: a buffer of the host emulation, see oracle/emu/ddc_host_emu.h)
#ifdef DDC_HOST_EMU
#define DDC_DYN_SHARED(T, name) T* name = reinterpret_cast<T*>(ddc_emu_dyn_smem())
#else
#define DDC_DYN_SHARED(T, name) extern __shared__ __align__(16) T name[]
#endif

namespace ddc {

struct Plan { // written by K2 (K4 adds iterations), copied into the host's pinned memory by K5
    int nlev, ix, iy, S;
    int xmin, xmax, ymin, ymax;
    long long W;
    int iters; // median iterations (x levels; K4 adds its own atomically)
    int mismatch; // (ix, iy) differ from what the host assumed when it sized the launches: the
                  // kernels after K2 do nothing and the host runs the step again with the real plan
    int fixup; // written by the kernel that ends the step (the labelling kernel's last CTA, or k_finalize):
               // 0 the tables are final; 1 nothing moved on any rank, the host has to run k_finalize for the
               // naive blocks; 2 nothing moved on THIS rank and the other ranks' verdicts were not awaited
    int pad_;
    // diagnostics (printed by the host when DDC_DEBUG_TS is set): %globaltimer stamps.
    //  0-5   K2: start, after the exchange barrier, prefix, plan, walks, end
    //  6-10  K4 block 0: start, after the barrier, after the prefix, end; 10: longest K4 block (ns)
    //  11-14 mask scan: first CTA past its dependency wait, last CTA out of its row loop, last column push
    //        performed, flag raised          15-16 strip rows: first CTA start, last CTA end
    //  17-19 labelling: first CTA start, last CTA out of its row loop, epilogue done
    //  20-27 K2 thread 0 after each level of its walk    28-35 the same for K4 block 0
    unsigned long long ts[44]; // 36-42: first block of k_sum_cols / K2 / row counts / K4 / labelling kernel on an SM (before its wait),
                               //        k_sum_cols past the flags, k_sum_cols done
};
constexpr int TS_SCAN = 11, TS_ROWS = 15, TS_LABEL = 17, TS_XLEV = 20, TS_YLEV = 28, TS_RES = 36;

struct NaiveParams { // Grid.cpp:150-166
    int np0, np1, lx, ly;
};

// ------------------------------------------------------------------------------------------------
// multi-GPU exchange over peer memory (NVLink / NVSwitch)
// ------------------------------------------------------------------------------------------------
// With several GPUs the three exchange steps of a decomposition (column counts, strip row counts,
// the `changes` flag) are not separate collectives.  The PRODUCING kernel pushes its histogram into
// a slot of every peer's exchange buffer (mapped with CUDA IPC; posted stores over NVLink, spread
// over all its CTAs), and the CONSUMING kernel waits for a flag in its prologue and then reads
// local memory only -- a remote LOAD costs a full NVLink round trip per dependent access, which a
// single cut CTA cannot hide (measured: 160 us to pull 8 x 128 KiB with one CTA, DESIGN.md 5).
//   signal  rank r stores 2 * step + bit into slot [stage][r] of EVERY rank's flag array
//           (st.release.sys over NVLink) once everything it pushed for the stage is performed;
//   wait    a rank polls its OWN flag array (local memory) until all G slots of the stage have
//           reached 2 * step.  Steps only grow, so flags are never reset, and the data slots
//           alternate between two copies by step parity, so a rank may run ahead into the next
//           step without overwriting what a slower peer is still reading.
// Each rank runs on its own GPU; a rank that does not show up within PEER_TIMEOUT_NS makes the
// others give up (Plan::mismatch = 3) instead of hanging.
constexpr int MAX_PEERS = 16;
constexpr int PEER_STAGES = 3; // 0 column counts, 1 strip row counts, 2 changes
constexpr unsigned long long PEER_TIMEOUT_NS = 2000000000ull;
struct PeerSync {
    unsigned* flags[MAX_PEERS]; // rank q's flag array [PEER_STAGES][MAX_PEERS], as mapped here
    int rank, G, enabled;
    unsigned step;
    // exchange step 2 with one flag per BLOCK of the row-count kernel (row_flags_*): rank q's array [G][flagcap], as
    // mapped here; rowflag[0] == nullptr: one flag per rank (stage 1 of `flags`), raised by the kernel's last block
    unsigned* rowflag[MAX_PEERS];
    int flagcap, rowblocks;
};
struct PeerCols { // column counts of every rank: slot g of MY exchange buffer (pushed there by rank g);
                  // n == 1: col[0] already holds global counts (single GPU, or after an all-reduce)
    const unsigned* col[MAX_PEERS];
    int n;
    int own, packed; // packed: every slot but col[own] holds 16-bit counts (see PeerPush)
};
struct PeerRows { // strip row counts of every rank: slot g of MY exchange buffer; n == 1: row[0] is
                  // the gathered [G][rank_stride] (or the only rank's block)
    const void* row[MAX_PEERS];
    int n;
};
struct PeerPush { // where a producing kernel stores its histogram: dst[q] = MY slot in rank q's exchange
                  // buffer (dst[rank] is local memory); n <= 1: nothing to push, dst[0] is the local buffer
    void* dst[MAX_PEERS];
    int n, rank;
    int packed; // column counts only: pushed as 16-bit values (every rank holds < 65536 rows)
};
#ifndef DDC_HOST_EMU
__device__ __forceinline__ unsigned long long global_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// thread q of a block tells rank q that this rank has reached `stage` of the current step.  The
// caller makes sure (fences + barriers) that everything pushed for the stage is ordered before.
// (st.release.sys is the fence: cumulative over the barriers and block counters the caller went through)
__device__ __forceinline__ void peer_signal(const PeerSync& ps, int stage, unsigned bit)
{
    const int q = threadIdx.x;
    unsigned* dst = ps.flags[q] + stage * MAX_PEERS + ps.rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(dst), "r"(2u * ps.step + bit) : "memory");
}
// the same for a stage whose flag IS the message (exchange step 3: the `changes` bit): nothing was pushed before it, so
// nothing has to be ordered before it -- the labelling kernel's last block does not wait for a round trip over NVLink
__device__ __forceinline__ void peer_signal_relaxed(const PeerSync& ps, int stage, unsigned bit)
{
    const int q = threadIdx.x;
    unsigned* dst = ps.flags[q] + stage * MAX_PEERS + ps.rank;
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(dst), "r"(2u * ps.step + bit) : "memory");
}
// thread q waits until rank q has reached `stage`.  Returns false on timeout; *seen = its flag value.
// this rank's own flag of a stage, for a consumer on the same GPU (one thread)
__device__ __forceinline__ void peer_signal_local(const PeerSync& ps, int stage)
{
    __threadfence();
    unsigned* dst = ps.flags[ps.rank] + stage * MAX_PEERS + ps.rank;
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(dst), "r"(2u * ps.step) : "memory");
}
__device__ __forceinline__ bool peer_wait(const PeerSync& ps, int stage, unsigned* seen)
{
    const int q = threadIdx.x;
    const unsigned want = 2u * ps.step;
    const unsigned* src = ps.flags[ps.rank] + stage * MAX_PEERS + q;
    const unsigned long long t0 = global_ns();
    unsigned v;
    for (;;) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
        if (v >= want)
            break;
        if (global_ns() - t0 > PEER_TIMEOUT_NS)
            return false;
    }
    *seen = v;
    return true;
}
#else
// test builds: the emulated ranks run phase by phase, a flag is either there or the test is wrong
inline unsigned long long global_ns()
{
    static unsigned long long t = 0;
    return t += 1000;
}
inline void peer_signal(const PeerSync& ps, int stage, unsigned bit)
{
    ps.flags[threadIdx.x][stage * MAX_PEERS + ps.rank] = 2u * ps.step + bit;
}
inline void peer_signal_relaxed(const PeerSync& ps, int stage, unsigned bit) { peer_signal(ps, stage, bit); }
inline void peer_signal_local(const PeerSync& ps, int stage)
{
    ps.flags[ps.rank][stage * MAX_PEERS + ps.rank] = 2u * ps.step;
}
inline bool peer_wait(const PeerSync& ps, int stage, unsigned* seen)
{
    const unsigned v = ps.flags[ps.rank][stage * MAX_PEERS + threadIdx.x];
    *seen = v;
    return v >= 2u * ps.step;
}
#endif
// Exchange step 1 travels as "data + flag" words (the LL protocol of collective libraries): every 8-byte word a rank
// stores into a peer's slot carries 32 bits of counts and, in its upper half, the step number.  An aligned 8-byte
// store is single-copy atomic, so the consumer polls the word itself -- data and "it has arrived" come together, and
// the producer needs no fence.sys before a separate flag (two of them sat on the critical path of every step: one
// per column block, one before the flag -- 10-14 us between the end of the scan and the flag on 8 GPUs, now the one-way
// latency of a store).  Steps only grow and a slot alternates by step parity, so a stale word is simply "not yet".
//   packed (every rank holds < 65536 rows): word i = { count[2 i] | count[2 i + 1] << 16, step }
//   else:                                   word i = { count[i], step }
//   behind the nw column words: the rank's dot y-range, { -(first ocean row), step } and { last ocean row, step }
__host__ __device__ __forceinline__ unsigned long long ll_word(unsigned data, unsigned step)
{
    return (unsigned long long)data | ((unsigned long long)step << 32);
}
__host__ __device__ __forceinline__ size_t ll_column_words(int yr_off, int packed) // yr_off = NX rounded up to 4
{
    return packed ? (size_t)yr_off / 2 : (size_t)yr_off;
}
#ifndef DDC_HOST_EMU
__device__ __forceinline__ void ll_store2(unsigned long long* dst, unsigned long long a, unsigned long long b)
{
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void ll_store1(unsigned long long* dst, unsigned long long a)
{
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(dst), "l"(a) : "memory");
}
__device__ __forceinline__ void ll_load2(const unsigned long long* src, unsigned long long& a, unsigned long long& b)
{
    asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(src) : "memory");
}
__device__ __forceinline__ unsigned long long ll_load1(const unsigned long long* src)
{
    unsigned long long a;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(a) : "l"(src) : "memory");
    return a;
}
#else
inline void ll_store2(unsigned long long* dst, unsigned long long a, unsigned long long b)
{
    dst[0] = a;
    dst[1] = b;
}
inline void ll_store1(unsigned long long* dst, unsigned long long a) { *dst = a; }
inline void ll_load2(const unsigned long long* src, unsigned long long& a, unsigned long long& b)
{
    a = src[0];
    b = src[1];
}
inline unsigned long long ll_load1(const unsigned long long* src) { return *src; }
#endif
// two / one words whose step halves must both read `step`; false: timed out
__device__ __forceinline__ bool ll_wait2(const unsigned long long* src, unsigned step, unsigned& d0, unsigned& d1)
{
    unsigned long long a, b;
    ll_load2(src, a, b);
    if ((unsigned)(a >> 32) != step || (unsigned)(b >> 32) != step) {
        const unsigned long long t0 = global_ns();
        do {
            if (global_ns() - t0 > PEER_TIMEOUT_NS)
                return false;
            ll_load2(src, a, b);
        } while ((unsigned)(a >> 32) != step || (unsigned)(b >> 32) != step);
    }
    d0 = (unsigned)a;
    d1 = (unsigned)b;
    return true;
}

// Programmatic dependent launch: the kernels of a step are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so a kernel may become resident while its predecessor
// in the stream is still running.  pdl_trigger() lets the NEXT kernel's CTAs be scheduled as soon as every CTA
// of this grid has called it (they then sit in their own pdl_wait()); pdl_wait() returns once the previous
// grid has completed and its memory operations are visible.  Every kernel of the chain calls pdl_wait() on
// every path before it touches global memory, so completion is transitive along the chain.  Without the
// launch attribute both are no-ops.
#ifndef DDC_HOST_EMU
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#else
inline void pdl_wait() { }
inline void pdl_trigger() { }
#endif
// diagnostic stamps (dbg == nullptr unless DDC_DEBUG_TS is set; the host zeroes them before the step)
__device__ __forceinline__ void stamp_first(unsigned long long* dbg, int i)
{
    if (dbg && dbg[i] == 0ull)
        atomicCAS(dbg + i, 0ull, global_ns());
}
__device__ __forceinline__ void stamp_last(unsigned long long* dbg, int i)
{
    if (dbg)
        atomicMax(dbg + i, global_ns());
}

// Flags instead of kernel boundaries.  griddepcontrol.wait returns when the previous GRID has completed and its memory
// is flushed -- 1.5 us after its last block on one GPU, but 5-8 us once the device maps peer memory (measured on 2 and
// 8 GPUs at every boundary of the chain, also behind kernels that store nothing remotely).  A consumer can do
// without the completion when the producer's LAST block publishes "my outputs are written" itself: it stores the step
// number into a word of device memory (release, gpu scope, after a barrier + fence that order the block's and -- through
// the block counter -- the grid's writes before it), and every block of the consumer polls that word (acquire) in
// place of griddepcontrol.wait.  Causality is cumulative, so whatever the producer had acquired (the completion of ITS
// predecessor, the peers' flags) is ordered before the consumer as well.  The consumer's blocks may be resident and
// polling while the producer runs; that is safe because a dependent grid is only launched once every block of the
// primary is resident (they all have executed griddepcontrol.launch_dependents).  word == nullptr: kernel boundary.
struct ChainWord {
    unsigned* word;
    unsigned step;
};
#ifndef DDC_HOST_EMU
// one thread, after a __syncthreads() behind the writes of its block
__device__ __forceinline__ void chain_signal(const ChainWord& c)
{
    if (!c.word)
        return;
    __threadfence();
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(c.word), "r"(c.step) : "memory");
}
// all threads of a block, first thing.  (Steps only grow and a word belongs to one boundary of one handle, so "==" and
// ">=" are the same; a word that never comes -- the producer died -- falls back to the kernel boundary.)
__device__ __forceinline__ void chain_wait(const ChainWord& c)
{
    if (!c.word) {
        pdl_wait();
        return;
    }
    if (threadIdx.x == 0) {
        const unsigned long long t0 = global_ns();
        unsigned v;
        for (;;) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(c.word) : "memory");
            if (v == c.step)
                break;
            if (global_ns() - t0 > PEER_TIMEOUT_NS) {
                pdl_wait();
                break;
            }
        }
    }
    __syncthreads();
}
#else
inline void chain_signal(const ChainWord& c)
{
    if (c.word)
        *c.word = c.step;
}
inline void chain_wait(const ChainWord& c)
{
    if (c.word && *c.word != c.step) // (the emulated launches run one after the other: the word must be there)
    {
        fprintf(stderr, "chain_wait: the producer did not publish its word (%u, step %u)\n", *c.word, c.step);
        abort();
    }
}
#endif

// Called by the first G threads of a block (thread q talks to rank q).  do_signal: exactly one
// block per rank sends.
__device__ __forceinline__ bool peer_barrier(const PeerSync& ps, int stage, unsigned bit, bool do_signal,
    unsigned* seen)
{
    if (do_signal)
        peer_signal(ps, stage, bit);
    return peer_wait(ps, stage, seen);
}

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }

// part loads -> global min / max (loadmm = {min, max}, pre-set to {LLONG_MAX, -1} by k_init); called by
// all threads of a block with the extremes of the parts each of them wrote (or the neutral values)
__device__ __forceinline__ void reduce_load_extremes(long long mn, long long mx, long long* loadmm)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
        mn = a < mn ? a : mn;
        mx = b > mx ? b : mx;
    }
    if (lane_id() == 0 && mx >= 0) {
        atomicMin(loadmm, mn);
        atomicMax(loadmm + 1, mx);
    }
}

// bits of a 32-column word that belong to word-relative columns [a, b), clipped to [0, 32]
__device__ __forceinline__ unsigned word_range_mask(int a, int b)
{
    a = max(a, 0);
    b = min(b, 32);
    if (b <= a)
        return 0u;
    const unsigned hi = b >= 32 ? 0xffffffffu : ((1u << b) - 1u);
    return hi & ~((1u << a) - 1u);
}

// exclusive block scan of one value per thread (blockDim.x <= 1024, multiple of 32)
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* total, T* warp_sums /* >= 33 entries */)
{
    unsigned lane = lane_id(), warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o)
            inc += t;
    }
    if (lane == 31)
        warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        T w = lane < nwarp ? warp_sums[lane] : T(0);
        T winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            T t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= (unsigned)o)
                winc += t;
        }
        warp_sums[lane] = winc - w; // exclusive
        if (lane == 31)
            warp_sums[32] = winc;
    }
    __syncthreads();
    T res = warp_sums[warp] + inc - v;
    *total = warp_sums[32];
    __syncthreads();
    return res;
}

// dst[i] = sum of src(0..i-1) for i in [0, n] (exclusive prefix, n + 1 outputs); every thread of the
// block calls it.  4 consecutive elements per thread and tile, so a warp reads 512 contiguous bytes.
// INCL_M1: write (inclusive prefix - 1 + bias) into dst[0..n) instead (used to turn "start flags"
// into "index of the last interval starting at or before i").
template <bool INCL_M1, typename F>
__device__ inline unsigned long long block_prefix(F src, int n, unsigned* dst, int bias,
    unsigned long long* wsum /* >= 33 */)
{
    unsigned long long carry = 0;
    const int tile = blockDim.x * 4;
    for (int base = 0; base < n; base += tile) {
        const int i0 = base + threadIdx.x * 4;
        unsigned v[4];
#pragma unroll
        for (int k = 0; k < 4; k++)
            v[k] = i0 + k < n ? src(i0 + k) : 0u;
        unsigned long long total;
        unsigned long long run
            = carry + block_exclusive_scan<unsigned long long>((unsigned long long)v[0] + v[1] + v[2] + v[3], &total, wsum);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (INCL_M1) {
                run += v[k];
                if (i0 + k < n)
                    dst[i0 + k] = (unsigned)((long long)run - 1 + bias);
            } else {
                if (i0 + k < n)
                    dst[i0 + k] = (unsigned)run;
                run += v[k];
            }
        }
        carry += total;
    }
    if (!INCL_M1 && threadIdx.x == 0)
        dst[n] = (unsigned)carry;
    __syncthreads();
    return carry;
}

// Same result as block_prefix<false> (dst[i] = sum of the first i elements, n + 1 outputs, 32-bit
// sums) for a 1024-thread block, built for the latency of the cut kernels: a tile of 32768 elements
// is ONE pass with two block barriers.  The tile is cut into 8 sub-tiles of 4096; thread t owns the 4
// consecutive elements [4 t, 4 t + 4) of every sub-tile, so that every load and every store of a warp
// is one contiguous 512-byte run (a single SM pulls the whole histogram out of L2: with 32
// consecutive elements per thread every load instruction touched 32 different lines and, because
// data written by other GPUs has to bypass L1, each line crossed the L2 interface 8 times).  The 8
// sub-tile scans run side by side: 8 independent shuffle chains per thread, then warp q scans the
// 32 warp totals of sub-tile q.
// load_tile(base, v) fills v[q] with elements base + q * 4096 .. + 3 (0 beyond n) for the 8 sub-tiles q, base
// a multiple of 4 -- all of a thread's loads are requested in ONE call, so that a loader that has to visit
// several buffers can keep 8 independent loads in flight per buffer; dst may be shared or global
// memory.  bitmap != nullptr: also writes the three-level bit map of the non-empty elements,
// l0 / l1 / l2 = bitmap + 0 / tiles * 1024 / tiles * (1024 + 32).   ws: >= 8 * 32 + 8 words.
constexpr int PFX_Q = 8; // sub-tiles of a tile
constexpr int PFX_WS = PFX_Q * 32 + PFX_Q;
template <typename F>
__device__ inline unsigned block_prefix_tiles(F load_tile, int n, unsigned* dst, unsigned* ws, unsigned* bitmap = nullptr)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tiles = (n + HIST_TILE - 1) / HIST_TILE;
    unsigned carry = 0;
    for (int t = 0; t < tiles; t++) {
        const int base = t * HIST_TILE + tid * 4;
        // sub-tiles of this tile that hold elements: a histogram of a few hundred bins (the small grids) pays for
        // one sub-tile scan, not for eight (the skipped ones are empty: sums 0, bit-map words 0)
        const int nq = min(PFX_Q, (n - t * HIST_TILE + 4095) >> 12);
        uint4 v[PFX_Q];
        unsigned s[PFX_Q], inc[PFX_Q];
        load_tile(base, v);
#pragma unroll
        for (int q = 0; q < PFX_Q; q++)
            inc[q] = s[q] = v[q].x + v[q].y + v[q].z + v[q].w;
#pragma unroll
        for (int q = 0; q < PFX_Q; q++) {
            if (q < nq) { // (uniform over the block)
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned u = __shfl_up_sync(0xffffffffu, inc[q], o);
                    if (lane >= o)
                        inc[q] += u;
                }
            }
        }
        if (bitmap) { // l0: one bit per element; 8 neighbouring lanes make one 32-bit word
#pragma unroll
            for (int q = 0; q < PFX_Q; q++) {
                if (q >= nq) {
                    if ((lane & 7) == 0 && (base + q * 4096) >> 5 < tiles * 1024)
                        bitmap[(base + q * 4096) >> 5] = 0u;
                    continue;
                }
                unsigned w = ((unsigned)(v[q].x != 0u) | ((unsigned)(v[q].y != 0u) << 1) | ((unsigned)(v[q].z != 0u) << 2)
                                 | ((unsigned)(v[q].w != 0u) << 3))
                    << (4 * (lane & 7));
                w |= __shfl_xor_sync(0xffffffffu, w, 1);
                w |= __shfl_xor_sync(0xffffffffu, w, 2);
                w |= __shfl_xor_sync(0xffffffffu, w, 4);
                if ((lane & 7) == 0)
                    bitmap[(base + q * 4096) >> 5] = w;
            }
        }
        if (lane == 31) {
#pragma unroll
            for (int q = 0; q < PFX_Q; q++)
                ws[q * 32 + warp] = inc[q];
        }
        __syncthreads();
        if (warp < PFX_Q) { // warp q: exclusive scan of the 32 warp totals of sub-tile q
            const unsigned w = ws[warp * 32 + lane];
            unsigned winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned u = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o)
                    winc += u;
            }
            ws[warp * 32 + lane] = winc - w;
            if (lane == 31)
                ws[PFX_Q * 32 + warp] = winc;
        }
        __syncthreads();
        unsigned run = carry;
#pragma unroll
        for (int q = 0; q < PFX_Q; q++) {
            const int i = base + q * 4096;
            if (q >= nq) // nothing of this sub-tile lies below n (and its total is 0)
                continue;
            uint4 o;
            o.x = run + ws[q * 32 + warp] + inc[q] - s[q];
            o.y = o.x + v[q].x;
            o.z = o.y + v[q].y;
            o.w = o.z + v[q].z;
            run += ws[PFX_Q * 32 + q];
            if (i + 4 <= n && ((uintptr_t)(dst + i) & 15) == 0)
                *reinterpret_cast<uint4*>(dst + i) = o;
            else {
                if (i < n)
                    dst[i] = o.x;
                if (i + 1 < n)
                    dst[i + 1] = o.y;
                if (i + 2 < n)
                    dst[i + 2] = o.z;
                if (i + 3 < n)
                    dst[i + 3] = o.w;
            }
        }
        carry = run;
        __syncthreads(); // ws is reused by the next tile
    }
    if (tid == 0)
        dst[n] = carry;
    if (bitmap) { // l1: one bit per l0 word, l2: one bit per l1 word
        unsigned* l1 = bitmap + tiles * 1024;
        unsigned* l2 = bitmap + tiles * (1024 + 32);
        for (int i = tid; i < tiles * 1024; i += 1024) {
            const unsigned b1 = __ballot_sync(0xffffffffu, bitmap[i] != 0u);
            if (lane == 0)
                l1[i >> 5] = b1;
        }
        __syncthreads();
        for (int i = tid; i < tiles * 32; i += 1024) { // whole warps: tiles * 32 is a multiple of 32
            const unsigned b2 = __ballot_sync(0xffffffffu, l1[i] != 0u);
            if (lane == 0)
                l2[i >> 5] = b2;
        }
    }
    __syncthreads();
    return carry;
}

// ------------------------------------------------------------------------------------------------
// K1: mask scan
// ------------------------------------------------------------------------------------------------
// One warp owns one 128-column group for `rows_per_cta` rows; the 8 warps of a CTA own 8 adjacent
// groups, i.e. 4 KiB contiguous per row.  Every lane issues 8 independent 16-byte loads (8 rows)
// before using any of them, then packs its 4 x 8 ocean flags into ONE register (nibble k = row k).
// Everything else is derived from that register once per 8 rows: the column counts (4 popcounts),
// the bit-map bytes (one shuffle pairs the nibbles of neighbouring lanes) and the rows that hold
// any ocean cell (one warp OR-reduction).  VEC: NX % 4 == 0 and a 16-byte aligned base pointer.
__device__ __forceinline__ unsigned ocean_nibble(const int4& v)
{
    return (unsigned)(v.x > 0) | ((unsigned)(v.y > 0) << 1) | ((unsigned)(v.z > 0) << 2)
        | ((unsigned)(v.w > 0) << 3);
}

constexpr int SCAN_STAGE_ROWS = 64; // bit-map rows staged in shared memory between flushes (power of 2)

template <bool VEC>
__global__ void __launch_bounds__(256, 4) k_scan_mask(const int32_t* __restrict__ mask, int NX, int rows,
    int y_begin, int NB, int rows_per_cta, uint8_t* __restrict__ bits, unsigned* __restrict__ colcount,
    int* __restrict__ yr /* this rank's {-(first ocean row), last ocean row}, max-reduced */,
    PeerPush push, PeerSync ps, unsigned* __restrict__ done /* [gridDim.x + 1], zeroed by k_init */, int yr_off,
    unsigned long long* dbg, int nbig /* row chunks of rows_per_cta rows; the chunks after them hold rows_small */,
    int rows_small)
{
    __shared__ __align__(16) uint8_t sbits[SCAN_STAGE_ROWS][128];
    __shared__ int s_last;
    pdl_trigger(); // the x-cut kernel may become resident (and warm up) while the scan is still running
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    // warps beyond the last 128-column group (last column block only) have no columns: they
    // load nothing (clamped, masked addresses below) but take part in the CTA barriers
    const int g = min(blockIdx.x * 8 + warp, NB / 16 - 1);
    const bool warp_valid = blockIdx.x * 8 + warp < NB / 16;
    // Blocks are scheduled in index order, and the last blocks of a grid run on a half-empty machine that no longer
    // saturates HBM: the last rows are therefore cut into smaller chunks (a fine-grained tail), the bulk into large
    // ones (fewer column atomics).
    const int big = (int)blockIdx.y < nbig;
    const int r0 = big ? blockIdx.y * rows_per_cta : nbig * rows_per_cta + ((int)blockIdx.y - nbig) * rows_small;
    const int r1 = min(rows, r0 + (big ? rows_per_cta : rows_small));
    const int x = g * 128 + lane * 4;
    unsigned c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    int ylo = 0x7fffffff, yhi = -1;

    // VEC: out-of-range lanes (x >= NX, only in the last group) re-read the last valid 16 bytes of
    // the row and are masked off below, so the main loop is branch-free.  The 8 rows of a batch
    // are loaded as two halves of 4; the next half is always requested before the current one
    // is consumed, so every lane keeps 4 to 8 independent 16-byte loads in flight at all times.
    const int xl = VEC ? min(x, NX - 4) : x;
    const unsigned lane_valid = ((VEC && x >= NX) || !warp_valid) ? 0u : 0xffffffffu;
    const size_t pitch4 = (size_t)NX >> 2;
    int4 h0[4], h1[4];
    const int4* pv = reinterpret_cast<const int4*>(mask + (size_t)r0 * NX + xl);
    const bool vec_first = VEC && r0 + 8 <= r1;
    // the previous step's labelling kernel still reads the bit map, and the mask may come from the caller's
    // kernel just before this one in the stream
    pdl_wait();
    if (threadIdx.x == 0)
        stamp_first(dbg, TS_SCAN);
    if (vec_first) {
#pragma unroll
        for (int k = 0; k < 4; k++)
            h0[k] = __ldcs(pv + k * pitch4);
    }
    for (int r = r0; r < r1; r += 8) {
        const bool full = r + 8 <= r1;
        unsigned packed = 0; // nibble k = the ocean flags of my 4 columns in row r + k
        if (VEC && full) {
            const int4* p = reinterpret_cast<const int4*>(mask + (size_t)r * NX + xl);
#pragma unroll
            for (int k = 0; k < 4; k++)
                h1[k] = __ldcs(p + (4 + k) * pitch4);
#pragma unroll
            for (int k = 0; k < 4; k++)
                packed |= ocean_nibble(h0[k]) << (4 * k);
            if (r + 16 <= r1) { // first half of the next batch
#pragma unroll
                for (int k = 0; k < 4; k++)
                    h0[k] = __ldcs(p + (8 + k) * pitch4);
            }
#pragma unroll
            for (int k = 0; k < 4; k++)
                packed |= ocean_nibble(h1[k]) << (16 + 4 * k);
        } else {
            int4 v[8];
#pragma unroll
            for (int k = 0; k < 8; k++) {
                v[k] = make_int4(0, 0, 0, 0);
                if (r + k < r1) {
                    const int32_t* p = mask + (size_t)(r + k) * NX + xl;
                    if (VEC) {
                        v[k] = __ldcs(reinterpret_cast<const int4*>(p));
                    } else {
                        if (x < NX)
                            v[k].x = __ldcs(p);
                        if (x + 1 < NX)
                            v[k].y = __ldcs(p + 1);
                        if (x + 2 < NX)
                            v[k].z = __ldcs(p + 2);
                        if (x + 3 < NX)
                            v[k].w = __ldcs(p + 3);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 8; k++)
                packed |= ocean_nibble(v[k]) << (4 * k);
        }
        packed &= lane_valid;
        c0 += __popc(packed & 0x11111111u);
        c1 += __popc(packed & 0x22222222u);
        c2 += __popc(packed & 0x44444444u);
        c3 += __popc(packed & 0x88888888u);
        // bit-map bytes: even lanes store [nibble of lane + 1 : own nibble]
        const unsigned other = __shfl_down_sync(0xffffffffu, packed, 1);
        const unsigned even = (packed & 0x0f0f0f0fu) | ((other & 0x0f0f0f0fu) << 4); // rows 0,2,4,6
        const unsigned odd = ((packed >> 4) & 0x0f0f0f0fu) | (other & 0xf0f0f0f0u); // rows 1,3,5,7
        // bit-map bytes go through shared memory so that the CTA writes whole 128-byte lines
        if (!(lane & 1)) {
            uint8_t* sp = &sbits[(r - r0) & (SCAN_STAGE_ROWS - 1)][warp * 16 + (lane >> 1)];
#pragma unroll
            for (int k = 0; k < 8; k++)
                sp[k * 128] = (uint8_t)(((k & 1) ? odd : even) >> (8 * (k >> 1)));
        }
        if ((((r - r0) + 8) & (SCAN_STAGE_ROWS - 1)) == 0 || r + 8 >= r1) {
            // flush the staged rows [rs, r + 8) as 16-byte chunks, 8 chunks (one line) per row
            const int rs = r0 + ((r - r0) & ~(SCAN_STAGE_ROWS - 1));
            const int nr = min(r + 8, r1) - rs;
            __syncthreads();
            for (int i = threadIdx.x; i < nr * 8; i += blockDim.x) {
                const int row = i >> 3, c = i & 7;
                if (blockIdx.x * 8 + c < NB / 16)
                    *reinterpret_cast<uint4*>(bits + (size_t)(rs + row) * NB + (size_t)blockIdx.x * 128 + c * 16)
                        = *reinterpret_cast<const uint4*>(&sbits[row][c * 16]);
            }
            __syncthreads();
        }
        // rows of this batch that hold an ocean cell in my 128 columns
        const unsigned any = __reduce_or_sync(0xffffffffu, packed);
        if (any) {
            ylo = min(ylo, r + ((__ffs(any) - 1) >> 2));
            yhi = r + ((31 - __clz(any)) >> 2);
        }
    }
    if (c0)
        atomicAdd(colcount + x, c0);
    if (c1)
        atomicAdd(colcount + x + 1, c1);
    if (c2)
        atomicAdd(colcount + x + 2, c2);
    if (c3)
        atomicAdd(colcount + x + 3, c3);
    if (lane == 0 && yhi >= 0) {
        const int ny0 = -(y_begin + ylo), y1 = y_begin + yhi;
        if (ny0 > yr[0])
            atomicMax(&yr[0], ny0);
        if (y1 > yr[1])
            atomicMax(&yr[1], y1);
    }
    if (threadIdx.x == 0)
        stamp_last(dbg, TS_SCAN + 1);
    if (push.n <= 1)
        return;
    // Exchange step 1 (several GPUs): the LAST CTA of a column block to finish pushes the block's final counts into
    // this rank's slot of every peer's exchange buffer as data + flag words (ll_word: no fence, the peers poll the
    // words themselves) -- so the counts travel while the rest of the scan is still running.  The last column block
    // to have done so sends the dot y-range the same way and tells this rank's own summing kernel (a flag in local
    // memory) that the local counts are final.
    __syncthreads(); // every thread's atomics are issued ...
    if (threadIdx.x == 0) {
        __threadfence(); // ... and performed (cumulative over the barrier) before this CTA is counted as done
        s_last = atomicAdd(&done[blockIdx.x], 1u) == gridDim.y - 1;
        if (s_last)
            __threadfence();
    }
    __syncthreads();
    if (!s_last)
        return;
    const int c = blockIdx.x * 1024 + threadIdx.x * 4;
    if (c < yr_off) {
        const uint4 v = __ldcg(reinterpret_cast<const uint4*>(colcount + c));
        if (push.packed) { // a rank holds < 65536 rows: two counts per word
            const unsigned long long w0 = ll_word(v.x | (v.y << 16), ps.step), w1 = ll_word(v.z | (v.w << 16), ps.step);
            for (int q = 0; q < push.n; q++)
                if (q != push.rank)
                    ll_store2(reinterpret_cast<unsigned long long*>(push.dst[q]) + (c >> 1), w0, w1);
        } else {
            const unsigned long long w0 = ll_word(v.x, ps.step), w1 = ll_word(v.y, ps.step), w2 = ll_word(v.z, ps.step),
                                     w3 = ll_word(v.w, ps.step);
            for (int q = 0; q < push.n; q++)
                if (q != push.rank) {
                    unsigned long long* d = reinterpret_cast<unsigned long long*>(push.dst[q]) + c;
                    ll_store2(d, w0, w1);
                    ll_store2(d + 2, w2, w3);
                }
        }
    }
    __syncthreads(); // (s_last is about to be written again)
    if (threadIdx.x == 0) {
        stamp_last(dbg, TS_SCAN + 2);
        s_last = atomicAdd(&done[gridDim.x], 1u) == gridDim.x - 1; // (this block has seen all CTAs of its columns)
        if (s_last)
            __threadfence();
    }
    __syncthreads();
    if (!s_last)
        return;
    if ((int)threadIdx.x < push.n) {
        const int q = threadIdx.x;
        if (q != push.rank) {
            unsigned long long* d = reinterpret_cast<unsigned long long*>(push.dst[q]) + ll_column_words(yr_off, push.packed);
            ll_store2(d, ll_word((unsigned)__ldcg(yr), ps.step), ll_word((unsigned)__ldcg(yr + 1), ps.step));
        } else
            peer_signal_local(ps, 0); // this rank's own counts: read in place by its summing kernel
        if (threadIdx.x == 0)
            stamp_last(dbg, TS_SCAN + 3);
    }
    // every CTA has been counted: the counters are ready for the next step (k_init is then only needed when
    // the geometry changes)
    for (unsigned i = threadIdx.x; i <= gridDim.x; i += blockDim.x)
        done[i] = 0u;
}

// ------------------------------------------------------------------------------------------------
// The RCB recursion level by level: ONE thread per set
// ------------------------------------------------------------------------------------------------
// The sets of one level (cell range [lo, hi) along the cut dimension, parts [plo, plo + n)) sit in shared memory
// in part order; every set is split by exactly one thread, and the threads that work are spread over the warps
// (set i -> thread i * spread), so that a level with up to 32 sets runs one median per warp: no divergence, no
// redundant work.  The barrier-free walks (rcb_walk: every leaf's thread group re-evaluates the medians of its
// whole path) issued ~7 x the instructions from all 32 warps at once and ran at 13 cycles per dependent
// instruction (ncu: "wait" stalls, 0.55 IPC); a level here costs one median's latency plus a block barrier.
// Because Zoltan_Divide_Machine halves the part counts (ceil / floor), the part counts of one level differ by at
// most one, which gives the position of a set's children in the next level in closed form: 2 i while every set
// still splits, and plo - root.plo once the sets hold one or two parts (a set of one part is carried down).
constexpr int LEVEL_NODES = 1024; // sets per level held in shared memory (more leaves: the walks below)
struct __align__(16) RcbNode {
    int lo, hi, plo, n;
};
constexpr size_t LEVEL_NODES_BYTES = 2 * LEVEL_NODES * sizeof(RcbNode) + 16;
// all threads of the block call it; returns the final sets (in part order) and their number through *count.
// iters: this thread's median iterations are added.  lvl_ts (diagnostics): thread 0 stamps the start of a level.
// FAST: the histogram is in shared memory with a bit map and at most FAST_HIST_BINS bins (median_boundary_fast)
template <bool FAST>
__device__ inline const RcbNode* rcb_levels(const Hist& H, RcbSet root, int levels, RcbNode* nodes /* [2][LEVEL_NODES] */,
    int* iters, unsigned long long* lvl_ts, int* count)
{
    FastHist F {};
    if (FAST)
        F = make_fast_hist(H);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    int cur = 0, cnt = 1;
    if (tid == 0) {
        const RcbNode r = { root.lo, root.hi, root.plo, root.n };
        nodes[0] = r;
    }
    __syncthreads();
    for (int l = 0; l < levels; l++) {
        // part counts of this level: floor and ceil of root.n / 2^l (uniform over the block)
        const int minn = l >= 31 ? 0 : root.n >> l;
        const int maxn = l >= 31 ? 1 : (int)(((long long)root.n + (1LL << l) - 1) >> l);
        if (maxn <= 1)
            break;
        if (lvl_ts && tid == 0 && l < 8)
            lvl_ts[l] = walk_clock();
        int shift = 0; // set i -> thread i << shift: the largest spread (<= 32) that still fits the block
        while (shift < 5 && (2 << shift) * cnt <= nthreads)
            shift++;
        const RcbNode* src = nodes + cur * LEVEL_NODES;
        RcbNode* dst = nodes + (cur ^ 1) * LEVEL_NODES;
        const int i = tid >> shift;
        if ((tid & ((1 << shift) - 1)) == 0 && i < cnt) {
            const RcbNode sset = src[i];
            const int off = minn >= 2 ? 2 * i : sset.plo - root.plo;
            if (sset.n > 1) {
                const int nlo = (sset.n - 1) / 2 + 1;
                int it = 0;
                const int cut = FAST ? median_boundary_fast(F, sset.lo, sset.hi - 1, nlo, sset.n, &it)
                                     : median_boundary(H, sset.lo, sset.hi - 1, nlo, sset.n, &it);
                *iters += it;
                const RcbNode a = { sset.lo, cut, sset.plo, nlo }, b = { cut, sset.hi, sset.plo + nlo, sset.n - nlo };
                dst[off] = a;
                dst[off + 1] = b;
            } else
                dst[off] = sset;
        }
        cnt = minn >= 2 ? 2 * cnt : root.n;
        cur ^= 1;
        __syncthreads();
    }
    *count = cnt;
    return nodes + cur * LEVEL_NODES;
}

// threads that share one leaf's walk: the largest power of two <= 32 with lanes * leaves <= threads
__device__ int g_walk_lanes = 32; // upper bound (tuning knob, set by the host)
__device__ __forceinline__ int walk_lanes(int leaves, int threads)
{
    int lanes = g_walk_lanes;
    while (lanes > 1 && (long long)lanes * leaves > threads)
        lanes >>= 1;
    return lanes;
}
// ------------------------------------------------------------------------------------------------
// K2: column prefix sums, preset directions, all x levels, strip table
// ------------------------------------------------------------------------------------------------
// the plan (levels, mismatch flag, iteration count, fix-up request) goes straight into the host's pinned copy,
// so that a step ends without a separate device -> host copy; called by all threads of a block (>= 128)
__device__ __forceinline__ void publish_plan(const Plan* plan, Plan* host_plan)
{
    static_assert(sizeof(Plan) % 4 == 0 && sizeof(Plan) / 4 <= 128, "Plan is copied word by word by one block");
    if (threadIdx.x < sizeof(Plan) / 4)
        reinterpret_cast<volatile unsigned*>(host_plan)[threadIdx.x]
            = reinterpret_cast<const volatile unsigned*>(plan)[threadIdx.x];
}

// Several GPUs, exchange step 1 on the consuming side.  The G slots of column counts that the ranks' mask scans
// pushed into this rank's buffer are summed by a GRID of blocks (one per 1024 columns, every thread requesting the
// G loads of its 4 columns together), so that the single x-cut block afterwards reads ONE buffer, as on one GPU:
// summing the slots itself cost that block G dependent round trips to L2 -- 24 us of a 58 us kernel on 8 GPUs.
// The peers' slots hold data + flag words (ll_word): a thread polls exactly the words it sums; this rank's own
// counts are plain 32-bit values in local memory, final once its scan has raised the local stage-0 flag.  Block 0
// also gathers the ranks' dot y-ranges behind the sums (sum[yr_off + 2 g ..], the layout K2 expects of a single
// global buffer).  A rank that does not show up raises Plan::mismatch to 3; K2 then gives up.
__global__ void __launch_bounds__(256) k_sum_cols(PeerCols pc, PeerSync ps, int NX, int yr_off, unsigned* __restrict__ sum,
    Plan* plan, int early /* the local flag stands in for the completion of the mask scan (see ChainWord) */,
    unsigned* __restrict__ done /* block counter, zero between steps */, ChainWord next, unsigned long long* dbg)
{
    __shared__ int s_last;
    pdl_trigger();
    if (dbg && threadIdx.x == 0)
        stamp_first(dbg, TS_RES);
    if (!early)
        pdl_wait(); // this rank's mask scan is complete
    bool ok = true;
    if ((int)threadIdx.x == ps.rank) { // (only the own flag: the peers' words are polled one by one below)
        unsigned seen;
        ok = peer_wait(ps, 0, &seen);
    }
    bool timed_out = __syncthreads_or(!ok);
    if (dbg && threadIdx.x == 0)
        stamp_first(dbg, TS_RES + 5);
    const int c = blockIdx.x * 1024 + threadIdx.x * 4;
    if (!timed_out && c < yr_off) {
        uint4 acc = __ldcg(reinterpret_cast<const uint4*>(pc.col[pc.own] + c)); // (zero between NX and yr_off)
        // all peers' words are requested together (one trip to L2); only a word that has not arrived is polled
        for (int g0 = 0; g0 < pc.n; g0 += 8) {
            unsigned long long w[8][4];
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int g = g0 + k;
                if (g >= pc.n || g == pc.own)
                    continue;
                const unsigned long long* src = reinterpret_cast<const unsigned long long*>(pc.col[g]);
                if (pc.packed)
                    ll_load2(src + (c >> 1), w[k][0], w[k][1]);
                else {
                    ll_load2(src + c, w[k][0], w[k][1]);
                    ll_load2(src + c + 2, w[k][2], w[k][3]);
                }
            }
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const int g = g0 + k;
                if (g >= pc.n || g == pc.own)
                    continue;
                const unsigned long long* src = reinterpret_cast<const unsigned long long*>(pc.col[g]);
                unsigned d0 = (unsigned)w[k][0], d1 = (unsigned)w[k][1], d2 = 0u, d3 = 0u;
                if (pc.packed) {
                    if (((unsigned)(w[k][0] >> 32) != ps.step || (unsigned)(w[k][1] >> 32) != ps.step)
                        && !ll_wait2(src + (c >> 1), ps.step, d0, d1))
                        ok = false;
                    acc.x += d0 & 0xffffu;
                    acc.y += d0 >> 16;
                    acc.z += d1 & 0xffffu;
                    acc.w += d1 >> 16;
                } else {
                    d2 = (unsigned)w[k][2];
                    d3 = (unsigned)w[k][3];
                    if (((unsigned)(w[k][0] >> 32) != ps.step || (unsigned)(w[k][1] >> 32) != ps.step)
                        && !ll_wait2(src + c, ps.step, d0, d1))
                        ok = false;
                    if (((unsigned)(w[k][2] >> 32) != ps.step || (unsigned)(w[k][3] >> 32) != ps.step)
                        && !ll_wait2(src + c + 2, ps.step, d2, d3))
                        ok = false;
                    acc.x += d0;
                    acc.y += d1;
                    acc.z += d2;
                    acc.w += d3;
                }
            }
            if (!ok)
                break;
        }
        *reinterpret_cast<uint4*>(sum + c) = acc;
    }
    if (!timed_out && blockIdx.x == 0 && (int)threadIdx.x < pc.n) {
        const int g = threadIdx.x;
        unsigned a = 0u, b = 0u;
        if (g == pc.own) {
            a = __ldcg(pc.col[g] + yr_off + 2 * g);
            b = __ldcg(pc.col[g] + yr_off + 2 * g + 1);
        } else if (!ll_wait2(reinterpret_cast<const unsigned long long*>(pc.col[g]) + ll_column_words(yr_off, pc.packed), ps.step,
                       a, b))
            ok = false;
        sum[yr_off + 2 * g] = a;
        sum[yr_off + 2 * g + 1] = b;
    }
    timed_out = __syncthreads_or(!ok) || timed_out;
    if (timed_out) {
        if (early)
            pdl_wait();
        if (threadIdx.x == 0)
            atomicMax(&plan->mismatch, 3);
    }
    if (dbg && threadIdx.x == 0)
        stamp_last(dbg, TS_RES + 6);
    if (!next.word)
        return;
    // the last block to finish tells the x-cut block that the sums are in place
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(done, 1u) == gridDim.x - 1u;
        if (s_last) {
            *done = 0u;
            chain_signal(next);
        }
    }
}

// the state a rank's column-count slot accumulates from: counts 0, its own y-range pair "no dot yet"
__device__ __forceinline__ unsigned column_slot_reset_value(int i, int yr_off, int rank)
{
    if (i == yr_off + 2 * rank)
        return 0x80000000u; // -(first ocean row) = INT_MIN
    if (i == yr_off + 2 * rank + 1)
        return 0xffffffffu; // last ocean row = -1
    return 0u;
}

// dynamic shared memory when SMEM: (NX + 1) unsigned, rounded up to 4, + hist_bitmap_words(NX).
// aix / aiy: the numbers of x / y levels the host assumed when it sized the launches that follow.
template <bool SMEM>
__global__ void __launch_bounds__(1024) k_xcuts(PeerCols pc, PeerSync ps, int NX, int NY, int P, unsigned* pfx_g,
    int yr_off, int G, int aix, int aiy, Plan* plan, StripTable st, BoxTable bx, long long* loads, long long* loadmm,
    DevScalars* sc, unsigned* own_col /* this rank's column counts: reset here once they are consumed */,
    int dbg, Plan* host_plan, int presummed /* k_sum_cols ran: pc is ONE buffer of global counts */,
    int reset_own /* put this rank's column counts back to zero here (else: the labelling kernel does it) */,
    ChainWord prev /* published by k_sum_cols */, ChainWord next /* polled by the row-count kernel */)
{
    DDC_DYN_SHARED(unsigned, smem_dyn);
    __shared__ unsigned wsum[PFX_WS];
    __shared__ int s_ix, s_iters;
    unsigned* pfx = SMEM ? smem_dyn : pfx_g;
    const int tid = threadIdx.x;
    pdl_trigger(); // the strip row-count kernel may become resident
    if (dbg && tid == 0)
        plan->ts[TS_RES + 1] = global_ns(); // (diagnostic only: the one word written before the wait)
    chain_wait(prev); // the mask scan (and k_sum_cols) is complete
    if (presummed && plan->mismatch == 3) { // a rank did not show up
        publish_plan(plan, host_plan);
        __syncthreads();
        if (tid == 0)
            chain_signal(next);
        return;
    }
    if (tid == 0) {
        plan->ts[0] = global_ns();
        // the per-step scalars: nothing before K2 touches them, everything after K2 accumulates into them
        sc->changes = 0;
        sc->changes_all = 0;
        sc->overflow = 0;
        sc->edge_cut = 0ull;
        loadmm[0] = 0x7fffffffffffffffLL;
        loadmm[1] = -1;
    }

    // 1. pfx[i] = ocean cells in columns [0, i)
    if (tid == 0)
        plan->ts[1] = global_ns();
    unsigned* bitmap = SMEM ? smem_dyn + (((size_t)NX + 1 + 3) & ~(size_t)3) : nullptr;
    // (ONE buffer of global counts: this GPU's own, an all-reduced one, or the sum k_sum_cols made of the ranks' slots;
    //  16-byte aligned, zero between NX and yr_off = NX rounded up to 4)
    const uint4* gcol = reinterpret_cast<const uint4*>(pc.col[0]);
    block_prefix_tiles(
        [&](int base, uint4 (&v)[PFX_Q]) {
#pragma unroll
            for (int q = 0; q < PFX_Q; q++) {
                const int i = base + q * 4096;
                v[q] = i < yr_off ? __ldcg(gcol + (i >> 2)) : make_uint4(0u, 0u, 0u, 0u);
            }
        },
        NX, pfx, wsum, bitmap);
    if (tid == 0)
        plan->ts[2] = global_ns();
    const Hist H = make_hist(pfx, bitmap, NX);

    // 2. the plan: bounding box of all dots -> preset direction of every level
    if (tid == 0) {
        const long long W = pfx[NX];
        int xmin = 0, xmax = 0, ymin = 0, ymax = 0;
        if (W > 0) {
            xmin = first_nonempty(H, 0, NX - 1);
            xmax = last_nonempty(H, 0, NX - 1);
            // every rank's {-(first ocean row), last ocean row} sits in slot g behind its column
            // counts (and, after an all-reduce, in slot g of the one global buffer)
            int a = (int)0x80000000, b = -1;
            for (int g = 0; g < G; g++) {
                const unsigned* src = pc.col[0] + yr_off + 2 * g;
                a = max(a, (int)__ldcg(src));
                b = max(b, (int)__ldcg(src + 1));
            }
            ymin = -a;
            ymax = b;
        }
        double wx = (double)(xmax - xmin), wy = (double)(ymax - ymin);
        int nlev = 0;
        for (int t = P; t > 1; t = (t + 1) / 2)
            nlev++;
        int ix = 0, iy = 0;
        for (int i = 0; i < nlev; i++) {
            if (wx > wy) { // a tie cuts y (Q1)
                ix++;
                wx = wx * 0.5; // exact, like the division by 2
            } else {
                iy++;
                wy = wy * 0.5;
            }
        }
        plan->nlev = nlev;
        plan->ix = ix;
        plan->iy = iy;
        plan->xmin = xmin;
        plan->xmax = xmax;
        plan->ymin = ymin;
        plan->ymax = ymax;
        plan->W = W;
        plan->mismatch = (ix != aix || iy != aiy) ? 1 : 0;
        plan->fixup = 0;
        s_ix = ix;
        s_iters = 0;
        plan->ts[3] = global_ns();
    }
    __syncthreads();
    // the column counts and the y-range pairs are consumed: this rank's buffer goes back to the state k_init
    // leaves it in, ready for the next step that accumulates into it
    // (With the peer exchange this rank's slot lives in memory the other GPUs map; a kernel that writes there
    //  completes microseconds later -- measured: 6.7 instead of 1.5 us until the next kernel of the chain runs.
    //  The labelling kernel, far off the critical path, resets the slot then.)
    for (int i = tid; reset_own && i < yr_off + 2 * G; i += blockDim.x)
        own_col[i] = column_slot_reset_value(i, yr_off, ps.rank);

    // 3. the x levels: a group of `lanes` adjacent threads walks to strip i, all of them evaluating
    //    the same medians (the block has more threads than strips; the fewer different medians the
    //    lanes of a warp work on, the less a warp waits for the slowest of them)
    const int ix = s_ix;
    const int nstrips = leaves_below(P, ix);
    const bool by_level = nstrips <= LEVEL_NODES;
    const int lanes = by_level ? 1 : walk_lanes(nstrips, blockDim.x);
    int my_iters = 0;
    long long lmn = 0x7fffffffffffffffLL, lmx = -1;
    const RcbNode* fin = nullptr;
    if (by_level) { // the sets of a level side by side, one thread each
        RcbNode* nodes = reinterpret_cast<RcbNode*>(
            (reinterpret_cast<uintptr_t>(SMEM ? bitmap + hist_bitmap_words(NX) : smem_dyn) + 15) & ~(uintptr_t)15);
        const RcbSet root = { 0, NX, 0, P };
        int cnt;
        fin = SMEM && NX <= FAST_HIST_BINS
            ? rcb_levels<true>(H, root, ix, nodes, &my_iters, dbg ? plan->ts + TS_XLEV : nullptr, &cnt)
            : rcb_levels<false>(H, root, ix, nodes, &my_iters, dbg ? plan->ts + TS_XLEV : nullptr, &cnt);
    }
    for (int i = tid / lanes; i < nstrips; i += blockDim.x / lanes) {
        RcbSet r;
        if (by_level) {
            const RcbNode f = fin[i];
            r.lo = f.lo;
            r.hi = f.hi;
            r.plo = f.plo;
            r.n = f.n;
        } else {
            const RcbSet root = { 0, NX, 0, P };
            int it = 0;
            r = rcb_walk(H, root, ix, i, &it, dbg && tid == 0 ? plan->ts + TS_XLEV : nullptr);
            if (tid % lanes)
                continue;
            my_iters += it;
        }
        // 4. the strip table, in ascending part order
        st.x0[i] = r.lo;
        st.x1[i] = r.hi;
        st.p0[i] = r.plo;
        if (r.n == 1) { // a leaf already: uncut in y
            bx.x0[r.plo] = r.lo;
            bx.ex[r.plo] = r.hi - r.lo;
            bx.y0[r.plo] = 0;
            bx.ey[r.plo] = NY;
            const long long w = (long long)hcnt(pfx, r.lo, r.hi - 1);
            loads[r.plo] = w;
            lmn = w < lmn ? w : lmn;
            lmx = w > lmx ? w : lmx;
        }
    }
    reduce_load_extremes(lmn, lmx, loadmm);
    if (my_iters)
        atomicAdd(&s_iters, my_iters);
    if (tid == 0) {
        st.p0[nstrips] = P;
        *st.S = nstrips;
        *st.always = 0;
        plan->S = nstrips;
    }
    if (tid == 0)
        plan->ts[4] = global_ns();
    __syncthreads();
    if (tid == 0) {
        plan->iters = s_iters;
        plan->ts[5] = global_ns();
        plan->ts[10] = 0ull;
    }
    if (plan->mismatch) { // (written by thread 0 before the barrier above) the kernels after this one do nothing:
        __syncthreads(); //   the host reads the real plan from its pinned copy and runs the step again
        publish_plan(plan, host_plan);
    }
    if (next.word) { // strip table, leaf boxes and plan are written: the row-count kernel's blocks may go
        __syncthreads();
        if (tid == 0)
            chain_signal(next);
    }
}

// strip of every column (read by the labelling kernel), for decompositions WITHOUT y levels; with y levels K4
// paints the table itself.
// The strips tile [0, NX) in order: one warp paints the column range of one strip; a zero-width
// strip paints nothing, the strip that follows it owns the shared start column.
__global__ void __launch_bounds__(256) k_paint_strips(StripTable st, const Plan* __restrict__ plan,
    int* __restrict__ strip_of_col)
{
    pdl_trigger();
    pdl_wait(); // the x-cut kernel is complete
    if (plan->mismatch)
        return;
    const int S = *st.S;
    const int lane = lane_id();
    for (int i = blockIdx.x * 8 + (threadIdx.x >> 5); i < S; i += gridDim.x * 8) {
        const int x0 = st.x0[i], x1 = st.x1[i];
        for (int x = x0 + lane; x < x1; x += 32)
            strip_of_col[x] = i;
    }
}

// ------------------------------------------------------------------------------------------------
// K3: per-strip row counts from the bit map
// ------------------------------------------------------------------------------------------------
// One warp = 32 consecutive rows of one strip; lane = row.  A lane reads the few 16-byte groups its
// strip overlaps straight from global memory (neighbouring strips share the boundary group, which
// L1 / L2 serve) and the warp writes 32 consecutive counts (layout: row_count_index), rows local
// to this rank.  Leaf strips (one part, never cut in y) are skipped.
// Layout of one rank's strip row counts: [row block][strip][RB rows], RB = 1 << rb_shift rows per
// block of the kernel that wrote them.  A block of the row-count kernels therefore writes ONE
// contiguous chunk of Scap * RB counts -- which is what makes pushing it to the other ranks cheap:
// whole 16-byte stores, 512 contiguous bytes per warp (exchange step 2; the y-cut kernels read
// their own copy).  With rows contiguous per strip every block scattered 16-byte fragments over all
// strips and all peers, and the push took 4 x longer than the counting (DESIGN.md 5).
__host__ __device__ __forceinline__ size_t row_count_index(int s, int yl, int Scap, int rb_shift)
{
    return ((((size_t)(yl >> rb_shift) * Scap + s) << rb_shift) + (yl & ((1 << rb_shift) - 1)));
}
// store 16 bytes of counts at element index idx of this rank's block -- in the buffer of every rank
// when the counts are exchanged through peer memory
__device__ __forceinline__ void store_row_counts16(const PeerPush& out, size_t byte_off, const uint4& v)
{
    if (out.n <= 1)
        *reinterpret_cast<uint4*>(reinterpret_cast<char*>(out.dst[0]) + byte_off) = v;
    else
        for (int q = 0; q < out.n; q++)
            *reinterpret_cast<uint4*>(reinterpret_cast<char*>(out.dst[q]) + byte_off) = v;
}
template <typename CT>
__device__ __forceinline__ void store_row_count(const PeerPush& out, size_t idx, CT v)
{
    if (out.n <= 1)
        reinterpret_cast<CT*>(out.dst[0])[idx] = v;
    else
        for (int q = 0; q < out.n; q++)
            reinterpret_cast<CT*>(out.dst[q])[idx] = v;
}

// Exchange step 2: the LAST block of a row-count kernel to finish raises this rank's flag at every peer -- the
// y-cut kernels only wait.  (Raised by the y-cut kernel's first block, the flag left one kernel boundary and a
// launch later.)  Called by all threads of every block; `done` is a counter that is zero between steps.
__device__ __forceinline__ void rows_pushed(const PeerSync& ps, unsigned* done, unsigned blocks, int* s_last)
{
    if (!ps.enabled)
        return;
    __syncthreads(); // every thread's stores are issued ...
    if (threadIdx.x == 0) {
        __threadfence_system(); // ... and performed at the peers (cumulative over the barrier) before the block is counted
        *s_last = atomicAdd(done, 1u) == blocks - 1u;
    }
    __syncthreads();
    if (*s_last) {
        if ((int)threadIdx.x < ps.G)
            peer_signal(ps, 1, 0u);
        if (threadIdx.x == 0)
            *done = 0u;
    }
}

// The same with one flag per block: a block of the row-count kernel tells every rank "my chunk is there" itself (the
// release store orders the block's pushes -- all threads', through the barrier -- before the flag), and the y-cut
// kernel polls the G x blocks flags.  No block counter, no last block that has to notice it is the last and then pay a
// second fence: the flags of a rank arrive as its blocks finish.
__device__ __forceinline__ void row_flags_raise(const PeerSync& ps)
{
    __syncthreads(); // every thread's stores are issued
    if ((int)threadIdx.x < ps.G) {
        unsigned* dst = ps.rowflag[threadIdx.x] + (size_t)ps.rank * ps.flagcap + blockIdx.x;
#ifndef DDC_HOST_EMU
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(dst), "r"(ps.step) : "memory");
#else
        *dst = ps.step;
#endif
    }
}
// all threads of a block; false: a flag did not arrive in time
__device__ __forceinline__ bool row_flags_wait(const PeerSync& ps)
{
    bool ok = true;
    const int n = ps.G * ps.rowblocks;
    for (int i = threadIdx.x; i < n && ok; i += blockDim.x) {
        const int g = i / ps.rowblocks, b = i - g * ps.rowblocks;
        const unsigned* src = ps.rowflag[ps.rank] + (size_t)g * ps.flagcap + b;
#ifndef DDC_HOST_EMU
        const unsigned long long t0 = global_ns();
        for (;;) {
            unsigned v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
            if (v == ps.step)
                break;
            if (global_ns() - t0 > PEER_TIMEOUT_NS) {
                ok = false;
                break;
            }
        }
#else
        ok = *src == ps.step;
#endif
    }
    return !__syncthreads_or(!ok);
}

// The grid covers Rmax rows (the rows of the largest shard): rows beyond this rank's `rows` are
// written as empty, so that a short last shard needs no separate clearing pass.
template <typename CT /* uint16_t when NX < 65536, else unsigned */>
__global__ void __launch_bounds__(256) k_strip_rows(const uint8_t* __restrict__ bits, int NB, int rows,
    const int* __restrict__ st_x0, const int* __restrict__ st_x1, const int* __restrict__ st_p0,
    const Plan* __restrict__ plan, int Scap, PeerPush out, int Rmax, PeerSync ps, unsigned* __restrict__ done,
    unsigned long long* dbg, ChainWord prev /* published by the x-cut block */)
{
    __shared__ int s_last;
    pdl_trigger();
    if (threadIdx.x == 0)
        stamp_first(dbg, TS_RES + 2);
    chain_wait(prev);
    if (plan->mismatch) { // (the flag is raised all the same: the y-cut kernel may wait for it before it looks at the plan)
        rows_pushed(ps, done, gridDim.x * gridDim.y, &s_last);
        return;
    }
    if (threadIdx.x == 0)
        stamp_first(dbg, TS_ROWS);
    const int S = plan->S;
    const int s = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int row = blockIdx.x * 32 + lane_id();
    const bool act = s < S && s < Scap && st_p0[min(s, Scap - 1) + 1] - st_p0[min(s, Scap - 1)] > 1 && row < Rmax;
    const int x0 = act ? st_x0[s] : 0, x1 = act ? st_x1[s] : 0;
    unsigned cnt = 0;
    if (x1 > x0 && row < rows) {
        const int g0 = x0 >> 7, g1 = (x1 - 1) >> 7;
        const uint4* rp = reinterpret_cast<const uint4*>(bits + (size_t)row * NB);
        for (int g = g0; g <= g1; g++) {
            const uint4 w = __ldg(rp + g);
            const int a = x0 - g * 128, b = x1 - g * 128; // group-relative column range
            if (a <= 0 && b >= 128)
                cnt += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
            else
                cnt += __popc(w.x & word_range_mask(a, b)) + __popc(w.y & word_range_mask(a - 32, b - 32))
                    + __popc(w.z & word_range_mask(a - 64, b - 64)) + __popc(w.w & word_range_mask(a - 96, b - 96));
        }
    }
    if (act)
        store_row_count<CT>(out, row_count_index(s, row, Scap, 5), (CT)cnt); // 32 consecutive counts per warp
    rows_pushed(ps, done, gridDim.x * gridDim.y, &s_last);
    if (threadIdx.x == 0)
        stamp_last(dbg, TS_ROWS + 1);
}

// The same counts, coalesced: a block takes 32 consecutive rows and streams them ONCE -- a warp
// reads a row 512 contiguous bytes at a time (lane = one 16-byte group of 128 columns), turns the
// per-group popcounts into a running prefix with one warp scan, and the lanes whose group holds a
// strip boundary record the prefix AT the boundary in shared memory.  The row count of strip s is the
// difference of two neighbouring boundary prefixes; the block writes them out with lanes along the
// rows (32 consecutive counts per strip).  Used when the boundary table fits shared memory.
// K = rows per warp (a block takes 8 K consecutive rows): small shards take fewer rows per block so
// that the grid still fills the SMs; every lane always has 2 K independent 16-byte loads in flight
// (the chunk being counted and the next one).
// dynamic smem (ints): gfirst[NG + 1] | xb[S + 1] | pb[8 K][PS], PS = (S + 1) | 1
__host__ __device__ inline size_t strip_scan_smem_words(int NG, int S, int K)
{
    return (size_t)(NG + 1) + (size_t)(S + 1) + 8 * (size_t)K * (size_t)((S + 1) | 1);
}
// FULL (K == 1, rows of at most 8 chunks = 32768 columns): a lane requests ALL chunks of its row before
// the boundary table is built, so that a block pays the memory latency once.
template <typename CT, int K, bool FULL>
__global__ void __launch_bounds__(256) k_strip_rows_scan(const uint8_t* __restrict__ bits, int NB, int NX, int rows,
    const int* __restrict__ st_x0, const int* __restrict__ st_p0, const Plan* __restrict__ plan, int Scap,
    PeerPush out, int Rmax, PeerSync ps, unsigned* __restrict__ done, unsigned long long* dbg,
    ChainWord prev /* published by the x-cut block */)
{
    DDC_DYN_SHARED(int, sm_scan);
    __shared__ int s_last;
    pdl_trigger();
    if (threadIdx.x == 0)
        stamp_first(dbg, TS_RES + 2);
    chain_wait(prev);
    if (plan->mismatch) { // (the flag is raised all the same: the y-cut kernel may wait for it before it looks at the plan)
        if (ps.enabled && ps.rowflag[0])
            row_flags_raise(ps);
        else
            rows_pushed(ps, done, gridDim.x, &s_last);
        return;
    }
    if (threadIdx.x == 0)
        stamp_first(dbg, TS_ROWS);
    static_assert(!FULL || K == 1, "FULL holds one row per warp in registers");
    constexpr int RB = 8 * K; // rows per block
    constexpr int KP = (K + 1) / 2; // packed scan registers (two 16-bit running sums each)
    constexpr int NCH = FULL ? 8 : 1; // chunks held in registers
    const int S = min(plan->S, Scap);
    const int NG = NB >> 4;
    const int PS = (S + 1) | 1;
    int* gfirst = sm_scan; // first boundary at or after column g * 128
    int* xb = sm_scan + NG + 1; // boundaries: xb[b] = first column of strip b (bit 31: leaf strip), xb[S] = NX
    unsigned* pb = reinterpret_cast<unsigned*>(xb + S + 1); // [RB][PS] ocean cells of the row left of boundary b
    const int tid = threadIdx.x, lane = lane_id(), warp = tid >> 5;
    // a warp owns rows warp, warp + 8, ... of the block and walks them in lockstep; their first
    // chunks are requested before the boundary table is built
    const int r_base = blockIdx.x * RB;
    const uint4* rp[K];
    bool live[K];
    unsigned carry[K];
    uint4 nxt[K], all[NCH];
#pragma unroll
    for (int k = 0; k < K; k++) {
        const int row = r_base + warp + 8 * k;
        live[k] = row < rows;
        rp[k] = reinterpret_cast<const uint4*>(bits + (size_t)(live[k] ? row : 0) * NB);
        carry[k] = 0u;
        nxt[k] = make_uint4(0u, 0u, 0u, 0u);
        if (!FULL && live[k] && lane < NG)
            nxt[k] = __ldg(rp[k] + lane);
    }
    if (FULL) {
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            all[c] = make_uint4(0u, 0u, 0u, 0u);
            if (live[0] && c * 32 + lane < NG)
                all[c] = __ldg(rp[0] + c * 32 + lane);
        }
    }
    for (int b = tid; b <= S; b += blockDim.x)
        xb[b] = b < S ? (st_x0[b] | (st_p0[b + 1] - st_p0[b] <= 1 ? (int)0x80000000 : 0)) : NX;
    __syncthreads();
    for (int g = tid; g <= NG; g += blockDim.x) {
        const int x = g * 128;
        int lo = 0, hi = S + 1; // first b in [0, S] with xb[b] >= x (S + 1 if none)
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((xb[mid] & 0x7fffffff) >= x)
                hi = mid;
            else
                lo = mid + 1;
        }
        gfirst[g] = lo;
    }
    __syncthreads();
    // The per-group popcounts (<= 128, their running sums over a chunk <= 4096) are scanned two to a register.
    const int nchunks = (NG + 31) >> 5;
#pragma unroll(FULL ? NCH : 1)
    for (int ch = 0; ch < (FULL ? NCH : nchunks); ch++) {
        const int g0 = ch * 32;
        if (FULL && g0 >= NG)
            break;
        const int g = g0 + lane;
        const bool in = g < NG;
        unsigned long long wl[K], wh[K]; // columns 0-63 and 64-127 of my group, per row
#pragma unroll
        for (int k = 0; k < K; k++) {
            if (FULL)
                nxt[k] = all[ch % NCH];
            wl[k] = (unsigned long long)nxt[k].x | ((unsigned long long)nxt[k].y << 32);
            wh[k] = (unsigned long long)nxt[k].z | ((unsigned long long)nxt[k].w << 32);
            if (!FULL) {
                nxt[k] = make_uint4(0u, 0u, 0u, 0u);
                if (live[k] && g + 32 < NG)
                    nxt[k] = __ldg(rp[k] + g + 32);
            }
        }
        unsigned pc[K], ip[KP];
#pragma unroll
        for (int k = 0; k < K; k++)
            pc[k] = __popcll(wl[k]) + __popcll(wh[k]);
#pragma unroll
        for (int j = 0; j < KP; j++)
            ip[j] = pc[2 * j] | (2 * j + 1 < K ? pc[(2 * j + 1) % K] << 16 : 0u);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int j = 0; j < KP; j++) {
                const unsigned u = __shfl_up_sync(0xffffffffu, ip[j], o);
                if (lane >= o)
                    ip[j] += u;
            }
        }
        unsigned inc[K];
#pragma unroll
        for (int k = 0; k < K; k++)
            inc[k] = (k & 1) ? ip[k / 2] >> 16 : ip[k / 2] & 0xffffu;
        if (in) {
            const int b1 = gfirst[g + 1];
            for (int b = gfirst[g]; b < b1; b++) {
                const int kk = (xb[b] & 0x7fffffff) - g * 128; // 0 .. 127: columns of my group left of the boundary
                const unsigned long long ml = kk >= 64 ? ~0ull : ((1ull << kk) - 1ull);
                const unsigned long long mh = kk > 64 ? ((1ull << (kk - 64)) - 1ull) : 0ull;
#pragma unroll
                for (int k = 0; k < K; k++)
                    pb[(warp + 8 * k) * PS + b] = carry[k] + inc[k] - pc[k] + __popcll(wl[k] & ml) + __popcll(wh[k] & mh);
            }
        }
#pragma unroll
        for (int j = 0; j < KP; j++) {
            const unsigned e = __shfl_sync(0xffffffffu, ip[j], 31);
            carry[2 * j] += e & 0xffffu;
            if (2 * j + 1 < K)
                carry[(2 * j + 1) % K] += e >> 16;
        }
    }
#pragma unroll
    for (int k = 0; k < K; k++) // boundaries at the very end of the padded row
        for (int b = gfirst[NG] + lane; b <= S; b += 32)
            pb[(warp + 8 * k) * PS + b] = carry[k];
    __syncthreads();
    // this block's chunk of the [row block][strip][RB] layout, written 16 bytes at a time
    constexpr int V = 16 / (int)sizeof(CT); // counts per store
    static_assert(RB % V == 0, "a 16-byte store must not straddle two strips");
    const size_t chunk = (size_t)blockIdx.x * Scap * RB;
    for (int i = tid; i < S * RB / V; i += blockDim.x) {
        const int e = i * V, s = e / RB, rl = e % RB;
        if (xb[s] < 0)
            continue; // leaf strips are never cut in y
        unsigned c[V];
#pragma unroll
        for (int v = 0; v < V; v++)
            c[v] = pb[(rl + v) * PS + s + 1] - pb[(rl + v) * PS + s]; // rows beyond `rows` count 0
        uint4 o;
        if (sizeof(CT) == 2) {
            o.x = c[0] | (c[1 % V] << 16);
            o.y = c[2 % V] | (c[3 % V] << 16);
            o.z = c[4 % V] | (c[5 % V] << 16);
            o.w = c[6 % V] | (c[7 % V] << 16);
        } else
            o = make_uint4(c[0], c[1 % V], c[2 % V], c[3 % V]);
        store_row_counts16(out, (chunk + e) * sizeof(CT), o);
    }
    if (ps.enabled && ps.rowflag[0])
        row_flags_raise(ps);
    else
        rows_pushed(ps, done, gridDim.x, &s_last);
    if (tid == 0)
        stamp_last(dbg, TS_ROWS + 1);
}

// ------------------------------------------------------------------------------------------------
// The gate between the cut kernels and the neighbour kernels on the second stream
// ------------------------------------------------------------------------------------------------
// The neighbour tables are built beside the labelling kernel, on a second stream.  Forking that stream with an
// event recorded behind K4 puts a stream operation between K4 and the labelling kernel: no programmatic launch
// there, and the largest kernel of the step started 6-7 us after the boxes were done.  Instead the second stream
// holds, from the start of the step, a one-warp kernel that waits for a word in device memory; the last block
// of K4 to finish writes the step number there once every box is in place.  Blocks of K4 that leave early (plan
// mismatch, exchange time-out) count themselves too, so the gate always opens.
struct BoxGate {
    unsigned* word; // nullptr: no gate (the stream is forked with an event)
    unsigned* done; // block counter, zero between steps
    unsigned step;
};
// called by all threads of a block of K4 on every path out
__device__ __forceinline__ void boxes_ready(const BoxGate& g)
{
    if (!g.word)
        return;
    __syncthreads(); // the block's boxes are written ...
    if (threadIdx.x == 0) {
        __threadfence(); // ... and visible to the device before the block is counted
        if (atomicAdd(g.done, 1u) == gridDim.x - 1u) {
            *g.done = 0u;
            __threadfence();
#ifndef DDC_HOST_EMU
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(g.word), "r"(g.step) : "memory");
#else
            *g.word = g.step;
#endif
        }
    }
}
__global__ void __launch_bounds__(32) k_gate(const unsigned* word, unsigned step, Plan* plan)
{
    if (threadIdx.x != 0)
        return;
#ifndef DDC_HOST_EMU
    const unsigned long long t0 = global_ns();
    for (;;) {
        unsigned v;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(word) : "memory");
        if ((int)(v - step) >= 0)
            return;
        if (global_ns() - t0 > 4 * PEER_TIMEOUT_NS) { // the cut kernels never ran to their end
            atomicMax(&plan->mismatch, 3);
            return;
        }
        __nanosleep(100);
    }
#else
    (void)word;
    (void)step;
    (void)plan;
#endif
}

// ------------------------------------------------------------------------------------------------
// K4: y levels, one CTA per strip (grid-stride), boxes out
// ------------------------------------------------------------------------------------------------
// Row counts of rank g: the block [row block][Scap][RB] described above (row_count_index); the blocks
// of all ranks are either the G slots of this rank's exchange buffer or, after an NCCL all-gather,
// one buffer [G][rank_stride].  Global row y lives at rank y / Rmax, local row y % Rmax.
// dynamic smem of k_ycuts: (NY + 1) unsigned + the bit map when use_smem, otherwise pfx_g holds
// gridDim.x slices of NY + 1.
template <typename CT>
__device__ __forceinline__ const CT* row_segment(const PeerRows& pr, size_t rank_stride, int g)
{
    return pr.n == 1 ? reinterpret_cast<const CT*>(pr.row[0]) + (size_t)g * rank_stride
                     : reinterpret_cast<const CT*>(pr.row[g]);
}
struct RowLayout {
    size_t rank_stride;
    int Rmax, Scap, rb_shift;
};
// 4 consecutive row counts of strip s starting at global row i (a multiple of 4)
// (g, yl): the rank holding global row i and the row's index there -- the caller keeps them up to date from one load
// of a thread to the next instead of dividing by Rmax for each of them
template <typename CT>
__device__ __forceinline__ uint4 load_row_counts4(const PeerRows& pr, const RowLayout& rl, int s, int i, int NY, int g, int yl)
{
    const CT* src = row_segment<CT>(pr, rl.rank_stride, g) + row_count_index(s, yl, rl.Scap, rl.rb_shift);
    if (i + 4 <= NY && yl + 4 <= rl.Rmax && (yl & 3) == 0 && ((uintptr_t)src & (4 * sizeof(CT) - 1)) == 0) {
        // the chunk lies inside one rank's rows and inside one row block (RB is a multiple of 4)
        if (sizeof(CT) == 4)
            return __ldcg(reinterpret_cast<const uint4*>(src));
        const uint2 t = __ldcg(reinterpret_cast<const uint2*>(src));
        return make_uint4(t.x & 0xffffu, t.x >> 16, t.y & 0xffffu, t.y >> 16);
    }
    unsigned c[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int y = i + k;
        c[k] = 0u;
        if (y < NY) {
            const int gg = y / rl.Rmax;
            c[k] = (unsigned)__ldcg(row_segment<CT>(pr, rl.rank_stride, gg)
                + row_count_index(s, y - gg * rl.Rmax, rl.Scap, rl.rb_shift));
        }
    }
    return make_uint4(c[0], c[1], c[2], c[3]);
}

template <typename CT, bool SMEM>
__global__ void __launch_bounds__(1024) k_ycuts(PeerRows pr, PeerSync ps, RowLayout rl, int NY, StripTable st,
    unsigned* pfx_g, BoxTable bx, long long* loads, long long* loadmm, Plan* plan, int* __restrict__ strip_of_col,
    int dbg, BoxGate gate, int* __restrict__ part_at /* [S][nchunk]: the part of a strip owning row 32 j (PartAt) */,
    int nchunk, int early /* the flags of exchange step 2 stand in for the completion of the row-count kernel */)
{
    DDC_DYN_SHARED(unsigned, smem_dyn);
    __shared__ unsigned wsum[PFX_WS];
    pdl_trigger(); // the labelling kernel may become resident
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0)
        plan->ts[TS_RES + 3] = global_ns(); // (diagnostic only)
    // Flags instead of a kernel boundary: a kernel that has stored into peer-mapped memory completes late -- the grid
    // is only done once every posted NVLink store is acknowledged -- and its successor in the stream starts 6-8 us
    // after its last block instead of 1.5 us.  This kernel needs nothing from that completion that the flags do not
    // give: this rank's own flag is raised by the last block of ITS row-count kernel (release, cumulative over the
    // block counter), which ran after the x-cut kernel had completed, so acquiring all G flags orders every input of
    // this kernel before it.  (The blocks may then be resident, polling, while the row counts are still written.)
    if (ps.enabled && early) {
        bool ok = true;
        unsigned seen;
        if (ps.rowflag[0])
            ok = row_flags_wait(ps);
        else if (threadIdx.x < ps.G)
            ok = peer_wait(ps, 1, &seen);
        if (__syncthreads_or(!ok)) {
            pdl_wait();
            if (threadIdx.x == 0)
                plan->mismatch = 3;
            boxes_ready(gate);
            return;
        }
    } else
        pdl_wait(); // the strip row-count kernel (and with it everything before) is complete
    // everything the block needs to know about its first strip is requested at once: one trip to L2 instead of a chain
    // of four (mismatch -> S -> p0 -> x0) in front of the row counts
    const int mism = plan->mismatch, S = *st.S, ylevels = plan->iy;
    const int first_plo = st.p0[blockIdx.x], first_pend = st.p0[blockIdx.x + 1];
    const int first_x0 = st.x0[blockIdx.x], first_x1 = st.x1[blockIdx.x];
    if (mism) {
        boxes_ready(gate); // (the kernels behind the gate look at the mismatch themselves)
        return;
    }
    const unsigned long long t_start = global_ns();
    if (blockIdx.x == 0 && threadIdx.x == 0)
        plan->ts[6] = t_start;
    // the column -> strip table the labelling kernel reads: the block of a strip paints the strip's columns
    // (while the other ranks' row counts are still on their way); a zero-width strip paints nothing, the strip
    // that follows it owns the shared start column
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        const bool f = s == (int)blockIdx.x;
        const int xa = f ? first_x0 : st.x0[s], xb = f ? first_x1 : st.x1[s];
        for (int x = xa + (int)threadIdx.x; x < xb; x += (int)blockDim.x)
            strip_of_col[x] = s;
    }
    // exchange step 2: every rank's strip row counts are written (the last block of its row-count kernel said so)
    if (ps.enabled && !early) {
        bool ok = true;
        unsigned seen;
        if (ps.rowflag[0])
            ok = row_flags_wait(ps);
        else if (threadIdx.x < ps.G)
            ok = peer_wait(ps, 1, &seen);
        if (__syncthreads_or(!ok)) {
            if (threadIdx.x == 0)
                plan->mismatch = 3;
            boxes_ready(gate);
            return;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        plan->ts[7] = global_ns();
    unsigned* pfx = SMEM ? smem_dyn : pfx_g + (size_t)blockIdx.x * (((size_t)NY + 1 + 3) & ~(size_t)3);
    unsigned* bitmap = SMEM ? smem_dyn + (((size_t)NY + 1 + 3) & ~(size_t)3) : nullptr;
    const Hist H = make_hist(pfx, bitmap, NY);
    const int tid = threadIdx.x;
    int my_iters = 0;
    long long lmn = 0x7fffffffffffffffLL, lmx = -1;
    for (int s = blockIdx.x; s < S; s += gridDim.x) {
        const bool f = s == (int)blockIdx.x;
        const int plo = f ? first_plo : st.p0[s], n = (f ? first_pend : st.p0[s + 1]) - plo;
        if (n <= 1) { // K2 already wrote the box of a leaf strip: its one part owns every row
            for (int j = tid; j < nchunk; j += blockDim.x)
                part_at[(size_t)s * nchunk + j] = plo;
            continue;
        }
        __syncthreads(); // previous strip done with pfx
        block_prefix_tiles(
            [&](int base, uint4 (&v)[PFX_Q]) {
                int g = base / rl.Rmax, yl = base - g * rl.Rmax; // one division per thread and tile
#pragma unroll
                for (int q = 0; q < PFX_Q; q++) {
                    const int i = base + q * 4096;
                    v[q] = i < NY ? load_row_counts4<CT>(pr, rl, s, i, NY, g, yl) : make_uint4(0u, 0u, 0u, 0u);
                    if (i + 4096 < NY) { // the next sub-tile's rows: a few ranks further when the ranks hold few rows
                        yl += 4096;
                        while (yl >= rl.Rmax) {
                            yl -= rl.Rmax;
                            g++;
                        }
                    }
                }
            },
            NY, pfx, wsum, bitmap);
        if (blockIdx.x == 0 && tid == 0)
            plan->ts[8] = global_ns();
        // a group of `lanes` threads walks to the j-th part of the strip (parts come out y-sorted)
        const int sx0 = f ? first_x0 : st.x0[s], sx1 = f ? first_x1 : st.x1[s];
        const int nleaves = leaves_below(n, ylevels);
        const bool by_level = nleaves <= LEVEL_NODES;
        const int lanes = by_level ? 1 : walk_lanes(nleaves, blockDim.x);
        const RcbSet root = { 0, NY, plo, n };
        const RcbNode* fin = nullptr;
        if (by_level) {
            RcbNode* nodes = reinterpret_cast<RcbNode*>(
                (reinterpret_cast<uintptr_t>(SMEM ? bitmap + hist_bitmap_words(NY) : smem_dyn) + 15) & ~(uintptr_t)15);
            int cnt;
            fin = SMEM && NY <= FAST_HIST_BINS
                ? rcb_levels<true>(H, root, ylevels, nodes, &my_iters, dbg && blockIdx.x == 0 ? plan->ts + TS_YLEV : nullptr, &cnt)
                : rcb_levels<false>(H, root, ylevels, nodes, &my_iters, dbg && blockIdx.x == 0 ? plan->ts + TS_YLEV : nullptr, &cnt);
        }
        for (int j = tid / lanes; j < nleaves; j += blockDim.x / lanes) {
            RcbSet r;
            if (by_level) {
                const RcbNode f = fin[j];
                r.lo = f.lo;
                r.hi = f.hi;
                r.plo = f.plo;
                r.n = f.n;
            } else {
                int it = 0;
                r = rcb_walk(H, root, ylevels, j, &it, dbg && tid == 0 && blockIdx.x == 0 ? plan->ts + TS_YLEV : nullptr);
                if (tid % lanes)
                    continue;
                my_iters += it;
            }
            bx.x0[r.plo] = sx0;
            bx.ex[r.plo] = sx1 - sx0;
            bx.y0[r.plo] = r.lo;
            bx.ey[r.plo] = r.hi - r.lo;
            const long long w = (long long)hcnt(pfx, r.lo, r.hi - 1);
            loads[r.plo] = w;
            lmn = w < lmn ? w : lmn;
            lmx = w > lmx ? w : lmx;
        }
        // the row -> part table of the strip for the labelling kernel: the first part whose rows end after row 32 j
        // (the last part if none does), exactly what seat_cursor's search over the boxes would find
        if (!by_level)
            __syncthreads(); // the boxes of this strip, written above by this block, are read back below
        for (int j = tid; j < nchunk; j += blockDim.x) {
            const int y = j << 5;
            int lo = 0, hi = nleaves - 1;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const int yend = by_level ? fin[mid].hi : bx.y0[plo + mid] + bx.ey[plo + mid];
                if (y < yend)
                    hi = mid;
                else
                    lo = mid + 1;
            }
            part_at[(size_t)s * nchunk + j] = plo + lo;
        }
    }
    reduce_load_extremes(lmn, lmx, loadmm);
    if (my_iters)
        atomicAdd(&plan->iters, my_iters);
    __syncthreads();
    if (tid == 0) {
        const unsigned long long t_end = global_ns();
        if (blockIdx.x == 0)
            plan->ts[9] = t_end;
        atomicMax(&plan->ts[10], t_end - t_start);
    }
    boxes_ready(gate);
}

// ------------------------------------------------------------------------------------------------
// K6: owner labelling + Zoltan's `changes`
// ------------------------------------------------------------------------------------------------
// Same thread mapping as K1: one warp = one 128-column group, walking down the rows 8 at a time.
// The part of a cell is strip_of_col[x] -> strip, then the part of that strip owning row y.  Parts
// of a strip are y-sorted and ~hundreds of rows tall, so a thread keeps a cursor (part, first row
// after it) for the strip of its first and of its last column (two cursors cover every thread that
// spans at most two strips; they coincide for the ~97 % of threads inside one strip).  While all 8
// rows of a batch stay inside both cursor parts -- the common case -- nothing is looked up at all;
// when a part boundary crosses the batch the cursors step forward row by row.
struct LabelCursor {
    int part; // part owning the current row
    int yend; // first row that no longer belongs to it
    int last; // last part of the strip
};
// first part of strip s whose rows end after y (binary search over the y-sorted parts)
__device__ __forceinline__ LabelCursor seat_cursor(const int* __restrict__ st_p0, const int* __restrict__ box_y0,
    const int* __restrict__ box_ey, int s, int y)
{
    LabelCursor c;
    int lo = st_p0[s];
    c.last = st_p0[s + 1] - 1;
    int hi = c.last;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (y < box_y0[mid] + box_ey[mid])
            hi = mid;
        else
            lo = mid + 1;
    }
    c.part = lo;
    c.yend = box_y0[lo] + box_ey[lo];
    return c;
}
__device__ __forceinline__ void advance_cursor(LabelCursor& c, const int* __restrict__ box_y0,
    const int* __restrict__ box_ey, int y)
{
    while (y >= c.yend && c.part < c.last) { // zero-height parts are stepped over
        c.part++;
        c.yend = box_y0[c.part] + box_ey[c.part];
    }
}

template <bool VEC>
__device__ __forceinline__ void store_pid_row(int32_t* __restrict__ q, int x, int NX, const int4& out)
{
    if (VEC) {
        if (x < NX)
            __stcs(reinterpret_cast<int4*>(q), out);
    } else {
        if (x < NX)
            q[0] = out.x;
        if (x + 1 < NX)
            q[1] = out.y;
        if (x + 2 < NX)
            q[2] = out.z;
        if (x + 3 < NX)
            q[3] = out.w;
    }
}

// The part of strip s that owns row y, for the start of a block's rows.  K4 leaves a table: part_at[s * nchunk + j] = the
// part of strip s owning row 32 j (PartAt below); from there the cursor steps forward (a block starts at most 31 rows
// further).  Without the table (no y levels) a binary search over the y-sorted parts.
struct PartAt {
    const int* table; // nullptr: search
    int nchunk; // = ceil(NY / 32)
};
__device__ __forceinline__ LabelCursor seat_cursor_at(const PartAt& pa, const int* __restrict__ st_p0,
    const int* __restrict__ box_y0, const int* __restrict__ box_ey, int s, int y)
{
    if (!pa.table)
        return seat_cursor(st_p0, box_y0, box_ey, s, y);
    LabelCursor c;
    c.part = pa.table[(size_t)s * pa.nchunk + (y >> 5)];
    c.last = st_p0[s + 1] - 1;
    c.yend = box_y0[c.part] + box_ey[c.part];
    advance_cursor(c, box_y0, box_ey, y);
    return c;
}

// the rows [r0, r1) of one thread's 4 columns; returns whether a moved cell was found
template <bool VEC, bool WRITE>
__device__ __forceinline__ bool label_rows(const uint8_t* __restrict__ bits, int NX, int y_begin, int NB, int g, int r0,
    int r1, const int* __restrict__ strip_of_col, const int* __restrict__ st_p0, const int* __restrict__ box_y0,
    const int* __restrict__ box_ey, const NaiveParams& nv, int32_t* __restrict__ pid, DevScalars* __restrict__ sc,
    const PartAt& pa)
{
    const int lane = lane_id();
    const int x = g * 128 + lane * 4;
    bool found = false;
    // everything that does not depend on anything else is requested first, together: the strips of my columns, the
    // first batch of bit-map bytes, the `changes` flag (a block lives for a few microseconds; a chain of dependent
    // trips to L2 at its start was a third of that)
    int sc4[4], nbx[4];
#pragma unroll
    for (int c = 0; c < 4; c++)
        sc4[c] = strip_of_col[min(x + c, NX - 1)];
    const uint8_t* brow = bits + (size_t)g * 16 + (lane >> 1);
    const int sh = (lane & 1) * 4;
    unsigned nb[8];
#pragma unroll
    for (int k = 0; k < 8; k++)
        nb[k] = r0 + k < r1 ? (unsigned)__ldg(brow + (size_t)(r0 + k) * NB) : 0u;
    // `changes` only ever goes 0 -> 1: stop looking as soon as anyone has found a moved cell
    bool check = *reinterpret_cast<volatile int*>(&sc->changes) == 0;
#pragma unroll
    for (int c = 0; c < 4; c++)
        nbx[c] = min(min(x + c, NX - 1) / nv.lx, nv.np0 - 1) * nv.np1;
    // columns 1, 2 belong to the strip of column 0 or of column 3 unless the thread spans > 2 strips
    const bool two = (sc4[1] == sc4[0] || sc4[1] == sc4[3]) && (sc4[2] == sc4[0] || sc4[2] == sc4[3]);
    const bool b1 = sc4[1] != sc4[0], b2 = sc4[2] != sc4[0], b3 = sc4[3] != sc4[0];
    LabelCursor A = seat_cursor_at(pa, st_p0, box_y0, box_ey, sc4[0], y_begin + r0);
    LabelCursor B = b3 ? seat_cursor_at(pa, st_p0, box_y0, box_ey, sc4[3], y_begin + r0) : A;
    int by = min((y_begin + r0) / nv.ly, nv.np1 - 1);
    int by_next = (by == nv.np1 - 1) ? 0x7fffffff : (by + 1) * nv.ly;
    for (int r = r0; r < r1; r += 8) {
        const int y = y_begin + r;
        const int nrow = min(8, r1 - r);
        unsigned packed = 0; // nibble k = ocean flags of my 4 columns in row r + k
#pragma unroll
        for (int k = 0; k < 8; k++)
            packed |= ((nb[k] >> sh) & 15u) << (4 * k);
        if (r + 8 < r1) {
#pragma unroll
            for (int k = 0; k < 8; k++)
                nb[k] = r + 8 + k < r1 ? (unsigned)__ldg(brow + (size_t)(r + 8 + k) * NB) : 0u;
        }
        const int ylast = y + nrow - 1;
        if (two && ylast < A.yend && ylast < B.yend) {
            // fast path: one part per column for the whole batch
            const int p0 = A.part, p1 = b1 ? B.part : A.part, p2 = b2 ? B.part : A.part, p3 = b3 ? B.part : A.part;
            if (check) {
                bool changed;
                if (ylast < by_next) {
                    const unsigned dm = (unsigned)(p0 != nbx[0] + by) | ((unsigned)(p1 != nbx[1] + by) << 1)
                        | ((unsigned)(p2 != nbx[2] + by) << 2) | ((unsigned)(p3 != nbx[3] + by) << 3);
                    changed = (packed & (dm * 0x11111111u)) != 0;
                } else { // the naive block row changes inside the batch: row by row
                    changed = false;
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        if (k < nrow) {
                            if (y + k >= by_next) {
                                by++;
                                by_next = (by == nv.np1 - 1) ? 0x7fffffff : by_next + nv.ly;
                            }
                            const unsigned nib = packed >> (4 * k);
                            changed |= ((nib & 1u) && p0 != nbx[0] + by) | ((nib & 2u) && p1 != nbx[1] + by)
                                | ((nib & 4u) && p2 != nbx[2] + by) | ((nib & 8u) && p3 != nbx[3] + by);
                        }
                    }
                }
                if (__any_sync(__activemask(), changed)) {
                    if (changed) {
                        atomicOr(&sc->changes, 1);
                        found = true;
                    }
                    check = false;
                }
            }
            if (WRITE) {
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if (k < nrow) {
                        const unsigned nib = packed >> (4 * k);
                        store_pid_row<VEC>(pid + (size_t)(r + k) * NX + x, x, NX,
                            make_int4((nib & 1u) ? p0 : -1, (nib & 2u) ? p1 : -1, (nib & 4u) ? p2 : -1,
                                (nib & 8u) ? p3 : -1));
                    }
                }
            }
        } else {
            // slow path: a part boundary crosses the batch (or the thread spans > 2 strips)
            bool changed = false;
            for (int k = 0; k < nrow; k++) {
                const int yy = y + k;
                advance_cursor(A, box_y0, box_ey, yy);
                advance_cursor(B, box_y0, box_ey, yy);
                int p0 = A.part, p1 = b1 ? B.part : A.part, p2 = b2 ? B.part : A.part, p3 = b3 ? B.part : A.part;
                if (!two) { // > 2 strips under one thread (strips narrower than 3 columns)
                    p1 = seat_cursor(st_p0, box_y0, box_ey, sc4[1], yy).part;
                    p2 = seat_cursor(st_p0, box_y0, box_ey, sc4[2], yy).part;
                }
                const unsigned nib = packed >> (4 * k);
                if (check) {
                    if (yy >= by_next) {
                        by++;
                        by_next = (by == nv.np1 - 1) ? 0x7fffffff : by_next + nv.ly;
                    }
                    changed |= ((nib & 1u) && p0 != nbx[0] + by) | ((nib & 2u) && p1 != nbx[1] + by)
                        | ((nib & 4u) && p2 != nbx[2] + by) | ((nib & 8u) && p3 != nbx[3] + by);
                }
                if (WRITE)
                    store_pid_row<VEC>(pid + (size_t)(r + k) * NX + x, x, NX,
                        make_int4((nib & 1u) ? p0 : -1, (nib & 2u) ? p1 : -1, (nib & 4u) ? p2 : -1,
                            (nib & 8u) ? p3 : -1));
            }
            if (check && changed) {
                atomicOr(&sc->changes, 1);
                found = true;
                check = false;
            }
        }
        if (check && (r & 63) == 0)
            check = *reinterpret_cast<volatile int*>(&sc->changes) == 0;
    }
    return found;
}

// The end of a step, folded into the labelling kernel (no separate launch behind the largest kernel of the
// step): every block adds itself -- and, in the upper half of the same 64-bit atomic, whether it found a moved
// cell -- to a counter; the block that completes the count knows this rank's `changes` without any fence,
// tells the other ranks (exchange step 3: the verdict rides in the low bit of the flag), and writes the plan
// into the host's pinned copy.  `changes` is an OR over the ranks, so a rank that found a moved cell knows the
// global answer already and does not wait for anybody.  Only when NOTHING moved here (all land, or the RCB
// reproduces the naive blocks) the answer is left open: the host then runs k_finalize (Plan::fixup).
struct LabelEnd {
    int fuse; // 0: k_finalize follows as a kernel of its own
    int P;
    PeerSync ps;
    unsigned long long* counter; // zero between steps
    Plan* host_plan;
    unsigned long long* dbg;
    PartAt part_at; // the row -> part table K4 left (table == nullptr: none)
    unsigned* reset_col; // != nullptr: this rank's column-count slot, consumed by k_sum_cols: zeroed here for the next step
    int reset_n, yr_off;
    ChainWord prev; // the gate word the last block of K4 writes (boxes_ready), polled instead of the kernel boundary
    ChainWord nbr; // published by the neighbour kernels on the second stream: the step ends when they have, too
};

template <bool VEC, bool WRITE>
__global__ void __launch_bounds__(256, 5) k_label(const uint8_t* __restrict__ bits, int NX, int rows,
    int y_begin, int NB, int rows_per_cta, const int* __restrict__ strip_of_col,
    const int* __restrict__ st_p0, const int* __restrict__ box_y0, const int* __restrict__ box_ey,
    NaiveParams nv, int32_t* __restrict__ pid, DevScalars* __restrict__ sc, Plan* __restrict__ plan, LabelEnd fin)
{
    __shared__ int s_changed, s_last;
    pdl_trigger(); // the next step's mask scan may become resident behind the last blocks of this grid
    if (threadIdx.x == 0)
        stamp_first(fin.dbg, TS_RES + 4);
    chain_wait(fin.prev);
    if (plan->mismatch) { // the host runs the step again with the real plan (or reports the time-out)
        if (fin.fuse && blockIdx.x == 0 && blockIdx.y == 0)
            publish_plan(plan, fin.host_plan);
        return;
    }
    if (threadIdx.x == 0)
        stamp_first(fin.dbg, TS_LABEL);
    if (fin.reset_col) { // (the first blocks of the grid take 256 entries each)
        const long long stride = (long long)gridDim.x * gridDim.y * blockDim.x;
        for (long long i = ((long long)blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x; i < fin.reset_n; i += stride)
            fin.reset_col[i] = column_slot_reset_value((int)i, fin.yr_off, fin.ps.rank);
    }
    const int g = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int r0 = blockIdx.y * rows_per_cta;
    const int r1 = min(rows, r0 + rows_per_cta);
    bool found = false;
    if (g * 128 < NX && r0 < r1)
        found = label_rows<VEC, WRITE>(bits, NX, y_begin, NB, g, r0, r1, strip_of_col, st_p0, box_y0, box_ey, nv, pid, sc,
            fin.part_at);
    if (!fin.fuse)
        return;
    const int any = __syncthreads_or(found ? 1 : 0); // (the one barrier of a block: its warps are done)
    if (threadIdx.x == 0) {
        stamp_last(fin.dbg, TS_LABEL + 1);
        const unsigned long long old = atomicAdd(fin.counter, 1ull | (any ? (1ull << 32) : 0ull));
        const unsigned blocks = gridDim.x * gridDim.y;
        s_last = (unsigned)(old & 0xffffffffull) == blocks - 1u;
        s_changed = (any || (old >> 32) != 0ull) ? 1 : 0; // only meaningful in the last block
    }
    __syncthreads();
    if (!s_last)
        return;
    const int changes = s_changed;
    if (fin.ps.enabled && (int)threadIdx.x < fin.ps.G)
        peer_signal_relaxed(fin.ps, 2, changes ? 1u : 0u);
    if (threadIdx.x == 0) {
        *fin.counter = 0ull;
        sc->changes = changes;
        sc->changes_all = changes;
        plan->fixup = (changes || fin.P <= 1) ? 0 : (fin.ps.enabled ? 2 : 1);
        // The neighbour tables are built beside this kernel on a second stream.  Instead of joining the streams with
        // an event (a stream operation between this kernel and the next step's scan: no programmatic launch there,
        // and ~2 us more per step), this block waits for the word their last block publishes: when this grid has
        // completed, the whole step has.
        if (fin.nbr.word) {
#ifndef DDC_HOST_EMU
            const unsigned long long t0 = global_ns();
            for (;;) {
                unsigned v;
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(fin.nbr.word) : "memory");
                if (v == fin.nbr.step)
                    break;
                if (global_ns() - t0 > PEER_TIMEOUT_NS) {
                    plan->mismatch = 3;
                    break;
                }
            }
#else
            if (*fin.nbr.word != fin.nbr.step)
                plan->mismatch = 3;
#endif
        }
        stamp_last(fin.dbg, TS_LABEL + 2);
    }
    __syncthreads();
    publish_plan(plan, fin.host_plan);
}

// ------------------------------------------------------------------------------------------------
// K7: neighbours and halos (interval intersection), count pass and fill pass
// ------------------------------------------------------------------------------------------------
// Two search strategies, same literal edge tests:
//  * structured (the normal case): the boxes are vertical strips, each holding y-sorted parts that
//    tile [0, NY).  One THREAD per (list, part): walk the strips in ascending order, keep those
//    whose x range satisfies the edge's x condition (exact at strip level, every part of a strip
//    has the strip's x range), binary-search the first part whose y range can match and scan the
//    short run that does.  ids come out ascending by construction.
//  * unstructured (`always`: caller-supplied boxes, degenerate naive blocks): one WARP per part,
//    all pairs, ballot compaction keeps ids ascending.
// list l = periodic * 4 + edge; counts/offsets [8][P]; ids/halos/starts [8][cap].
template <bool FILL>
__device__ __forceinline__ void neighbours_all_pairs(const BoxTable& bx, int P, int NX, int NY, int px, int py,
    int me, int* __restrict__ counts, const int* __restrict__ offsets, int cap, int* __restrict__ ids,
    int* __restrict__ halos, int* __restrict__ starts, DevScalars* sc)
{
    const int lane = lane_id();
    Dom d1;
    d1.x1 = bx.x0[me];
    d1.y1 = bx.y0[me];
    d1.x2 = d1.x1 + bx.ex[me];
    d1.y2 = d1.y1 + bx.ey[me];
    int cnt[8];
    int base[8];
#pragma unroll
    for (int l = 0; l < 8; l++) {
        cnt[l] = 0;
        base[l] = FILL ? offsets[l * (P + 1) + me] : 0;
    }
    unsigned long long cut = 0;
    for (int qb = 0; qb < P; qb += 32) {
        const int q = qb + lane;
        const bool valid = q < P;
        Dom d2 = { 0, 0, 0, 0 };
        if (valid) {
            d2.x1 = bx.x0[q];
            d2.y1 = bx.y0[q];
            d2.x2 = d2.x1 + bx.ex[q];
            d2.y2 = d2.y1 + bx.ey[q];
        }
#pragma unroll
        for (int l = 0; l < 8; l++) {
            const int per = l >> 2, edge = l & 3;
            const bool lr = edge < 2;
            bool pass = valid;
            if (per) // filter of get_neighbour_info_periodic (Partitioner.cpp:116)
                pass = pass && ((lr && px) || (!lr && py));
            else // a subdomain is not its own interior neighbour (Partitioner.cpp:408)
                pass = pass && q != me;
            int halo = 0;
            if (pass) {
                pass = is_neighbour(d1, d2, edge, per && px, per && py, NX, NY);
                if (pass) {
                    halo = domain_overlap(d1, d2, edge);
                    pass = halo > 0;
                }
            }
            const unsigned b = __ballot_sync(0xffffffffu, pass);
            if (FILL && pass) {
                const int pos = base[l] + cnt[l] + __popc(b & ((1u << lane) - 1u));
                ids[(size_t)l * cap + pos] = q;
                halos[(size_t)l * cap + pos] = halo;
                starts[(size_t)l * cap + pos] = halo_start(d1, d2, edge);
                if (!per)
                    cut += (unsigned long long)halo;
            }
            cnt[l] += __popc(b);
        }
    }
    if (!FILL) {
        if (lane == 0) {
#pragma unroll
            for (int l = 0; l < 8; l++)
                counts[l * P + me] = cnt[l];
        }
    } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
            cut += __shfl_xor_sync(0xffffffffu, cut, o);
        if (lane == 0 && cut)
            atomicAdd(&sc->edge_cut, cut);
    }
}

// launched with enough threads for one warp per part (P * 32); the structured mode only uses the
// first 8 * P of them (thread = list * P + part, so a warp works on 32 consecutive parts of one list)
template <bool FILL>
__global__ void __launch_bounds__(256) k_neighbours(BoxTable bx, int P, int NX, int NY, int px, int py,
    StripTable st, int* __restrict__ counts, const int* __restrict__ offsets,
    const int* __restrict__ totals, int cap, int* __restrict__ ids, int* __restrict__ halos,
    int* __restrict__ starts, DevScalars* sc, const Plan* __restrict__ plan,
    ChainWord tables_done /* FILL: published by the last block on every path (the labelling kernel's last block waits
                             for it: no join of the two streams between two steps) */,
    unsigned* __restrict__ done_ctr)
{
    // (the scan of the counts is launched programmatically behind the count kernel; the count and the fill kernel
    //  themselves follow their predecessors with plain launches: P / 8 blocks waiting behind the gate kernel would hold
    //  SMs that the y-cut kernel, which opens the gate, still needs, and waiting behind the scan they take them from
    //  the labelling kernel)
    pdl_trigger();
    pdl_wait();
    bool run = !(plan && plan->mismatch);
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (run && FILL) {
        bool over = false;
#pragma unroll
        for (int l = 0; l < 8; l++)
            over |= totals[l] > cap;
        if (over) {
            if (t == 0)
                sc->overflow = 1;
            run = false;
        }
    }
    if (run) {
        if (*st.always) {
            const int me = (int)(t >> 5);
            if (me < P)
                neighbours_all_pairs<FILL>(bx, P, NX, NY, px, py, me, counts, offsets, cap, ids, halos, starts, sc);
        } else {
            // thread = list * Ppad + part with Ppad a multiple of 32: a warp works on 32 consecutive
            // parts of ONE list (uniform control flow, coalesced box loads)
            const int Ppad = (P + 31) & ~31;
            if (t < 8LL * Ppad)
                neighbours_structured<FILL>(bx, P, NX, NY, px, py, st, (int)(t / Ppad), (int)(t % Ppad), counts,
                    offsets, cap, ids, halos, starts, sc);
        }
    }
    if (FILL && tables_done.word) {
        __syncthreads(); // the block's entries are written ...
        if (threadIdx.x == 0) {
            __threadfence(); // ... and visible to the device before the block is counted
            if (atomicAdd(done_ctr, 1u) == gridDim.x - 1u) {
                *done_ctr = 0u;
                chain_signal(tables_done);
            }
        }
    }
}

// exclusive scan of each of the 8 count lists (one CTA per list)
__global__ void __launch_bounds__(1024) k_scan_counts(const int* __restrict__ counts, int P,
    int* __restrict__ offsets, int* __restrict__ totals, const Plan* __restrict__ plan)
{
    __shared__ unsigned long long wsum64[33];
    pdl_trigger();
    pdl_wait();
    if (plan && plan->mismatch)
        return;
    const int l = blockIdx.x;
    const int* c = counts + (size_t)l * P;
    // writes P + 1 values; offsets has one spare slot after every list
    const unsigned long long total = block_prefix<false>([&](int i) { return (unsigned)c[i]; }, P,
        reinterpret_cast<unsigned*>(offsets) + (size_t)l * (P + 1), 0, wsum64);
    if (threadIdx.x == 0)
        totals[l] = (int)total;
}

// ------------------------------------------------------------------------------------------------
// K5: the end of a step as a kernel of its own, ONE block
// ------------------------------------------------------------------------------------------------
// Normally the labelling kernel's last block ends the step (LabelEnd above).  This kernel runs
//  (a) in the stream, when there is no labelling kernel (a rank without rows; one part and no pid wanted) or
//      when the exchange goes through NCCL, and
//  (b) from the host's validate(), when the labelling kernel left the verdict open (Plan::fixup != 0).
//  * exchange step 3: `changes` of every rank (it rides in the low bit of the flag);
//  * `changes == 0`  =>  the naive blocks are reported (ZoltanPartitioner.cpp:182-187).  The neighbour
//    tables were built speculatively from the RCB boxes, beside the labelling kernel that was still
//    looking for `changes`; in this rare case they are built again here from the naive blocks
//    (count, scan and fill in this one block);
//  * the plan (levels, mismatch flag, iteration count) is written straight into the host's pinned
//    copy, so that the step ends without a separate device -> host copy.
struct NbrTables {
    int* counts;
    int* offsets;
    int* totals;
    int cap;
    int* ids;
    int* halos;
    int* starts;
};
__global__ void __launch_bounds__(1024) k_finalize(PeerSync ps, int P, int NX, int NY, int px, int py, NaiveParams nv,
    DevScalars* __restrict__ sc, Plan* __restrict__ plan, StripTable st, BoxTable bx,
    int want_nbr, NbrTables nb, Plan* __restrict__ host_plan)
{
    __shared__ unsigned long long wsum64[33];
    __shared__ int s_over;
    const int tid = threadIdx.x;
    if (plan->mismatch) {
        publish_plan(plan, host_plan);
        return;
    }
    int changes = sc->changes;
    if (ps.enabled) {
        bool ok = true;
        unsigned seen = 0u;
        if (tid < ps.G)
            ok = peer_barrier(ps, 2, changes ? 1u : 0u, true, &seen);
        if (__syncthreads_or(!ok)) {
            if (tid == 0)
                plan->mismatch = 3;
            __syncthreads();
            publish_plan(plan, host_plan);
            return;
        }
        changes = __syncthreads_or(tid < ps.G && (seen & 1u));
    }
    if (tid == 0) {
        sc->changes_all = changes;
        plan->fixup = 0; // whatever is left to do is done below
    }
    __syncthreads();
    publish_plan(plan, host_plan); // K4 is done: the iteration count is final
    if (P == 1 || changes != 0)
        return;
    // ---- nothing moved: the naive blocks (Grid.cpp:150-166) replace the RCB boxes ----
    for (int p = tid; p < P; p += blockDim.x) {
        const int bxi = p / nv.np1, byi = p % nv.np1; // Grid.cpp:158-159
        int ex = nv.lx, ey = nv.ly;
        if (bxi == nv.np0 - 1)
            ex = NX - bxi * nv.lx;
        if (byi == nv.np1 - 1)
            ey = NY - byi * nv.ly;
        bx.x0[p] = bxi * nv.lx;
        bx.y0[p] = byi * nv.ly;
        bx.ex[p] = ex;
        bx.ey[p] = ey;
        if (byi == 0) {
            st.x0[bxi] = bxi * nv.lx;
            st.x1[bxi] = bxi * nv.lx + ex;
            st.p0[bxi] = p;
        }
        if (p == 0) {
            st.p0[nv.np0] = P;
            *st.S = nv.np0;
            // ceil() over-covering makes trailing blocks start beyond the extent (non-positive
            // extents, y no longer sorted): let the neighbour search test all pairs then
            *st.always = ((nv.np0 - 1) * nv.lx >= NX || (nv.np1 - 1) * nv.ly >= NY) ? 1 : 0;
            sc->edge_cut = 0ull;
            sc->overflow = 0;
            s_over = 0;
        }
    }
    __syncthreads(); // the boxes and the strip table are in place (same block: visible after the barrier)
    if (!want_nbr)
        return;
    const bool all = *st.always != 0;
    const int Ppad = (P + 31) & ~31;
    if (all) {
        for (int me = tid >> 5; me < P; me += blockDim.x >> 5)
            neighbours_all_pairs<false>(bx, P, NX, NY, px, py, me, nb.counts, nb.offsets, nb.cap, nb.ids, nb.halos,
                nb.starts, sc);
    } else {
        for (int t = tid; t < 8 * Ppad; t += blockDim.x)
            neighbours_structured<false>(bx, P, NX, NY, px, py, st, t / Ppad, t % Ppad, nb.counts, nb.offsets, nb.cap,
                nb.ids, nb.halos, nb.starts, sc);
    }
    __syncthreads();
    for (int l = 0; l < 8; l++) {
        const int* c = nb.counts + (size_t)l * P;
        const unsigned long long total = block_prefix<false>([&](int i) { return (unsigned)c[i]; }, P,
            reinterpret_cast<unsigned*>(nb.offsets) + (size_t)l * (P + 1), 0, wsum64);
        if (tid == 0) {
            nb.totals[l] = (int)total;
            if ((long long)total > nb.cap)
                s_over = 1;
        }
    }
    __syncthreads();
    if (s_over) {
        if (tid == 0)
            sc->overflow = 1;
        return;
    }
    if (all) {
        for (int me = tid >> 5; me < P; me += blockDim.x >> 5)
            neighbours_all_pairs<true>(bx, P, NX, NY, px, py, me, nb.counts, nb.offsets, nb.cap, nb.ids, nb.halos,
                nb.starts, sc);
    } else {
        for (int t = tid; t < 8 * Ppad; t += blockDim.x)
            neighbours_structured<true>(bx, P, NX, NY, px, py, st, t / Ppad, t % Ppad, nb.counts, nb.offsets, nb.cap,
                nb.ids, nb.halos, nb.starts, sc);
    }
}

// resets the per-call accumulators: column counts, the per-rank y-range slots that follow them
// (this rank's slot to "no dot yet", the others to 0 so that the SUM all-reduce of the whole
// buffer delivers every rank's pair), scalars, load min / max
__global__ void __launch_bounds__(256) k_init(unsigned* __restrict__ colcount, int n, int yr_off, int rank,
    DevScalars* __restrict__ sc, long long* __restrict__ loadmm, unsigned* __restrict__ done, int ndone)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ndone)
        done[i] = 0u;
    if (i < n) {
        unsigned v = 0u;
        if (i == yr_off + 2 * rank)
            v = 0x80000000u; // -(first ocean row) = INT_MIN
        if (i == yr_off + 2 * rank + 1)
            v = 0xffffffffu; // last ocean row = -1
        colcount[i] = v;
    }
    if (i == 0) {
        sc->changes = 0;
        sc->changes_all = 0;
        sc->overflow = 0;
        sc->edge_cut = 0ull;
        loadmm[0] = 0x7fffffffffffffffLL;
        loadmm[1] = -1;
    }
}

// ------------------------------------------------------------------------------------------------
// Halo exchange: a consumer of the neighbour tables
// ------------------------------------------------------------------------------------------------
// The reference's only in-tree consumer of get_neighbour_info is examples/zoltan_comm.cpp:84-246: every rank
// holds its box as a (ext + 2)^2-framed array, builds one MPI subarray type per neighbour from the halo sizes and
// exchanges the frames with MPI_Neighbor_alltoallw.  Here all parts of a decomposition live in one device buffer
// -- tile p is a row-major (ext_y + 2) x (ext_x + 2) array with a ghost frame of one cell, at tiles[off[p]] -- and one
// warp per (edge list, part) walks the part's CSR entries: neighbour id, halo size and halo START (the index of
// the first shared cell in the neighbour's flattened box, Partitioner.cpp:55-80) locate the source cells, the
// overlap of the two boxes the ghost cells.  Corners are not exchanged (a corner-touching box is no neighbour,
// DomainUtils.cpp:15-35).  lists: bit l set = use list l (l = periodic * 4 + edge).
template <typename T>
__global__ void __launch_bounds__(256) k_halo_exchange(BoxTable bx, int P, const int* __restrict__ counts,
    const int* __restrict__ offsets, int cap, const int* __restrict__ ids, const int* __restrict__ halos,
    const int* __restrict__ starts, const long long* __restrict__ off, T* __restrict__ tiles, unsigned lists)
{
    const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = lane_id();
    if (w >= 8LL * P)
        return;
    const int l = (int)(w / P), p = (int)(w % P);
    if (!((lists >> l) & 1u))
        return;
    const int edge = l & 3;
    const int px0 = bx.x0[p], py0 = bx.y0[p], pex = bx.ex[p], pey = bx.ey[p];
    T* mine = tiles + off[p];
    const int n = counts[l * P + p], first = offsets[l * (P + 1) + p];
    for (int k = 0; k < n; k++) {
        const size_t e = (size_t)l * cap + first + k;
        const int q = ids[e], h = halos[e], st = starts[e];
        const int qw = bx.ex[q];
        const T* theirs = tiles + off[q];
        const bool lr = edge < 2; // left / right: the shared cells run along y
        const int along = lr ? max(py0, bx.y0[q]) - py0 : max(px0, bx.x0[q]) - px0; // first shared cell along my edge
        for (int i = lane; i < h; i += 32) {
            const int s = st + (lr ? i * qw : i); // the neighbour's cell, in its flattened box
            const T v = theirs[(size_t)(s / qw + 1) * (qw + 2) + (s % qw + 1)];
            int row, col; // my ghost cell
            if (edge == 0) {
                row = along + i + 1;
                col = 0;
            } else if (edge == 1) {
                row = along + i + 1;
                col = pex + 1;
            } else if (edge == 2) {
                row = 0;
                col = along + i + 1;
            } else {
                row = pey + 1;
                col = along + i + 1;
            }
            mine[(size_t)row * (pex + 2) + col] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Halo exchange across ranks: parts sharded over the ranks, ghost cells pushed over peer memory
// ------------------------------------------------------------------------------------------------
// Rank r owns parts [r P / G, (r + 1) P / G) and holds their framed tiles, in the layout of k_halo_exchange restricted
// to those parts and rebased to 0, behind a head of HALO_HEAD_BYTES in a buffer of its own that every rank maps.  One
// exchange is three plain launches with halo step k:
//   k_halo_open   one block: R = k into slot [0][rank] of every rank's flags, then wait for R >= k of every rank
//                 (nothing earlier on any rank's stream still reads the ghosts that are about to be overwritten);
//   k_halo_push   every ghost cell whose SOURCE part this rank owns, read locally and stored into the receiving
//                 part's tile wherever it lives (posted remote stores: no NVLink round trip per access); the last
//                 block stores D = k into slot [1][rank] of every rank's flags;
//   k_halo_close  one block: wait for D >= k of every rank (every ghost of this rank's tiles has arrived).
// The flags are PeerSync flags ([stage][MAX_PEERS], value 2 k), never reset.  A wait that times out sets the
// handle's error word (host memory, read by ddc_synchronize); a push whose open timed out stores nothing and raises
// no flag, so the ranks that wait for it time out too instead of reading stale ghosts.
constexpr size_t HALO_HEAD_BYTES = 256; // [flags: 2 x MAX_PEERS u32][block counter][opened step] ... tiles
struct HaloShards {
    PeerSync ps; // flags[q] = rank q's head as mapped here; step = the exchange number k
    double* tiles[MAX_PEERS]; // rank q's tiles as mapped here (tiles[rank]: this rank's)
    unsigned* done; // this rank's block counter of k_halo_push, zero between exchanges
    unsigned* opened; // this rank's word: the last step whose k_halo_open saw every rank
    int* err; // host-mapped error word (1: a rank did not reach the exchange in time)
    int P, p_begin, p_count; // all parts; this rank's range
};
__device__ __forceinline__ void halo_timed_out(const HaloShards& hs)
{
#ifndef DDC_HOST_EMU
    *(volatile int*)hs.err = 1;
    __threadfence_system();
#else
    *hs.err = 1;
#endif
}
// phases: 1 signal, 2 wait, 3 both (the device always runs both; the CPU emulation runs its ranks phase by phase)
__global__ void __launch_bounds__(32) k_halo_open(HaloShards hs, int phases)
{
    const int q = threadIdx.x;
    if (phases & 1) {
        __threadfence_system(); // everything this rank did before is complete (plain launch) and performed
        if (q < hs.ps.G)
            peer_signal(hs.ps, 0, 0u);
    }
    if (phases & 2) {
        unsigned seen = 0;
        const bool ok = q >= hs.ps.G || peer_wait(hs.ps, 0, &seen);
        if (!__syncthreads_or(!ok)) {
            if (q == 0)
                *hs.opened = hs.ps.step;
        } else if (q == 0)
            halo_timed_out(hs);
    }
}

// The end of every middle kernel of the sharded protocol (all threads of the block): once every block has counted
// itself, the last one stores D = k into slot [1][rank] of every rank's flags, for k_halo_close, and resets the counter.
__device__ __forceinline__ void halo_block_done(const HaloShards& hs)
{
    __shared__ int s_last;
    __syncthreads(); // every thread's accesses are issued ...
    if (threadIdx.x == 0) {
        __threadfence_system(); // ... and performed at the peers before the block is counted
        s_last = atomicAdd(hs.done, 1u) == gridDim.x - 1u;
    }
    __syncthreads();
    if (s_last) {
        if ((int)threadIdx.x < hs.ps.G)
            peer_signal(hs.ps, 1, 0u);
        if (threadIdx.x == 0)
            *hs.done = 0u;
    }
}

// One warp per (list l, owned part q): q's neighbours p in list l receive q's cells in their ghosts on the opposite
// edge.  The lists are symmetric (p is in q's edge-e list iff q is in p's opposite-edge list, same periodic flag), so
// q's entry in p's list -- found by binary search, the lists are id-ascending -- gives the halo size and start that
// k_halo_exchange uses for that ghost run, and the cells and values written are exactly the ones it writes.
__global__ void __launch_bounds__(256) k_halo_push(HaloShards hs, BoxTable bx, const int* __restrict__ counts,
    const int* __restrict__ offsets, int cap, const int* __restrict__ ids, const int* __restrict__ halos,
    const int* __restrict__ starts, const long long* __restrict__ off, unsigned lists)
{
    const int P = hs.P, G = hs.ps.G;
    const bool go = *(volatile unsigned*)hs.opened == hs.ps.step;
    // grid-stride over the warps: few enough blocks that the system fence each one pays below stays cheap
    const long long nw = go ? 8LL * hs.p_count : 0, stride = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < nw; w += stride) {
        const int l = (int)(w / hs.p_count), q = hs.p_begin + (int)(w % hs.p_count);
        if ((lists >> l) & 1u) {
            const int lane = lane_id();
            const int lp = (l & 4) | ((l & 3) ^ 1); // the list of p that holds q
            const int edge = lp & 3; // p's edge that faces q
            const int qw = bx.ex[q];
            const double* theirs = hs.tiles[hs.ps.rank] + (off[q] - off[hs.p_begin]);
            const int n = counts[l * P + q], first = offsets[l * (P + 1) + q];
            for (int k = 0; k < n; k++) {
                const int p = ids[(size_t)l * cap + first + k];
                const int m = counts[lp * P + p];
                const size_t base = (size_t)lp * cap + offsets[lp * (P + 1) + p];
                int lo = 0, hi = m;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (ids[base + mid] < q)
                        lo = mid + 1;
                    else
                        hi = mid;
                }
                if (lo == m || ids[base + lo] != q)
                    continue; // (not symmetric: k_halo_exchange would write nothing for this pair either)
                const int h = halos[base + lo], st = starts[base + lo];
                const int owner = (int)(((long long)(p + 1) * G - 1) / P), pb = (int)((long long)owner * P / G);
                double* mine = hs.tiles[owner] + (off[p] - off[pb]);
                const int px0 = bx.x0[p], py0 = bx.y0[p], pex = bx.ex[p], pey = bx.ey[p];
                const bool lr = edge < 2;
                const int along = lr ? max(py0, bx.y0[q]) - py0 : max(px0, bx.x0[q]) - px0;
                for (int i = lane; i < h; i += 32) {
                    const int s = st + (lr ? i * qw : i);
                    const double v = theirs[(size_t)(s / qw + 1) * (qw + 2) + (s % qw + 1)];
                    const int row = lr ? along + i + 1 : (edge == 2 ? 0 : pey + 1);
                    const int col = lr ? (edge == 0 ? 0 : pex + 1) : along + i + 1;
                    mine[(size_t)row * (pex + 2) + col] = v;
                }
            }
        }
    }
    if (!go)
        return; // (block-uniform) k_halo_open timed out: no stores, no flag
    halo_block_done(hs);
}

__global__ void __launch_bounds__(32) k_halo_close(HaloShards hs)
{
    if (*(volatile unsigned*)hs.opened != hs.ps.step)
        return; // k_halo_open timed out and said so
    const int q = threadIdx.x;
    unsigned seen = 0;
    const bool ok = q >= hs.ps.G || peer_wait(hs.ps, 1, &seen);
    if (__syncthreads_or(!ok) && q == 0)
        halo_timed_out(hs);
}

// ------------------------------------------------------------------------------------------------
// Halo scatter / gather: a field between its rows (double [ny][nx], x fastest) and the parts' tile interiors
// ------------------------------------------------------------------------------------------------
// Scatter stores field[y0 + j][x0 + i] into row j + 1, column i + 1 of part p's tile; gather is the inverse.  The work
// is (part, interior row) items, one warp each: at C5 a part row is ~256 cells, so every warp instruction moves 256
// contiguous bytes on both sides, and there are millions of items for 148 SMs instead of one long walk per part.
// The host lists, per part, the interior rows that meet the field rows at hand (all of them for one buffer, the rank's
// ddc_shard_rows block when sharded): range k is part[k]'s rows j0[k] ... for first[k + 1] - first[k] items, and its
// tile is at element base[k] of the buffer of rank owner[k] (one buffer: owner 0, base = the ddc_halo_tile_offsets
// offset; sharded: rebased to the owner's first part).  The host computes both: in a kernel, the 64-bit divisions that
// find the owner are a subroutine call, and the registers saved around it spill.
// Only non-empty ranges are listed, so first[] is strictly increasing.
struct HaloItems {
    const int* part; // [n]
    const int* j0; // [n]
    const int* owner; // [n]
    const int* first; // [n + 1], first[0] = 0, first[n] = all items
    const long long* base; // [n]
    int n;
};
// the ranges of the field rows [lo, hi) with the parts sharded over G ranks (G = 1: one buffer) into
// out[4 P + 1] = [part: P][j0: P][owner: P][first: P + 1] and base[P]; y0 / ex / ey: the boxes, off: the
// ddc_halo_tile_offsets offsets.  Returns n.  Host code, shared by ddc_api.cu and the emulation harness of the tests.
inline int halo_item_ranges(int P, int G, const int* y0, const int* ex, const int* ey, const long long* off, int lo, int hi,
    int* out, long long* base)
{
    int n = 0, run = 0;
    for (int p = 0; p < P; p++) {
        const int a = (y0[p] > lo ? y0[p] : lo) - y0[p], b = (y0[p] + ey[p] < hi ? y0[p] + ey[p] : hi) - y0[p];
        if (ex[p] > 0 && b > a) {
            const int owner = (int)(((long long)(p + 1) * G - 1) / P);
            out[n] = p;
            out[P + n] = a;
            out[2 * P + n] = owner;
            out[3 * P + n] = run;
            base[n] = off[p] - off[(long long)owner * P / G];
            run += b - a;
            n++;
        }
    }
    out[3 * P + n] = run;
    return n;
}

constexpr int HALO_ROW_LOADS = 8; // loads in flight per lane: a 256-cell row in one round
// n cells between a tile row and a field row, as 64-bit words (no arithmetic: NaN payloads, -0.0, subnormals stay).
// Every load of a round is issued before its stores: over NVLink (the sharded gather) a load is a round trip, and
// 8 independent ones per lane keep the link busy where one dependent load at a time would not.
template <bool kScatter>
__device__ __forceinline__ void halo_copy_row(unsigned long long* tile, unsigned long long* row, int n, int lane)
{
    const unsigned long long* __restrict__ src = kScatter ? row : tile;
    unsigned long long* __restrict__ dst = kScatter ? tile : row;
    for (int c0 = 0; c0 < n; c0 += 32 * HALO_ROW_LOADS) {
        unsigned long long v[HALO_ROW_LOADS];
#pragma unroll
        for (int u = 0; u < HALO_ROW_LOADS; u++) {
            const int c = c0 + 32 * u + lane;
            if (c < n)
                v[u] = src[c];
        }
#pragma unroll
        for (int u = 0; u < HALO_ROW_LOADS; u++) {
            const int c = c0 + 32 * u + lane;
            if (c < n)
                dst[c] = v[u];
        }
    }
}
// every item of `it`.  Warp g takes the contiguous items [g c, (g + 1) c), c = ceil(items / warps): one binary search
// for its first range, then row after row -- the next row's addresses are arithmetic, so its loads issue right behind
// the previous row's stores, and a part's box and tile are looked up only when the walk enters the part (DESIGN.md 7).
// tile_of(k): the tile of range k; field: the row y_base of the field
template <bool kScatter, typename TileOf>
__device__ __forceinline__ void halo_copy_items(const HaloItems& it, BoxTable bx, TileOf tile_of, double* field, int nx, int y_base)
{
    const unsigned total = (unsigned)it.first[it.n], warps = gridDim.x * (blockDim.x >> 5);
    const unsigned chunk = total / warps + (total % warps != 0u);
    const unsigned g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long w0 = (unsigned long long)g * chunk;
    if (w0 >= total)
        return;
    const int end = (int)min((unsigned long long)total, w0 + chunk), lane = lane_id();
    int w = (int)w0, k = 0, hi = it.n - 1; // k: the range with first[k] <= w < first[k + 1]
    while (k < hi) {
        const int mid = (k + hi + 1) >> 1;
        if (it.first[mid] <= w)
            k = mid;
        else
            hi = mid - 1;
    }
    while (w < end) {
        const int p = it.part[k], ex = bx.ex[p], stop = min(end, it.first[k + 1]);
        int j = it.j0[k] + (w - it.first[k]);
        unsigned long long* tile = reinterpret_cast<unsigned long long*>(tile_of(k)) + (size_t)(j + 1) * (ex + 2) + 1;
        unsigned long long* row = reinterpret_cast<unsigned long long*>(field) + (size_t)(bx.y0[p] + j - y_base) * nx + bx.x0[p];
        for (; w < stop; w++, tile += ex + 2, row += nx)
            halo_copy_row<kScatter>(tile, row, ex, lane);
        k++;
    }
}

// one buffer with every part's tile at tiles + off[p] (ddc_halo_tile_offsets); field: the whole double [ny][nx]
template <bool kScatter>
__global__ void __launch_bounds__(256) k_halo_field(HaloItems it, BoxTable bx, double* tiles, double* field, int nx)
{
    halo_copy_items<kScatter>(it, bx, [&](int k) { return tiles + it.base[k]; }, field, nx, 0);
}

// The sharded scatter / gather: the middle kernel between k_halo_open and k_halo_close.  rows: this rank's
// ddc_shard_rows block, starting at field row y_begin; `it` lists the parts' rows inside it, whoever owns the part.
// Scatter reads the rows locally and stores into the owners' tiles (posted remote stores, as k_halo_push); gather
// loads from the owners' tiles and stores into the rows, which only this rank maps (they are the caller's memory).
// Its D flag therefore also says "this rank has finished reading every rank's tiles": after k_halo_close no kernel a
// caller runs next on any rank can overwrite a cell that is still being read.
template <bool kScatter>
__global__ void __launch_bounds__(256) k_halo_field_shards(HaloShards hs, HaloItems it, BoxTable bx, double* rows, int nx,
    int y_begin)
{
    if (*(volatile unsigned*)hs.opened != hs.ps.step)
        return; // (grid-uniform) k_halo_open timed out: nothing touched, no flag
    halo_copy_items<kScatter>(it, bx, [&](int k) { return hs.tiles[it.owner[k]] + it.base[k]; }, rows, nx, y_begin);
    halo_block_done(hs);
}

// ------------------------------------------------------------------------------------------------
// synthetic land-sea mask: two octaves of integer value noise (bit-identical on host and device)
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline uint64_t splitmix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__host__ __device__ inline uint64_t lattice16(uint64_t seed, uint64_t oct, uint64_t ix, uint64_t iy)
{
    return splitmix64(seed ^ splitmix64((oct << 60) ^ (ix << 30) ^ iy)) >> 48;
}
__host__ __device__ inline uint64_t octave16(uint64_t seed, uint64_t oct, uint64_t L, uint64_t x, uint64_t y)
{
    const uint64_t cx = x / L, fx = x % L, cy = y / L, fy = y % L;
    const uint64_t v00 = lattice16(seed, oct, cx, cy), v10 = lattice16(seed, oct, cx + 1, cy);
    const uint64_t v01 = lattice16(seed, oct, cx, cy + 1), v11 = lattice16(seed, oct, cx + 1, cy + 1);
    const uint64_t top = v00 * (L - fx) + v10 * fx, bot = v01 * (L - fx) + v11 * fx;
    return (top * (L - fy) + bot * fy) / (L * L); // < 65536
}
// value in [0, 4 * 65536): ocean <=> value >= threshold
__host__ __device__ inline uint32_t synth_value(uint64_t seed, uint64_t L1, uint64_t L2, uint64_t x, uint64_t y)
{
    return (uint32_t)(3 * octave16(seed, 1, L1, x, y) + octave16(seed, 2, L2, x, y));
}

__global__ void __launch_bounds__(256) k_generate_mask(int32_t* __restrict__ out, int NX, int rows,
    int y_begin, uint64_t seed, uint64_t L1, uint64_t L2, uint32_t thresh)
{
    const size_t n = (size_t)NX * rows;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint64_t y = i / NX + y_begin, x = i % NX;
        out[i] = synth_value(seed, L1, L2, x, y) >= thresh ? 1 : 0;
    }
}

} // namespace ddc
