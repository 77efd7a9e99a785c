// emu_pipeline.cpp -- TEST INFRASTRUCTURE.  One decomposition through the product's REAL kernels
// (domain_decomp_b200/csrc/ddc_kernels.cuh compiled with -DDDC_HOST_EMU) on the host emulation of the CUDA
// execution model (cuda_emu.cpp), for G emulated ranks: the launch sequence, grid sizes and buffer layouts
// follow enqueue_partition() of ddc_api.cu, the ranks run phase by phase (all mask scans, then all x cuts, ...),
// and with G > 1 the kernels exchange their histograms exactly as on NVLink: the producers push into the
// other ranks' slots, the consumers check the flags and read their own buffers.
//
// What it is for: the CPU suite runs whole decompositions of small masks through the kernels' own code --
// every kernel, both exchange layouts, the variants of the strip row-count kernel -- and compares them with
// the oracle, on a machine without a GPU.  It says nothing about speed.
#include "cuda_emu.h"
#include "ddc_kernels.cuh"

#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace ddc;
using cuda_emu::Dim3;

namespace {
std::string g_err;

struct Rank {
    int rank = 0, y_begin = 0, rows = 0;
    const int32_t* mask = nullptr;
    std::vector<uint8_t> bits;
    std::vector<unsigned> flags; // [PEER_STAGES][MAX_PEERS]
    std::vector<unsigned> rowflags; // [G][flagcap]: one flag per block of the row-count kernel
    std::vector<unsigned> colslots, rowslots; // G slots each (slot g is written by rank g)
    std::vector<unsigned> colpfx, ypfx, done, colsum;
    std::vector<int> strips, boxes, strip_of_col, part_at;
    std::vector<long long> loads, loadmm;
    std::vector<int32_t> pid;
    std::vector<int> nbr_counts, nbr_offsets, nbr_totals, nbr_ids, nbr_halos, nbr_starts;
    DevScalars sc {};
    unsigned gate_word = 0;
    unsigned sum_word = 0; // k_sum_cols -> K2 (ChainWord)
    Plan plan {}, host_plan {};
};

#define LAUNCH(grid, block, smem, call)                                                            \
    do {                                                                                           \
        if (!cuda_emu::launch(grid, block, smem, [&] { call; })) {                                  \
            g_err = std::string(#call) + ": " + cuda_emu::last_error();                            \
            return false;                                                                          \
        }                                                                                          \
    } while (0)

struct Options {
    int strip_k = 0; // 0 auto, 1 / 2 / 4 rows per warp, 16 the kernel for boundary tables beyond shared memory
    int scan_rpc = 64; // rows per CTA of the mask scan
    int smem_limit = 232448; // bytes of dynamic shared memory a block may use (B200: 227 KB)
    bool collectives = false; // G > 1: the NCCL fallback of ddc_api.cu (all-reduce / all-gather between the kernels,
                              // emulated by host loops) instead of the slot exchange inside the kernels
};

bool run_step(std::vector<Rank>& R, int NX, int NY, int P, int px, int py, int aix, int aiy, unsigned step,
    const Options& opt, int cap, bool skip_init)
{
    const int G = (int)R.size();
    const int NG = (NX + 127) / 128, NB = NG * 16;
    const int yr_off = (NX + 3) & ~3, ncol = yr_off + 2 * G;
    const int Rmax = (NY + G - 1) / G;
    const int Scap = (int)std::min<long long>(P, 1LL << std::min(aix, 30));
    const bool ycuts = aiy > 0 && P > 1, narrow = NX < 65536, p2p = G > 1 && !opt.collectives;
    const size_t rc_elems = (size_t)Scap * (((size_t)Rmax + 31) & ~(size_t)31);
    const size_t rc_words = narrow ? (rc_elems + 1) / 2 : rc_elems;
    const size_t rank_stride = narrow ? rc_words * 2 : rc_words;
    const size_t colcap = ((std::max<size_t>(ncol, 2 * ((size_t)yr_off + 2)) + 3) & ~(size_t)3), rowcap = (rc_words + 4 + 3) & ~(size_t)3;
    const size_t xneed = sizeof(unsigned) * ((((size_t)NX + 1 + 3) & ~(size_t)3) + hist_bitmap_words(NX)) + LEVEL_NODES_BYTES;
    const size_t yneed = sizeof(unsigned) * ((((size_t)NY + 1 + 3) & ~(size_t)3) + hist_bitmap_words(NY)) + LEVEL_NODES_BYTES;
    const bool x_smem = xneed + 1024 <= (size_t)opt.smem_limit, y_smem = yneed + 1024 <= (size_t)opt.smem_limit;
    const int ygrid = std::max(1, std::min(Scap, 148 * 2));
    const int gridx = (NG + 7) / 8;
    const int d_rows = gridx + 1, d_label = (gridx + 3) & ~1, d_ycuts = d_label + 2, d_sum = d_ycuts + 1, ndone = d_sum + 1; // ddc_api.cu: the "last block" counters
    const NaiveParams nv = naive_params(P, NX, NY);
    const int nchunk = (NY + 31) / 32;
    const int par = (int)(step & 1u);
    const bool want_nbr = P > 1;

    auto tables = [&](Rank& r, StripTable& st, BoxTable& bx) {
        int* q = r.strips.data();
        st.x0 = q;
        st.x1 = q + (P + 1);
        st.p0 = q + 2 * (P + 1);
        st.S = q + 3 * (P + 1) + 1;
        st.always = q + 3 * (P + 1) + 2;
        int* b = r.boxes.data();
        bx = { b, b + P, b + 2 * P, b + 3 * P };
    };
    auto colslot = [&](Rank& r, int slot) { return r.colslots.data() + ((size_t)par * G + slot) * colcap; };
    auto rowslot = [&](Rank& r, int slot) { return r.rowslots.data() + ((size_t)par * G + slot) * rowcap; };
    const size_t flagcap = (size_t)(Rmax + 7) / 8 + 4;
    auto sync_of = [&](Rank& r) {
        PeerSync ps {};
        ps.rank = r.rank;
        ps.G = G;
        ps.enabled = p2p ? 1 : 0;
        ps.step = step;
        for (int q = 0; q < G; q++)
            ps.flags[q] = R[q].flags.data();
        return ps;
    };

    for (Rank& r : R) { // buffers
        r.bits.resize((size_t)std::max(r.rows, 1) * NB);
        r.flags.resize((size_t)PEER_STAGES * MAX_PEERS, 0u);
        r.rowflags.resize((size_t)G * flagcap, 0u);
        r.colslots.resize(2 * (size_t)G * colcap, 0xdeadbeefu);
        r.rowslots.resize(2 * (size_t)G * rowcap, 0xdeadbeefu);
        r.colpfx.resize((size_t)NX + 1);
        r.ypfx.resize((size_t)ygrid * (((size_t)NY + 1 + 3) & ~(size_t)3));
        r.done.resize((size_t)ndone);
        r.strips.assign((size_t)3 * (P + 1) + 3, 0);
        r.boxes.assign((size_t)4 * P, 0);
        r.strip_of_col.assign(NX, 0);
        r.part_at.assign((size_t)std::max(Scap, 1) * nchunk, -12345);
        r.loads.assign(P, 0);
        r.loadmm.assign(2, 0);
        r.pid.assign((size_t)std::max(r.rows, 1) * NX, INT_MIN);
        r.nbr_counts.assign((size_t)8 * P, 0);
        r.nbr_offsets.assign((size_t)8 * (P + 1), 0);
        r.nbr_totals.assign(8, 0);
        r.nbr_ids.assign((size_t)8 * cap, 0);
        r.nbr_halos.assign((size_t)8 * cap, 0);
        r.nbr_starts.assign((size_t)8 * cap, 0);
    }
    // ---- K1: mask scan (with G > 1: pushes the column counts and raises the stage-0 flag) ----
    for (Rank& r : R) {
        unsigned* colcount = colslot(r, r.rank);
        if (!skip_init) // the product launches k_init only for buffers K2 / the scan have not left clean
            LAUNCH(Dim3((std::max(ncol, ndone) + 255) / 256), Dim3(256), 0,
                k_init(colcount, ncol, yr_off, r.rank, &r.sc, r.loadmm.data(), r.done.data(), ndone));
        PeerPush push {};
        push.rank = r.rank;
        push.n = p2p ? G : 1;
        push.packed = p2p && Rmax < 65536 ? 1 : 0;
        for (int q = 0; q < G; q++)
            push.dst[q] = p2p ? (void*)colslot(R[q], r.rank) : (void*)colcount;
        const PeerSync ps = sync_of(r);
        const bool vec = (NX % 4 == 0) && (((uintptr_t)r.mask) % 16 == 0);
        int* yr = reinterpret_cast<int*>(colcount + yr_off + 2 * r.rank);
        if (r.rows > 0 || p2p) {
            const int rpc = opt.scan_rpc;
            const int small = std::max(8, (rpc / 4) & ~7); // ddc_api.cu: the last quarter of the rows in smaller chunks
            int nbig = (r.rows + rpc - 1) / rpc, nsmall = 0;
            if (small < rpc && r.rows >= 4 * rpc) {
                nbig = (int)((long long)r.rows * 75 / 100) / rpc;
                nsmall = (r.rows - nbig * rpc + small - 1) / small;
            }
            const Dim3 grid(gridx, std::max(1, nbig + nsmall));
            if (vec)
                LAUNCH(grid, Dim3(256), 0,
                    k_scan_mask<true>(r.mask, NX, r.rows, r.y_begin, NB, rpc, r.bits.data(), colcount, yr, push, ps,
                        r.done.data(), yr_off, nullptr, nbig, small));
            else
                LAUNCH(grid, Dim3(256), 0,
                    k_scan_mask<false>(r.mask, NX, r.rows, r.y_begin, NB, rpc, r.bits.data(), colcount, yr, push, ps,
                        r.done.data(), yr_off, nullptr, nbig, small));
        }
    }
    if (G > 1 && !p2p) { // ncclAllReduce(SUM) of the column counts and the y-range pairs, in place on every rank
        std::vector<unsigned> sum((size_t)ncol, 0u);
        for (Rank& r : R)
            for (int i = 0; i < ncol; i++)
                sum[i] += colslot(r, r.rank)[i];
        for (Rank& r : R)
            std::copy(sum.begin(), sum.end(), colslot(r, r.rank));
    }
    // odd steps poll flags / words in place of the kernel boundaries between k_sum_cols and K2, as a step with
    // programmatic launches does on the device; even steps wait for the boundaries, as a DDC_PROFILE step does
    const bool chained = (step & 1u) != 0u;
    // ---- K2: x cuts ----
    for (Rank& r : R) {
        StripTable st;
        BoxTable bx;
        tables(r, st, bx);
        PeerCols pc {};
        pc.n = p2p ? G : 1;
        pc.own = r.rank;
        pc.packed = p2p && Rmax < 65536 ? 1 : 0;
        for (int q = 0; q < G; q++)
            pc.col[q] = colslot(r, p2p ? q : r.rank);
        PeerSync ps = sync_of(r);
        const ChainWord w_sum = chained && p2p ? ChainWord { &r.sum_word, step } : ChainWord { nullptr, 0u };
        if (p2p) { // the ranks' slots summed by a grid of blocks first (k_sum_cols), K2 reads one buffer
            r.colsum.assign((size_t)ncol + 4, 0xdeadbeefu);
            LAUNCH(Dim3(gridx), Dim3(256), 0,
                k_sum_cols(pc, ps, NX, yr_off, r.colsum.data(), &r.plan, chained ? 1 : 0, r.done.data() + d_sum, w_sum, nullptr));
            pc = PeerCols {};
            pc.col[0] = r.colsum.data();
            pc.n = 1;
            ps.enabled = 0;
        }
        if (x_smem)
            LAUNCH(Dim3(1), Dim3(1024), xneed,
                k_xcuts<true>(pc, ps, NX, NY, P, nullptr, yr_off, G, aix, aiy, &r.plan, st, bx, r.loads.data(), r.loadmm.data(),
                    &r.sc, colslot(r, r.rank), 0, &r.host_plan, p2p ? 1 : 0, (p2p && r.rows > 0) ? 0 : 1, w_sum));
        else
            LAUNCH(Dim3(1), Dim3(1024), LEVEL_NODES_BYTES,
                k_xcuts<false>(pc, ps, NX, NY, P, r.colpfx.data(), yr_off, G, aix, aiy, &r.plan, st, bx, r.loads.data(),
                    r.loadmm.data(), &r.sc, colslot(r, r.rank), 0, &r.host_plan, p2p ? 1 : 0, (p2p && r.rows > 0) ? 0 : 1, w_sum));
        if (!ycuts) // with y levels K4 paints the column -> strip table
            LAUNCH(Dim3(std::max(1, std::min((Scap + 7) / 8, 148 * 4))), Dim3(256), 0,
                k_paint_strips(st, &r.plan, r.strip_of_col.data()));
    }
    // ---- K3: strip row counts (pushed to every rank) ----
    int rb_shift = 5, row_blocks = 0;
    auto row_sync = [&](PeerSync& ps) {
        for (int q = 0; q < G; q++)
            ps.rowflag[q] = R[q].rowflags.data();
        ps.flagcap = (int)flagcap;
        ps.rowblocks = row_blocks;
    };
    if (ycuts) {
        for (Rank& r : R) {
            StripTable st;
            BoxTable bx;
            tables(r, st, bx);
            PeerPush out {};
            out.rank = r.rank;
            out.n = p2p ? G : 1;
            for (int q = 0; q < G; q++)
                out.dst[q] = rowslot(R[p2p ? q : r.rank], r.rank);
            PeerSync ps = sync_of(r);
            int K = Rmax >= 32 * 4 * 148 ? 4 : 2;
            if (opt.strip_k)
                K = opt.strip_k;
            while (K > 1 && sizeof(int) * strip_scan_smem_words(NG, Scap, K) > 48 * 1024)
                K >>= 1;
            const size_t scan_smem = sizeof(int) * strip_scan_smem_words(NG, Scap, K);
            if (scan_smem <= 48 * 1024 && opt.strip_k != 16) {
                const Dim3 grid((Rmax + 8 * K - 1) / (8 * K));
                rb_shift = K == 4 ? 5 : (K == 2 ? 4 : 3);
                if (p2p && G <= 2) { // one flag per block instead of one per rank (row_flags_raise), as on 2 GPUs
                    row_blocks = (int)grid.x;
                    row_sync(ps);
                }
#define SCAN(CT, KK)                                                                               \
    LAUNCH(grid, Dim3(256), scan_smem,                                                             \
        (k_strip_rows_scan<CT, KK>(r.bits.data(), NB, NX, r.rows, st.x0, st.p0, &r.plan, Scap, out, Rmax, ps,          \
            r.done.data() + d_rows, nullptr)))
                if (narrow) {
                    if (K == 4)
                        SCAN(uint16_t, 4);
                    else if (K == 2)
                        SCAN(uint16_t, 2);
                    else
                        SCAN(uint16_t, 1);
                } else {
                    if (K == 4)
                        SCAN(unsigned, 4);
                    else if (K == 2)
                        SCAN(unsigned, 2);
                    else
                        SCAN(unsigned, 1);
                }
#undef SCAN
            } else { // strip_k == 16: the kernel for boundary tables that do not fit shared memory
                rb_shift = 5;
                const Dim3 grid((Rmax + 31) / 32, (Scap + 7) / 8);
                if (narrow)
                    LAUNCH(grid, Dim3(256), 0,
                        k_strip_rows<uint16_t>(r.bits.data(), NB, r.rows, st.x0, st.x1, st.p0, &r.plan, Scap, out, Rmax, ps,
                            r.done.data() + d_rows, nullptr));
                else
                    LAUNCH(grid, Dim3(256), 0,
                        k_strip_rows<unsigned>(r.bits.data(), NB, r.rows, st.x0, st.x1, st.p0, &r.plan, Scap, out, Rmax, ps,
                            r.done.data() + d_rows, nullptr));
            }
        }
        std::vector<std::vector<unsigned>> gathered;
        if (G > 1 && !p2p) { // ncclAllGather of every rank's block: [G][rc_words]
            gathered.assign(G, std::vector<unsigned>(rc_words * G + 4, 0u));
            for (Rank& dst : R)
                for (Rank& src : R)
                    std::copy(rowslot(src, src.rank), rowslot(src, src.rank) + rc_words,
                        gathered[dst.rank].begin() + (size_t)src.rank * rc_words);
        }
        // (the last block of every rank's K3 has raised the rank's stage-1 flag at every peer)
        // ---- K4: y cuts ----
        for (Rank& r : R) {
            StripTable st;
            BoxTable bx;
            tables(r, st, bx);
            PeerRows pr {};
            pr.n = p2p ? G : 1;
            for (int q = 0; q < G; q++)
                pr.row[q] = rowslot(r, p2p ? q : r.rank);
            if (G > 1 && !p2p)
                pr.row[0] = gathered[r.rank].data();
            PeerSync ps = sync_of(r);
            if (row_blocks)
                row_sync(ps);
            const RowLayout rl = { rank_stride, Rmax, Scap, rb_shift };
            BoxGate gate {}; // as in ddc_api.cu: K4's last block opens the gate of the second stream
            gate.word = &r.gate_word;
            gate.done = r.done.data() + d_ycuts;
            gate.step = step;
#define YCUTS(CT, SM)                                                                              \
    LAUNCH(Dim3(ygrid), Dim3(1024), SM ? yneed : LEVEL_NODES_BYTES,                                                \
        (k_ycuts<CT, SM>(pr, ps, rl, NY, st, r.ypfx.data(), bx, r.loads.data(), r.loadmm.data(), &r.plan,                    \
            r.strip_of_col.data(), 0, gate, r.part_at.data(), nchunk)))
            if (narrow) {
                if (y_smem)
                    YCUTS(uint16_t, true);
                else
                    YCUTS(uint16_t, false);
            } else {
                if (y_smem)
                    YCUTS(unsigned, true);
                else
                    YCUTS(unsigned, false);
            }
#undef YCUTS
        }
    }
    // ---- K7 (speculative), K6 ----
    for (Rank& r : R) {
        StripTable st;
        BoxTable bx;
        tables(r, st, bx);
        const int ngrid = (std::max(P, 8) + 7) / 8;
        if (want_nbr) {
            if (ycuts) {
                if (r.gate_word != step) {
                    g_err = "K4 did not open the gate of the second stream";
                    return false;
                }
                LAUNCH(Dim3(1), Dim3(32), 0, k_gate(&r.gate_word, step, &r.plan));
            }
            LAUNCH(Dim3(ngrid), Dim3(256), 0,
                k_neighbours<false>(bx, P, NX, NY, px, py, st, r.nbr_counts.data(), nullptr, nullptr, cap, nullptr, nullptr,
                    nullptr, &r.sc, &r.plan));
            LAUNCH(Dim3(8), Dim3(1024), 0,
                k_scan_counts(r.nbr_counts.data(), P, r.nbr_offsets.data(), r.nbr_totals.data(), &r.plan));
            LAUNCH(Dim3(ngrid), Dim3(256), 0,
                k_neighbours<true>(bx, P, NX, NY, px, py, st, r.nbr_counts.data(), r.nbr_offsets.data(), r.nbr_totals.data(),
                    cap, r.nbr_ids.data(), r.nbr_halos.data(), r.nbr_starts.data(), &r.sc, &r.plan));
        }
        if (r.rows > 0) {
            const bool vecp = (NX % 4 == 0) && (((uintptr_t)r.pid.data()) % 16 == 0);
            const int rpc = 32;
            const Dim3 grid(gridx, (r.rows + rpc - 1) / rpc);
            LabelEnd fin {};
            fin.fuse = (G == 1 || p2p) ? 1 : 0;
            fin.P = P;
            fin.ps = sync_of(r);
            fin.counter = reinterpret_cast<unsigned long long*>(r.done.data() + d_label);
            fin.host_plan = &r.host_plan;
            fin.dbg = nullptr;
            fin.part_at.table = ycuts ? r.part_at.data() : nullptr;
            fin.part_at.nchunk = nchunk;
            fin.reset_col = p2p ? colslot(r, r.rank) : nullptr;
            fin.reset_n = ncol;
            fin.yr_off = yr_off;
            if (vecp)
                LAUNCH(grid, Dim3(256), 0,
                    (k_label<true, true>(r.bits.data(), NX, r.rows, r.y_begin, NB, rpc, r.strip_of_col.data(), st.p0, bx.y0,
                        bx.ey, nv, r.pid.data(), &r.sc, &r.plan, fin)));
            else
                LAUNCH(grid, Dim3(256), 0,
                    (k_label<false, true>(r.bits.data(), NX, r.rows, r.y_begin, NB, rpc, r.strip_of_col.data(), st.p0, bx.y0,
                        bx.ey, nv, r.pid.data(), &r.sc, &r.plan, fin)));
        }
    }
    if (G > 1 && !p2p) { // ncclAllReduce(MAX) of `changes`
        int any = 0;
        for (Rank& r : R)
            any = std::max(any, r.sc.changes);
        for (Rank& r : R)
            r.sc.changes = any;
    }
    // ---- K5: in the stream for ranks without a labelling kernel and for the NCCL exchange; otherwise from
    //      validate() when the labelling kernel's last block left the verdict open (Plan::fixup) ----
    auto finalize = [&](Rank& r) {
        StripTable st;
        BoxTable bx;
        tables(r, st, bx);
        const PeerSync ps = sync_of(r);
        const NbrTables nb = { r.nbr_counts.data(), r.nbr_offsets.data(), r.nbr_totals.data(), cap, r.nbr_ids.data(),
            r.nbr_halos.data(), r.nbr_starts.data() };
        LAUNCH(Dim3(1), Dim3(1024), 0,
            k_finalize(ps, P, NX, NY, px, py, nv, &r.sc, &r.plan, st, bx, want_nbr ? 1 : 0, nb, &r.host_plan));
        return true;
    };
    // ranks whose K5 is in the stream raise their stage-2 flag there; on the GPU a peer that needs it polls until it
    // arrives, the emulation runs these ranks first
    for (Rank& r : R)
        if (!(r.rows > 0 && (G == 1 || p2p)))
            if (p2p && r.rows == 0) // (with NCCL there are no flags)
                for (int q = 0; q < G; q++)
                    R[q].flags[2 * MAX_PEERS + r.rank] = 2u * step + (r.sc.changes ? 1u : 0u);
    for (Rank& r : R)
        if (!(r.rows > 0 && (G == 1 || p2p)))
            if (!finalize(r))
                return false;
    for (Rank& r : R)
        if (r.rows > 0 && (G == 1 || p2p) && !r.host_plan.mismatch && r.host_plan.fixup)
            if (!finalize(r))
                return false;
    return true;
}
} // namespace

extern "C" {
__attribute__((visibility("default"))) const char* emu_last_error(void) { return g_err.c_str(); }

// One decomposition of mask[NY][NX] into P parts on G emulated ranks (row-sharded like ddc_shard_rows).
// boxes[P*4] = x0 y0 ex ey; pid[NY*NX]; nbr_counts[8*P]; nbr_flat[3][sum of list totals] = ids, halos, starts of
// the eight lists one after the other (list l = periodic * 4 + edge), nbr_cap = entries available per array;
// out[0..7] = changes, median iterations, n_ocean, strips, x levels, y levels, load min, load max.
// strip_k: 0 the product's choice; 1 / 2 / 4 rows per warp of the streaming row-count kernel; 16: the non-streaming one.
// smem_limit: 0 = B200's 227 KB; smaller values force the global-memory prefix paths of the cut kernels.
// Returns 0, or -1 (emu_last_error()).  Every rank must end with identical boxes and tables (checked).
__attribute__((visibility("default"))) int emu_partition(const int32_t* mask, int NX, int NY, int P, int px, int py, int G,
    int strip_k, int scan_rpc, int smem_limit, int32_t* boxes, int32_t* pid, int32_t* nbr_counts, int32_t* nbr_flat,
    long nbr_cap, long long* out)
{
    g_err.clear();
    if (std::getenv("DDC_EMU_OOB_SELFTEST")) { // proves that an AddressSanitizer build of this library is live
        std::vector<int> v(4);
        volatile int* q = v.data();
        q[4] = 1;
    }
    if (const char* e = std::getenv("DDC_EMU_SCHED_SEED")) // random block / thread schedules (race shaking)
        cuda_emu::set_schedule_seed(std::strtoull(e, nullptr, 10));
    else
        cuda_emu::set_schedule_seed(0);
    if (G < 1 || G > MAX_PEERS || NX < 1 || NY < 1 || P < 1
        || !(strip_k == 0 || strip_k == 1 || strip_k == 2 || strip_k == 4 || strip_k == 16)) {
        g_err = "bad arguments";
        return -1;
    }
    Options opt;
    opt.strip_k = strip_k;
    if (scan_rpc > 0)
        opt.scan_rpc = scan_rpc;
    if (smem_limit > 0)
        opt.smem_limit = smem_limit;
    opt.collectives = std::getenv("DDC_EMU_COLLECTIVES") != nullptr;
    // the masks of the ranks: 16-byte aligned copies of their row blocks (like a cudaMalloc'ed shard)
    std::vector<Rank> R(G);
    std::vector<std::vector<int32_t>> shard(G);
    const int rpr = (NY + G - 1) / G;
    for (int g = 0; g < G; g++) {
        const int b = std::min(NY, g * rpr), e = std::min(NY, b + rpr);
        R[g].rank = g;
        R[g].y_begin = b;
        R[g].rows = e - b;
        shard[g].assign((size_t)std::max(1, e - b) * NX + 4, 0);
        int32_t* base = shard[g].data();
        while ((uintptr_t)base % 16)
            base++;
        std::memcpy(base, mask + (size_t)b * NX, sizeof(int32_t) * (size_t)(e - b) * NX);
        R[g].mask = base;
    }
    int aix, aiy;
    guess_plan(P, NX, NY, &aix, &aiy);
    unsigned step = 0;
    int cap = 3 * P + 64; // entries per neighbour list, as the product sizes them
    // DDC_EMU_REPEAT=n: the decomposition is enqueued n more times first, like back-to-back calls on one handle --
    // from the third step on WITHOUT k_init: K2 and the scan's last CTA must have left every accumulator clean
    if (const char* e = std::getenv("DDC_EMU_REPEAT"))
        for (int i = std::atoi(e); i > 0; i--) {
            step++;
            if (!run_step(R, NX, NY, P, px, py, aix, aiy, step, opt, cap, step > 2))
                return -1;
            if (R[0].plan.mismatch == 1) { // settle the plan as validate() would
                aix = R[0].plan.ix;
                aiy = R[0].plan.iy;
            }
        }
    for (int attempt = 0;; attempt++) {
        step++;
        if (!run_step(R, NX, NY, P, px, py, aix, aiy, step, opt, cap, step > 2))
            return -1;
        const Plan& pl = R[0].host_plan;
        if (!pl.mismatch && R[0].sc.overflow && attempt < 4) {
            // the bounded lists overflowed (tiny grids cut into many empty parts): the product re-runs the fill
            // pass with the exact capacity (fetch_totals), the emulation re-runs the step
            for (int l = 0; l < 8; l++)
                cap = std::max(cap, R[0].nbr_totals[l] + 1);
            continue;
        }
        if (!pl.mismatch)
            break;
        if (pl.mismatch == 3 || attempt >= 2) {
            g_err = pl.mismatch == 3 ? "a rank missed an exchange flag" : "the RCB plan did not settle";
            return -1;
        }
        aix = pl.ix;
        aiy = pl.iy;
    }
    // results: replicated tables from rank 0 (and they must be identical on every rank), pid from every rank
    const Rank& r0 = R[0];
    for (int g = 1; g < G; g++) {
        if (R[g].boxes != r0.boxes || R[g].nbr_counts != r0.nbr_counts || R[g].nbr_totals != r0.nbr_totals
            || R[g].sc.changes_all != r0.sc.changes_all || R[g].host_plan.iters != r0.host_plan.iters) {
            g_err = "rank " + std::to_string(g) + " ended with other boxes / tables than rank 0";
            return -1;
        }
    }
    for (int p = 0; p < P; p++)
        for (int i = 0; i < 4; i++)
            boxes[4 * p + i] = r0.boxes[(size_t)i * P + p];
    for (int g = 0; g < G; g++)
        if (R[g].rows > 0)
            std::memcpy(pid + (size_t)R[g].y_begin * NX, R[g].pid.data(), sizeof(int32_t) * (size_t)R[g].rows * NX);
    std::memset(nbr_counts, 0, sizeof(int32_t) * 8 * (size_t)P);
    long pos = 0;
    if (P > 1) {
        if (r0.sc.overflow) {
            g_err = "neighbour lists overflowed their capacity";
            return -1;
        }
        std::memcpy(nbr_counts, r0.nbr_counts.data(), sizeof(int32_t) * 8 * (size_t)P);
        long total = 0;
        for (int l = 0; l < 8; l++)
            total += r0.nbr_totals[l];
        if (total > nbr_cap) {
            g_err = "nbr_flat too small";
            return -1;
        }
        for (int l = 0; l < 8; l++)
            for (int k = 0; k < r0.nbr_totals[l]; k++, pos++) {
                nbr_flat[pos] = r0.nbr_ids[(size_t)l * cap + k];
                nbr_flat[nbr_cap + pos] = r0.nbr_halos[(size_t)l * cap + k];
                nbr_flat[2 * nbr_cap + pos] = r0.nbr_starts[(size_t)l * cap + k];
            }
    }
    out[0] = P > 1 ? r0.sc.changes_all : 0;
    out[1] = r0.host_plan.iters;
    out[2] = r0.host_plan.W;
    out[3] = r0.host_plan.S;
    out[4] = r0.host_plan.ix;
    out[5] = r0.host_plan.iy;
    out[6] = r0.loadmm[0];
    out[7] = r0.loadmm[1];
    return 0;
}
}
