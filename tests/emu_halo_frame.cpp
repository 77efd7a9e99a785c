// emu_halo_frame.cpp -- TEST INFRASTRUCTURE.  The full-frame halo exchange (ddc_halo_exchange_full_f64 and
// ddc_halo_exchange_full_shards_f64: edges plus corner ghosts) through the product's REAL kernels and host tables
// (halo_corner_sources / halo_corner_items, k_halo_exchange + k_halo_corners on one buffer, k_halo_push_full between
// k_halo_open and k_halo_close on the shards; ddc_kernels.cuh compiled with -DDDC_HOST_EMU) on the host emulation of
// the CUDA execution model, for G emulated ranks, mixed with edge exchanges (k_halo_push), scatters and gathers on one
// halo step counter.  Structured as tests/emu_halo_fields.cpp: the buffers, item tables and launches follow
// ddc_api.cu, the ranks run phase by phase, and beside them the single-buffer kernels run on one buffer holding all
// parts.  It says nothing about speed.
// Compiled by tests/test_halo_frame_on_cpu_emulator.py (into a temporary directory) against oracle/emu/cuda_emu.cpp.
#include "cuda_emu.h"
#include "ddc_kernels.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace ddc;
using cuda_emu::Dim3;

namespace {
std::string g_err;
constexpr int GRID_MAX = 4; // few blocks: the grid-stride loops and the block counter see several rounds and blocks
}

#define LAUNCH(grid, block, call)                                                                  \
    do {                                                                                           \
        if (!cuda_emu::launch(grid, block, 0, [&] { call; })) {                                    \
            g_err = std::string(#call) + ": " + cuda_emu::last_error();                            \
            return -1;                                                                             \
        }                                                                                          \
    } while (0)

extern "C" {
__attribute__((visibility("default"))) const char* emu_halo_frame_last_error(void) { return g_err.c_str(); }

// boxes[P][4] = x0 y0 ex ey; counts / ids / halos / starts: the neighbour lists as in emu_halo_shards (used by 'x' and
// 'f'); px / py: the decomposition's periodic flags (the corner table).  rows_b[G], rows_c[G]: every rank's
// ddc_shard_rows block.  ops: a string of 's' (scatter), 'x' (edge exchange), 'f' (full-frame exchange), 'g' (gather),
// run in order on the sharded buffers AND on the single buffer, with one halo step counter.
// corner_ids / corner_starts [2][4][P]: the corner table of halo_corner_sources, as ddc_api.cu builds it.
// field[ny * nx]: what each rank's rows hold for a scatter (rank r: rows rows_b[r] ...), and what the single-buffer
// scatter reads.  tiles_in[total]: the tiles before the first op (every buffer); rows_in[ny * nx]: the rows (and the
// single-buffer field) a gather writes into before the first op.  After op i: tiles_out[i] = the ranks' buffers
// concatenated, single_out[i] = the single buffer, rows_out[i] = the ranks' rows concatenated, field_out[i] = the
// single-buffer field.  stall: a rank that runs none of the kernels (-1: none).  err_out[G]: the error words at the end.
// Returns 0, or -1 (emu_halo_frame_last_error()).
__attribute__((visibility("default"))) int emu_halo_frame(int P, const int32_t* boxes, const int32_t* counts,
    const int32_t* ids, const int32_t* halos, const int32_t* starts, int nx, int ny, int px, int py, int G,
    const int32_t* rows_b, const int32_t* rows_c, int periodic, const char* ops, int stall, const double* field,
    const double* tiles_in, const double* rows_in, double* tiles_out, double* single_out, double* rows_out,
    double* field_out, int32_t* err_out, int32_t* corner_ids, int32_t* corner_starts)
{
    g_err.clear();
    if (const char* e = std::getenv("DDC_EMU_SCHED_SEED"))
        cuda_emu::set_schedule_seed(std::strtoull(e, nullptr, 10));
    else
        cuda_emu::set_schedule_seed(0);
    if (P < 1 || G < 1 || G > MAX_PEERS || nx < 1 || ny < 1) {
        g_err = "bad arguments";
        return -1;
    }
    // device layout of the tables (ddc_api.cu): counts [8][P], offsets [8][P + 1], ids / halos / starts [8][cap]
    std::vector<int> bxv((size_t)4 * P), cnt(counts, counts + (size_t)8 * P), offs((size_t)8 * (P + 1));
    for (int p = 0; p < P; p++)
        for (int i = 0; i < 4; i++)
            bxv[(size_t)i * P + p] = boxes[4 * p + i];
    int cap = 1;
    std::vector<int> tot(8, 0);
    for (int l = 0; l < 8; l++) {
        for (int p = 0; p < P; p++) {
            offs[(size_t)l * (P + 1) + p] = tot[l];
            tot[l] += cnt[(size_t)l * P + p];
        }
        offs[(size_t)l * (P + 1) + P] = tot[l];
        cap = std::max(cap, tot[l]);
    }
    std::vector<int> vid((size_t)8 * cap, -1), vh((size_t)8 * cap, 0), vs((size_t)8 * cap, 0);
    for (int l = 0, pos = 0; l < 8; l++)
        for (int k = 0; k < tot[l]; k++, pos++) {
            vid[(size_t)l * cap + k] = ids[pos];
            vh[(size_t)l * cap + k] = halos[pos];
            vs[(size_t)l * cap + k] = starts[pos];
        }
    const bool have_nbr = P > 1; // ddc_api.cu: no neighbour tables for one part, and the exchange does nothing
    BoxTable bx = { bxv.data(), bxv.data() + P, bxv.data() + 2 * P, bxv.data() + 3 * P };
    std::vector<long long> off((size_t)P + 1, 0);
    for (int p = 0; p < P; p++)
        off[p + 1] = off[p] + (long long)(std::max(bxv[(size_t)2 * P + p], 0) + 2) * (std::max(bxv[(size_t)3 * P + p], 0) + 2);
    const long long total = off[P];
    const size_t cells = (size_t)nx * ny;

    // the item tables of ddc_api.cu's tile_offsets(): every row (single buffer), each rank's rows (sharded)
    auto table = [&](int g, int lo, int hi, std::vector<int>& t, std::vector<long long>& base) {
        t.assign((size_t)4 * P + 1, 0);
        base.assign((size_t)P, 0);
        const int n = halo_item_ranges(P, g, bx.y0, bx.ex, bx.ey, off.data(), lo, hi, t.data(), base.data());
        return HaloItems { t.data(), t.data() + P, t.data() + 2 * P, t.data() + 3 * P, base.data(), n };
    };
    auto grid_of = [](const HaloItems& it) { return (unsigned)std::max(1, std::min((it.first[it.n] + 7) / 8, GRID_MAX)); };
    std::vector<int> single_t;
    std::vector<long long> single_b;
    const HaloItems single_items = table(1, 0, ny, single_t, single_b);

    // the corner table and items of ddc_api.cu's tile_offsets(): all items on one buffer, each rank's own sources
    halo_corner_sources(P, nx, ny, px, py, bx.x0, bx.y0, bx.ex, bx.ey, corner_ids, corner_starts);
    const size_t cp = (size_t)4 * P;
    std::vector<std::vector<long long>> cix(G + 1, std::vector<long long>(2 * cp));
    std::vector<std::vector<int>> crank(G + 1, std::vector<int>(cp));
    std::vector<HaloCorners> corners(G + 1); // [G]: the single buffer
    for (int r = 0; r <= G; r++) {
        int n[2];
        halo_corner_items(P, r < G ? G : 1, r < G ? r : 0, corner_ids, corner_starts, bx.ex, bx.ey, off.data(),
            cix[r].data(), cix[r].data() + cp, crank[r].data(), n);
        corners[r] = HaloCorners { cix[r].data(), cix[r].data() + cp, crank[r].data(), n[periodic ? 1 : 0] };
    }
    std::vector<std::vector<int>> rank_t(G);
    std::vector<std::vector<long long>> rank_b(G);
    std::vector<HaloItems> rank_items(G);
    for (int r = 0; r < G; r++)
        rank_items[r] = table(G, rows_b[r], rows_b[r] + rows_c[r], rank_t[r], rank_b[r]);

    // the ranks' halo buffers (head + tiles, 256-byte aligned like cudaMalloc), rows with guard bands, error words
    const size_t head = HALO_HEAD_BYTES / sizeof(double), guard = (size_t)nx + 40;
    const double GUARD = -1234.5;
    std::vector<std::vector<double>> buf(G), rows(G), src(G);
    std::vector<char*> base(G);
    std::vector<int> pb(G), pc(G), err(G, 0);
    for (int r = 0; r < G; r++) {
        pb[r] = (int)((long long)r * P / G);
        pc[r] = (int)((long long)(r + 1) * P / G) - pb[r];
        buf[r].assign(head + (size_t)(off[pb[r] + pc[r]] - off[pb[r]]) + 32, 0.0);
        char* b = reinterpret_cast<char*>(buf[r].data());
        while ((uintptr_t)b % 256)
            b += 8;
        base[r] = b;
        std::memcpy(b + HALO_HEAD_BYTES, tiles_in + off[pb[r]], sizeof(double) * (size_t)(off[pb[r] + pc[r]] - off[pb[r]]));
        const size_t n = (size_t)rows_c[r] * nx;
        rows[r].assign(n + 2 * guard, GUARD);
        src[r].assign(n + 2 * guard, GUARD);
        std::memcpy(rows[r].data() + guard, rows_in + (size_t)rows_b[r] * nx, sizeof(double) * n);
        std::memcpy(src[r].data() + guard, field + (size_t)rows_b[r] * nx, sizeof(double) * n);
    }
    std::vector<double> single(tiles_in, tiles_in + total), single_field(rows_in, rows_in + cells),
        single_src(field, field + cells);
    unsigned step = 0;
    auto shards_of = [&](int r) {
        HaloShards hs {};
        hs.ps.rank = r;
        hs.ps.G = G;
        hs.ps.enabled = 1;
        hs.ps.step = step;
        for (int q = 0; q < G; q++) {
            hs.ps.flags[q] = reinterpret_cast<unsigned*>(base[q]);
            hs.tiles[q] = reinterpret_cast<double*>(base[q] + HALO_HEAD_BYTES);
        }
        hs.done = reinterpret_cast<unsigned*>(base[r]) + 2 * MAX_PEERS;
        hs.opened = hs.done + 1;
        hs.err = &err[r];
        hs.P = P;
        hs.p_begin = pb[r];
        hs.p_count = pc[r];
        return hs;
    };
    const unsigned lists = periodic ? 0xffu : 0x0fu;
    const int nops = (int)std::strlen(ops);
    for (int i = 0; i < nops; i++) {
        const char op = ops[i];
        if (op != 's' && op != 'x' && op != 'g' && op != 'f') {
            g_err = std::string("unknown op ") + op;
            return -1;
        }
        const bool exchange = op == 'x' || op == 'f';
        if (!exchange || have_nbr) { // (an exchange without neighbour tables takes no step: ddc_api.cu returns first)
            step++;
            for (int phase = 1; phase <= 2; phase++)
                for (int r = 0; r < G; r++)
                    if (r != stall)
                        LAUNCH(Dim3(1), Dim3(32), k_halo_open(shards_of(r), phase));
            for (int r = 0; r < G; r++) {
                if (r == stall)
                    continue;
                if (op == 'x')
                    LAUNCH(Dim3(std::max(1, std::min(pc[r], GRID_MAX))), Dim3(256),
                        k_halo_push(shards_of(r), bx, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(),
                            off.data(), lists));
                else if (op == 'f')
                    LAUNCH(Dim3(std::max(1, std::min(std::max(pc[r], (corners[r].n + 255) / 256), GRID_MAX))), Dim3(256),
                        k_halo_push_full(shards_of(r), bx, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(),
                            off.data(), lists, corners[r]));
                else if (op == 's')
                    LAUNCH(Dim3(grid_of(rank_items[r])), Dim3(256),
                        k_halo_field_shards<true>(shards_of(r), rank_items[r], bx, src[r].data() + guard, nx, rows_b[r]));
                else
                    LAUNCH(Dim3(grid_of(rank_items[r])), Dim3(256),
                        k_halo_field_shards<false>(shards_of(r), rank_items[r], bx, rows[r].data() + guard, nx, rows_b[r]));
            }
            for (int r = 0; r < G; r++)
                if (r != stall)
                    LAUNCH(Dim3(1), Dim3(32), k_halo_close(shards_of(r)));
        }
        if (exchange && have_nbr) {
            const long long warps = 8LL * P;
            LAUNCH(Dim3((unsigned)((warps * 32 + 255) / 256)), Dim3(256),
                k_halo_exchange<double>(bx, P, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(), off.data(),
                    single.data(), lists));
            if (op == 'f' && corners[G].n > 0)
                LAUNCH(Dim3((unsigned)std::min((corners[G].n + 255) / 256, GRID_MAX)), Dim3(256),
                    k_halo_corners(corners[G], single.data()));
        } else if (op == 's')
            LAUNCH(Dim3(grid_of(single_items)), Dim3(256), k_halo_field<true>(single_items, bx, single.data(), single_src.data(), nx));
        else if (op == 'g')
            LAUNCH(Dim3(grid_of(single_items)), Dim3(256), k_halo_field<false>(single_items, bx, single.data(), single_field.data(), nx));
        for (int r = 0; r < G; r++) {
            std::memcpy(tiles_out + (size_t)i * total + off[pb[r]], base[r] + HALO_HEAD_BYTES,
                sizeof(double) * (size_t)(off[pb[r] + pc[r]] - off[pb[r]]));
            std::memcpy(rows_out + (size_t)i * cells + (size_t)rows_b[r] * nx, rows[r].data() + guard,
                sizeof(double) * (size_t)rows_c[r] * nx);
            if (r != stall && reinterpret_cast<unsigned*>(base[r])[2 * MAX_PEERS] != 0u) {
                g_err = "rank " + std::to_string(r) + " left its block counter set after op " + std::to_string(i);
                return -1;
            }
            for (size_t k = 0; k < guard; k++)
                for (const std::vector<double>* v : { &rows[r], &src[r] })
                    if ((*v)[k] != GUARD || (*v)[v->size() - 1 - k] != GUARD) {
                        g_err = "rank " + std::to_string(r) + " wrote outside its rows in op " + std::to_string(i);
                        return -1;
                    }
        }
        std::memcpy(single_out + (size_t)i * total, single.data(), sizeof(double) * (size_t)total);
        std::memcpy(field_out + (size_t)i * cells, single_field.data(), sizeof(double) * cells);
    }
    for (int r = 0; r < G; r++)
        err_out[r] = err[r];
    return 0;
}
}
