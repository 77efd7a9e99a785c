// emu_halo.cpp -- TEST INFRASTRUCTURE.  The halo calls (scatter, edge exchange, full-frame exchange and gather, on
// one buffer and sharded) with frames of width w (ddc_halo_set_width), through the product's REAL kernels and host code
// (halo_plan with the width and halo_shards; at w = 1 k_halo_exchange + k_halo_corners on one buffer and k_halo_push /
// k_halo_push_full between k_halo_open and k_halo_close on the shards, at w >= 2 k_halo_rects and k_halo_push_rects;
// k_halo_field / k_halo_field_shards at the width; ddc_kernels.cuh compiled with -DDDC_HOST_EMU) on the host emulation
// of the CUDA execution model, for G emulated ranks on one halo step counter.  The buffers and launches follow
// ddc_api.cu: each rank's buffer is [HALO_HEAD_BYTES head][tiles of its parts], every tile sized for the width, and the
// kernels receive every rank's buffer as "mapped" and push into them.  The ranks run phase by phase (all signal R, all
// wait for R, all run the middle kernel, all wait for D), as oracle/emu/emu_pipeline.cpp runs the decomposition's
// kernels.  Beside them the single-buffer kernels run on one buffer holding all parts and one whole field.  Every rank's
// rows live in an allocation of their own with a guard band on either side, so a store outside the rank's block is
// seen.  It says nothing about speed.  Compiled by tests/halo_emu.py (into a temporary directory) against
// oracle/emu/cuda_emu.cpp.
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
}

#define LAUNCH(grid, block, call)                                                                  \
    do {                                                                                           \
        if (!cuda_emu::launch(grid, block, 0, [&] { call; })) {                                    \
            g_err = std::string(#call) + ": " + cuda_emu::last_error();                            \
            return -1;                                                                             \
        }                                                                                          \
    } while (0)

extern "C" {
__attribute__((visibility("default"))) const char* emu_halo_last_error(void) { return g_err.c_str(); }

// boxes[P][4] = x0 y0 ex ey; counts[8][P]; ids / halos / starts: the eight lists one after the other (list l =
// periodic * 4 + edge, each the concatenation over parts of the part's id-ascending list), as oracle.Neighbours (used
// by 'x' and 'f'); px / py: the decomposition's periodic flags (the corner table).  rows_b[G], rows_c[G]: every rank's
// ddc_shard_rows block.  ops: a string of 's' (scatter), 'x' (edge exchange), 'f' (full-frame exchange), 'g' (gather),
// run in order on the sharded buffers AND on the single buffer, with one halo step counter.
// grid_cap: 0 the library's grids, else at most that many blocks for the grid-stride kernels (few blocks: the loops
// and the block counter see several rounds and blocks).
// corner_ids / corner_starts [2][4][P]: the plan's corner table (ddc_get_corner_neighbours).  w: the frame width
// (ddc_halo_set_width); at w >= 2 the exchanges run k_halo_rects / k_halo_push_rects, as ddc_api.cu does.
// fields[k][ny * nx]: what each rank's rows hold for the k-th scatter (rank r: rows rows_b[r] ...), and what the
// single-buffer scatter reads.  tiles_in[total]: the tiles before the first op (every buffer); rows_in[ny * nx]: the
// rows (and the single-buffer field) a gather writes into before the first op.  After op i: tiles_out[i] = the ranks'
// buffers concatenated, single_out[i] = the single buffer, rows_out[i] = the ranks' rows concatenated, field_out[i] =
// the single-buffer field.  stall: a rank that runs none of the kernels (-1: none).  err_out[G]: the error words at
// the end.  Returns 0, or -1 (emu_halo_last_error()).
__attribute__((visibility("default"))) int emu_halo(int P, const int32_t* boxes, const int32_t* counts,
    const int32_t* ids, const int32_t* halos, const int32_t* starts, int nx, int ny, int px, int py, int G,
    const int32_t* rows_b, const int32_t* rows_c, int periodic, const char* ops, int stall, int grid_cap,
    const double* fields, const double* tiles_in, const double* rows_in, double* tiles_out, double* single_out,
    double* rows_out, double* field_out, int32_t* err_out, int32_t* corner_ids, int32_t* corner_starts, int w)
{
    g_err.clear();
    if (const char* e = std::getenv("DDC_EMU_SCHED_SEED"))
        cuda_emu::set_schedule_seed(std::strtoull(e, nullptr, 10));
    else
        cuda_emu::set_schedule_seed(0);
    if (P < 1 || G < 1 || G > MAX_PEERS || nx < 1 || ny < 1 || w < 1) {
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

    // every rank's halo plan, as ddc_api.cu's tile_offsets() builds it; the single buffer uses view 0 of rank 0's
    std::vector<HaloPlan> plan(G);
    for (int r = 0; r < G; r++)
        plan[r] = halo_plan(P, G, r, nx, ny, px, py, bx.x0, bx.y0, bx.ex, bx.ey, rows_b[r], rows_c[r], w);
    std::memcpy(corner_ids, plan[0].corner_ids.data(), sizeof(int32_t) * 8 * P);
    std::memcpy(corner_starts, plan[0].corner_starts.data(), sizeof(int32_t) * 8 * P);
    const long long* off = plan[0].off();
    const long long total = off[P];
    const size_t cells = (size_t)nx * ny;
    const auto grid = [&](unsigned g) { return Dim3(grid_cap > 0 ? std::min(g, (unsigned)grid_cap) : g); };

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
    }
    std::vector<double> single(tiles_in, tiles_in + total), single_field(rows_in, rows_in + cells), single_src(cells);
    void* single_plan = plan[0].block.data();
    const HaloItems single_items = plan[0].items(single_plan, 0);
    const HaloCorners single_corners = plan[0].corners(single_plan, 0, periodic);
    unsigned step = 0;
    const unsigned lists = periodic ? 0xffu : 0x0fu;
    const int nops = (int)std::strlen(ops);
    for (int i = 0, scatters = 0; i < nops; i++) {
        const char op = ops[i];
        if (op != 's' && op != 'x' && op != 'g' && op != 'f') {
            g_err = std::string("unknown op ") + op;
            return -1;
        }
        if (op == 's') { // this scatter's field
            const double* field = fields + (size_t)scatters++ * cells;
            for (int r = 0; r < G; r++)
                std::memcpy(src[r].data() + guard, field + (size_t)rows_b[r] * nx, sizeof(double) * rows_c[r] * nx);
            single_src.assign(field, field + cells);
        }
        const bool exchange = op == 'x' || op == 'f';
        if (!exchange || have_nbr) { // (an exchange without neighbour tables takes no step: ddc_api.cu returns first)
            step++;
            std::vector<HaloShards> hs(G);
            for (int r = 0; r < G; r++)
                hs[r] = halo_shards(P, G, r, step, base.data(), &err[r]);
            for (int phase = 1; phase <= 2; phase++)
                for (int r = 0; r < G; r++)
                    if (r != stall)
                        LAUNCH(Dim3(1), Dim3(32), k_halo_open(hs[r], phase));
            for (int r = 0; r < G; r++) {
                if (r == stall)
                    continue;
                void* at = plan[r].block.data();
                const HaloItems items = plan[r].items(at, 1);
                const HaloCorners corners = plan[r].corners(at, 1, periodic);
                const HaloRects rects = plan[r].rects(at, 1, periodic, op == 'f');
                if (exchange && w > 1)
                    LAUNCH(grid(halo_field_grid(rects.n)), Dim3(256), k_halo_push_rects(hs[r], rects));
                else if (op == 'x')
                    LAUNCH(grid(halo_push_grid(pc[r], 0)), Dim3(256),
                        k_halo_push(hs[r], bx, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(), off, lists));
                else if (op == 'f')
                    LAUNCH(grid(halo_push_grid(pc[r], corners.n)), Dim3(256),
                        k_halo_push_full(hs[r], bx, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(), off,
                            lists, corners));
                else if (op == 's')
                    LAUNCH(grid(halo_field_grid(plan[r].items_total[1])), Dim3(256),
                        k_halo_field_shards<true>(hs[r], items, bx, src[r].data() + guard, nx, rows_b[r]));
                else
                    LAUNCH(grid(halo_field_grid(plan[r].items_total[1])), Dim3(256),
                        k_halo_field_shards<false>(hs[r], items, bx, rows[r].data() + guard, nx, rows_b[r]));
            }
            for (int r = 0; r < G; r++)
                if (r != stall)
                    LAUNCH(Dim3(1), Dim3(32), k_halo_close(hs[r]));
        }
        if (exchange && have_nbr && w > 1) {
            const HaloRects rects = plan[0].rects(single_plan, 0, periodic, op == 'f');
            if (rects.n > 0)
                LAUNCH(grid(halo_field_grid(rects.n)), Dim3(256), k_halo_rects(rects, single.data()));
        } else if (exchange && have_nbr) {
            LAUNCH(Dim3(halo_exchange_grid(P)), Dim3(256), // (not grid-stride: never capped)
                k_halo_exchange<double>(bx, P, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(), off,
                    single.data(), lists));
            if (op == 'f' && single_corners.n > 0)
                LAUNCH(grid(halo_corner_grid(single_corners.n)), Dim3(256), k_halo_corners(single_corners, single.data()));
        } else if (op == 's')
            LAUNCH(grid(halo_field_grid(plan[0].items_total[0])), Dim3(256),
                k_halo_field<true>(single_items, bx, single.data(), single_src.data(), nx));
        else if (op == 'g')
            LAUNCH(grid(halo_field_grid(plan[0].items_total[0])), Dim3(256),
                k_halo_field<false>(single_items, bx, single.data(), single_field.data(), nx));
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
