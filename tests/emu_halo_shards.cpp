// emu_halo_shards.cpp -- TEST INFRASTRUCTURE.  The sharded halo exchange (ddc_halo_exchange_shards_f64) through the
// product's REAL kernels (k_halo_open, k_halo_push, k_halo_close of ddc_kernels.cuh compiled with -DDDC_HOST_EMU) on
// the host emulation of the CUDA execution model, for G emulated ranks.  The buffers and launches follow ddc_api.cu:
// each rank's buffer is [HALO_HEAD_BYTES head][tiles of its parts], the kernels receive every rank's buffer as
// "mapped" and push into them.  The ranks run phase by phase (all signal R, all wait for R, all push, all wait for D),
// as oracle/emu/emu_pipeline.cpp runs the decomposition's kernels.  Beside the ranks, k_halo_exchange runs on one buffer holding
// all parts, the single-GPU exchange the sharded one must reproduce bit for bit.  It says nothing about speed.
// Compiled by tests/halo_emu.py (into a temporary directory) against oracle/emu/cuda_emu.cpp, the fiber emulation.
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
// periodic * 4 + edge, each the concatenation over parts of the part's id-ascending list), as oracle.Neighbours.
// tiles_in[nsteps][total]: before exchange k the INTERIORS of tiles_in[k] are copied into the buffers (the whole tiles
// before the first), so that a ghost not written by exchange k keeps whatever it held.
// tiles_out[nsteps][total]: the ranks' buffers concatenated in rank order after each exchange; single_out the same
// for k_halo_exchange on one buffer.  stall: a rank that runs none of the kernels (-1: none).  err_out[G]: the error
// word of every rank after the last exchange.  Returns 0, or -1 (emu_halo_last_error()).
__attribute__((visibility("default"))) int emu_halo_shards(int P, const int32_t* boxes, const int32_t* counts,
    const int32_t* ids, const int32_t* halos, const int32_t* starts, int G, int periodic, int nsteps, int stall,
    const double* tiles_in, double* tiles_out, double* single_out, int32_t* err_out)
{
    g_err.clear();
    if (const char* e = std::getenv("DDC_EMU_SCHED_SEED"))
        cuda_emu::set_schedule_seed(std::strtoull(e, nullptr, 10));
    else
        cuda_emu::set_schedule_seed(0);
    if (P < 1 || G < 1 || G > MAX_PEERS || nsteps < 1) {
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
    BoxTable bx = { bxv.data(), bxv.data() + P, bxv.data() + 2 * P, bxv.data() + 3 * P };
    std::vector<long long> off((size_t)P + 1, 0);
    for (int p = 0; p < P; p++)
        off[p + 1] = off[p] + (long long)(bxv[(size_t)2 * P + p] + 2) * (bxv[(size_t)3 * P + p] + 2);
    const long long total = off[P];

    // the ranks' buffers (head + tiles, 256-byte aligned like cudaMalloc), their error words
    const size_t head = HALO_HEAD_BYTES / sizeof(double);
    std::vector<std::vector<double>> buf(G);
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
    }
    auto shards_of = [&](int r, unsigned step) {
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
    std::vector<double> single((size_t)total);
    const unsigned lists = periodic ? 0xffu : 0x0fu;
    for (int k = 0; k < nsteps; k++) {
        const double* in = tiles_in + (size_t)k * total;
        for (int p = 0; p < P; p++) { // interiors (whole tiles before the first exchange)
            const int ex = bxv[(size_t)2 * P + p], ey = bxv[(size_t)3 * P + p];
            const int r = (int)(((long long)(p + 1) * G - 1) / P);
            double* mine = reinterpret_cast<double*>(base[r] + HALO_HEAD_BYTES) + (off[p] - off[pb[r]]);
            for (int y = 0; y < ey + 2; y++)
                for (int x = 0; x < ex + 2; x++) {
                    const bool interior = y >= 1 && y <= ey && x >= 1 && x <= ex;
                    if (k == 0 || interior) {
                        const size_t i = (size_t)y * (ex + 2) + x;
                        mine[i] = in[off[p] + i];
                        single[off[p] + i] = in[off[p] + i];
                    }
                }
        }
        const unsigned step = (unsigned)k + 1;
        for (int phase = 1; phase <= 2; phase++)
            for (int r = 0; r < G; r++)
                if (r != stall)
                    LAUNCH(Dim3(1), Dim3(32), k_halo_open(shards_of(r, step), phase));
        for (int r = 0; r < G; r++)
            if (r != stall)
                LAUNCH(Dim3(std::max(1, pc[r])), Dim3(256),
                    k_halo_push(shards_of(r, step), bx, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(),
                        off.data(), lists));
        for (int r = 0; r < G; r++)
            if (r != stall)
                LAUNCH(Dim3(1), Dim3(32), k_halo_close(shards_of(r, step)));
        const long long warps = 8LL * P;
        LAUNCH(Dim3((unsigned)((warps * 32 + 255) / 256)), Dim3(256),
            k_halo_exchange<double>(bx, P, cnt.data(), offs.data(), cap, vid.data(), vh.data(), vs.data(), off.data(),
                single.data(), lists));
        double* out = tiles_out + (size_t)k * total;
        for (int r = 0; r < G; r++)
            std::memcpy(out + off[pb[r]], base[r] + HALO_HEAD_BYTES, sizeof(double) * (size_t)(off[pb[r] + pc[r]] - off[pb[r]]));
        std::memcpy(single_out + (size_t)k * total, single.data(), sizeof(double) * (size_t)total);
        for (int r = 0; r < G; r++) // the block counter is zero between exchanges
            if (r != stall && reinterpret_cast<unsigned*>(base[r])[2 * MAX_PEERS] != 0u) {
                g_err = "rank " + std::to_string(r) + " left its block counter set";
                return -1;
            }
    }
    for (int r = 0; r < G; r++)
        err_out[r] = err[r];
    return 0;
}
}
