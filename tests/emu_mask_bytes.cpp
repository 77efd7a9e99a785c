// emu_mask_bytes.cpp -- TEST INFRASTRUCTURE.  Emulated multi-rank decompositions in which chosen ranks scan a byte
// mask (k_scan_mask_u8) and the others the int32 mask (k_scan_mask).
//
// This is oracle/emu/emu_pipeline.cpp -- the launch sequence of ddc_api.cu on G emulated ranks, unchanged -- with
// its mask-scan launch routed through scan_dispatch below: a rank that has a byte shard scans it with the byte
// kernel, with the same grid and arguments, and the pipeline after the scan runs as it always does.  Every byte
// shard is an allocation of exactly `offset + rows * nx` bytes with the rows at `offset`, so an AddressSanitizer
// build sees a read past the last row's nx bytes.
#include "cuda_emu.h"
#include "ddc_kernels.cuh"

#include <cstdlib>
#include <cstring>

namespace {
const uint8_t* g_u8[ddc::MAX_PEERS]; // rank -> its byte rows (nullptr: the rank scans the int32 mask)

template <bool VEC>
void scan_dispatch(const int32_t* mask, int NX, int rows, int y_begin, int NB, int rpc, uint8_t* bits, unsigned* colcount,
    int* yr, ddc::PeerPush push, ddc::PeerSync ps, unsigned* done, int yr_off, unsigned long long* dbg, int nbig, int small)
{
    if (const uint8_t* m = g_u8[ps.rank]) { // (the condition ddc_api.cu uses for the byte kernel)
        if (NX % 4 == 0 && (uintptr_t)m % 4 == 0)
            ddc::k_scan_mask_u8<true>(m, NX, rows, y_begin, NB, rpc, bits, colcount, yr, push, ps, done, yr_off, dbg, nbig, small);
        else
            ddc::k_scan_mask_u8<false>(m, NX, rows, y_begin, NB, rpc, bits, colcount, yr, push, ps, done, yr_off, dbg, nbig, small);
    } else
        ddc::k_scan_mask<VEC>(mask, NX, rows, y_begin, NB, rpc, bits, colcount, yr, push, ps, done, yr_off, dbg, nbig, small);
}
} // namespace

#define k_scan_mask scan_dispatch
#include "emu_pipeline.cpp"
#undef k_scan_mask

extern "C" {
// bytes[NY][NX]: the byte mask; ranks whose bit is set in u8_ranks scan their rows of it, the others scan the int32
// mask passed to emu_partition.  offset: where the rows start in each byte shard's allocation (0..15).  The shards
// live until the next call.
__attribute__((visibility("default"))) int emu_set_byte_mask(const uint8_t* bytes, int NX, int NY, int G, unsigned u8_ranks,
    int offset)
{
    static uint8_t* shard[MAX_PEERS];
    for (int g = 0; g < MAX_PEERS; g++) {
        std::free(shard[g]);
        shard[g] = nullptr;
        g_u8[g] = nullptr;
    }
    if (G < 1 || G > MAX_PEERS || offset < 0 || offset > 15)
        return -1;
    const int rpr = (NY + G - 1) / G;
    for (int g = 0; g < G; g++) {
        if (!(u8_ranks >> g & 1u))
            continue;
        const int b = std::min(NY, g * rpr), e = std::min(NY, b + rpr);
        const size_t n = (size_t)(e - b) * NX;
        shard[g] = static_cast<uint8_t*>(std::malloc(offset + n + (offset + n == 0))); // malloc: 16-byte aligned
        std::memcpy(shard[g] + offset, bytes + (size_t)b * NX, n);
        g_u8[g] = shard[g] + offset;
    }
    return 0;
}
}
