// inflate_kernels.cuh -- sm_100a BGZF inflate (device side of msnv_inflate, include/msnv.h).
//
// inflate_kernel: one warp per member. DEFLATE's symbols form one serial bit stream, so lane 0 builds the Huffman tables
// in the warp's slice of shared memory and decodes symbols (inflate_member.h, msnv_inflate_step: the code the CPU tests
// check against zlib), writing literals at once and queueing up to 32 checked matches. The warp then copies the queued
// matches in order, a lane per byte (a match of length L takes ceil(L / 32) steps, whatever its distance), while lane 0
// waits; then lane 0 decodes on. At the end every lane takes 1/32 of the member's bytes, computes their CRC-32, shifts it
// to the end of the member (msnv_crc32_shift) and the warp XORs the 32 pieces into the member's CRC, which is compared
// with the trailer. Residency is bound by the ~8.8 KB of tables and queue per member: see DESIGN.md §3.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "inflate_member.h"

namespace msnv_gpu {

constexpr int INFLATE_WARPS = 4;                // warps (members in flight) per CTA
constexpr uint32_t INFLATE_QUEUE = 32;          // matches lane 0 queues before the warp copies them

__global__ void __launch_bounds__(INFLATE_WARPS * 32)
inflate_kernel(const uint8_t* __restrict__ comp, const msnv_bgzf_member* __restrict__ members, uint32_t n,
               uint8_t* __restrict__ out, int32_t* __restrict__ status)
{
    __shared__ MsnvInflateScratch scratch[INFLATE_WARPS];
    __shared__ MsnvInfMatch queue[INFLATE_WARPS][INFLATE_QUEUE];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t i = blockIdx.x * INFLATE_WARPS + warp;
    if (i >= n) return;
    const msnv_bgzf_member m = members[i];
    uint8_t* dst = out + m.ooff;
    MsnvInfState st;
    if (lane == 0) msnv_inflate_begin(st, comp + m.coff, m.clen);
    int r;
    do {
        uint32_t nq = 0;
        r = 0;
        if (lane == 0) r = msnv_inflate_step(st, dst, m.isize, &scratch[warp], queue[warp], INFLATE_QUEUE, &nq);
        r = __shfl_sync(0xffffffffu, r, 0);
        nq = __shfl_sync(0xffffffffu, nq, 0);
        __syncwarp();                               // lane 0's literals and queue are visible to the warp from here
        for (uint32_t k = 0; k < nq; ++k) {
            const MsnvInfMatch q = queue[warp][k];
            for (uint32_t j = lane; j < q.len; j += 32) msnv_inf_match_byte(dst, q, j);
            __syncwarp();                           // a later match may read this one's bytes
        }
    } while (r == MSNV_INF_RUNNING);
    if (r == MSNV_INFLATE_OK) {
        const uint32_t piece = (m.isize + 31) / 32;
        const uint32_t lo = min(m.isize, lane * piece), hi = min(m.isize, lo + piece);
        uint32_t c = msnv_crc32_shift(msnv_crc32_piece(dst + lo, hi - lo), m.isize - hi);
        for (int k = 16; k; k >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, k);
        if (c != m.crc) r = MSNV_INFLATE_BAD_CRC;
    }
    if (lane == 0) status[i] = r;
}

}  // namespace msnv_gpu
