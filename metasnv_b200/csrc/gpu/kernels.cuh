// kernels.cuh -- sm_100a kernels of the pileup + call path (device side of include/msnv.h).
//
// Data flow for one shard (all samples of one genome bin, see DESIGN.md):
//   index_kernel     (tile, sample) pairs that have reads  -> ordered work items (ballot compaction)
//   pileup_kernel    persistent CTAs: a producer warp stages the items' position-aligned reads through a
//                    ring of TMA bulk copies; consumer warps apply the mate-overlap quality correction
//                    (SURVEY.md Annex A.2) in shared memory and scatter sixteen positions per thread and
//                    step into byte-lane count planes -> 6 B per sample-position     [dominant kernel]
//   call_kernel      per tile: reduce over samples, snpCall thresholds (call_vC.cpp:545-601)
//   compact_kernel   ordered stream compaction of called positions (warp ballot + block scan)
//   gather_kernel    per hit: per-sample coverage / allele counts for the host formatter
//
// The reference computes the same quantities one text character at a time
// (call_vC.cpp:503-535 over the columns rendered by `samtools mpileup`).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/msnv.h"
#include "overlap_rule.h"

namespace msnv_gpu {

constexpr int TILE = MSNV_TILE;                 // positions per tile

struct SampleDev {
    const int32_t*  pos;
    const uint32_t* seg_off;
    const uint32_t* q4_off;
    const int32_t*  mate;
    const int32_t*  seg_pos;
    const uint16_t* seg_len;
    const uint8_t*  seq2;
    const uint8_t*  qual;
    uint8_t*        fix;          // samples with mate links: per quad, the verdict of the mate-overlap rule (mate_kernel), else null
    uint32_t        n_reads, max_span;
};

struct Item { uint32_t sample, tile, r_lo, r_hi; };   // reads [r_lo, r_hi) of `sample` may overlap `tile`

// Per-position population result of call_kernel.
struct CallParamsDev { int32_t min_cov; int32_t thr; double frac; };

// ------------------------------------------------------------------------------------------------
// small PTX helpers (mbarrier + 1-D TMA bulk copy), see blackwell_cuda_programming.md G3/G15
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
// global -> shared bulk copy (TMA, SASS UBLKCP); dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ uint32_t lower_bound_i32(const int32_t* __restrict__ a, uint32_t n, int64_t key)
{
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if ((int64_t)__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// lower_bound_i32 when the answer is expected near `guess`: gallop away from the guess in doubling steps,
// then bisect the bracket. A good guess costs ~8 probes that share one or two cache lines instead of
// log2(n) scattered ones; a bad one costs 2*log2(error).
__device__ __forceinline__ uint32_t lower_bound_near_i32(const int32_t* __restrict__ a, uint32_t n, int64_t key, uint32_t guess)
{
    uint32_t lo, hi, cur = guess < n ? guess : n, step = 16;
    if (cur < n && (int64_t)__ldg(a + cur) < key) {            // the answer lies above the guess
        lo = cur + 1;
        for (;;) {
            const uint32_t c = cur + step;
            if (c >= n) { hi = n; break; }
            if ((int64_t)__ldg(a + c) >= key) { hi = c; break; }
            lo = c + 1; cur = c; step <<= 1;
        }
    } else {                                                   // at or below it
        hi = cur;
        for (;;) {
            if (cur < step) { lo = 0; break; }
            const uint32_t c = cur - step;
            if ((int64_t)__ldg(a + c) < key) { lo = c + 1; break; }
            hi = c; cur = c; step <<= 1;
        }
    }
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if ((int64_t)__ldg(a + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Block-wide exclusive rank of `flag` among the block's threads (thread order) and the block total.
// blockDim.x must be a multiple of 32 and at most 1024.
__device__ __forceinline__ uint32_t block_rank(bool flag, uint32_t* s_warp /*[33]*/, uint32_t& total)
{
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    uint32_t bal = __ballot_sync(0xffffffffu, flag);
    uint32_t r = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        uint32_t v = lane < nwarp ? s_warp[lane] : 0;
        uint32_t incl = v;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        s_warp[lane] = incl - v;
        if (lane == 31) s_warp[32] = incl;
    }
    __syncthreads();
    total = s_warp[32];
    uint32_t base = s_warp[warp];
    __syncthreads();
    return base + r;
}

// ------------------------------------------------------------------------------------------------
// index: which (tile, sample) pairs have reads. Pairs are enumerated tile-major so that the
// compacted item list is grouped by tile (call_kernel reads one contiguous run of slots per tile).
// Two passes over the same predicate: COUNT writes per-block totals, EMIT writes the items at the
// scanned offsets (ordered stream compaction by warp ballot).
// ------------------------------------------------------------------------------------------------
// Occupancy bitmap for sparse shards (most (tile, sample) pairs have no reads at all, e.g. a sample that
// carries 10 % of the genomes of its bin): one bit per (sample, tile), set for the tile a read starts in.
// index_kernel then skips the two binary searches of every pair whose tile and the tiles a read could
// reach it from are all clear.
__global__ void __launch_bounds__(256) mark_kernel(const SampleDev* __restrict__ samples, uint32_t words_per_sample,
                                                   uint32_t tile0, uint32_t n_tiles, uint32_t* __restrict__ bitmap)
{
    const SampleDev sd = samples[blockIdx.y];
    uint32_t* bm = bitmap + (size_t)blockIdx.y * words_per_sample;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < sd.n_reads; i += gridDim.x * blockDim.x) {
        // tile of the window the read starts in; reads that start in front of the window (they reach into it) count for its
        // first tile, reads behind it for none
        const int64_t ta = (int64_t)__ldg(sd.pos + i) / TILE - (int64_t)tile0;
        if (ta >= (int64_t)n_tiles) continue;
        const uint32_t t = ta < 0 ? 0u : (uint32_t)ta;
        // consecutive reads mostly share a tile: one atomic per (warp, tile)
        const uint32_t peers = __match_any_sync(__activemask(), t);
        if ((threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicOr(bm + (t >> 5), 1u << (t & 31));
    }
}

// The index searches every sample's `pos`: refuse samples whose reads are not in coordinate order (err_flag = 3).
__global__ void __launch_bounds__(256) order_check_kernel(const SampleDev* __restrict__ samples, int* __restrict__ err_flag)
{
    const SampleDev sd = samples[blockIdx.y];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i + 1 < sd.n_reads; i += gridDim.x * blockDim.x)
        if (__ldg(sd.pos + i) > __ldg(sd.pos + i + 1)) atomicExch(err_flag, 3);
}

template <bool EMIT>
__global__ void __launch_bounds__(256) index_kernel(const SampleDev* __restrict__ samples, uint32_t n_samples,
                                                    uint32_t tile0 /* first tile of the window */, uint32_t n_tiles /* tiles of the window */,
                                                    uint32_t* __restrict__ block_sums,
                                                    Item* __restrict__ items, uint32_t* __restrict__ tile_begin,
                                                    uint2* __restrict__ range_cache /* [tiles*samples] or null: COUNT stores, EMIT reloads */,
                                                    const uint32_t* __restrict__ bitmap /* mark_kernel's, or null */, uint32_t words_per_sample,
                                                    unsigned long long* __restrict__ item_reads /* COUNT: [0] sum, [1] maximum of r_hi - r_lo over the items */)
{
    __shared__ uint32_t s_warp[33];
    const uint64_t pair = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    const uint64_t n_pairs = (uint64_t)n_tiles * n_samples;
    bool active = false;
    uint32_t s = 0, t = 0, r_lo = 0, r_hi = 0;
    if (pair < n_pairs) {
        t = (uint32_t)(pair / n_samples);
        s = (uint32_t)(pair - (uint64_t)t * n_samples);
        if (EMIT && range_cache) {
            const uint2 c = range_cache[pair];
            r_lo = c.x; r_hi = c.y;
        } else {
            const uint32_t n = samples[s].n_reads;
            bool maybe = n != 0;
            if (maybe && bitmap) {                       // any read starting in a tile that can reach tile t?
                const uint32_t back = (samples[s].max_span + TILE - 2) / TILE;      // tiles a read can reach back from
                const uint32_t* bm = bitmap + (size_t)s * words_per_sample;
                maybe = false;
                for (uint32_t u = t >= back ? t - back : 0; u <= t && !maybe; ++u) maybe = (__ldg(bm + (u >> 5)) >> (u & 31)) & 1u;
            }
            if (maybe) {
                const int32_t* pos = samples[s].pos;
                const int64_t t0 = (int64_t)(tile0 + t) * TILE, k_lo = t0 - (int64_t)samples[s].max_span + 1;
                if (bitmap) {
                    // sparse shard: the sample covers a few contigs of many, its read density is anything but even
                    r_lo = lower_bound_i32(pos, n, k_lo);
                    r_hi = lower_bound_near_i32(pos, n, t0 + TILE, r_lo + 32);          // ... but the end is close to the start
                } else {
                    // reads are spread fairly evenly over what the sample covers: interpolate, then search near the guess
                    const int64_t first = __ldg(pos), extent = (int64_t)__ldg(pos + n - 1) - first + 1;
                    const int64_t g = k_lo <= first ? 0 : (k_lo - first) * (int64_t)n / extent;
                    r_lo = lower_bound_near_i32(pos, n, k_lo, (uint32_t)(g < (int64_t)n ? g : (int64_t)n));
                    const int64_t w = ((int64_t)TILE + samples[s].max_span) * (int64_t)n / extent;
                    r_hi = lower_bound_near_i32(pos, n, t0 + TILE, r_lo + (uint32_t)(w < (int64_t)n ? w : (int64_t)n));
                }
            }
            if (!EMIT && range_cache) range_cache[pair] = make_uint2(r_lo, r_hi);
        }
        active = r_hi > r_lo;
    }
    uint32_t total;
    uint32_t rank = block_rank(active, s_warp, total);
    if (!EMIT) {
        if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
        // reads staged over all items: sizes the pileup kernel's staging buffers
        uint32_t nr = active ? r_hi - r_lo : 0u, nmax = nr;
        #pragma unroll
        for (int d = 16; d > 0; d >>= 1) { nr += __shfl_down_sync(0xffffffffu, nr, d); nmax = max(nmax, __shfl_down_sync(0xffffffffu, nmax, d)); }
        if ((threadIdx.x & 31) == 0 && nr) { atomicAdd(item_reads, (unsigned long long)nr); atomicMax(item_reads + 1, (unsigned long long)nmax); }
    } else {
        const uint32_t slot = block_sums[blockIdx.x] + rank;     // block_sums holds exclusive offsets now
        if (active) items[slot] = Item{s, tile0 + t, r_lo, r_hi};
        if (pair < n_pairs && s == 0) tile_begin[t] = slot;          // tile_begin is indexed by the window's tiles
    }
}

// Work items of dense count tiles handed in by the host (classic text mode): every sample on every tile.
__global__ void dense_items_kernel(uint32_t n_samples, uint32_t n_tiles, Item* __restrict__ items, uint32_t* __restrict__ tile_begin)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t n = (uint64_t)n_samples * n_tiles;
    if (i < n) {
        const uint32_t t = (uint32_t)(i / n_samples), s = (uint32_t)(i - (uint64_t)t * n_samples);
        items[i] = Item{s, t, 0u, 0xffffffffu};             // "wide": the planes handed in are 16-bit
        if (s == 0) tile_begin[t] = (uint32_t)i;
    }
    if (i == n) tile_begin[n_tiles] = (uint32_t)n;
}

// Exclusive scan of `v[0..n)` in place by one CTA; total to *total.
__global__ void __launch_bounds__(1024) scan_kernel(uint32_t* __restrict__ v, uint32_t n, uint32_t* __restrict__ total)
{
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_carry;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        uint32_t i = base + threadIdx.x;
        uint32_t x = i < n ? v[i] : 0;
        uint32_t incl = x;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane], wi = w;
            #pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                uint32_t o = __shfl_up_sync(0xffffffffu, wi, d);
                if (lane >= d) wi += o;
            }
            s_warp[lane] = wi - w;
        }
        __syncthreads();
        const uint32_t carry = s_carry;
        if (i < n) v[i] = carry + s_warp[warp] + incl - x;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[warp] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

// ------------------------------------------------------------------------------------------------
// expand: reads as BAM stores them -> position-aligned segments (include/msnv.h). This is the column builder's
// per-read half - the CIGAR walk of htslib's resolve_cigar2 and the base / quality look-up of pileup_seq,
// which `samtools mpileup` performs once per COLUMN upstream of snpCall (metaSNV.py:160-165) - done once per
// read: every M/=/X operation becomes a segment whose bases (4-bit -> 2-bit, anything but A/C/G/T flagged) and
// qualities (capped at 127) are stored at their reference position modulo four.
// One warp per read: every lane walks the (short) CIGAR, lane 0 writes the segment records, the lanes share the
// segment's quads - consecutive lanes write consecutive bytes / words.
// ------------------------------------------------------------------------------------------------
struct RawDev {
    const int32_t* pos; const uint32_t* seg_off; const uint32_t* q4_off;      // in the sample's block
    const uint32_t* raw_off; const uint16_t* n_cigar; const uint16_t* l_seq; const uint32_t* raw;      // staged
    uint32_t n_reads;
};

// xstat: [0] bases that are neither A/C/G/T nor N, [1] != 0: a record is inconsistent (CIGAR longer than the sequence, blob
// shorter than the record, more segments or quads than the offsets say); aligned: the sample's aligned bases (statistics)
__global__ void __launch_bounds__(256) expand_kernel(const RawDev in, int32_t* __restrict__ seg_pos, uint16_t* __restrict__ seg_len,
                                                     uint8_t* __restrict__ seq2, uint32_t* __restrict__ qual32, unsigned long long* __restrict__ xstat,
                                                     unsigned long long* __restrict__ aligned)
{
    const uint32_t lane = threadIdx.x & 31u, r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= in.n_reads) return;
    const uint32_t b0 = __ldg(in.raw_off + r), b1 = __ldg(in.raw_off + r + 1);
    const uint32_t* blob = in.raw + b0;
    const uint32_t nc = __ldg(in.n_cigar + r), ls = __ldg(in.l_seq + r);
    const uint8_t* seq4 = reinterpret_cast<const uint8_t*>(blob + nc);
    const uint8_t* ql = seq4 + (ls + 1u) / 2u;
    uint32_t rx = (uint32_t)__ldg(in.pos + r), qy = 0, k = __ldg(in.seg_off + r), Q = __ldg(in.q4_off + r);
    const uint32_t k_end = __ldg(in.seg_off + r + 1), Q_end = __ldg(in.q4_off + r + 1);
    uint32_t n_iupac = 0, n_al = 0;
    if (b1 < b0 || (size_t)(b1 - b0) * 4u < 4u * (size_t)nc + (ls + 1u) / 2u + ls) { if (lane == 0) atomicExch(xstat + 1, 1ull); return; }
    for (uint32_t c = 0; c < nc; ++c) {
        const uint32_t w = __ldg(blob + c), op = w & 15u, len = w >> 4;
        if (op == 0u || op == 7u || op == 8u) {                                  // M, =, X: aligned bases
            if (len) {
                const uint32_t a = rx & 3u, nq = (a + len + 3u) >> 2;
                if (qy + len > ls || k >= k_end || Q + nq > Q_end) { if (lane == 0) atomicExch(xstat + 1, 1ull); return; }
                n_al += len;
                if (lane == 0) { seg_pos[k] = (int32_t)rx; seg_len[k] = (uint16_t)len; }
                for (uint32_t i = lane; i < nq; i += 32u) {
                    uint32_t sb = 0, qw = 0;
                    #pragma unroll
                    for (uint32_t j = 0; j < 4u; ++j) {
                        const int32_t o = (int32_t)(4u * i + j) - (int32_t)a;    // offset in the segment (padding in front of / behind it stays 0)
                        if (o >= 0 && (uint32_t)o < len) {
                            const uint32_t q = qy + (uint32_t)o;
                            const uint32_t b4 = (__ldg(seq4 + (q >> 1)) >> ((~q & 1u) << 2)) & 15u;    // "=ACMGRSVTWYHKDBN": A, C, G, T are the one-hot codes
                            const bool other = __popc(b4) != 1;
                            const uint32_t ph = __ldg(ql + q);
                            sb |= (other ? 0u : (uint32_t)__ffs((int)b4) - 1u) << (2u * j);
                            qw |= ((ph < 127u ? ph : 127u) | (other ? 0x80u : 0u)) << (8u * j);
                            n_iupac += (other && b4 != 15u) ? 1u : 0u;
                        }
                    }
                    seq2[Q + i] = (uint8_t)sb;
                    qual32[Q + i] = qw;
                }
                ++k; Q += nq;
            }
            rx += len; qy += len;
        } else if (op == 2u || op == 3u) rx += len;                              // D, N: reference only
        else if (op == 1u || op == 4u) qy += len;                                // I, S: query only (H, P: neither)
    }
    if (n_iupac) atomicAdd(xstat, (unsigned long long)n_iupac);
    if (lane == 0 && n_al) atomicAdd(aligned, (unsigned long long)n_al);
}

// ------------------------------------------------------------------------------------------------
// mate overlap (htslib tweak_overlap_quality, SURVEY.md Annex A.2): for every pair the host linked, at every
// reference position both mates align a base to, the rule decides which of the two bases is still counted
// (overlap_rule.h: a corrected quality is only ever compared with the threshold, so its verdict is one bit).
// The uploaded reads are never modified: the verdicts go to a side array `fix`, one byte per quad of the
// sample - low nibble: positions the rule overrides, high nibble: whether the base passes there - which the
// pileup kernel stages next to the bases. Cleared and rebuilt by every run (fix_clear_kernel, mate_kernel).
// ------------------------------------------------------------------------------------------------
// bit 0 of the four byte lanes -> a nibble, and back
__device__ __forceinline__ uint32_t lanes_to_nibble(uint32_t x) { return ((x & 0x01010101u) * 0x01020408u) >> 24; }
__device__ __forceinline__ uint32_t nibble_to_lanes(uint32_t n) { return ((n & 0xfu) * 0x00204081u) & 0x01010101u; }

// `which`: the samples that have mate links (blockIdx.y indexes it)
__global__ void __launch_bounds__(256) fix_clear_kernel(const SampleDev* __restrict__ samples, const uint32_t* __restrict__ which)
{
    const SampleDev sd = samples[which[blockIdx.y]];
    if (!sd.fix || sd.n_reads == 0) return;
    const uint32_t n16 = (__ldg(sd.q4_off + sd.n_reads) + 15u) / 16u;        // the array has spare bytes behind it
    uint4* f = reinterpret_cast<uint4*>(sd.fix);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += gridDim.x * blockDim.x) f[i] = make_uint4(0u, 0u, 0u, 0u);
}

// A warp takes 32 consecutive reads, picks the ones that open a pair (the earlier mate) by ballot and hands them out eight
// at a time to its eight groups of four lanes: every lane works on a pair, one quad of both mates per lane and step. The
// mates are stored position-aligned, so their quads line up word for word; a step of a pair is two coalesced 16-byte loads
// per mate and one 4-byte store of verdicts per mate. (Four lanes rather than eight per pair: a 100-base overlap is 18 quads,
// and the per-pair set-up - offsets, segment records - is paid once per warp pass however many pairs share it.)
constexpr uint32_t MATE_LANES = 4;

__global__ void __launch_bounds__(256) mate_kernel(const SampleDev* __restrict__ samples, const uint32_t* __restrict__ which)
{
    const SampleDev sd = samples[which[blockIdx.y]];
    if (!sd.fix) return;
    const uint32_t* __restrict__ qual32 = reinterpret_cast<const uint32_t*>(sd.qual);
    uint32_t* __restrict__ fix32 = reinterpret_cast<uint32_t*>(sd.fix);
    const uint32_t nq_total = sd.n_reads ? __ldg(sd.q4_off + sd.n_reads) : 0u;
    constexpr uint32_t GROUPS = 32u / MATE_LANES;
    const uint32_t lane = threadIdx.x & 31u, lg = lane % MATE_LANES, grp = lane / MATE_LANES;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5, warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    // the quads [lo, hi) (positions) that a segment of a at (ax, first quad qa) and one of b at (bx, qb) share
    auto overlap = [&](int32_t ax, uint32_t qa, int32_t bx, uint32_t qb, int32_t lo, int32_t hi) {
        const uint32_t ia0 = qa - (uint32_t)(ax >> 2), ib0 = qb - (uint32_t)(bx >> 2);                  // quad index of position quad P: i0 + P
        for (int32_t P = (lo >> 2) + (int32_t)lg; P < ((hi + 3) >> 2); P += (int32_t)MATE_LANES) {      // (empty when the segments share no position)
            const uint32_t ia = ia0 + (uint32_t)P, ib = ib0 + (uint32_t)P;
            if (ia >= nq_total || ib >= nq_total) continue;           // segments and offsets disagree (the pileup kernel reports it)
            const uint32_t va = __ldg(qual32 + ia), vb = __ldg(qual32 + ib);
            const uint32_t d = msnv_spread_bases((uint32_t)__ldg(sd.seq2 + ia) ^ (uint32_t)__ldg(sd.seq2 + ib));
            uint32_t pa7, pb7;
            msnv_overlap_verdict4(va, vb, d, pa7, pb7);               // bit 7 of a lane: that mate's base still passes
            const uint32_t na = ((pa7 >> 7) * 0x01020408u) >> 24, nb = ((pb7 >> 7) * 0x01020408u) >> 24;     // ... as nibbles
            // a quad the rule covers whole belongs to this segment combination alone: plain byte stores. Two
            // combinations can meet in a quad at their ends (with disjoint positions): OR into the byte there.
            if ((P << 2) >= lo && (P << 2) + 4 <= hi) { sd.fix[ia] = (uint8_t)(0xfu | na << 4); sd.fix[ib] = (uint8_t)(0xfu | nb << 4); }
            else {
                const uint32_t ovr = lanes_to_nibble(msnv_quad_mask(P << 2, lo, hi));
                atomicOr(fix32 + (ia >> 2), (ovr | (na & ovr) << 4) << (8u * (ia & 3u)));
                atomicOr(fix32 + (ib >> 2), (ovr | (nb & ovr) << 4) << (8u * (ib & 3u)));
            }
        }
    };
    for (uint32_t base = warp0 * 32u; base < sd.n_reads; base += warps * 32u) {
        const uint32_t r_l = base + lane;
        const int32_t mt_l = r_l < sd.n_reads ? __ldg(sd.mate + r_l) : -1;
        uint32_t open = __ballot_sync(0xffffffffu, mt_l > (int32_t)r_l && (uint32_t)mt_l < sd.n_reads);     // the earlier mate (a) handles the pair
        while (open) {
            // the grp-th of the next (up to) GROUPS pairs
            const uint32_t src = __fns(open, 0u, grp + 1u);                                                   // 0xffffffff when there are fewer
            const bool have = src < 32u;
            const int32_t mt = __shfl_sync(0xffffffffu, mt_l, have ? src : 0u);
            const uint32_t r = base + (have ? src : 0u);
            { uint32_t k = __popc(open); k = k < GROUPS ? k : GROUPS; for (uint32_t i = 0; i < k; ++i) open &= open - 1u; }
            if (!have) continue;
            const uint32_t sa0 = __ldg(sd.seg_off + r), sa1 = __ldg(sd.seg_off + r + 1), sb0 = __ldg(sd.seg_off + mt), sb1 = __ldg(sd.seg_off + mt + 1);
            uint32_t qa = __ldg(sd.q4_off + r);                                   // first quad of a's next segment
            const uint32_t qb0 = __ldg(sd.q4_off + mt);
            if (sa1 - sa0 == 1u && sb1 - sb0 == 1u) {                             // the common case: both mates are one segment
                const int32_t ax = __ldg(sd.seg_pos + sa0), bx = __ldg(sd.seg_pos + sb0);
                const int32_t ae = ax + (int32_t)__ldg(sd.seg_len + sa0), be = bx + (int32_t)__ldg(sd.seg_len + sb0);
                overlap(ax, qa, bx, qb0, max(ax, bx), min(ae, be));
                continue;
            }
            for (uint32_t ka = sa0; ka < sa1; ++ka) {
                const int32_t ax = __ldg(sd.seg_pos + ka);
                const uint32_t al = __ldg(sd.seg_len + ka);
                uint32_t qb = qb0;
                for (uint32_t kb = sb0; kb < sb1; ++kb) {
                    const int32_t bx = __ldg(sd.seg_pos + kb);
                    const uint32_t bl = __ldg(sd.seg_len + kb);
                    overlap(ax, qa, bx, qb, max(ax, bx), min(ax + (int32_t)al, bx + (int32_t)bl));
                    qb += (((uint32_t)bx & 3u) + bl + 3u) >> 2;
                }
                qa += (((uint32_t)ax & 3u) + al + 3u) >> 2;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// count tiles: what the pileup kernel writes and the call / gather kernels read.
// Every work item (sample, tile) owns a slot of SLOT_BYTES in HBM holding six count planes of
// TILE positions:
//   D   bases counted at the position (quality >= 13 after the mate-overlap correction, base A/C/G/T)
//   A, C, G, T   those of them that DIFFER from the position's expected letter e (expect[]: the
//       reference base, A where the reference is not A/C/G/T); the plane of letter e stays 0
//   N   counted bases that are not A/C/G/T
// so count[e] = D - (A + C + G + T) and count[x != e] = plane x. Nearly every aligned base equals the
// reference, so the pileup does ONE shared-memory atomic per four positions instead of four.
// Narrow items (at most 255 reads touch the tile: no counter can pass 255) store the planes as
// bytes (6 B per sample-position), wide items (deep coverage) as 16-bit values (12 B).
// ------------------------------------------------------------------------------------------------
constexpr int TILE_QUADS = TILE / 4;
constexpr int N_PLANES = 6;
constexpr int PLANE_D = 0, PLANE_A = 1, PLANE_N = 5;
constexpr uint32_t NARROW_MAX_READS = 255;
constexpr size_t SLOT_BYTES = 2 * N_PLANES * TILE;
static_assert(TILE_QUADS == 256, "a staged quad is tagged with one byte");

__host__ __device__ __forceinline__ bool item_is_wide(uint32_t r_lo, uint32_t r_hi) { return r_hi - r_lo > NARROW_MAX_READS; }

// expected letter per position (0..3 = A,C,G,T) from the reference characters
__global__ void expect_kernel(const uint8_t* __restrict__ ref, uint32_t n, uint8_t* __restrict__ expect)
{
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    uint32_t e = 0;
    switch (ref[p]) {
        case 'C': case 'c': e = 1; break;
        case 'G': case 'g': e = 2; break;
        case 'T': case 't': e = 3; break;
        default: break;
    }
    expect[p] = (uint8_t)e;
}

// ------------------------------------------------------------------------------------------------
// pileup: persistent CTAs, one producer warp + four consumer warps each, walking the work items
// blockIdx.x, blockIdx.x + gridDim.x, ... (items are tile-major, so the CTAs resident at any time
// work on neighbouring tiles and the reads of a sample stream through L2 once).
//
// Producer warp. Item records and the four offsets that size an item are fetched 32 items at a time
// (one per lane: the dependent global loads of 32 items overlap). An item whose reads fit one stage
// (the common case) becomes one chunk; otherwise the warp searches the longest prefix of reads that
// fits (32 probes at a time) and sends several chunks. For a chunk the warp waits for a free stage of
// the ring, writes a header and issues eight TMA bulk copies (UBLKCP) that complete on the stage's
// mbarrier: the reads' offsets and mate links, the segment records, the 2-bit bases, the qualities
// and the tile's expected letters. Consumers therefore never wait for HBM, only for the barrier.
//
// Consumer warps, per chunk (reads arrive as position-aligned segments, include/msnv.h: a staged
// quad holds four consecutive positions starting at a multiple of four, so a quad is either on the
// tile or off it and its four bases are handled with byte-lane arithmetic):
//   1. one thread per read: every staged quad that lies on the tile is tagged with its tile-relative
//      index (four tags per store), the qualities of the few quads off the tile are zeroed (the
//      scatter's threshold test then rejects them like any poor base)
//   2. scatter: a thread takes FOUR consecutive staged quads per step (one 128-bit load of the
//      qualities, one word each of bases, tags and - for samples with mates - overlap verdicts).
//      Per quad: quality test on four byte lanes (overridden where mate_kernel left a verdict), one
//      shared-memory atomic into plane D, and a compare with the expected letters; only lanes that
//      hold a mismatch loop over their set bits and add to a letter plane.
//   3. last chunk of an item: narrow items copy the byte planes to HBM (6 KB, 128-bit stores) and
//      clear them; wide items fold every chunk into 16-bit lanes held in registers (a chunk stages
//      at most 255 reads) and store those.
// The mate-overlap rule itself runs before this kernel (mate_kernel): no read ever waits for its mate here.
//
// Shared memory (dynamic, see pileup_smem_layout): mbarriers | 6 count planes | quad tags |
// stages x { header, q4_off, seg_off, seg_pos, seg_len, expected letters, bases, overlap
// verdicts, qualities }. Every TMA destination is 16-byte aligned; sources are the 16-byte
// aligned addresses at or below the first element needed (the arrays are 256-byte aligned and have
// 32 spare bytes behind them), so a stage holds a few elements in front of and behind the chunk.
// ------------------------------------------------------------------------------------------------
// consumer threads per CTA: a template parameter of the kernel (128 or 256; the CTA has one more warp, the producer)
constexpr uint32_t PL_STAGES_MAX = 8;          // stages of the ring: PileupShape::stages (2 unless the host chose otherwise)
constexpr uint32_t CHUNK_Q4_MIN = MSNV_MAX_READ_BASES / 4 + 2 * MSNV_MAX_READ_SEGMENTS;   // a single read always fits
constexpr uint32_t CHUNK_SEGS_MIN = MSNV_MAX_READ_SEGMENTS;
constexpr uint32_t CHUNK_FIRST = 1u, CHUNK_LAST = 2u, CHUNK_WIDE = 4u, CHUNK_STOP = 8u, CHUNK_FIX = 16u /* the sample has mate verdicts */;

// limits of one staged chunk, chosen per launch from the shape of the shard
struct PileupShape { uint32_t max_reads, max_segs, chunk_q4, has_fix /* some sample carries mate verdicts */,
                     gather /* stages carry the gather kernel's segment records and ranges instead of the scatter kernel's tags */,
                     stages /* of the ring, 2 .. PL_STAGES_MAX */; };

struct ChunkHdr { uint32_t m, nq4, q4_0, sg_0, nseg, c0, item, sample, tile, flags, pad[6]; };
static_assert(sizeof(ChunkHdr) == 64, "header is one 64-byte block");

struct PileupSmem {
    uint32_t bar, cnt, tags, stage0, stage_bytes;                               // byte offsets
    uint32_t o_hdr, o_q4, o_sg, o_sp, o_sl, o_exp, o_seq, o_fix, o_qual;        // within a stage
    uint32_t o_set, o_rec, o_lohi;                                              // within a stage, gather kernel only (written by its consumers)
    uint32_t total;
};

__host__ __device__ constexpr uint32_t up_to(uint32_t v, uint32_t a) { return (v + a - 1) / a * a; }

__host__ __device__ inline PileupSmem pileup_smem_layout(const PileupShape sh)
{
    PileupSmem L{};
    uint32_t o = 0;
    L.bar = o;   o += 128;
    L.cnt = o;   o += N_PLANES * TILE;
    L.tags = o;  o += sh.gather ? 0u : up_to(sh.chunk_q4, 16) + 16;
    L.stage0 = up_to(o, 128);
    uint32_t s = 0;
    const uint32_t mw = up_to(sh.max_reads + 1, 4) + 8;
    L.o_hdr = s;  s += 64;
    L.o_q4 = s;   s += mw * 4;
    L.o_sg = s;   s += mw * 4;
    L.o_sp = s;   s += (up_to(sh.max_segs, 4) + 8) * 4;
    L.o_sl = s;   s += (up_to(sh.max_segs, 8) + 16) * 2;
    L.o_exp = s;  s += TILE;
    L.o_seq = s;  s += up_to(sh.chunk_q4, 16) + 32;
    L.o_fix = s;  s += sh.has_fix ? up_to(sh.chunk_q4, 16) + 32 : 0;
    L.o_qual = s; s += 4 * up_to(sh.chunk_q4, 16) + 32;
    if (sh.gather) {
        L.o_set = s;  s += 64;
        L.o_rec = s;  s += (up_to(sh.max_segs, 4) + 8) * 8;
        L.o_lohi = s; s += TILE_QUADS * 4;
    }
    L.stage_bytes = up_to(s, 128);
    L.total = L.stage0 + sh.stages * L.stage_bytes;
    return L;
}

// explicit shared-window accesses (32-bit addresses) for the scatter loop
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint4 lds_v4(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void red_shared_add(uint32_t a, uint32_t v) { asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t and3(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm("lop3.b32 %0, %1, %2, %3, 0x80;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// barrier among the consumer warps only (the producer warp never joins it)
template <int CONSUMERS>
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory"); }

// the arrays of one sample the producer copies from
struct SrcPtrs {
    const uint32_t* q4_off; const uint32_t* seg_off; const int32_t* seg_pos; const uint16_t* seg_len;
    const uint8_t* seq2; const uint8_t* qual; const uint8_t* fix;
};
__device__ __forceinline__ SrcPtrs load_src_ptrs(const SampleDev* __restrict__ sd)
{
    SrcPtrs p;
    p.q4_off = sd->q4_off; p.seg_off = sd->seg_off; p.seg_pos = sd->seg_pos; p.seg_len = sd->seg_len;
    p.seq2 = sd->seq2; p.qual = sd->qual; p.fix = sd->fix;
    return p;
}

// source address and size of the seven bulk copies of a chunk (16-byte aligned addresses at or below the first element
// needed, sizes rounded up to 16 bytes)
struct ChunkCopies { const void* src[7]; uint32_t bytes[7]; };
__device__ __forceinline__ ChunkCopies chunk_copies(const SrcPtrs& p, uint32_t c0, uint32_t m, uint32_t q4_0, uint32_t nq4, uint32_t sg_0, uint32_t nseg)
{
    const uint32_t dm = c0 & 3u, ds = sg_0 & 3u, dl = sg_0 & 7u, dq = q4_0 & 3u, d16 = q4_0 & 15u;
    ChunkCopies c;
    c.src[0] = p.q4_off + (c0 - dm);             c.bytes[0] = up_to(dm + m + 1u, 4) * 4u;
    c.src[1] = p.seg_off + (c0 - dm);            c.bytes[1] = c.bytes[0];
    c.src[2] = p.fix ? p.fix + (q4_0 - d16) : nullptr; c.bytes[2] = p.fix ? up_to(d16 + nq4, 16) : 0u;   // same geometry as the bases
    c.src[3] = p.seg_pos + (sg_0 - ds);          c.bytes[3] = up_to(ds + nseg, 4) * 4u;
    c.src[4] = p.seg_len + (sg_0 - dl);          c.bytes[4] = up_to(dl + nseg, 8) * 2u;
    c.src[5] = p.seq2 + (q4_0 - d16);            c.bytes[5] = up_to(d16 + nq4, 16);
    c.src[6] = p.qual + 4u * (size_t)(q4_0 - dq); c.bytes[6] = up_to(dq + nq4, 4) * 4u;
    return c;
}

// ---- producer: one chunk of sample `sd` into the next stage of the ring (whole warp waits; lane `issuer` reads the sample's
// array pointers, writes the header and issues: no lane holds seven pointers across the producer's loops)
__device__ __forceinline__ void pileup_issue_chunk(uint8_t* smem, const PileupSmem& L, const PileupShape& sh, uint32_t& chunk_no, uint32_t issuer, const SampleDev* __restrict__ sd,
                                                   const uint8_t* __restrict__ expect, uint32_t item, uint32_t sample, uint32_t tile, uint32_t c0,
                                                   uint32_t m, uint32_t q4_0, uint32_t nq4, uint32_t sg_0, uint32_t nseg, uint32_t flags)
{
    uint64_t* full = (uint64_t*)(smem + L.bar);
    uint64_t* empty = full + sh.stages;
    const uint32_t s = chunk_no % sh.stages, ph = (chunk_no / sh.stages) & 1u;
    // the producer spins for a free stage: sleeping 200 or 1000 ns between polls measured the same, 3000 ns slower
    // (profiles/r02_pileup_ablations.txt, D)
    mbar_wait(empty + s, ph ^ 1u);
    if ((threadIdx.x & 31) == issuer) {
        const SrcPtrs src = load_src_ptrs(sd);
        uint8_t* stage = smem + L.stage0 + s * L.stage_bytes;
        ChunkHdr* h = (ChunkHdr*)(stage + L.o_hdr);
        h->m = m; h->nq4 = nq4; h->q4_0 = q4_0; h->sg_0 = sg_0; h->nseg = nseg; h->c0 = c0;
        h->item = item; h->sample = sample; h->tile = tile; h->flags = flags | (src.fix ? CHUNK_FIX : 0u);
        const ChunkCopies c = chunk_copies(src, c0, m, q4_0, nq4, sg_0, nseg);
        const uint32_t dst[7] = {L.o_q4, L.o_sg, L.o_fix, L.o_sp, L.o_sl, L.o_seq, L.o_qual};
        uint32_t total = (uint32_t)TILE;
        #pragma unroll
        for (int i = 0; i < 7; ++i) total += c.bytes[i];
        fence_proxy_async();
        mbar_expect_tx(full + s, total);
        #pragma unroll
        for (int i = 0; i < 7; ++i) if (c.bytes[i]) tma_load_1d(stage + dst[i], c.src[i], c.bytes[i], full + s);
        tma_load_1d(stage + L.o_exp, expect + (size_t)tile * TILE, TILE, full + s);
    }
    __syncwarp();
    ++chunk_no;
}

__device__ __forceinline__ void pileup_producer(uint8_t* smem, const PileupSmem& L, const PileupShape sh, const SampleDev* __restrict__ samples,
                                                const Item* __restrict__ items, uint32_t n_items, const uint8_t* __restrict__ expect,
                                                int* __restrict__ err_flag)
{
    const uint32_t lane = threadIdx.x & 31, G = gridDim.x;
    uint32_t chunk_no = 0;
    for (uint64_t base = blockIdx.x; base < n_items; base += 32ull * G) {
        // ---- 32 upcoming items of this CTA, one per lane: item record and the offsets that size the item
        const uint64_t mine = base + (uint64_t)lane * G;
        uint4 it = make_uint4(0u, 0u, 0u, 0u);
        uint32_t q_lo = 0, q_hi = 0, g_lo = 0, g_hi = 0;
        bool whole = false;                  // the item fits one stage
        if (mine < n_items) {
            it = __ldg(reinterpret_cast<const uint4*>(items) + mine);
            const SrcPtrs src = load_src_ptrs(samples + it.x);
            q_lo = __ldg(src.q4_off + it.z); q_hi = __ldg(src.q4_off + it.w);
            g_lo = __ldg(src.seg_off + it.z); g_hi = __ldg(src.seg_off + it.w);
            whole = it.w - it.z <= sh.max_reads && q_hi - q_lo <= sh.chunk_q4 && g_hi - g_lo <= sh.max_segs;
        }
        for (uint32_t k = 0; k < 32u; ++k) {
            const uint64_t idx = base + (uint64_t)k * G;
            if (idx >= n_items) break;
            if (__shfl_sync(0xffffffffu, (int)whole, k)) {                   // the lane that owns the item issues it from its own registers
                pileup_issue_chunk(smem, L, sh, chunk_no, k, samples + it.x, expect, (uint32_t)mine, it.x, it.y, it.z, it.w - it.z, q_lo, q_hi - q_lo, g_lo,
                                   g_hi - g_lo, CHUNK_FIRST | CHUNK_LAST | (item_is_wide(it.z, it.w) ? CHUNK_WIDE : 0u));
                continue;
            }
            // ---- the item needs several chunks: longest prefix of the remaining reads within the three limits
            const uint32_t sample = __shfl_sync(0xffffffffu, it.x, k), tile = __shfl_sync(0xffffffffu, it.y, k);
            const uint32_t r_lo = __shfl_sync(0xffffffffu, it.z, k), r_hi = __shfl_sync(0xffffffffu, it.w, k);
            const uint32_t ql = __shfl_sync(0xffffffffu, q_lo, k), gl = __shfl_sync(0xffffffffu, g_lo, k);
            const uint32_t* q4p = samples[sample].q4_off; const uint32_t* sgp = samples[sample].seg_off;
            const uint32_t wide = item_is_wide(r_lo, r_hi) ? CHUNK_WIDE : 0u;
            uint32_t c0 = r_lo, qc = ql, gc = gl;
            while (c0 < r_hi) {
                // Optimistic sizing of the next 32 chunks at once: max_reads reads each, one probe per lane (the stage is
                // sized so that this many reads normally fit). A deep item takes hundreds of chunks; sizing them one by one
                // would put two or three dependent global round trips between any two copies.
                const uint32_t b_l = min(c0 + lane * sh.max_reads, r_hi), e_l = min(b_l + sh.max_reads, r_hi);
                const uint32_t qe = __ldg(q4p + e_l), ge = __ldg(sgp + e_l);
                uint32_t qb = __shfl_up_sync(0xffffffffu, qe, 1), gb = __shfl_up_sync(0xffffffffu, ge, 1);
                if (lane == 0) { qb = qc; gb = gc; }
                const bool fit = e_l == b_l || (qe - qb <= sh.chunk_q4 && ge - gb <= sh.max_segs);
                const uint32_t okmask = __ballot_sync(0xffffffffu, fit);
                const uint32_t n_ok = okmask == 0xffffffffu ? 32u : (uint32_t)__ffs((int)~okmask) - 1u;      // leading chunks that fit
                if (n_ok) {
                    const uint32_t fl = (b_l == r_lo ? CHUNK_FIRST : 0u) | (e_l == r_hi ? CHUNK_LAST : 0u) | wide;
                    uint32_t done_to = c0, done_q = qc, done_g = gc;
                    for (uint32_t kk = 0; kk < n_ok; ++kk) {
                        const uint32_t bk = __shfl_sync(0xffffffffu, b_l, kk), ek = __shfl_sync(0xffffffffu, e_l, kk);
                        if (ek == bk) break;                                             // past the end of the item
                        pileup_issue_chunk(smem, L, sh, chunk_no, kk, samples + sample, expect, (uint32_t)idx, sample, tile, b_l, e_l - b_l, qb, qe - qb, gb, ge - gb, fl);
                        done_to = ek; done_q = __shfl_sync(0xffffffffu, qe, kk); done_g = __shfl_sync(0xffffffffu, ge, kk);
                    }
                    c0 = done_to; qc = done_q; gc = done_g;
                    continue;
                }
                // the first of them does not fit (long reads, many segments): longest prefix of reads within the three limits
                const uint32_t cap = min(sh.max_reads, r_hi - c0), step = (cap + 31u) / 32u;
                const uint32_t pi = min((lane + 1u) * step, cap);
                bool fits = __ldg(q4p + c0 + pi) - qc <= sh.chunk_q4 && __ldg(sgp + c0 + pi) - gc <= sh.max_segs;
                const uint32_t cnt = __popc(__ballot_sync(0xffffffffu, fits));
                uint32_t m = cap;
                if (cnt < 32u) {                     // lanes 0..cnt-1 fit, lane cnt does not: refine between the two probes
                    const uint32_t b0 = cnt * step, pj = b0 + lane + 1u;
                    fits = false;
                    if (lane + 1u < step && pj <= cap) fits = __ldg(q4p + c0 + pj) - qc <= sh.chunk_q4 && __ldg(sgp + c0 + pj) - gc <= sh.max_segs;
                    m = b0 + __popc(__ballot_sync(0xffffffffu, fits));
                }
                const uint32_t first = c0 == r_lo ? CHUNK_FIRST : 0u;
                if (m == 0) {                        // a single read over the documented limits: host validation failed
                    if (lane == 0) atomicExch(err_flag, 1);
                    pileup_issue_chunk(smem, L, sh, chunk_no, 0u, samples + sample, expect, (uint32_t)idx, sample, tile, c0, 0u, qc, 0u, gc, 0u, first | CHUNK_LAST | wide);
                    break;
                }
                const uint32_t qn = __ldg(q4p + c0 + m), gn = __ldg(sgp + c0 + m);
                pileup_issue_chunk(smem, L, sh, chunk_no, 0u, samples + sample, expect, (uint32_t)idx, sample, tile, c0, m, qc, qn - qc, gc, gn - gc,
                                   first | (c0 + m == r_hi ? CHUNK_LAST : 0u) | wide);
                c0 += m; qc = qn; gc = gn;
            }
        }
    }
    // ---- no more items: tell the consumers
    uint64_t* full = (uint64_t*)(smem + L.bar);
    uint64_t* empty = full + sh.stages;
    const uint32_t s = chunk_no % sh.stages, ph = (chunk_no / sh.stages) & 1u;
    mbar_wait(empty + s, ph ^ 1u);
    if (lane == 0) {
        ((ChunkHdr*)(smem + L.stage0 + s * L.stage_bytes + L.o_hdr))->flags = CHUNK_STOP;
        mbar_arrive(full + s);
    }
}

// ---- what both forms share
// CTA start: the ring's barriers (a stage is free again after `empty_count` arrivals) and cleared count planes; then the
// producer warp runs the producer. Returns true to the producer warp, which leaves the kernel.
template <int CONSUMERS>
__device__ __forceinline__ bool pileup_cta_start(uint8_t* smem, const PileupSmem& L, const PileupShape& sh, uint32_t empty_count,
                                                 const SampleDev* __restrict__ samples, const Item* __restrict__ items, uint32_t n_items,
                                                 const uint8_t* __restrict__ expect, int* __restrict__ err_flag)
{
    uint64_t* full = (uint64_t*)(smem + L.bar);
    uint64_t* empty = full + sh.stages;
    uint32_t* s_cnt = (uint32_t*)(smem + L.cnt);
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < sh.stages; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, empty_count); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t k = threadIdx.x; k < (uint32_t)(N_PLANES * TILE_QUADS); k += CONSUMERS + 32) s_cnt[k] = 0;
    __syncthreads();
    if (threadIdx.x < CONSUMERS) return false;
    pileup_producer(smem, L, sh, samples, items, n_items, expect, err_flag);
    return true;
}

// Wide items (more than 255 reads) are counted in 16-bit lanes held in registers, per plane and owned quad QPT * tid + k
// (QPT = TILE_QUADS / CONSUMERS, 2 or 1): [0] = positions 0 and 2, [1] = positions 1 and 3. HAS_WIDE: the shard has such
// items (deep coverage); without them one plane's worth is declared and never used.
template <int CONSUMERS, bool HAS_WIDE> using WideAcc = uint32_t[HAS_WIDE ? N_PLANES : 1][TILE_QUADS / CONSUMERS][2];

// this thread's words of the byte planes into its 16-bit lanes (a chunk stages at most 255 reads: no byte lane has
// overflowed); the words are cleared
template <int CONSUMERS, bool HAS_WIDE>
__device__ __forceinline__ void wide_fold(WideAcc<CONSUMERS, HAS_WIDE>& acc, uint32_t* s_cnt, uint32_t tid)
{
    constexpr int QPT = TILE_QUADS / CONSUMERS;
    #pragma unroll
    for (int c = 0; c < (HAS_WIDE ? N_PLANES : 1); ++c)
        #pragma unroll
        for (int k = 0; k < QPT; ++k) {
            const uint32_t slot = c * TILE_QUADS + QPT * tid + k;
            const uint32_t w = s_cnt[slot];
            s_cnt[slot] = 0;
            acc[c][k][0] += w & 0x00ff00ffu; acc[c][k][1] += (w >> 8) & 0x00ff00ffu;
        }
}

// the item's 16-bit planes from this thread's lanes to its slot in HBM; the lanes are cleared
template <int CONSUMERS, bool HAS_WIDE>
__device__ __forceinline__ void wide_store(WideAcc<CONSUMERS, HAS_WIDE>& acc, uint8_t* slot, uint32_t tid)
{
    constexpr int QPT = TILE_QUADS / CONSUMERS;
    uint2* dst = reinterpret_cast<uint2*>(slot);
    #pragma unroll
    for (int c = 0; c < (HAS_WIDE ? N_PLANES : 1); ++c)
        #pragma unroll
        for (int k = 0; k < QPT; ++k) {
            // 16-bit plane c, positions 4 * (QPT * tid + k) .. + 3
            dst[c * (TILE / 4) + QPT * tid + k] = make_uint2((acc[c][k][0] & 0xffffu) | (acc[c][k][1] << 16), (acc[c][k][0] >> 16) | (acc[c][k][1] & 0xffff0000u));
            acc[c][k][0] = acc[c][k][1] = 0;
        }
}

// The pass test of one staged quad, on byte lanes (bit 0 of each): ok = the base counts (quality >= 13, A/C/G/T), nn = it
// counts as N (it passes, but is not A/C/G/T). q: the four qualities, bit 7 of a lane set where the base is not A/C/G/T.
// FIX (the sample carries mate verdicts): where the overlap rule spoke (low nibble of the verdict byte f) its verdict (high
// nibble) replaces the quality test.
template <bool FIX>
__device__ __forceinline__ void quad_pass(uint32_t q, uint32_t f, uint32_t& ok, uint32_t& nn)
{
    if (!FIX) {
        const uint32_t v = (q & 0x7f7f7f7fu) + 0x73737373u;                     // bit 7 of a lane: quality >= 13
        asm("lop3.b32 %0, %1, %2, 0x80808080, 0x20;" : "=r"(ok) : "r"(v), "r"(q));    // v & ~q & 0x80808080: ... and A/C/G/T
        ok >>= 7;
        nn = and3(v, q, 0x80808080u) >> 7;
    } else {
        const uint32_t ovr = nibble_to_lanes(f), val = nibble_to_lanes(f >> 4);
        const uint32_t qp = (((q & 0x7f7f7f7fu) + 0x73737373u) >> 7) & 0x01010101u;
        const uint32_t pass = (qp & ~ovr) | (val & ovr);
        const uint32_t fl = (q >> 7) & 0x01010101u;
        ok = pass & ~fl;
        nn = pass & fl;
    }
}

// CONSUMERS: consumer threads (128: four CTAs per SM at the standard shape; 256: three larger ones).
// HAS_WIDE: the shard has items with more than 255 reads (see WideAcc).
template <int CONSUMERS, bool HAS_WIDE>
__global__ void __launch_bounds__(CONSUMERS + 32, CONSUMERS == 128 ? 4 : 3)
pileup_kernel(const SampleDev* __restrict__ samples, const Item* __restrict__ items, uint32_t n_items, const PileupShape sh,
              const uint8_t* __restrict__ expect, uint8_t* __restrict__ tiles /*[n_items][SLOT_BYTES]*/, int* __restrict__ err_flag)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const PileupSmem L = pileup_smem_layout(sh);
    if (pileup_cta_start<CONSUMERS>(smem, L, sh, 1u, samples, items, n_items, expect, err_flag)) return;

    // ------------------------------------------------------------------------------------ consumers
    uint64_t* full = (uint64_t*)(smem + L.bar);
    uint64_t* empty = full + sh.stages;
    uint32_t* s_cnt = (uint32_t*)(smem + L.cnt);
    const uint32_t tid = threadIdx.x;
    uint8_t* s_tags = smem + L.tags;
    WideAcc<CONSUMERS, HAS_WIDE> acc = {};

    for (uint32_t chunk_no = 0;; ++chunk_no) {
        const uint32_t st = chunk_no % sh.stages, ph = (chunk_no / sh.stages) & 1u;
        uint8_t* stage = smem + L.stage0 + st * L.stage_bytes;
        mbar_wait(full + st, ph);
        const ChunkHdr* h = (const ChunkHdr*)(stage + L.o_hdr);
        const uint32_t flags = h->flags;
        if (flags & CHUNK_STOP) break;
        const uint32_t m = h->m, nq4 = h->nq4, q4_0 = h->q4_0, sg_0 = h->sg_0, nseg = h->nseg, c0 = h->c0, item = h->item;
        const int32_t p0 = (int32_t)(h->tile * TILE);
        const uint32_t dm = c0 & 3u, dq = q4_0 & 3u, c12 = q4_0 & 12u;
        const uint32_t* s_q4 = (const uint32_t*)(stage + L.o_q4) + dm;          // s_q4[t] = q4_off[c0 + t], t <= m
        const uint32_t* s_sgo = (const uint32_t*)(stage + L.o_sg) + dm;
        const int32_t* s_sp = (const int32_t*)(stage + L.o_sp) + (sg_0 & 3u);   // s_sp[k] = seg_pos[sg_0 + k], k < nseg
        const uint16_t* s_sl = (const uint16_t*)(stage + L.o_sl) + (sg_0 & 7u);
        uint32_t* s_qw = (uint32_t*)(stage + L.o_qual);                         // qualities of buffer quad B in word B
        uint8_t* s_fx = stage + L.o_fix + c12;                                  // overlap verdicts of buffer quad B (samples with mates)
        const bool has_fix = (flags & CHUNK_FIX) != 0;
        const uint32_t nbq = dq + nq4, ngroups = (nbq + 3u) >> 2;               // staged quad g is buffer quad g + dq
        // a quad that must not count (off the tile, in front of or behind the chunk): no quality passes and no verdict overrides
        auto mute = [&](uint32_t g) { s_qw[g] = 0; if (has_fix) s_fx[g] = 0; };

        // ---- 1. one thread per read: tags of the quads on the tile, zeroed qualities off it
        for (uint32_t t = tid; t < m; t += CONSUMERS) {
            const uint32_t k0 = s_sgo[t] - sg_0, k1 = s_sgo[t + 1] - sg_0;
            uint32_t B = s_q4[t] - q4_0 + dq;                                   // first buffer quad of the next segment
            const uint32_t B_end = s_q4[t + 1] - q4_0 + dq;
            if (k1 < k0 || k1 > nseg || B_end < B || B_end > nbq) { atomicExch(err_flag, 2); continue; }   // offsets not prefix sums
            for (uint32_t k = k0; k < k1; ++k) {
                const int32_t p = s_sp[k];
                const uint32_t len = s_sl[k];
                const uint32_t a = (uint32_t)p & 3u;
                const int32_t nq = (int32_t)((a + len + 3u) >> 2);
                const int32_t jw = (p - (int32_t)a - p0) >> 2;                  // tile-relative index of the segment's first quad
                if (B + (uint32_t)nq > B_end) break;                            // segments and offsets disagree: flagged below
                int32_t i_lo = jw < 0 ? -jw : 0; if (i_lo > nq) i_lo = nq;
                int32_t i_hi = TILE_QUADS - jw; if (i_hi > nq) i_hi = nq; if (i_hi < i_lo) i_hi = i_lo;
                for (int32_t i = 0; i < i_lo; ++i) mute(B + (uint32_t)i);
                for (int32_t i = i_hi; i < nq; ++i) mute(B + (uint32_t)i);
                uint32_t g = B + (uint32_t)i_lo, tv = (uint32_t)(jw + i_lo);
                const uint32_t e = B + (uint32_t)i_hi;                          // tags tv .. tv + (e - g) - 1 are within 0..255
                // up to three single tags to a word boundary, words of four consecutive tags, up to three single tags
                uint32_t hn = (0u - g) & 3u; if (hn > e - g) hn = e - g;
                if (hn > 0u) s_tags[g] = (uint8_t)tv;
                if (hn > 1u) s_tags[g + 1] = (uint8_t)(tv + 1u);
                if (hn > 2u) s_tags[g + 2] = (uint8_t)(tv + 2u);
                g += hn; tv += hn;
                uint32_t wv = tv * 0x01010101u + 0x03020100u;                       // no lane passes 255: all four quads are on the tile
                uint32_t* tw = reinterpret_cast<uint32_t*>(s_tags + g);
                const uint32_t nw = (e - g) >> 2;
                uint32_t w = 0;
                for (; w + 2u <= nw; w += 2u, wv += 0x08080808u) { tw[w] = wv; tw[w + 1] = wv + 0x04040404u; }
                if (w < nw) { tw[w] = wv; ++w; }
                g += 4u * nw; tv += 4u * nw;
                const uint32_t tn = e - g;
                if (tn > 0u) s_tags[g] = (uint8_t)tv;
                if (tn > 1u) s_tags[g + 1] = (uint8_t)(tv + 1u);
                if (tn > 2u) s_tags[g + 2] = (uint8_t)(tv + 2u);
                B += (uint32_t)nq;
            }
            if (B != B_end) {                                                   // quads no segment owns: keep them out of the counts
                atomicExch(err_flag, 2);
                for (uint32_t g = B; g < B_end; ++g) mute(g);
            }
        }
        if (tid == CONSUMERS - 1) {                                             // elements in front of and behind the chunk in the buffer
            for (uint32_t g = 0; g < dq; ++g) mute(g);
            for (uint32_t g = nbq; g < 4u * ngroups; ++g) mute(g);
        }
        consumer_sync<CONSUMERS>();

        // ---- 2. scatter: four consecutive buffer quads per thread and step
        {
            const uint32_t a_q = smem_u32(s_qw), a_s = smem_u32(stage + L.o_seq) + c12, a_f = smem_u32(stage + L.o_fix) + c12, a_g = smem_u32(s_tags);
            const uint32_t a_c = smem_u32(s_cnt), a_e = smem_u32(stage + L.o_exp);
            for (uint32_t u = tid; u < ngroups; u += CONSUMERS) {
                const uint4 qv = lds_v4(a_q + 16u * u);
                const uint32_t sw = lds_u32(a_s + 4u * u), tw = lds_u32(a_g + 4u * u);
                const uint32_t qa[4] = {qv.x, qv.y, qv.z, qv.w};
                uint32_t xs[4], mm[4], ac[4], nn[4], nn_any = 0, mm_any = 0;
                if (!has_fix) {
                    #pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t j = __byte_perm(tw, 0u, 0x4440u + k);                // tile-relative quad
                        ac[k] = a_c + 4u * j;                                               // its word in plane D
                        xs[k] = msnv_spread_bases(__byte_perm(sw, 0u, 0x4440u + k));        // one 2-bit base per byte lane
                        uint32_t ok;
                        quad_pass<false>(qa[k], 0u, ok, nn[k]);
                        const uint32_t d = xs[k] ^ lds_u32(a_e + 4u * j);                   // differs from the expected letter?
                        red_shared_add(ac[k], ok);
                        mm[k] = (d | (d >> 1)) & ok;
                        mm_any |= mm[k];
                        nn_any |= nn[k];
                    }
                } else {
                    const uint32_t fw = lds_u32(a_f + 4u * u);                              // the quads' verdict bytes
                    #pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t j = __byte_perm(tw, 0u, 0x4440u + k);
                        ac[k] = a_c + 4u * j;
                        xs[k] = msnv_spread_bases(__byte_perm(sw, 0u, 0x4440u + k));
                        uint32_t ok;
                        quad_pass<true>(qa[k], __byte_perm(fw, 0u, 0x4440u + k), ok, nn[k]);
                        const uint32_t d = xs[k] ^ lds_u32(a_e + 4u * j);
                        red_shared_add(ac[k], ok);
                        mm[k] = (d | (d >> 1)) & ok;
                        mm_any |= mm[k];
                        nn_any |= nn[k];
                    }
                }
                if (mm_any) {                                                           // counted bases that are not the expected letter:
                    #pragma unroll                                                      // only the lanes that hold one loop over their set bits
                    for (int k = 0; k < 4; ++k) {
                        uint32_t r = mm[k];
                        while (r) {
                            const uint32_t b = (uint32_t)__ffs((int)r) - 1u;            // 0, 8, 16 or 24
                            red_shared_add(ac[k] + (PLANE_A + ((xs[k] >> b) & 3u)) * (uint32_t)TILE, 1u << b);
                            r &= r - 1u;
                        }
                    }
                }
                if (nn_any) {                                                           // rare: counted non-ACGT bases
                    #pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (nn[k]) red_shared_add(ac[k] + PLANE_N * (uint32_t)TILE, nn[k]);
                }
            }
        }
        fence_proxy_async();                // this thread's writes to the stage are ordered before the copies that refill it
        consumer_sync<CONSUMERS>();
        if (tid == 0) mbar_arrive(empty + st);

        // ---- 4. counts of the chunk
        if (HAS_WIDE && (flags & CHUNK_WIDE)) {
            wide_fold<CONSUMERS, HAS_WIDE>(acc, s_cnt, tid);
            if (flags & CHUNK_LAST) wide_store<CONSUMERS, HAS_WIDE>(acc, tiles + (size_t)item * SLOT_BYTES, tid);
        } else if (flags & CHUNK_LAST) {
            uint4* cnt4 = reinterpret_cast<uint4*>(s_cnt);
            uint4* dst = reinterpret_cast<uint4*>(tiles + (size_t)item * SLOT_BYTES);
            for (uint32_t i = tid; i < (uint32_t)(N_PLANES * TILE / 16); i += CONSUMERS) {
                const uint4 w = cnt4[i];
                cnt4[i] = make_uint4(0u, 0u, 0u, 0u);
                dst[i] = w;
            }
        }
        // no barrier here: the next chunk touches the counters again only after its own barriers
    }
}

// ------------------------------------------------------------------------------------------------
// pileup, gather form. Same ring, same stages, same count planes as pileup_kernel; what differs is who adds what:
// a consumer thread OWNS tile quads (four positions each) and walks the aligned segments that cover them, so the counts
// live in registers - no shared-memory atomics, no tags, no cleared planes - and go straight from the registers to HBM.
// A consumer warp releases the stage on its own when it has read it (the stage's "empty" barrier counts warps).
//
// The geometry the consumers need is built per chunk by the consumers themselves, a thread per read (gather_setup, two
// CTA-wide barriers: a single warp doing it - tried first, in the producer - takes longer than the counting):
//   * a record per segment, clipped to the tile: first and last+1 tile quad, and the buffer quad that holds tile quad 0
//   * per tile quad j the range [lo_j, hi_j) of segments that can cover it. Reads are in coordinate order, so
//     hi_j = first segment of the first read that starts behind j, and lo_j = first segment of the first read r whose
//     running maximum of read ends (a warp scan, block maxima through shared memory) passes j. Both are written as runs
//     by the thread that owns the read.
// For a read that covers j the segments in between are its neighbours in the file: at 10x and 100-base reads a thread
// looks at ~12 records to find its ~10.
//
// Per (quad, segment) step: one 64-bit record, the quad's four qualities and its base byte; quality test on byte lanes;
// D += pass; the letters are counted as three bit-plane sums (bit 0 set, bit 1 set, both set) from which the four letter
// counts follow at the end of the item by subtraction - the expected letter is not needed inside the loop at all. With 128
// consumers a thread owns two neighbouring quads, which share the record and its range test.
//
// Narrow items (at most 255 reads: a byte lane cannot overflow) stay in the registers of the threads that own their quads
// over as many chunks as the item takes. Deep items (cut into chunks of 255 reads that start within a few positions of each
// other): a chunk then spans only part of the tile, so the 256 quad slots are dealt out as G groups of W quads (W = the
// chunk's span rounded up to a power of two), group g taking every G-th segment; the partial sums are added to the shared
// planes (one atomic per non-zero word instead of one per staged quad) and the planes are folded as in pileup_kernel.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int32_t clamp_quad(int32_t v) { return v < 0 ? 0 : (v > TILE_QUADS ? TILE_QUADS : v); }

// Layout of a stage's "set" block (16 words): [0] jmin, [1] jmax (quads [jmin, jmax) can be covered), [2..9] maximum of the
// read ends per block of 32 reads, [10] != 0: the ranges are not usable (see below).
template <int CONSUMERS>
__device__ __forceinline__ void gather_setup(uint8_t* stage, const PileupSmem& L, int* __restrict__ err_flag)
{
    constexpr int RPT = (int)(NARROW_MAX_READS + CONSUMERS) / CONSUMERS;    // reads per thread (a chunk stages at most 255)
    constexpr int N_WARPS = CONSUMERS / 32;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const ChunkHdr* h = (const ChunkHdr*)(stage + L.o_hdr);
    const uint32_t m = h->m, nq4 = h->nq4, q4_0 = h->q4_0, sg_0 = h->sg_0, nseg = h->nseg, c0 = h->c0;
    const int32_t p0 = (int32_t)(h->tile * TILE);
    const uint32_t dm = c0 & 3u, dq = q4_0 & 3u;
    const uint32_t* s_q4 = (const uint32_t*)(stage + L.o_q4) + dm;          // s_q4[t] = q4_off[c0 + t], t <= m
    const uint32_t* s_sgo = (const uint32_t*)(stage + L.o_sg) + dm;
    const int32_t* s_sp = (const int32_t*)(stage + L.o_sp) + (sg_0 & 3u);   // s_sp[k] = seg_pos[sg_0 + k], k < nseg
    const uint16_t* s_sl = (const uint16_t*)(stage + L.o_sl) + (sg_0 & 7u);
    uint2* recs = (uint2*)(stage + L.o_rec);
    uint16_t* lohi = (uint16_t*)(stage + L.o_lohi);                         // [2 j] = lo_j, [2 j + 1] = hi_j
    int32_t* set = (int32_t*)(stage + L.o_set);
    const uint32_t nbq = dq + nq4;
    // first tile quad (clipped) of read t's first segment; 256 behind the last read
    auto read_start = [&](uint32_t t) -> int32_t {
        if (t >= m) return TILE_QUADS;
        const uint32_t k = s_sgo[t] - sg_0;
        if (k >= nseg) return TILE_QUADS;
        return clamp_quad((s_sp[k] - p0) >> 2);
    };
    int32_t aq[RPT], pb[RPT];
    uint32_t k0[RPT], k1[RPT];
    // ---- records; per block of 32 reads the maximum of the read ends
    #pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const uint32_t t = tid + (uint32_t)i * CONSUMERS;
        int32_t eq = 0;
        aq[i] = TILE_QUADS; k0[i] = k1[i] = 0;
        if (t < m) {
            k0[i] = s_sgo[t] - sg_0; k1[i] = s_sgo[t + 1] - sg_0;
            uint32_t B = s_q4[t] - q4_0 + dq;                                   // first buffer quad of the next segment
            const uint32_t B_end = s_q4[t + 1] - q4_0 + dq;
            if (k1[i] < k0[i] || k1[i] > nseg || B_end < B || B_end > nbq) { atomicExch(err_flag, 2); k0[i] = k1[i] = 0; }   // offsets not prefix sums
            aq[i] = read_start(t);
            for (uint32_t k = k0[i]; k < k1[i]; ++k) {
                const int32_t p = s_sp[k];
                const uint32_t len = s_sl[k];
                const uint32_t a = (uint32_t)p & 3u;
                const int32_t nq = (int32_t)((a + len + 3u) >> 2);
                const int32_t jw = (p - (int32_t)a - p0) >> 2;                  // tile-relative index of the segment's first quad
                int32_t lo = clamp_quad(jw), hi = clamp_quad(jw + nq);
                if (B + (uint32_t)nq > B_end) { atomicExch(err_flag, 2); lo = hi = 0; }    // segments and offsets disagree: the run fails
                recs[k] = make_uint2((uint32_t)((int32_t)B - jw), hi > lo ? (uint32_t)lo | (uint32_t)hi << 16 : 0u);
                if (hi > lo && hi > eq) eq = hi;
                B += (uint32_t)nq;
            }
            if (B != B_end) atomicExch(err_flag, 2);                            // quads no segment owns
            if (t == 0) { set[0] = aq[i]; set[10] = 0; }                        // jmin; "ranges are valid"
        }
        if ((uint32_t)i * CONSUMERS < m) {                                      // (uniform)
            int32_t v = eq;
            #pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int32_t o = __shfl_up_sync(0xffffffffu, v, d); if ((int)lane >= d && o > v) v = o; }
            pb[i] = v;
            if (lane == 31) set[2 + i * N_WARPS + (int)warp] = v;
        } else pb[i] = 0;
    }
    if (m == 0 && tid == 0) { set[0] = 0; set[1] = 0; }
    consumer_sync<CONSUMERS>();
    // ---- running maximum over the blocks in front, then the two ranges as runs
    const int32_t jmin = m ? set[0] : 0;
    #pragma unroll
    for (int i = 0; i < RPT; ++i) {
        const uint32_t t = tid + (uint32_t)i * CONSUMERS;
        if ((uint32_t)i * CONSUMERS >= m) break;                                // (uniform)
        const int b = i * N_WARPS + (int)warp;
        int32_t carry = jmin;
        for (int bb = 0; bb < b; ++bb) { const int32_t v = set[2 + bb]; if (v > carry) carry = v; }
        int32_t p = pb[i] > carry ? pb[i] : carry;
        int32_t p_prev = __shfl_up_sync(0xffffffffu, p, 1);
        if (lane == 0) p_prev = carry;
        if (t < m) {
            for (int32_t j = p_prev; j < p; ++j) lohi[2 * j] = (uint16_t)k0[i];
            const int32_t upper = t + 1 < m ? read_start(t + 1) : p;
            // first segments out of coordinate order (the reads are in order of `pos`, but a CIGAR may open with a deletion): the
            // runs of hi would overlap. Such a chunk is counted with every record offered to every quad instead.
            if (t + 1 < m && upper < aq[i]) set[10] = 1;
            for (int32_t j = aq[i]; j < upper; ++j) lohi[2 * j + 1] = (uint16_t)k1[i];
            if (t + 1 == m) set[1] = p;                                         // jmax (>= jmin)
        }
    }
    consumer_sync<CONSUMERS>();
}

__device__ __forceinline__ uint2 lds_v2(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
template <int OFF> __device__ __forceinline__ uint32_t lds_u32_at(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF)); return v; }
template <int OFF> __device__ __forceinline__ uint32_t lds_u8_at(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF)); return v; }

// The records at shared addresses a_rec, a_rec + stride, ... < a_end against the NQ consecutive tile quads j0, j0 + 1, ...
// of this thread (FIX: the sample carries mate verdicts). a_qj / a_sj / a_fj: shared addresses of the qualities / bases /
// verdicts of "buffer quad j0". One record fetch and one range test serve all NQ quads (neighbouring quads are covered by
// the same segments except at a segment's ends, where the quad outside is read - the byte in front of or behind the
// segment is inside the stage - and then ignored).
template <bool FIX, int NQ>
__device__ __forceinline__ void gather_quads(uint32_t j0, uint32_t a_rec, uint32_t a_end, uint32_t stride, uint32_t a_qj, uint32_t a_sj, uint32_t a_fj,
                                             uint32_t (&D)[NQ], uint32_t (&N)[NQ], uint32_t (&X0)[NQ], uint32_t (&X1)[NQ], uint32_t (&X01)[NQ])
{
    static_assert(NQ == 1 || NQ == 2, "one or two quads per thread");
    // No branch inside: a record that covers none of this thread's quads is read at offset 0 (inside the stage) and its
    // qualities are replaced by 0, which no test passes (some lane of the warp is covered in nearly every step anyway).
    // Software pipeline, two deep: the record of step i + 2 and the quads of step i + 1 are on their way while step i is
    // counted - a thread's steps are otherwise one chain of dependent shared-memory round trips.
    struct Step { uint32_t q[NQ], sv[NQ], f[NQ]; };
    auto fetch_rec = [&](uint32_t addr) { uint2 r = make_uint2(0u, 0u); if (addr < a_end) r = lds_v2(addr); return r; };       // behind the end: an empty record
    auto issue = [&](const uint2 rec, Step& st) {
        const uint32_t a = rec.y & 0xffffu, len = (rec.y >> 16) - a, t0 = j0 - a;   // quad q is covered iff t0 + q < len (an empty record has len = 0)
        const bool in0 = t0 < len, in1 = NQ > 1 && t0 + 1u < len;
        const uint32_t x = (in0 || in1) ? rec.x : 0u;                               // rec.x + j = buffer quad of tile quad j
        const uint32_t aq = a_qj + 4u * x, as = a_sj + x, af = a_fj + x;
        st.q[0] = lds_u32_at<0>(aq); st.sv[0] = lds_u8_at<0>(as);
        if (NQ > 1) { st.q[NQ - 1] = lds_u32_at<4>(aq); st.sv[NQ - 1] = lds_u8_at<1>(as); }
        if (FIX) { st.f[0] = lds_u8_at<0>(af); if (NQ > 1) st.f[NQ - 1] = lds_u8_at<1>(af); }
        if (!in0) { st.q[0] = 0; if (FIX) st.f[0] = 0; }                            // quality 0 and no verdict: nothing counts
        if (NQ > 1 && !in1) { st.q[NQ - 1] = 0; if (FIX) st.f[NQ - 1] = 0; }
    };
    auto count = [&](const Step& st) {
        #pragma unroll
        for (int i = 0; i < NQ; ++i) {
            const uint32_t xs = msnv_spread_bases(st.sv[i]);                        // one 2-bit base per byte lane
            uint32_t ok, nn;
            quad_pass<FIX>(st.q[i], FIX ? st.f[i] : 0u, ok, nn);
            const uint32_t s1 = xs >> 1;
            D[i] += ok; N[i] += nn;
            X0[i] += xs & ok; X1[i] += s1 & ok; X01[i] += and3(xs, s1, ok);
        }
    };
    if (a_rec >= a_end) return;
    Step cur, nxt;
    uint2 r1;
    { const uint2 r0 = fetch_rec(a_rec); r1 = fetch_rec(a_rec + stride); issue(r0, cur); }
    uint32_t a_next = a_rec + 2u * stride;                                          // record of the step after next
    #pragma unroll 2
    for (; a_rec < a_end; a_rec += stride, a_next += stride) {
        issue(r1, nxt);                     // (behind the end: the empty record, offset 0, counted by nobody)
        r1 = fetch_rec(a_next);
        count(cur);
        cur = nxt;
    }
}

template <int CONSUMERS, bool HAS_WIDE>
__global__ void __launch_bounds__(CONSUMERS + 32, CONSUMERS == 128 ? 4 : 3)
pileup_gather_kernel(const SampleDev* __restrict__ samples, const Item* __restrict__ items, uint32_t n_items, const PileupShape sh,
                     const uint8_t* __restrict__ expect, uint8_t* __restrict__ tiles /*[n_items][SLOT_BYTES]*/, int* __restrict__ err_flag)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const PileupSmem L = pileup_smem_layout(sh);
    // records and ranges start out empty: a failed consistency check (which fails the run) must not leave wild indices behind
    for (uint32_t s = 0; s < sh.stages; ++s) {
        uint32_t* z = (uint32_t*)(smem + L.stage0 + s * L.stage_bytes + L.o_set);
        for (uint32_t k = threadIdx.x; k < (L.stage_bytes - L.o_set) / 4u; k += CONSUMERS + 32) z[k] = 0;
    }
    if (pileup_cta_start<CONSUMERS>(smem, L, sh, CONSUMERS / 32, samples, items, n_items, expect, err_flag)) return;   // (a stage is free when every consumer warp has read it)

    // ------------------------------------------------------------------------------------ consumers
    uint64_t* full = (uint64_t*)(smem + L.bar);
    uint64_t* empty = full + sh.stages;
    uint32_t* s_cnt = (uint32_t*)(smem + L.cnt);
    const uint32_t tid = threadIdx.x, lane = tid & 31u;
    constexpr int QPT = TILE_QUADS / CONSUMERS;                 // quad slots per thread (2 or 1): slots QPT * tid, QPT * tid + 1
    WideAcc<CONSUMERS, HAS_WIDE> acc = {};
    uint32_t D[QPT], N[QPT], X0[QPT], X1[QPT], X01[QPT];        // counts of this thread's quads (see gather_quads)
    #pragma unroll
    for (int i = 0; i < QPT; ++i) D[i] = N[i] = X0[i] = X1[i] = X01[i] = 0;

    for (uint32_t chunk_no = 0;; ++chunk_no) {
        const uint32_t st = chunk_no % sh.stages, ph = (chunk_no / sh.stages) & 1u;
        uint8_t* stage = smem + L.stage0 + st * L.stage_bytes;
        mbar_wait(full + st, ph);
        const ChunkHdr* h = (const ChunkHdr*)(stage + L.o_hdr);
        const uint32_t flags = h->flags;
        if (flags & CHUNK_STOP) break;
        gather_setup<CONSUMERS>(stage, L, err_flag);
        const uint32_t nseg = h->nseg, item = h->item, c12 = h->q4_0 & 12u;
        const uint2* recs = (const uint2*)(stage + L.o_rec);
        const uint32_t* lohi = (const uint32_t*)(stage + L.o_lohi);
        const uint32_t* s_qw = (const uint32_t*)(stage + L.o_qual);            // qualities of buffer quad B in word B
        const uint8_t* s_sq = stage + L.o_seq + c12;
        const uint8_t* s_fx = stage + L.o_fix + c12;
        const uint32_t* s_exp = (const uint32_t*)(stage + L.o_exp);
        const uint32_t* set = (const uint32_t*)(stage + L.o_set);
        const bool no_ranges = set[10] != 0;                                    // (rare: see gather_setup)
        const uint32_t jmin = no_ranges ? 0u : set[0], jmax = set[1];
        const bool has_fix = (flags & CHUNK_FIX) != 0;
        // narrow items (at most 255 reads: a byte lane cannot overflow) stay in the registers of the threads that own their
        // quads, over as many chunks as the item takes, and go from there to HBM; deep items go through the shared planes
        const bool direct = !(flags & CHUNK_WIDE);
        uint32_t wsh = 8;                                                       // log2 of the quads per group of slots
        if (!direct) { const uint32_t span = jmax - jmin; wsh = span <= 32u ? 5u : span <= 64u ? 6u : span <= 128u ? 7u : 8u; }
        const uint32_t G = (uint32_t)TILE_QUADS >> wsh;
        uint32_t* dst = reinterpret_cast<uint32_t*>(tiles + (size_t)item * SLOT_BYTES);
        const uint32_t a_recs = smem_u32(recs), a_q = smem_u32(s_qw), a_s = smem_u32(s_sq), a_f = smem_u32(s_fx);

        // this thread's QPT consecutive quad slots
        const uint32_t v0 = (uint32_t)QPT * tid;
        const uint32_t j0 = direct ? v0 : jmin + (v0 & ((1u << wsh) - 1u)), grp = direct ? 0u : v0 >> wsh;
        if (!direct || (flags & CHUNK_FIRST)) {
            #pragma unroll
            for (int i = 0; i < QPT; ++i) D[i] = N[i] = X0[i] = X1[i] = X01[i] = 0;
        }
        {
            // the quads of this thread that a segment of the chunk can cover: [ja, jb)
            const uint32_t ja = j0 > jmin ? j0 : jmin, jb = j0 + QPT < jmax ? j0 + QPT : jmax;
            if (ja < jb) {
                const uint32_t lo = no_ranges ? 0u : lohi[ja] & 0xffffu;
                uint32_t hi = no_ranges ? nseg : lohi[jb - 1u] >> 16;
                if (hi > nseg) hi = nseg;
                const uint32_t k = lo + ((grp - lo) & (G - 1u));                // first segment of this group at or behind lo
                if (has_fix) gather_quads<true, QPT>(j0, a_recs + 8u * k, a_recs + 8u * hi, 8u * G, a_q + 4u * j0, a_s + j0, a_f + j0, D, N, X0, X1, X01);
                else         gather_quads<false, QPT>(j0, a_recs + 8u * k, a_recs + 8u * hi, 8u * G, a_q + 4u * j0, a_s + j0, a_f + j0, D, N, X0, X1, X01);
            }
        }
        uint32_t out[QPT][N_PLANES];
        if (!direct || (flags & CHUNK_LAST)) {
            // letter counts from the bit-plane sums; the planes hold only the bases that DIFFER from the expected letter
            #pragma unroll
            for (int i = 0; i < QPT; ++i) {
                const uint32_t e = j0 + i < (uint32_t)TILE_QUADS ? s_exp[j0 + i] : 0u;
                const uint32_t cnt[4] = {D[i] - X0[i] - X1[i] + X01[i], X0[i] - X01[i], X1[i] - X01[i], X01[i]};
                out[i][PLANE_D] = D[i];
                #pragma unroll
                for (uint32_t l = 0; l < 4u; ++l) {
                    const uint32_t x = e ^ (l * 0x01010101u);
                    const uint32_t nz = (x | (x >> 1)) & 0x01010101u;           // lanes whose expected letter is not l
                    out[i][PLANE_A + l] = cnt[l] & (nz * 255u);
                }
                out[i][PLANE_N] = N[i];
            }
        }
        // ---- the stage is read: hand it back (per warp, no CTA-wide barrier)
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + st);

        if (direct) {
            if (flags & CHUNK_LAST) {
                #pragma unroll
                for (int c = 0; c < N_PLANES; ++c) {
                    if (QPT == 2) reinterpret_cast<uint2*>(dst)[(c * TILE_QUADS + j0) >> 1] = make_uint2(out[0][c], out[QPT - 1][c]);     // (j0 is even)
                    else dst[c * TILE_QUADS + j0] = out[0][c];
                }
            }
            continue;
        }
        // ---- deep items: partial sums into the shared planes, folded into 16-bit lanes held in registers
        #pragma unroll
        for (int i = 0; i < QPT; ++i)
            if (j0 + i < (uint32_t)TILE_QUADS) {
                #pragma unroll
                for (int c = 0; c < N_PLANES; ++c)
                    if (out[i][c]) red_shared_add(smem_u32(s_cnt) + 4u * (uint32_t)(c * TILE_QUADS + j0 + i), out[i][c]);
            }
        consumer_sync<CONSUMERS>();
        if (HAS_WIDE) {
            wide_fold<CONSUMERS, HAS_WIDE>(acc, s_cnt, tid);
            if (flags & CHUNK_LAST) wide_store<CONSUMERS, HAS_WIDE>(acc, tiles + (size_t)item * SLOT_BYTES, tid);
        }
        consumer_sync<CONSUMERS>();             // the planes are folded and cleared before the next chunk adds to them
    }
}

// ------------------------------------------------------------------------------------------------
// call: one CTA per tile, one thread per position. Sums the per-sample counts of the tile's items
// and applies snpCall's tests (call_vC.cpp:545-601). Output: one flag byte per position
// (low nibble: population mask, high nibble: individual mask, allele order A,C,G,T).
// ------------------------------------------------------------------------------------------------
// reference character -> channel of the base mpileup renders as '.'/',' (0..3 = A,C,G,T, 4 = N-like,
// 5 = none: IUPAC ambiguity codes match no read base). Derived from SAMv1's nt16 coding, the table
// mpileup's pileup_seq compares with (SURVEY.md Annex A.4).
__device__ __forceinline__ uint32_t ref_channel(uint32_t c)
{
    switch (c) {
        case 'A': case 'a': case '0': return 0;
        case 'C': case 'c': case '1': return 1;
        case 'G': case 'g': case '2': return 2;
        case 'T': case 't': case '3': return 3;
        case 'M': case 'm': case 'R': case 'r': case 'S': case 's': case 'V': case 'v': case 'W': case 'w':
        case 'Y': case 'y': case 'H': case 'h': case 'K': case 'k': case 'D': case 'd': case 'B': case 'b':
        case '=': return 5;
        default: return 4;
    }
}

// Per-position verdict from the population sums of a position (call_vC.cpp:545-601).
//   sum[a]   population count of letter a (A,C,G,T), extra = what else counts as coverage (N bases under an N-like
//   reference; the '.'/',' matches in text mode), any = bit a set when some sample has count[a] >= thr
// Returns the flag byte: low nibble population mask, high nibble individual mask.
__device__ __forceinline__ uint32_t call_position(uint32_t rc, uint32_t ch, const uint32_t sum[4], uint32_t extra, uint32_t any,
                                                  const CallParamsDev& prm)
{
    const int32_t thr = prm.thr;
    uint32_t flag = 0;
    const int64_t cov = (int64_t)sum[0] + sum[1] + sum[2] + sum[3] + extra;
    int64_t nonref = 0;
    #pragma unroll
    for (int a = 0; a < 4; ++a) if ((uint32_t)a != ch) nonref += sum[a];
    // call_vC.cpp:547-552
    if (cov >= prm.min_cov && nonref >= thr) {
        const double lim = __dmul_rn((double)cov, prm.frac);       // cov*calling_min_fraction, no FMA contraction
        #pragma unroll
        for (int a = 0; a < 4; ++a) {
            // call_vC.cpp:580: the allele is skipped only when the reference character is its lower-case letter
            const uint32_t lower = a == 0 ? 'a' : a == 1 ? 'c' : a == 2 ? 'g' : 't';
            if (rc == lower) continue;
            const int64_t n = ((uint32_t)a == ch) ? 0 : (int64_t)sum[a];
            if (n >= thr && (double)n >= lim) flag |= 1u << a;                       // population variant
            else {
                const bool indiv = ((uint32_t)a == ch) ? (0 >= thr) : ((any >> a) & 1u);
                if (indiv) flag |= 16u << a;                                         // individual variant
            }
        }
    }
    return flag;
}

// ------------------------------------------------------------------------------------------------
// call: one CTA per tile, one thread per quad of four positions. Sums the count planes of the
// tile's items over the samples (byte lanes -> 16-bit lanes -> 32 bits), tracks per letter whether
// some sample reaches the threshold, and applies snpCall's tests (call_vC.cpp:545-601).
// Output: one flag byte per position (low nibble: population mask, high nibble: individual mask,
// allele order A,C,G,T) and the number of flagged positions of the tile.
// HI_THR: the calling threshold lies in 129..255 (the byte-lane ">= thr" test needs a different
// combination); thresholds above 255 can only be met by wide items, which are compared as integers.
// ------------------------------------------------------------------------------------------------
constexpr int CALL_THREADS = TILE_QUADS;

template <bool HI_THR>
__global__ void __launch_bounds__(CALL_THREADS, 3)
call_kernel(const uint8_t* __restrict__ tiles /* slot of item `item0` first */, const Item* __restrict__ items, uint32_t item0,
            const uint32_t* __restrict__ tile_begin /* of this launch's first tile */, uint32_t tile_abs0 /* its shard tile index */,
            const uint8_t* __restrict__ ref, const uint8_t* __restrict__ expect, CallParamsDev prm, int text_mode,
            uint8_t* __restrict__ flags /* of this launch's first tile */, uint32_t* __restrict__ tile_hits)
{
    __shared__ uint32_t s_hits;
    const uint32_t t = blockIdx.x, tid = threadIdx.x;
    const uint32_t i0 = tile_begin[t], i1 = tile_begin[t + 1];
    const int32_t thr = prm.thr;
    if (tid == 0) s_hits = 0;
    // byte-lane test "lane >= thr": bit 7 of ((x & 0x7f) + tb) combined with bit 7 of x (OR for thr <= 128, AND above)
    const uint32_t tb = (HI_THR ? (thr <= 255 ? 256u - (uint32_t)thr : 0u) : (thr >= 1 ? 128u - (uint32_t)thr : 0u)) * 0x01010101u;
    uint32_t s32[N_PLANES][4];
    #pragma unroll
    for (int c = 0; c < N_PLANES; ++c) { s32[c][0] = s32[c][1] = s32[c][2] = s32[c][3] = 0; }
    uint32_t any7[5] = {0, 0, 0, 0, 0};            // bit 7 of lane p: some sample has >= thr of A, C, G, T, expected letter at position p
    const size_t lane_off = 4u * (size_t)tid;

    for (uint32_t i = i0; i < i1;) {
        const uint32_t blk_end = min(i1, i + 256u);   // 16-bit lanes hold the sums of 256 narrow items
        uint32_t s16[N_PLANES][2];
        #pragma unroll
        for (int c = 0; c < N_PLANES; ++c) { s16[c][0] = s16[c][1] = 0; }
        for (; i < blk_end; i += 4) {
            uint4 it[4]; uint32_t w[4][N_PLANES];
            #pragma unroll
            for (int u = 0; u < 4; ++u)
                it[u] = i + u < blk_end ? __ldg(reinterpret_cast<const uint4*>(items) + (i + u)) : make_uint4(0u, 0u, 0u, 0u);
            #pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool live = i + u < blk_end && !item_is_wide(it[u].z, it[u].w);
                const uint8_t* base = tiles + (size_t)(i + u - item0) * SLOT_BYTES + lane_off;
                #pragma unroll
                for (int c = 0; c < N_PLANES; ++c) w[u][c] = live ? __ldg(reinterpret_cast<const uint32_t*>(base + c * TILE)) : 0u;
            }
            #pragma unroll
            for (int u = 0; u < 4; ++u) {
                const uint32_t R = w[u][0] - (w[u][1] + w[u][2] + w[u][3] + w[u][4]);     // lane-wise: D >= A + C + G + T
                #pragma unroll
                for (int a = 0; a < 5; ++a) {
                    const uint32_t x = a < 4 ? w[u][1 + a] : R;
                    const uint32_t g = (x & 0x7f7f7f7fu) + tb;
                    any7[a] |= HI_THR ? (g & x) : (g | x);
                }
                #pragma unroll
                for (int c = 0; c < N_PLANES; ++c) { s16[c][0] += w[u][c] & 0x00ff00ffu; s16[c][1] += (w[u][c] >> 8) & 0x00ff00ffu; }
                if (i + u < blk_end && item_is_wide(it[u].z, it[u].w)) {                  // deep coverage: 16-bit planes, compared as integers
                    const uint8_t* base = tiles + (size_t)(i + u - item0) * SLOT_BYTES + 2u * lane_off;
                    uint32_t v[N_PLANES][4];
                    #pragma unroll
                    for (int c = 0; c < N_PLANES; ++c) {
                        const uint2 ww = __ldg(reinterpret_cast<const uint2*>(base + c * 2 * TILE));
                        v[c][0] = ww.x & 0xffffu; v[c][1] = ww.x >> 16; v[c][2] = ww.y & 0xffffu; v[c][3] = ww.y >> 16;
                    }
                    #pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        const uint32_t Rp = v[0][p] - (v[1][p] + v[2][p] + v[3][p] + v[4][p]);
                        #pragma unroll
                        for (int a = 0; a < 5; ++a) {
                            const uint32_t x = a < 4 ? v[1 + a][p] : Rp;
                            if ((int64_t)x >= (int64_t)thr) any7[a] |= 0x80u << (8 * p);
                        }
                        #pragma unroll
                        for (int c = 0; c < N_PLANES; ++c) s32[c][p] += v[c][p];
                    }
                }
            }
        }
        i = blk_end;
        #pragma unroll
        for (int c = 0; c < N_PLANES; ++c) {
            s32[c][0] += s16[c][0] & 0xffffu; s32[c][2] += s16[c][0] >> 16;
            s32[c][1] += s16[c][1] & 0xffffu; s32[c][3] += s16[c][1] >> 16;
        }
    }

    uint32_t out = 0, n_flagged = 0;
    if (i1 > i0) {
        const size_t p4 = (size_t)(tile_abs0 + t) * TILE + lane_off;
        const uint32_t rw = *reinterpret_cast<const uint32_t*>(ref + p4), ew = *reinterpret_cast<const uint32_t*>(expect + p4);
        #pragma unroll
        for (int p = 0; p < 4; ++p) {
            const uint32_t rc = (rw >> (8 * p)) & 0xffu, e = (ew >> (8 * p)) & 3u;
            if (rc == 0) continue;
            uint32_t sum[4] = {s32[1][p], s32[2][p], s32[3][p], s32[4][p]};
            const uint32_t rest = s32[0][p] - (sum[0] + sum[1] + sum[2] + sum[3]);      // bases equal to the expected letter / text mode: '.' and ','
            uint32_t any = 0;
            #pragma unroll
            for (int a = 0; a < 4; ++a) any |= ((any7[a] >> (8 * p + 7)) & 1u) << a;
            uint32_t ch, extra;
            if (text_mode) {
                // counts parsed from mpileup text: letters are never the reference's own base and `rest` holds the
                // '.'/',' matches, so nothing is masked (call_vC.cpp:545,550,583-584)
                ch = 6u; extra = rest;
            } else {
                #pragma unroll
                for (int a = 0; a < 4; ++a) if ((uint32_t)a == e) { sum[a] += rest; any |= ((any7[4] >> (8 * p + 7)) & 1u) << a; }
                ch = ref_channel(rc);
                extra = ch == 4u ? s32[PLANE_N][p] : 0u;
            }
            if (thr <= 0) any = 15u;
            const uint32_t f = call_position(rc, ch, sum, extra, any, prm);
            out |= f << (8 * p);
            n_flagged += f != 0;
        }
    }
    *reinterpret_cast<uint32_t*>(flags + (size_t)t * TILE + lane_off) = out;
    __syncthreads();
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) n_flagged += __shfl_down_sync(0xffffffffu, n_flagged, d);
    if ((tid & 31) == 0 && n_flagged) atomicAdd(&s_hits, n_flagged);
    __syncthreads();
    if (tid == 0) tile_hits[t] = s_hits;
}
// ordered compaction of the flagged positions: tile_hits holds exclusive offsets on entry
__global__ void __launch_bounds__(TILE)
compact_kernel(const uint8_t* __restrict__ flags, const uint32_t* __restrict__ tile_hits, uint32_t tile_abs0, uint32_t* __restrict__ hit_pos,
               uint8_t* __restrict__ hit_pop, uint8_t* __restrict__ hit_ind)
{
    __shared__ uint32_t s_warp[33];
    const uint32_t t = blockIdx.x, tid = threadIdx.x;
    const size_t p = (size_t)(tile_abs0 + t) * TILE + tid;        // shard coordinate; flags and tile_hits are this launch's
    const uint32_t f = flags[(size_t)t * TILE + tid];
    uint32_t total;
    const uint32_t r = block_rank(f != 0, s_warp, total);
    if (f) {
        const uint32_t slot = tile_hits[t] + r;
        hit_pos[slot] = (uint32_t)p;
        hit_pop[slot] = (uint8_t)(f & 15u);
        hit_ind[slot] = (uint8_t)(f >> 4);
    }
}

// the six plane values of one position of one item (bytes for narrow items, 16-bit values for wide ones)
__device__ __forceinline__ void load_planes(const uint8_t* __restrict__ tiles, uint32_t item, bool wide, uint32_t off, uint32_t v[N_PLANES])
{
    const uint8_t* base = tiles + (size_t)item * SLOT_BYTES;
    #pragma unroll
    for (int c = 0; c < N_PLANES; ++c)
        v[c] = wide ? (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(base) + c * TILE + off) : (uint32_t)__ldg(base + c * TILE + off);
}

// per hit: per-sample coverage and allele counts (zero for samples without an item on the tile)
// plus population totals. One CTA of 128 threads per hit; outputs were zero-filled by the host side.
__global__ void __launch_bounds__(128)
gather_kernel(const uint8_t* __restrict__ tiles, const Item* __restrict__ items, uint32_t item0,
              const uint32_t* __restrict__ tile_begin /* of the window's first tile */, uint32_t win_tile0, const uint8_t* __restrict__ ref, const uint8_t* __restrict__ expect, const uint32_t* __restrict__ hit_pos,
              uint32_t n_samples, int text_mode, uint16_t* __restrict__ cov, uint16_t* __restrict__ allele, uint32_t* __restrict__ total)
{
    __shared__ uint32_t s_tot[5];
    const uint32_t h = blockIdx.x, tid = threadIdx.x;
    const uint32_t p = hit_pos[h];
    const uint32_t t = p / TILE - win_tile0, off = p % TILE;
    const uint32_t ch = text_mode ? 6u : ref_channel(ref[p]);
    const uint32_t e = expect[p] & 3u;
    if (tid < 5) s_tot[tid] = 0;
    __syncthreads();
    uint32_t tc = 0, ta[4] = {0, 0, 0, 0};
    for (uint32_t i = tile_begin[t] + tid; i < tile_begin[t + 1]; i += blockDim.x) {
        const uint4 it = __ldg(reinterpret_cast<const uint4*>(items) + i);
        uint32_t v[N_PLANES];
        load_planes(tiles, i - item0, item_is_wide(it.z, it.w), off, v);
        const uint32_t rest = v[0] - (v[1] + v[2] + v[3] + v[4]);
        uint32_t c[4] = {v[1], v[2], v[3], v[4]}, cv;
        if (text_mode) cv = rest;
        else {
            #pragma unroll
            for (int a = 0; a < 4; ++a) if ((uint32_t)a == e) c[a] += rest;
            cv = ch == 4u ? v[PLANE_N] : 0u;
        }
        #pragma unroll
        for (int a = 0; a < 4; ++a) { cv += c[a]; if ((uint32_t)a == ch) c[a] = 0; }
        cov[(size_t)h * n_samples + it.x] = (uint16_t)cv;
        #pragma unroll
        for (int a = 0; a < 4; ++a) { allele[((size_t)h * 4 + a) * n_samples + it.x] = (uint16_t)c[a]; ta[a] += c[a]; }
        tc += cv;
    }
    atomicAdd(&s_tot[0], tc);
    #pragma unroll
    for (int a = 0; a < 4; ++a) atomicAdd(&s_tot[1 + a], ta[a]);
    __syncthreads();
    if (tid < 5) total[(size_t)h * 5 + tid] = s_tot[tid];
}

// inspection hook: one sample's counts for a position range as [n][5] u16 (A, C, G, T, non-ACGT)
__global__ void counts_kernel(const uint8_t* __restrict__ tiles, const Item* __restrict__ items, uint32_t item0,
                              const uint32_t* __restrict__ tile_begin /* of the window's first tile */, uint32_t win_tile0,
                              const uint8_t* __restrict__ expect, uint32_t sample, uint32_t first, uint32_t n, uint16_t* __restrict__ out)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t p = first + k, t = p / TILE - win_tile0, off = p % TILE;
    uint32_t r[5] = {0, 0, 0, 0, 0};
    for (uint32_t i = tile_begin[t]; i < tile_begin[t + 1]; ++i) {
        const uint4 it = __ldg(reinterpret_cast<const uint4*>(items) + i);
        if (it.x != sample) continue;
        uint32_t v[N_PLANES];
        load_planes(tiles, i - item0, item_is_wide(it.z, it.w), off, v);
        const uint32_t e = expect[p] & 3u;
        for (int a = 0; a < 4; ++a) r[a] = v[1 + a] + ((uint32_t)a == e ? v[0] - (v[1] + v[2] + v[3] + v[4]) : 0u);
        r[4] = v[PLANE_N];
        break;
    }
    for (int a = 0; a < 5; ++a) out[(size_t)k * 5 + a] = (uint16_t)r[a];
}

// classic text mode: counts parsed by the host from mpileup text ([item][TILE]: packed letter counts and '.'/','
// matches) -> wide count planes. D holds everything counted, so "D - letters" gives the matches back.
__global__ void text_tiles_kernel(const uint64_t* __restrict__ acgt, const uint16_t* __restrict__ matches, uint64_t n_cells,
                                  uint8_t* __restrict__ tiles)
{
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_cells) return;
    const uint64_t item = g / TILE; const uint32_t off = (uint32_t)(g % TILE);
    const uint64_t w = acgt[g];
    uint32_t c[4], sum = matches[g];
    for (int a = 0; a < 4; ++a) { c[a] = (uint32_t)(w >> (16 * a)) & 0xffffu; sum += c[a]; }
    uint16_t* base = reinterpret_cast<uint16_t*>(tiles + item * SLOT_BYTES);
    base[off] = (uint16_t)(sum > 0xffffu ? 0xffffu : sum);
    for (int a = 0; a < 4; ++a) base[(1 + a) * TILE + off] = (uint16_t)c[a];
    base[PLANE_N * TILE + off] = 0;
}

// ------------------------------------------------------------------------------------------------
// coverage (qaCompute.cpp:530-552 scatter, :142-165 prefix sum + histogram).
// Contigs that have reads are laid out in a "coverage coordinate" space, each starting at a multiple
// of COV_CHUNK. A block [beg,end) contributes +1 at beg and -1 at end like the reference's
// difference array, but every chunk it enters gets its own +1 at the chunk's first index, so each
// chunk is prefix-summed independently by one CTA: no carries between CTAs, one pass over HBM.
// The histogram's first COV_MAX_BINS bins are collected in shared memory; coverage values above
// them (qaCompute -c 1024 and more, deep spots only) go straight to the global histogram.
// ------------------------------------------------------------------------------------------------
constexpr int COV_CHUNK = 4096;
constexpr int COV_THREADS = 256;              // x 16 positions per thread = one chunk
constexpr int COV_MAX_BINS = 1024;            // bins held in shared memory

__global__ void __launch_bounds__(256)
cov_scatter_kernel(const uint32_t* __restrict__ beg, const uint32_t* __restrict__ end, const uint64_t* __restrict__ blk_off,
                   const uint32_t* __restrict__ contig_chunk0, uint32_t n_contigs, uint64_t n_blocks, int32_t* __restrict__ diff)
{
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_blocks) return;
    uint32_t lo = 0, hi = n_contigs;                       // contig of this block: blk_off[lo] <= g < blk_off[lo+1]
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (__ldg(blk_off + mid) <= g) lo = mid; else hi = mid; }
    const uint32_t b = __ldg(beg + g), e = __ldg(end + g);
    if (e <= b) return;
    int32_t* d = diff + (size_t)__ldg(contig_chunk0 + lo) * COV_CHUNK;
    for (uint32_t c = b / COV_CHUNK; c <= (e - 1) / COV_CHUNK; ++c) {
        const uint32_t c0 = c * COV_CHUNK;
        atomicAdd(d + (b > c0 ? b : c0), 1);
        if (e < c0 + COV_CHUNK) atomicAdd(d + e, -1);
    }
}

__global__ void __launch_bounds__(COV_THREADS)
cov_scan_kernel(const int32_t* __restrict__ diff, const uint32_t* __restrict__ chunk_contig, const uint32_t* __restrict__ contig_chunk0,
                const uint32_t* __restrict__ contig_len, uint32_t max_cov, unsigned long long* __restrict__ cov_sum,
                unsigned long long* __restrict__ hist /*[n_contigs][max_cov+1]*/)
{
    // 256 threads x 16 consecutive positions: many small CTAs per SM (the scan needs two barriers, and a CTA of 1024
    // threads spent most of its life in them), four 16-byte loads in flight per thread
    static_assert(COV_THREADS * 16 == COV_CHUNK, "a CTA scans one chunk");
    __shared__ int32_t s_warp[COV_THREADS / 32];
    __shared__ uint32_t s_hist[COV_MAX_BINS];
    __shared__ unsigned long long s_sum;
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t k = chunk_contig[blockIdx.x];
    const uint32_t first = (blockIdx.x - contig_chunk0[k]) * COV_CHUNK;        // contig coordinate of the chunk's first index
    const uint32_t len = contig_len[k];
    const uint32_t n_shared = max_cov < (uint32_t)COV_MAX_BINS ? max_cov + 1u : (uint32_t)COV_MAX_BINS;
    unsigned long long* const g_hist = hist + (size_t)k * ((size_t)max_cov + 1);
    for (uint32_t i = tid; i < n_shared; i += COV_THREADS) s_hist[i] = 0;
    if (tid == 0) s_sum = 0;
    const int4* src = reinterpret_cast<const int4*>(diff + (size_t)blockIdx.x * COV_CHUNK) + 4 * tid;
    const int4 v[4] = {src[0], src[1], src[2], src[3]};
    int32_t c[16];
    int32_t run = 0;
    #pragma unroll
    for (int i = 0; i < 4; ++i) { c[4 * i] = run += v[i].x; c[4 * i + 1] = run += v[i].y; c[4 * i + 2] = run += v[i].z; c[4 * i + 3] = run += v[i].w; }
    int32_t incl = run;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int32_t base = incl - run;
    #pragma unroll
    for (int w = 0; w < COV_THREADS / 32; ++w) if ((uint32_t)w < warp) base += s_warp[w];
    unsigned long long local = 0;
    #pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t p = first + tid * 16 + j;
        const bool valid = p < len;
        const int32_t cv = base + c[j];
        // negative coverage cannot occur for blocks that satisfy the ABI contract (beg < end)
        uint32_t bin = cv < 0 ? 0u : ((uint32_t)cv > max_cov ? max_cov : (uint32_t)cv);
        if (!valid) bin = 0xffffffffu;
        else local += (unsigned long long)(cv < 0 ? 0 : cv);
        const uint32_t peers = __match_any_sync(0xffffffffu, bin);
        if (valid && lane == (uint32_t)(__ffs(peers) - 1)) {
            if (bin < n_shared) atomicAdd(&s_hist[bin], (uint32_t)__popc(peers));
            else atomicAdd(g_hist + bin, (unsigned long long)__popc(peers));
        }
    }
    #pragma unroll
    for (int d = 16; d > 0; d >>= 1) local += __shfl_down_sync(0xffffffffu, local, d);
    if (lane == 0 && local) atomicAdd(&s_sum, local);
    __syncthreads();
    for (uint32_t i = tid; i < n_shared; i += COV_THREADS)
        if (s_hist[i]) atomicAdd(g_hist + i, (unsigned long long)s_hist[i]);
    if (tid == 0 && s_sum) atomicAdd(cov_sum + k, s_sum);
}

}  // namespace msnv_gpu


