// msnv_gpu.cu -- implementation of the C ABI in include/msnv.h (libmsnv_gpu.so).
// Host-side orchestration only: device memory, streams, kernel launches, result copies.
// Kernels are in kernels.cuh. There is no CPU fallback: every entry point needs a CUDA device.
//
// A shard is processed as one or more position WINDOWS. The reads of a window live in one of two
// window slots, so the upload of the next window (copy stream) overlaps the kernels of the current
// one (compute stream). Within a window the index runs once; pileup, call, compaction and gather
// then run over ranges of tiles sized so that the count planes of a range fit the tile budget
// (free device memory, or MSNV_TILE_BUDGET_MB): neither the reads nor the counts of a whole shard
// have to fit the device (the reference streams with O(samples) memory, call_vC.cpp:466-479).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "inflate_kernels.cuh"
#include "kernels.cuh"
#include "synth_kernels.cuh"
#include "../host/sample_layout.hpp"

using namespace msnv_gpu;
using msnv::BlockLayout; using msnv::ReadGroup; using msnv::SegmentGroup; using msnv::RawGroup;

// A block of device (cudaMalloc) or pinned host (cudaMallocHost) memory that this object owns, with its capacity in
// elements. ensure() frees the old block before it allocates the new one, so growing never holds both. A failed
// allocation leaves the buffer empty and clears the runtime's last error: the caller reports it, and a later call that
// needs the buffer allocates it again.
template <class T, cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
struct Buf {
    T* p = nullptr;
    uint64_t cap = 0;
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { reset(); }
    operator T*() const { return p; }
    void reset() { if (p) Free(p); p = nullptr; cap = 0; }
    // room for n elements; `want` (>= n) of them when it has to grow. With `keep` the first keep elements survive: the
    // new block is then allocated and filled before the old one is freed (pinned memory only).
    cudaError_t ensure(uint64_t n, uint64_t want, uint64_t keep = 0)
    {
        if (n <= cap) return cudaSuccess;
        if (!keep) reset();
        T* q = nullptr;
        const cudaError_t e = Alloc((void**)&q, (size_t)want * sizeof(T));
        if (e != cudaSuccess) { cudaGetLastError(); reset(); return e; }
        if (keep) memcpy(q, p, (size_t)keep * sizeof(T));
        reset();
        p = q; cap = want;
        return cudaSuccess;
    }
    cudaError_t ensure(uint64_t n) { return ensure(n, n); }
};
template <class T> using DevBuf = Buf<T, cudaMalloc, cudaFree>;
template <class T> using PinnedBuf = Buf<T, cudaMallocHost, cudaFreeHost>;

// f(a.pos, b.pos, ..., w) for each of the six arrays of the hit sets a, b, ...; w is the array's elements per hit
template <class F, class... H>
void each_hit_array(uint64_t S, F f, H&... h)
{
    f(h.pos..., 1); f(h.total..., 5); f(h.pop..., 1); f(h.ind..., 1); f(h.cov..., S); f(h.allele..., 4 * S);
}

// The called positions as six parallel arrays: position, totals, population and individual masks, and per sample the
// coverage and the allele counts. One set on the device holds the hits of a range, one pinned set those of a window.
template <template <class> class B>
struct HitArrays {
    B<uint32_t> pos, total; B<uint8_t> pop, ind; B<uint16_t> cov, allele;
    // room for n hits of S samples, `cap` hits when it grows; the first `keep` hits survive the growth (pinned sets).
    // Without hits to keep every old block is freed before the first new one is allocated.
    cudaError_t ensure(uint64_t n, uint64_t S, uint64_t cap, uint64_t keep = 0)
    {
        bool fits = true;
        each_hit_array(S, [&](auto& b, uint64_t w) { fits = fits && n * w <= b.cap; }, *this);
        if (fits) return cudaSuccess;
        if (!keep) each_hit_array(S, [](auto& b, uint64_t) { b.reset(); }, *this);
        cudaError_t e = cudaSuccess;
        each_hit_array(S, [&](auto& b, uint64_t w) { if (e == cudaSuccess) e = b.ensure(n * w, cap * w, keep * w); }, *this);
        return e;
    }
};

constexpr int N_SLOTS = 2;

struct msnv_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;        // kernels and result copies
    cudaStream_t copy_stream = nullptr;   // uploads of the reads
    std::string err;

    struct Block { void* p; size_t bytes; bool in_slab; uint64_t gen; };
    struct Slab { uint8_t* base; size_t size, used; };
    // the reads of one window
    struct Window {
        bool open = false;
        uint32_t t0 = 0, t1 = 0;                    // tiles [t0, t1) of the shard
        std::vector<SampleDev> h_samples;           // [S]
        std::vector<msnv_sample_sizes> sizes;       // [S]
        std::vector<Block> allocs;                  // device blocks holding the samples
        uint64_t n_reads = 0, n_bases = 0, n_segs = 0;
        DevBuf<SampleDev> d_samples;
        DevBuf<unsigned long long> d_aligned; bool has_raw = false;     // aligned bases per sample (samples expanded on the device)
        cudaEvent_t uploaded = nullptr;
    };

    // ---- shard state
    bool open = false, has_run = false;
    uint32_t S = 0, P = 0, n_tiles = 0;
    Window win[N_SLOTS];
    std::vector<Block> pool;            // blocks of finished windows / shards, reused by later ones
    std::vector<Slab> slabs;            // small blocks are carved out of large allocations
    uint64_t gen = 0;                   // counts msnv_window_begin calls: pool entries unused for a while are freed
    DevBuf<uint8_t> d_ref;
    DevBuf<uint8_t> d_expect;           // expected letter per position (derived from d_ref)

    // ---- work buffers (grown on demand, kept across windows and shards)
    DevBuf<Item> d_items;
    DevBuf<uint8_t> d_tiles;            // count planes, SLOT_BYTES per item of a range
    DevBuf<uint64_t> d_text_acgt; DevBuf<uint16_t> d_text_match;   // classic text mode staging
    int sm_count = 0;
    DevBuf<uint32_t> d_tile_begin, d_tile_hits; DevBuf<uint8_t> d_flags;
    std::vector<uint32_t> h_tile_begin;
    DevBuf<uint32_t> d_block_sums;
    DevBuf<uint2> d_range_cache;
    DevBuf<uint32_t> d_bitmap;
    DevBuf<uint32_t> d_scalar; DevBuf<int> d_err;
    DevBuf<uint32_t> d_fix_list;        // samples with mate links
    // raw (BAM-shaped) reads of the sample being expanded: one staging buffer, reused in stream order
    DevBuf<uint8_t> d_raw;
    DevBuf<unsigned long long> d_xstat;  // [0] IUPAC bases seen by expand_kernel, [1] inconsistent record flag
    // what msnv_shard_counts can still look at: the last range of the last run
    uint32_t last_slot = 0, last_item0 = 0, last_ta = 0, last_tb = 0;

    // ---- hits: device buffers for one range, pinned host arrays for the whole window
    HitArrays<DevBuf> d_hits;
    HitArrays<PinnedBuf> h_hits;
    PinnedBuf<uint32_t> h_scalar;       // 8 words

    // coverage pass: work buffers grown on demand and kept (one call per BAM, hundreds of calls per job)
    DevBuf<int32_t> d_cov_diff;
    DevBuf<uint32_t> d_cov_beg, d_cov_end;
    DevBuf<uint32_t> d_cov_meta;        // chunk0 | chunk_contig | contig_len | blk_off (as 2 words each)
    DevBuf<unsigned long long> d_cov_out;  // cov_sum | hist
    cudaEvent_t ev[8] = {};
    msnv_timings tm = {};
};

namespace {

// records the error on a context or an inflater and returns `code`
template <class Obj>
int fail(Obj* o, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (o) o->err = buf;
    return code;
}

// (the object the error is recorded on is `ctx`, a context or an inflater)
#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return fail(ctx, MSNV_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Blocks of a finished window go to a pool: the next window (or the next genome bin of the same sample set)
// reuses them instead of paying cudaFree (a device-wide sync) and cudaMalloc per sample. Blocks below
// SLAB_BYTES / 4 are carved out of SLAB_BYTES allocations: a job with hundreds of small samples would
// otherwise make hundreds of cudaMalloc calls while the decoder threads fault pages in, and the two
// contend for the process's address-space lock (measured: 0.7 s vs 3.4 s for 400 samples). Carved blocks
// are never given back individually; they stay in the pool and are reused by best fit.
constexpr size_t SLAB_BYTES = 256u << 20;

void release_window(msnv_ctx* ctx, msnv_ctx::Window& w)
{
    for (auto& b : w.allocs) { b.gen = ctx->gen; ctx->pool.push_back(b); }
    w.allocs.clear();
    w.h_samples.clear(); w.sizes.clear();
    w.n_reads = w.n_bases = w.n_segs = 0;
    w.open = false; w.has_raw = false;
    // plain blocks nobody has reused for a few windows are returned to the driver
    size_t k = 0;
    for (size_t i = 0; i < ctx->pool.size(); ++i) {
        const msnv_ctx::Block& b = ctx->pool[i];
        if (!b.in_slab && b.gen + 4 < ctx->gen) cudaFree(b.p);
        else ctx->pool[k++] = b;
    }
    ctx->pool.resize(k);
}

void drop_pool(msnv_ctx* ctx)
{
    for (auto& b : ctx->pool) if (!b.in_slab) cudaFree(b.p);
    ctx->pool.clear();
}

void* take_block(msnv_ctx* ctx, msnv_ctx::Window& w, size_t bytes)
{
    size_t best = (size_t)-1, bi = 0;
    for (size_t i = 0; i < ctx->pool.size(); ++i)
        if (ctx->pool[i].bytes >= bytes && ctx->pool[i].bytes < best) { best = ctx->pool[i].bytes; bi = i; }
    if (best != (size_t)-1 && best <= bytes + bytes / 4 + (1u << 20)) {
        void* p = ctx->pool[bi].p;
        w.allocs.push_back(ctx->pool[bi]);
        ctx->pool[bi] = ctx->pool.back(); ctx->pool.pop_back();
        return p;
    }
    if (bytes <= SLAB_BYTES / 4) {
        const size_t need = align_up(bytes, 256);
        for (int attempt = 0; attempt < 2; ++attempt) {
            for (auto& sl : ctx->slabs)
                if (sl.size - sl.used >= need) {
                    void* p = sl.base + sl.used;
                    sl.used += need;
                    w.allocs.push_back({p, need, true, ctx->gen});
                    return p;
                }
            void* base = nullptr;
            if (attempt || cudaMalloc(&base, SLAB_BYTES) != cudaSuccess) { cudaGetLastError(); break; }   // fall through to a plain block
            ctx->slabs.push_back({(uint8_t*)base, SLAB_BYTES, 0});
        }
    }
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        drop_pool(ctx);                                      // give the pool back and retry once
        if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    w.allocs.push_back({p, bytes, false, ctx->gen});
    return p;
}

// count-plane slots one range may use: what the device has free (less a reserve), or MSNV_TILE_BUDGET_MB
uint64_t tile_budget_slots(msnv_ctx* ctx)
{
    size_t budget;
    if (const char* e = getenv("MSNV_TILE_BUDGET_MB")) budget = (size_t)(atof(e) * 1048576.0);
    else {
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { cudaGetLastError(); fr = (size_t)8 << 30; }
        fr += ctx->d_tiles.cap;                                 // what the buffer holds already is ours to use
        // the called positions of a range need buffers too (10 bytes per hit and sample): a third of what is free stays for them
        const size_t reserve = (size_t)2 << 30;
        budget = fr > 3 * reserve ? (fr - reserve) / 3 * 2 : fr / 2;
    }
    return budget / SLOT_BYTES;
}

int ensure_tile_slots(msnv_ctx* ctx, uint64_t n)
{
    if (ctx->d_tiles.ensure(n * SLOT_BYTES, (n + n / 16 + 16) * SLOT_BYTES) != cudaSuccess && ctx->d_tiles.ensure(n * SLOT_BYTES) != cudaSuccess)
        return fail(ctx, MSNV_E_NOMEM, "count planes for %llu (sample, tile) items do not fit device memory", (unsigned long long)n);
    return MSNV_OK;
}

int ensure_window_buffers(msnv_ctx* ctx, uint32_t n_tiles_w)
{
    CU(ctx->d_tile_begin.ensure((uint64_t)n_tiles_w + 1));
    CU(ctx->d_tile_hits.ensure((uint64_t)n_tiles_w + 1));
    CU(ctx->d_flags.ensure((uint64_t)n_tiles_w * TILE));
    return MSNV_OK;
}

}  // namespace

// Staging limits of the pileup kernel for a shard (PileupShape) and the CTAs per SM they allow. A stage should hold
// a whole item in the common case: the limits follow the mean number of reads per item (measured by the index pass)
// with head-room for its spread; what is left of the SM's shared memory after fitting `ctas` CTAs goes into larger
// quad buffers. MSNV_MAX_READS / MSNV_CHUNK_Q4 / MSNV_PILEUP_CTAS override the choice (tuning hooks).
constexpr size_t SMEM_PER_SM = 233472, SMEM_PER_CTA_MAX = 232448, SMEM_CTA_RESERVED = 1024;
constexpr uint32_t CHUNK_Q4_CAP = 16384;

// Which pileup kernel: the gather form (counts in registers, kernels.cuh) for ordinary depth, the scatter form for deep shards
// (hundreds of reads per position: a chunk of 255 reads then covers ~30 quads and the scatter's one atomic per staged quad
// costs less than the gather's record per (quad, segment) step; measured at C4, profiles/r02_pileup_ablations.txt).
// MSNV_PILEUP=gather|scatter overrides.
static bool pileup_gather_mode(bool deep)
{
    if (const char* e = getenv("MSNV_PILEUP")) {
        if (!strcmp(e, "scatter")) return false;
        if (!strcmp(e, "gather")) return true;
    }
    return !deep;
}

// the pileup kernel of a form, a number of consumer threads per CTA (128 or 256) and with or without the 16-bit accumulators
using PileupKernelFn = void (*)(const SampleDev*, const Item*, uint32_t, const PileupShape, const uint8_t*, uint8_t*, int*);
static PileupKernelFn pileup_kernel_for(bool gather, int consumers, bool has_wide)
{
    if (gather) {
        if (consumers == 256) return has_wide ? pileup_gather_kernel<256, true> : pileup_gather_kernel<256, false>;
        return has_wide ? pileup_gather_kernel<128, true> : pileup_gather_kernel<128, false>;
    }
    if (consumers == 256) return has_wide ? pileup_kernel<256, true> : pileup_kernel<256, false>;
    return has_wide ? pileup_kernel<128, true> : pileup_kernel<128, false>;
}

// deep: the shard averages more than 200 reads per item (items take several chunks whatever the limits)
static PileupShape choose_pileup_shape(uint64_t n_reads, uint64_t n_bases, uint64_t n_segs, uint64_t n_items, uint64_t item_reads, uint32_t item_reads_max, bool has_fix, bool deep,
                                       int max_ctas, int& ctas)
{
    const double reads_per_item = (double)item_reads / (double)(n_items ? n_items : 1);
    const double q4_per_read = (double)n_bases / 4.0 / (double)(n_reads ? n_reads : 1);
    const double segs_per_read = (double)n_segs / (double)(n_reads ? n_reads : 1);
    PileupShape sh{};
    sh.gather = pileup_gather_mode(deep) ? 1u : 0u;
    sh.has_fix = has_fix ? 1u : 0u;
    sh.stages = 2;
    if (const char* e = getenv("MSNV_STAGES")) { const int v = atoi(e); if (v >= 2 && v <= (int)PL_STAGES_MAX) sh.stages = (uint32_t)v; }
    uint32_t mr = deep ? (max_ctas <= 3 ? NARROW_MAX_READS : 96u) : (uint32_t)(reads_per_item * 1.3 + 24.0);
    if (!deep && item_reads_max && mr > item_reads_max) mr = item_reads_max;      // no item has more reads than this
    if (const char* e = getenv("MSNV_MAX_READS")) mr = (uint32_t)atoi(e);
    if (mr < 16) mr = 16;
    if (mr > NARROW_MAX_READS) mr = NARROW_MAX_READS;
    sh.max_reads = mr;
    uint32_t ms = (uint32_t)(mr * segs_per_read * 1.1 + 16.0);
    if (ms < CHUNK_SEGS_MIN) ms = CHUNK_SEGS_MIN;
    sh.max_segs = up_to(ms, 8);
    // quads per stage: `want` holds a whole item with head-room for the spread of the items' sizes, `least` is what is
    // accepted for the sake of one more CTA per SM (a few per cent of the items then take a second chunk)
    auto clampq = [](double q) { uint32_t v = q < 0 ? 0u : (uint32_t)q; if (v < CHUNK_Q4_MIN) v = CHUNK_Q4_MIN; if (v > CHUNK_Q4_CAP) v = CHUNK_Q4_CAP; return up_to(v, 16); };
    uint32_t want = deep ? clampq(mr * q4_per_read * 1.15 + 64.0) : clampq((reads_per_item * 1.25 + 4.0) * q4_per_read + 64.0);
    uint32_t least = deep ? want : clampq(reads_per_item * 1.12 * q4_per_read);
    if (!deep && item_reads_max) least = std::min(least, clampq((item_reads_max + 1.0) * q4_per_read + 32.0));      // (the largest item, with a little slack)
    if (const char* e = getenv("MSNV_CHUNK_Q4")) want = least = clampq((double)atoi(e));
    auto total_at = [&](uint32_t cq) { PileupShape t = sh; t.chunk_q4 = cq; return (size_t)pileup_smem_layout(t).total; };
    if (const char* e = getenv("MSNV_PILEUP_CTAS")) { const int v = atoi(e); if (v >= 1 && v < max_ctas) max_ctas = v; }
    ctas = 1;
    for (int c = max_ctas; c >= 1; --c)
        if (total_at(least) + SMEM_CTA_RESERVED <= SMEM_PER_SM / c && total_at(least) <= SMEM_PER_CTA_MAX) { ctas = c; break; }
    // the largest stage that keeps this many CTAs per SM, up to `want` (deep shards: exactly the read limit's worth)
    const size_t budget = std::min<size_t>(SMEM_PER_SM / ctas - SMEM_CTA_RESERVED, SMEM_PER_CTA_MAX);
    uint32_t cq = least;
    while (cq + 16 <= (getenv("MSNV_CHUNK_Q4") || deep ? want : CHUNK_Q4_CAP) && total_at(cq + 16) <= budget) cq += 16;
    while (cq > CHUNK_Q4_MIN && total_at(cq) > budget) cq -= 16;
    sh.chunk_q4 = cq;
    return sh;
}


// One range of a window: items [a, b) = tiles [ta, tb) of the window. The caller has filled the range's count
// planes (slot of item `a` first). call -> ordered compaction -> per-hit gather -> copy to the host arrays behind
// the `n_before` hits of earlier ranges. `acc` collects the device times of the phases.
struct PhaseTimes { float call = 0, compact = 0, gather = 0, d2h = 0; };

static int call_range(msnv_ctx* ctx, const msnv_ctx::Window& w, uint32_t a, uint32_t ta, uint32_t tb, const msnv_call_params* prm,
                      int text_mode, uint32_t n_before, uint32_t& n_range, uint32_t& launches, PhaseTimes& acc)
{
    cudaStream_t st = ctx->stream;
    const uint32_t S = ctx->S, nt = tb - ta;
    CallParamsDev cp{prm->min_coverage, prm->calling_threshold, prm->min_fraction};
    CU(cudaEventRecord(ctx->ev[3], st));
    if (cp.thr > 128)
        call_kernel<true><<<nt, CALL_THREADS, 0, st>>>(ctx->d_tiles, ctx->d_items, a, ctx->d_tile_begin + ta, w.t0 + ta, ctx->d_ref, ctx->d_expect, cp,
                                                       text_mode, ctx->d_flags + (size_t)ta * TILE, ctx->d_tile_hits + ta);
    else
        call_kernel<false><<<nt, CALL_THREADS, 0, st>>>(ctx->d_tiles, ctx->d_items, a, ctx->d_tile_begin + ta, w.t0 + ta, ctx->d_ref, ctx->d_expect, cp,
                                                        text_mode, ctx->d_flags + (size_t)ta * TILE, ctx->d_tile_hits + ta);
    ++launches;
    CU(cudaEventRecord(ctx->ev[4], st));

    // ---- ordered compaction of the called positions
    scan_kernel<<<1, 1024, 0, st>>>(ctx->d_tile_hits + ta, nt, ctx->d_scalar + 1);
    ++launches;
    CU(cudaMemcpyAsync(ctx->h_scalar + 1, ctx->d_scalar + 1, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ctx->h_scalar + 6, ctx->d_err, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (ctx->h_scalar[6]) return fail(ctx, MSNV_E_LIMIT, "a read exceeds MSNV_MAX_READ_BASES / MSNV_MAX_READ_SEGMENTS, or its offsets and segments disagree");
    const uint32_t n_hits = ctx->h_scalar[1];
    n_range = n_hits;
    const uint64_t n_window = (uint64_t)n_before + n_hits;
    CU(ctx->d_hits.ensure(n_hits, S, (uint64_t)n_hits + n_hits / 4 + 1024));
    CU(ctx->h_hits.ensure(n_window, S, n_window + n_window / 2 + 1024, n_before));
    HitArrays<DevBuf>& d = ctx->d_hits;
    if (n_hits) {
        compact_kernel<<<nt, TILE, 0, st>>>(ctx->d_flags + (size_t)ta * TILE, ctx->d_tile_hits + ta, w.t0 + ta, d.pos, d.pop, d.ind);
        ++launches;
    }
    CU(cudaEventRecord(ctx->ev[5], st));

    // ---- per-hit, per-sample numbers for the formatter
    if (n_hits) {
        CU(cudaMemsetAsync(d.cov, 0, (size_t)n_hits * S * 2, st));
        CU(cudaMemsetAsync(d.allele, 0, (size_t)n_hits * S * 8, st));
        gather_kernel<<<n_hits, 128, 0, st>>>(ctx->d_tiles, ctx->d_items, a, ctx->d_tile_begin, w.t0, ctx->d_ref, ctx->d_expect, d.pos, S,
                                               text_mode, d.cov, d.allele, d.total);
        ++launches;
    }
    CU(cudaEventRecord(ctx->ev[6], st));
    if (n_hits) {
        cudaError_t e = cudaSuccess;
        each_hit_array(S, [&](auto& h, auto& dv, uint64_t k) {
            if (e == cudaSuccess) e = cudaMemcpyAsync(h.p + n_before * k, dv.p, n_hits * k * sizeof *dv.p, cudaMemcpyDeviceToHost, st);
        }, ctx->h_hits, d);
        if (e != cudaSuccess) return fail(ctx, MSNV_E_CUDA, "copy of the hits to the host failed: %s", cudaGetErrorString(e));
    }
    CU(cudaEventRecord(ctx->ev[7], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    float ms;
    cudaEventElapsedTime(&ms, ctx->ev[3], ctx->ev[4]); acc.call += ms;
    cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]); acc.compact += ms;
    cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[6]); acc.gather += ms;
    cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]); acc.d2h += ms;
    return MSNV_OK;
}

static void publish_hits(msnv_ctx* ctx, uint32_t n_hits, msnv_hits* hits)
{
    hits->n_hits = n_hits;
    hits->n_samples = ctx->S;
    const HitArrays<PinnedBuf>& h = ctx->h_hits;
    hits->pos = h.pos; hits->pop_mask = h.pop; hits->ind_mask = h.ind; hits->cov = h.cov; hits->allele = h.allele; hits->total = h.total;
}

// the pileup kernel over items [a, a + n) of the window, count planes to d_tiles (slot 0 = item a)
static int launch_pileup(msnv_ctx* ctx, const msnv_ctx::Window& w, uint32_t a, uint32_t n, uint64_t n_items_window, uint64_t item_reads,
                         uint32_t item_reads_max, uint32_t& launches)
{
    // consumer threads per CTA (MSNV_CONSUMERS overrides); the 16-bit accumulators only where an item can need them
    // (measured: four CTAs of 128 consumers for shallow shards, larger CTAs with 255-read chunks for deep ones)
    const bool deep = (double)item_reads > 200.0 * (double)(n_items_window ? n_items_window : 1);
    int consumers = deep ? 256 : 128;
    if (const char* e = getenv("MSNV_CONSUMERS")) consumers = atoi(e) == 256 ? 256 : 128;
    int ctas = 1;
    bool has_fix = false;
    for (const SampleDev& sd : w.h_samples) has_fix = has_fix || sd.fix;
    const PileupShape sh = choose_pileup_shape(w.n_reads, w.n_bases, w.n_segs, n_items_window, item_reads, item_reads_max, has_fix, deep, consumers == 256 ? 3 : 4, ctas);   // register-bound CTA counts
    const size_t smem = pileup_smem_layout(sh).total;
    const bool has_wide = item_reads_max > NARROW_MAX_READS;
    const int threads = consumers + 32;
    const PileupKernelFn K = pileup_kernel_for(sh.gather, consumers, has_wide);
    int fit = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, K, threads, smem));
    if (fit < 1) return fail(ctx, MSNV_E_CUDA, "pileup kernel does not fit an SM (%zu bytes of shared memory)", smem);
    if (fit < ctas) ctas = fit;
    uint64_t grid = (uint64_t)ctas * (uint64_t)ctx->sm_count;
    if (grid > n) grid = n;
    K<<<(unsigned)grid, threads, smem, ctx->stream>>>(w.d_samples, ctx->d_items + a, n, sh, ctx->d_expect, ctx->d_tiles, ctx->d_err);
    ++launches;
    if (getenv("MSNV_VERBOSE"))
        fprintf(stderr, "msnv: pileup (%s) %u items (%.1f reads each, at most %u), %u CTAs (%d per SM) x %d threads%s, stage limits %u reads / %u segments / %u quads, %zu B shared memory\n",
                sh.gather ? "gather" : "scatter", n, (double)item_reads / (double)n_items_window, item_reads_max, (unsigned)grid, ctas, threads, has_wide ? " (wide items)" : "", sh.max_reads,
                sh.max_segs, sh.chunk_q4, smem);
    return MSNV_OK;
}

// index -> [pileup -> call -> compaction -> gather -> copy back] per range of tiles
static int run_window(msnv_ctx* ctx, uint32_t slot, const msnv_call_params* prm, msnv_hits* hits)
{
    msnv_ctx::Window& w = ctx->win[slot];
    cudaStream_t st = ctx->stream;
    const uint32_t S = ctx->S, nt = w.t1 - w.t0;
    uint32_t launches = 0;
    memset(hits, 0, sizeof *hits);
    hits->n_samples = S;

    // the window's reads are on the device once the copy stream reaches this point
    CU(cudaEventRecord(w.uploaded, ctx->copy_stream));
    CU(cudaStreamWaitEvent(st, w.uploaded, 0));
    CU(w.d_samples.ensure(S));
    CU(cudaMemcpyAsync(w.d_samples, w.h_samples.data(), sizeof(SampleDev) * S, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(ctx->d_err, 0, 4, st));
    CU(cudaMemsetAsync(ctx->d_scalar, 0, 32, st));
    if (int rc = ensure_window_buffers(ctx, nt)) return rc;

    // ---- mate overlap: verdicts per quad for the samples that have pairs (read by the pileup kernel)
    uint64_t max_reads = 0, max_fix_reads = 0;
    std::vector<uint32_t> fix_samples;
    for (uint32_t s = 0; s < S; ++s) {
        if (w.h_samples[s].n_reads > max_reads) max_reads = w.h_samples[s].n_reads;
        if (w.h_samples[s].fix) { fix_samples.push_back(s); if (w.h_samples[s].n_reads > max_fix_reads) max_fix_reads = w.h_samples[s].n_reads; }
    }
    unsigned gx = (unsigned)((max_reads + 256 * 8 - 1) / (256 * 8)); if (gx < 1) gx = 1; if (gx > 1024) gx = 1024;
    cudaEvent_t ev_m0 = ctx->ev[2], ev_m1 = ctx->ev[3];
    CU(cudaEventRecord(ev_m0, st));
    if (!fix_samples.empty()) {
        CU(ctx->d_fix_list.ensure(fix_samples.size(), fix_samples.size() + 64));
        // (pageable source: the copy is staged before the call returns)
        CU(cudaMemcpyAsync(ctx->d_fix_list, fix_samples.data(), fix_samples.size() * 4, cudaMemcpyHostToDevice, st));
        unsigned gc = (unsigned)((max_fix_reads * 2 + 255) / 256); if (gc < 1) gc = 1; if (gc > 1024) gc = 1024;          // ~27 bytes per read, 16 per thread
        unsigned gm = (unsigned)((max_fix_reads + 255) / 256); if (gm < 1) gm = 1; if (gm > 4096) gm = 4096;              // a warp per 32 reads
        fix_clear_kernel<<<dim3(gc, (unsigned)fix_samples.size()), 256, 0, st>>>(w.d_samples, ctx->d_fix_list);
        mate_kernel<<<dim3(gm, (unsigned)fix_samples.size()), 256, 0, st>>>(w.d_samples, ctx->d_fix_list);
        launches += 2;
    }
    CU(cudaEventRecord(ev_m1, st));

    CU(cudaEventRecord(ctx->ev[0], st));
    // expected letter per position of the window (msnv_shard_mask_position may have changed the reference since the last run)
    expect_kernel<<<(nt * TILE + 255) / 256, 256, 0, st>>>(ctx->d_ref + (size_t)w.t0 * TILE, nt * TILE, ctx->d_expect + (size_t)w.t0 * TILE);
    ++launches;
    // ---- index
    const uint64_t n_pairs_idx = (uint64_t)nt * S;
    const uint64_t n_blocks = (n_pairs_idx + 255) / 256;
    if (n_blocks > 0x7fffffffull) return fail(ctx, MSNV_E_LIMIT, "window too large: %u tiles x %u samples", nt, S);
    CU(ctx->d_block_sums.ensure(n_blocks));
    // the (r_lo, r_hi) of every pair found by the counting pass is kept for the emitting pass when it fits 1 GiB
    uint2* cache = nullptr;
    if (n_pairs_idx * 8 <= (1ull << 30)) {
        CU(ctx->d_range_cache.ensure(n_pairs_idx));
        cache = ctx->d_range_cache;
    }
    // the index and the pileup rely on coordinate order within a sample; checked on the device (0.3 ms for 5e8 reads)
    order_check_kernel<<<dim3(gx, S), 256, 0, st>>>(w.d_samples, ctx->d_err);
    ++launches;
    // sparse windows (fewer than ~1/3 of the pairs can be active): occupancy bitmap first
    uint32_t* bitmap = nullptr;
    const uint32_t words_per_sample = (nt + 31) / 32;
    const bool sparse = getenv("MSNV_INDEX_BITMAP") ? atoi(getenv("MSNV_INDEX_BITMAP")) != 0
                                                     : w.n_reads / 20 < n_pairs_idx;     // < 20 reads per (tile, sample) pair on average
    if (sparse) {
        const uint64_t words = (uint64_t)words_per_sample * S;
        CU(ctx->d_bitmap.ensure(words));
        CU(cudaMemsetAsync(ctx->d_bitmap, 0, words * 4, st));
        mark_kernel<<<dim3(gx, S), 256, 0, st>>>(w.d_samples, words_per_sample, w.t0, nt, ctx->d_bitmap);
        ++launches;
        bitmap = ctx->d_bitmap;
    }
    unsigned long long* d_item_reads = reinterpret_cast<unsigned long long*>(ctx->d_scalar + 2);
    index_kernel<false><<<(unsigned)n_blocks, 256, 0, st>>>(w.d_samples, S, w.t0, nt, ctx->d_block_sums, nullptr, nullptr, cache, bitmap, words_per_sample,
                                                            d_item_reads);
    scan_kernel<<<1, 1024, 0, st>>>(ctx->d_block_sums, (uint32_t)n_blocks, ctx->d_scalar);
    launches += 2;
    CU(cudaMemcpyAsync(ctx->h_scalar, ctx->d_scalar, 24, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ctx->h_scalar + 6, ctx->d_err, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ctx->h_scalar + 7, reinterpret_cast<const uint32_t*>(ctx->d_xstat + 1), 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (ctx->h_scalar[7]) return fail(ctx, MSNV_E_ARG, "a BAM-shaped record is inconsistent: CIGAR longer than the sequence, blob shorter than the record, or offsets that disagree with the CIGAR");
    float ms_mate = 0;
    cudaEventElapsedTime(&ms_mate, ev_m0, ev_m1);          // (the events are reused by the ranges below)
    if (ctx->h_scalar[6] == 3) return fail(ctx, MSNV_E_ARG, "the reads of a sample are not in coordinate order (pos must be ascending)");
    const uint32_t n_items = ctx->h_scalar[0];
    const uint64_t item_reads = (uint64_t)ctx->h_scalar[2] | (uint64_t)ctx->h_scalar[3] << 32;
    const uint32_t item_reads_max = ctx->h_scalar[4];
    CU(ctx->d_items.ensure(n_items, (uint64_t)n_items + n_items / 8 + 64));
    index_kernel<true><<<(unsigned)n_blocks, 256, 0, st>>>(w.d_samples, S, w.t0, nt, ctx->d_block_sums, ctx->d_items, ctx->d_tile_begin, cache, bitmap,
                                                           words_per_sample, nullptr);
    ++launches;
    CU(cudaMemcpyAsync(ctx->d_tile_begin + nt, ctx->d_scalar, 4, cudaMemcpyDeviceToDevice, st));
    CU(cudaEventRecord(ctx->ev[1], st));

    // ---- ranges of tiles whose count planes fit the budget (one range in the common case)
    const uint64_t budget = tile_budget_slots(ctx);
    std::vector<uint32_t> cuts{0u};
    if ((uint64_t)n_items <= budget) cuts.push_back(nt);
    else {
        ctx->h_tile_begin.resize((size_t)nt + 1);
        CU(cudaMemcpyAsync(ctx->h_tile_begin.data(), ctx->d_tile_begin, ((size_t)nt + 1) * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const std::vector<uint32_t>& tb = ctx->h_tile_begin;
        uint32_t ta = 0;
        while (ta < nt) {
            uint32_t te = ta + 1;
            if ((uint64_t)(tb[te] - tb[ta]) > budget)
                return fail(ctx, MSNV_E_NOMEM, "the count planes of one tile (%u samples) do not fit the tile budget", tb[te] - tb[ta]);
            while (te < nt && (uint64_t)(tb[te + 1] - tb[ta]) <= budget) ++te;
            cuts.push_back(te);
            ta = te;
        }
    }
    uint64_t max_range = 0;
    if (cuts.size() == 2) max_range = n_items;
    else for (size_t k = 0; k + 1 < cuts.size(); ++k) max_range = std::max<uint64_t>(max_range, ctx->h_tile_begin[cuts[k + 1]] - ctx->h_tile_begin[cuts[k]]);
    if (int rc = ensure_tile_slots(ctx, max_range)) return rc;

    float ms_pileup = 0;
    PhaseTimes acc;
    uint32_t n_hits = 0;
    for (size_t k = 0; k + 1 < cuts.size(); ++k) {
        const uint32_t ta = cuts[k], tb = cuts[k + 1];
        const uint32_t a = cuts.size() == 2 ? 0u : ctx->h_tile_begin[ta], b = cuts.size() == 2 ? n_items : ctx->h_tile_begin[tb];
        CU(cudaEventRecord(ctx->ev[2], st));
        if (b > a) if (int rc = launch_pileup(ctx, w, a, b - a, n_items, item_reads, item_reads_max, launches)) return rc;
        uint32_t n_range = 0;
        if (int rc = call_range(ctx, w, a, ta, tb, prm, 0, n_hits, n_range, launches, acc)) return rc;     // records ev[3] first
        float ms; cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]); ms_pileup += ms;
        n_hits += n_range;
        ctx->last_slot = slot; ctx->last_item0 = a; ctx->last_ta = ta; ctx->last_tb = tb;
    }
    publish_hits(ctx, n_hits, hits);

    msnv_timings& tm = ctx->tm;
    tm = msnv_timings{};
    cudaEventElapsedTime(&tm.ms_index, ctx->ev[0], ctx->ev[1]);
    tm.ms_mate = ms_mate;
    tm.ms_pileup = ms_pileup + ms_mate; tm.ms_call = acc.call; tm.ms_compact = acc.compact; tm.ms_gather = acc.gather; tm.ms_d2h = acc.d2h;
    tm.ms_total = tm.ms_index + tm.ms_pileup + tm.ms_call + tm.ms_compact + tm.ms_gather;
    tm.n_items = n_items; tm.n_reads = w.n_reads; tm.n_bases = w.n_bases; tm.n_tiles = nt;
    tm.kernel_launches = launches;
    tm.n_ranges = (uint32_t)cuts.size() - 1;
    ctx->has_run = true;
    return MSNV_OK;
}

// the checks of msnv_window_add_sample / _raw: an open window in `slot`, a sample in range that was not added yet,
// and a reference span within the limit
static int check_add(msnv_ctx* ctx, uint32_t slot, uint32_t sample, uint32_t n_reads, uint32_t max_span, const char* fn)
{
    if (!ctx->open || slot >= (uint32_t)N_SLOTS || !ctx->win[slot].open) return fail(ctx, MSNV_E_STATE, "%s: no open window in this slot", fn);
    if (sample >= ctx->S) return fail(ctx, MSNV_E_ARG, "%s: sample %u out of range", fn, sample);
    if (ctx->win[slot].h_samples[sample].n_reads) return fail(ctx, MSNV_E_STATE, "%s: sample %u added twice", fn, sample);
    if (n_reads && max_span > (uint32_t)MSNV_MAX_READ_SPAN)
        return fail(ctx, MSNV_E_LIMIT, "sample %u: reference span %u exceeds the limit of %u", sample, max_span, (uint32_t)MSNV_MAX_READ_SPAN);
    return MSNV_OK;
}

// whether a caller's array p sits at offset o of its batch starting at b (then a group goes up in one copy)
static bool at(const void* p, const void* b, size_t o) { return static_cast<const uint8_t*>(p) == static_cast<const uint8_t*>(b) + o; }

// a sample whose read group is in block rb and segment group in block sb joins the window
static void attach_sample(msnv_ctx::Window& w, uint32_t sample, uint8_t* rb, const ReadGroup& g, uint8_t* sb, const SegmentGroup& sg,
                          const msnv_sample_sizes& z)
{
    SampleDev& d = w.h_samples[sample];
    d.pos = (const int32_t*)(rb + g.pos);
    d.seg_off = (const uint32_t*)(rb + g.seg_off); d.q4_off = (const uint32_t*)(rb + g.q4_off);
    d.mate = (const int32_t*)(rb + g.mate);
    d.seg_pos = (const int32_t*)(sb + sg.seg_pos);  d.seg_len = (const uint16_t*)(sb + sg.seg_len);
    d.seq2 = sb + sg.seq2;                         d.qual = sb + sg.qual;
    d.fix = sg.fix ? sb + sg.fix : nullptr;
    d.n_reads = z.n_reads; d.max_span = z.max_span;
    w.n_reads += z.n_reads; w.n_bases += 4 * z.n_q4; w.n_segs += z.n_segs;
    w.sizes[sample] = z;
}

extern "C" {

int msnv_abi_version(void) { return MSNV_ABI_VERSION; }
int msnv_tile(void) { return MSNV_TILE; }

int msnv_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int msnv_create(int device, msnv_ctx** out)
{
    if (!out) return MSNV_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device < 0 || device >= n) return MSNV_E_CUDA;
    msnv_ctx* ctx = new msnv_ctx();
    ctx->device = device;
    *out = ctx;                                   // returned even on failure so the caller can read the error
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (auto& e : ctx->ev) CU(cudaEventCreate(&e));
    for (auto& w : ctx->win) CU(cudaEventCreateWithFlags(&w.uploaded, cudaEventDisableTiming));
    CU(ctx->d_scalar.ensure(8));
    CU(ctx->d_err.ensure(1));
    CU(ctx->d_xstat.ensure(2));
    CU(cudaMemset(ctx->d_xstat, 0, 16));
    CU(ctx->h_scalar.ensure(8));
    for (bool gather : {false, true})
        for (int consumers : {128, 256})
            for (bool has_wide : {false, true})
                CU(cudaFuncSetAttribute(pileup_kernel_for(gather, consumers, has_wide), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_PER_CTA_MAX));
    CU(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));
    return MSNV_OK;
}

void msnv_destroy(msnv_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& w : ctx->win) { release_window(ctx, w); if (w.uploaded) cudaEventDestroy(w.uploaded); }
    drop_pool(ctx);
    for (auto& sl : ctx->slabs) cudaFree(sl.base);
    for (auto& e : ctx->ev) if (e) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;                                   // (the work buffers free themselves)
}

void* msnv_pinned_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void msnv_pinned_free(void* p) { if (p) cudaFreeHost(p); }

const char* msnv_last_error(const msnv_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (no CUDA device?)"; }

int msnv_shard_begin(msnv_ctx* ctx, uint32_t n_samples, uint32_t n_positions, const uint8_t* ref)
{
    if (!ctx) return MSNV_E_ARG;
    if (!ref || n_samples == 0 || n_positions == 0 || n_positions % TILE != 0)
        return fail(ctx, MSNV_E_ARG, "msnv_shard_begin: n_samples and n_positions must be positive, n_positions a multiple of %d", TILE);
    if (n_samples > 65535) return fail(ctx, MSNV_E_LIMIT, "msnv_shard_begin: at most 65535 samples (32-bit population sums)");
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->copy_stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ++ctx->gen;
    for (auto& w : ctx->win) release_window(ctx, w);
    ctx->S = n_samples; ctx->P = n_positions; ctx->n_tiles = n_positions / TILE;
    ctx->open = ctx->has_run = false;             // (a failure below leaves no shard open)
    ctx->d_ref.reset(); ctx->d_expect.reset();
    CU(ctx->d_ref.ensure(n_positions));
    CU(ctx->d_expect.ensure(n_positions));
    CU(cudaMemcpyAsync(ctx->d_ref, ref, n_positions, cudaMemcpyHostToDevice, ctx->stream));
    ctx->open = true;
    // the whole shard as one window in slot 0 until msnv_window_begin says otherwise
    msnv_ctx::Window& w = ctx->win[0];
    w.open = true; w.t0 = 0; w.t1 = ctx->n_tiles;
    w.h_samples.assign(n_samples, SampleDev{});
    w.sizes.assign(n_samples, msnv_sample_sizes{});
    return MSNV_OK;
}

int msnv_window_begin(msnv_ctx* ctx, uint32_t slot, uint32_t pos_lo, uint32_t pos_hi)
{
    if (!ctx) return MSNV_E_ARG;
    if (!ctx->open) return fail(ctx, MSNV_E_STATE, "msnv_window_begin: no open shard");
    if (slot >= (uint32_t)N_SLOTS || pos_lo >= pos_hi || pos_hi > ctx->P || pos_lo % TILE || pos_hi % TILE)
        return fail(ctx, MSNV_E_ARG, "msnv_window_begin: slot 0 or 1, and 0 <= pos_lo < pos_hi <= n_positions in multiples of %d", TILE);
    CU(cudaSetDevice(ctx->device));
    ++ctx->gen;
    msnv_ctx::Window& w = ctx->win[slot];
    release_window(ctx, w);              // (the kernels that read the slot's previous window finished inside msnv_window_run)
    w.open = true; w.t0 = pos_lo / TILE; w.t1 = pos_hi / TILE;
    w.h_samples.assign(ctx->S, SampleDev{});
    w.sizes.assign(ctx->S, msnv_sample_sizes{});
    return MSNV_OK;
}

int msnv_window_add_sample(msnv_ctx* ctx, uint32_t slot, uint32_t sample, const msnv_sample_reads* r)
{
    if (!ctx || !r) return MSNV_E_ARG;
    if (int rc = check_add(ctx, slot, sample, r->n_reads, r->max_span, __func__)) return rc;
    if (r->n_reads == 0) return MSNV_OK;
    msnv_ctx::Window& w = ctx->win[slot];
    CU(cudaSetDevice(ctx->device));
    const size_t n = r->n_reads, n1 = n + 1;
    const size_t n_seg = r->seg_off[n] - r->seg_off[0], n_q4 = r->q4_off[n] - r->q4_off[0];
    if (r->seg_off[0] != 0 || r->q4_off[0] != 0) return fail(ctx, MSNV_E_ARG, "sample %u: seg_off / q4_off must start at 0", sample);
    if (n_seg < n || n_q4 < n_seg) return fail(ctx, MSNV_E_ARG, "sample %u: inconsistent offsets (%zu reads, %zu segments, %zu quads)", sample, n, n_seg, n_q4);
    bool has_mates = false;
    for (size_t i = 0; i < n && !has_mates; ++i) has_mates = r->mate[i] >= 0;
    // one allocation per sample (the fix verdicts of the mate-overlap rule are rebuilt by every run)
    BlockLayout layout;
    const ReadGroup g(layout, n);
    const SegmentGroup sg(layout, n_seg, n_q4, has_mates);
    uint8_t* base = (uint8_t*)take_block(ctx, w, layout.size);
    if (!base) return fail(ctx, MSNV_E_NOMEM, "sample %u: cannot allocate %zu bytes of device memory; process the shard in smaller windows (msnv_window_begin) or smaller genome bins (metaSNV.py --n_splits)", sample, layout.size);
    cudaStream_t st = ctx->copy_stream;
    // a caller that packed the arrays the way this block is laid out gets ONE copy instead of eight
    const void* h0 = r->pos;
    if (at(r->seg_off, h0, g.seg_off) && at(r->q4_off, h0, g.q4_off) && at(r->mate, h0, g.mate) && at(r->seg_pos, h0, sg.seg_pos) &&
        at(r->seg_len, h0, sg.seg_len) && at(r->seq2, h0, sg.seq2) && at(r->qual, h0, sg.qual)) {
        CU(cudaMemcpyAsync(base + g.pos, h0, sg.end - g.pos, cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemcpyAsync(base + g.pos, r->pos, n * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.seg_off, r->seg_off, n1 * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.q4_off, r->q4_off, n1 * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.mate, r->mate, n * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + sg.seg_pos, r->seg_pos, n_seg * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + sg.seg_len, r->seg_len, n_seg * 2, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + sg.seq2, r->seq2, n_q4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + sg.qual, r->qual, n_q4 * 4, cudaMemcpyHostToDevice, st));
    }
    uint64_t n_aligned = 0;
    for (size_t k = 0; k < n_seg; ++k) n_aligned += r->seg_len[k];
    attach_sample(w, sample, base, g, base, sg, msnv_sample_sizes{r->n_reads, 0, r->max_span ? r->max_span : 1, 0, (uint64_t)n_seg, (uint64_t)n_q4, n_aligned});
    return MSNV_OK;
}

int msnv_window_add_sample_raw(msnv_ctx* ctx, uint32_t slot, uint32_t sample, const msnv_raw_reads* r)
{
    if (!ctx || !r) return MSNV_E_ARG;
    if (int rc = check_add(ctx, slot, sample, r->n_reads, r->max_span, __func__)) return rc;
    if (r->n_reads == 0) return MSNV_OK;
    msnv_ctx::Window& w = ctx->win[slot];
    CU(cudaSetDevice(ctx->device));
    const size_t n = r->n_reads, n1 = n + 1;
    if (r->seg_off[0] != 0 || r->q4_off[0] != 0 || r->raw_off[0] != 0) return fail(ctx, MSNV_E_ARG, "sample %u: seg_off / q4_off / raw_off must start at 0", sample);
    const size_t n_seg = r->seg_off[n], n_q4 = r->q4_off[n], raw_words = r->raw_off[n];
    if (n_seg < n || n_q4 < n_seg) return fail(ctx, MSNV_E_ARG, "sample %u: inconsistent offsets (%zu reads, %zu segments, %zu quads)", sample, n, n_seg, n_q4);
    // (the records themselves are checked by expand_kernel: CIGAR against sequence length, blob size, offsets)
    bool has_mates = false;
    for (size_t i = 0; i < n && !has_mates; ++i) has_mates = r->mate[i] >= 0;
    CU(w.d_aligned.ensure(ctx->S));
    if (!w.has_raw) { CU(cudaMemsetAsync(w.d_aligned, 0, (size_t)ctx->S * 8, ctx->copy_stream)); w.has_raw = true; }
    BlockLayout layout;
    const ReadGroup g(layout, n);
    const SegmentGroup sg(layout, n_seg, n_q4, has_mates);
    uint8_t* base = (uint8_t*)take_block(ctx, w, layout.size);
    if (!base) return fail(ctx, MSNV_E_NOMEM, "sample %u: cannot allocate %zu bytes of device memory; process the shard in smaller windows (msnv_window_begin) or smaller genome bins (metaSNV.py --n_splits)", sample, layout.size);
    // staging of the BAM-shaped arrays
    BlockLayout staging;
    const RawGroup x(staging, n, raw_words);
    CU(ctx->d_raw.ensure(staging.size, staging.size + staging.size / 4 + (1u << 20)));
    uint8_t* raw = ctx->d_raw;
    cudaStream_t st = ctx->copy_stream;
    // packed callers (same order and spacing as the device side): two copies instead of eight
    const void* h0 = r->pos;
    const void* g0 = r->raw_off;
    if (at(r->seg_off, h0, g.seg_off) && at(r->q4_off, h0, g.q4_off) && at(r->mate, h0, g.mate)) {
        CU(cudaMemcpyAsync(base + g.pos, h0, g.end - g.pos, cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemcpyAsync(base + g.pos, r->pos, n * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.seg_off, r->seg_off, n1 * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.q4_off, r->q4_off, n1 * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(base + g.mate, r->mate, n * 4, cudaMemcpyHostToDevice, st));
    }
    if (at(r->raw, g0, x.raw) && at(r->n_cigar, g0, x.n_cigar) && at(r->l_seq, g0, x.l_seq)) {
        CU(cudaMemcpyAsync(raw + x.raw_off, g0, x.end - x.raw_off, cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemcpyAsync(raw + x.raw_off, r->raw_off, n1 * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(raw + x.raw, r->raw, raw_words * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(raw + x.n_cigar, r->n_cigar, n * 2, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(raw + x.l_seq, r->l_seq, n * 2, cudaMemcpyHostToDevice, st));
    }
    // the aligned arrays are built in place: padding bytes must be 0
    CU(cudaMemsetAsync(base + sg.seq2, 0, n_q4 + 32, st));
    RawDev in;
    in.pos = (const int32_t*)(base + g.pos); in.seg_off = (const uint32_t*)(base + g.seg_off); in.q4_off = (const uint32_t*)(base + g.q4_off);
    in.raw_off = (const uint32_t*)(raw + x.raw_off); in.raw = (const uint32_t*)(raw + x.raw);
    in.n_cigar = (const uint16_t*)(raw + x.n_cigar); in.l_seq = (const uint16_t*)(raw + x.l_seq); in.n_reads = r->n_reads;
    expand_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(in, (int32_t*)(base + sg.seg_pos), (uint16_t*)(base + sg.seg_len), base + sg.seq2, (uint32_t*)(base + sg.qual), ctx->d_xstat, w.d_aligned + sample);
    CU(cudaGetLastError());
    // n_aligned: see msnv_window_sample_sizes
    attach_sample(w, sample, base, g, base, sg, msnv_sample_sizes{r->n_reads, 0, r->max_span ? r->max_span : 1, 0, (uint64_t)n_seg, (uint64_t)n_q4, 0});
    return MSNV_OK;
}

int msnv_expand_stats(msnv_ctx* ctx, uint64_t* iupac_bases)
{
    if (!ctx || !iupac_bases) return MSNV_E_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->copy_stream));
    unsigned long long v = 0;
    CU(cudaMemcpy(&v, ctx->d_xstat, 8, cudaMemcpyDeviceToHost));
    *iupac_bases = v;
    return MSNV_OK;
}

int msnv_window_run(msnv_ctx* ctx, uint32_t slot, const msnv_call_params* prm, msnv_hits* hits)
{
    if (!ctx || !prm || !hits) return MSNV_E_ARG;
    if (!ctx->open || slot >= (uint32_t)N_SLOTS || !ctx->win[slot].open) return fail(ctx, MSNV_E_STATE, "msnv_window_run: no open window in this slot");
    CU(cudaSetDevice(ctx->device));
    return run_window(ctx, slot, prm, hits);
}

int msnv_shard_add_sample(msnv_ctx* ctx, uint32_t sample, const msnv_sample_reads* r) { return msnv_window_add_sample(ctx, 0, sample, r); }

int msnv_shard_mask_position(msnv_ctx* ctx, uint32_t pos)
{
    if (!ctx) return MSNV_E_ARG;
    if (!ctx->open || pos >= ctx->P) return fail(ctx, MSNV_E_ARG, "msnv_shard_mask_position: position out of range");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemsetAsync(ctx->d_ref + pos, 0, 1, ctx->stream));
    return MSNV_OK;
}

int msnv_shard_sync(msnv_ctx* ctx)
{
    if (!ctx) return MSNV_E_ARG;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->copy_stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return MSNV_OK;
}

int msnv_shard_run(msnv_ctx* ctx, const msnv_call_params* prm, msnv_hits* hits) { return msnv_window_run(ctx, 0, prm, hits); }

int msnv_call_counts(msnv_ctx* ctx, uint32_t n_samples, uint32_t n_positions, const uint8_t* ref, const uint64_t* acgt,
                     const uint16_t* matches, const msnv_call_params* prm, msnv_hits* hits)
{
    if (!ctx || !ref || !acgt || !matches || !prm || !hits) return MSNV_E_ARG;
    if (int rc = msnv_shard_begin(ctx, n_samples, n_positions, ref)) return rc;
    cudaStream_t st = ctx->stream;
    msnv_ctx::Window& w = ctx->win[0];
    const uint32_t nt = ctx->n_tiles;
    const uint64_t n_items = (uint64_t)nt * n_samples;
    if (n_items > 0xffffffffull) return fail(ctx, MSNV_E_LIMIT, "msnv_call_counts: batch too large");
    CU(ctx->d_items.ensure(n_items, n_items + 64));
    if (int rc = ensure_tile_slots(ctx, n_items)) return rc;
    if (int rc = ensure_window_buffers(ctx, nt)) return rc;
    memset(hits, 0, sizeof *hits);
    uint32_t launches = 0;
    CU(cudaMemsetAsync(ctx->d_err, 0, 4, st));
    CU(ctx->d_text_acgt.ensure(n_items * TILE));
    CU(ctx->d_text_match.ensure(n_items * TILE));
    CU(cudaMemcpyAsync(ctx->d_text_acgt, acgt, n_items * TILE * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_text_match, matches, n_items * TILE * 2, cudaMemcpyHostToDevice, st));
    expect_kernel<<<(ctx->P + 255) / 256, 256, 0, st>>>(ctx->d_ref, ctx->P, ctx->d_expect);
    text_tiles_kernel<<<(unsigned)((n_items * TILE + 255) / 256), 256, 0, st>>>(ctx->d_text_acgt, ctx->d_text_match, n_items * TILE, ctx->d_tiles);
    dense_items_kernel<<<(unsigned)((n_items + 1 + 255) / 256), 256, 0, st>>>(n_samples, nt, ctx->d_items, ctx->d_tile_begin);
    launches += 3;
    PhaseTimes acc;
    uint32_t n_hits = 0;
    if (int rc = call_range(ctx, w, 0, 0, nt, prm, 1, 0, n_hits, launches, acc)) return rc;
    publish_hits(ctx, n_hits, hits);
    msnv_timings& tm = ctx->tm;
    tm = msnv_timings{};
    tm.ms_call = acc.call; tm.ms_compact = acc.compact; tm.ms_gather = acc.gather; tm.ms_d2h = acc.d2h;
    tm.ms_total = acc.call + acc.compact + acc.gather;
    tm.n_items = n_items; tm.n_tiles = nt; tm.kernel_launches = launches; tm.n_ranges = 1;
    ctx->last_slot = 0; ctx->last_item0 = 0; ctx->last_ta = 0; ctx->last_tb = nt;
    ctx->has_run = true;
    return MSNV_OK;
}

static int synth_model(msnv_ctx* ctx, const msnv_synth_desc* d, msnv::synth::Model& m, std::vector<uint32_t>& off)
{
    if (!ctx || !d || !d->contig_len || !d->contig_genome || !d->genome_n_sub) return MSNV_E_ARG;
    if (d->n_samples == 0 || d->n_contigs == 0 || d->read_len < 20 || d->read_len > 1000)
        return fail(ctx, MSNV_E_ARG, "msnv_shard_synth: bad description");
    m.seed = d->seed; m.n_samples = (int32_t)d->n_samples; m.read_len = (int32_t)d->read_len; m.depth_x100 = d->depth_x100;
    m.presence_ppm = d->presence_ppm; m.paired_pct = d->paired_pct; m.site_ppm = d->site_ppm; m.err_ppm = d->err_ppm;
    m.nbase_ppm = d->nbase_ppm; m.refn_ppm = d->refn_ppm; m.indel_pct_x10 = d->indel_pct_x10; m.clip_pct_x10 = d->clip_pct_x10;
    m.mapq0_pct_x10 = d->mapq0_pct_x10;
    const uint32_t K = d->n_contigs;
    off.assign(K + 1, 0);
    uint64_t P = 0;
    for (uint32_t k = 0; k < K; ++k) {
        off[k] = (uint32_t)P;
        P += ((uint64_t)d->contig_len[k] + TILE - 1) / TILE * TILE + (d->contig_len[k] == 0 ? TILE : 0);
        if (P > 0x7ff00000ull) return fail(ctx, MSNV_E_LIMIT, "msnv_shard_synth: shard larger than 2^31 positions");
        if (d->contig_genome[k] >= d->n_genomes) return fail(ctx, MSNV_E_ARG, "msnv_shard_synth: contig_genome out of range");
    }
    off[K] = (uint32_t)P;
    return MSNV_OK;
}

int msnv_shard_synth_ref(msnv_ctx* ctx, const msnv_synth_desc* d, int64_t* first_column)
{
    msnv::synth::Model m;
    std::vector<uint32_t> off;
    if (int rc = synth_model(ctx, d, m, off)) return rc;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint32_t K = d->n_contigs, S = d->n_samples, L = d->read_len;
    const uint64_t P = off[K];
    {
        // msnv_shard_begin wants a host reference; give it a zero page and overwrite on the device
        std::vector<uint8_t> zero((size_t)P, 0);
        if (int rc = msnv_shard_begin(ctx, S, (uint32_t)P, zero.data())) return rc;
        CU(cudaStreamSynchronize(st));
    }
    {
        DevBuf<uint32_t> d_off, d_len;
        CU(d_off.ensure((uint64_t)K + 1));
        CU(d_len.ensure(K));
        CU(cudaMemcpyAsync(d_off, off.data(), ((size_t)K + 1) * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_len, d->contig_len, (size_t)K * 4, cudaMemcpyHostToDevice, st));
        synth_ref_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(m, d_off, d_len, K, (uint32_t)P, ctx->d_ref);
        CU(cudaStreamSynchronize(st));
    }
    // first pileup column of the shard: the smallest first fragment start over the samples' first contigs
    int64_t first_col = -1;
    for (uint32_t s = 0; s < S; ++s) {
        const bool paired = msnv::synth::sample_paired(m, (int)s);
        const int32_t D = paired ? msnv::synth::sample_mate_offset(m, (int)s) : 0;
        const uint32_t span = msnv::synth::frag_span(m, paired, D);
        for (uint32_t k = 0; k < K; ++k) {
            if (!msnv::synth::sample_has_genome(m, (int)s, (int)d->contig_genome[k]) || d->contig_len[k] <= span) continue;
            const uint32_t nf = msnv::synth::n_fragments(m, d->contig_len[k], paired);
            if (!nf) continue;
            const int64_t c = (int64_t)off[k] + msnv::synth::frag_start(m, (int)s, k, d->contig_len[k], span, nf, 0);
            if (first_col < 0 || c < first_col) first_col = c;
            break;
        }
    }
    (void)L;
    if (first_column) *first_column = first_col;
    return MSNV_OK;
}

int msnv_window_synth(msnv_ctx* ctx, uint32_t slot, const msnv_synth_desc* d, uint32_t ctg_lo, uint32_t ctg_hi)
{
    msnv::synth::Model m;
    std::vector<uint32_t> off;
    if (int rc = synth_model(ctx, d, m, off)) return rc;
    if (!ctx->open || ctx->S != d->n_samples || ctx->P != off[d->n_contigs]) return fail(ctx, MSNV_E_STATE, "msnv_window_synth: call msnv_shard_synth_ref for this description first");
    if (ctg_lo >= ctg_hi || ctg_hi > d->n_contigs) return fail(ctx, MSNV_E_ARG, "msnv_window_synth: bad contig range");
    CU(cudaSetDevice(ctx->device));
    if (int rc = msnv_window_begin(ctx, slot, off[ctg_lo], off[ctg_hi])) return rc;
    cudaStream_t st = ctx->copy_stream;           // the stream msnv_window_run() waits for
    msnv_ctx::Window& w = ctx->win[slot];
    const uint32_t S = d->n_samples, L = d->read_len, q4 = (L + 3) / 4;
    std::vector<SynthSampleCtg> blocks;
    std::vector<uint32_t> frag0;
    for (uint32_t s = 0; s < S; ++s) {
        const bool paired = msnv::synth::sample_paired(m, (int)s);
        const int32_t D = paired ? msnv::synth::sample_mate_offset(m, (int)s) : 0;
        const bool overlap = paired && D < (int32_t)L;
        const uint32_t span = msnv::synth::frag_span(m, paired, D);
        blocks.clear(); frag0.assign(1, 0);
        uint64_t n_reads = 0, n_mated = 0;
        for (uint32_t k = ctg_lo; k < ctg_hi; ++k) {
            const uint32_t g = d->contig_genome[k];
            if (!msnv::synth::sample_has_genome(m, (int)s, (int)g) || d->contig_len[k] <= span) continue;
            const uint32_t nf = msnv::synth::n_fragments(m, d->contig_len[k], paired);
            if (!nf) continue;
            SynthSampleCtg b{k, d->contig_len[k], off[k], g, d->genome_n_sub[g], nf, (uint32_t)n_reads};
            blocks.push_back(b);
            frag0.push_back(frag0.back() + nf);
            n_reads += (uint64_t)nf * (paired ? 2 : 1);
            if (overlap) n_mated += 2ull * nf;
            if (n_reads > 0x7fffffffull) return fail(ctx, MSNV_E_LIMIT, "msnv_shard_synth: more than 2^31 reads in one sample");
        }
        if (blocks.empty()) continue;
        const size_t n = (size_t)n_reads, nb = blocks.size(), nft = frag0.back();
        // ---- phase 1: per-read metadata (segments and quads per read, then their prefix sums)
        BlockLayout meta_layout;
        const ReadGroup g(meta_layout, n);
        uint8_t* meta = (uint8_t*)take_block(ctx, w, meta_layout.size);
        if (!meta) return fail(ctx, MSNV_E_NOMEM, "msnv_shard_synth: out of device memory (sample %u)", s);
        DevBuf<SynthSampleCtg> d_blocks;
        DevBuf<uint32_t> d_frag0, d_nq, d_nsegs, d_for;
        CU(d_blocks.ensure(nb));
        CU(d_frag0.ensure(nb + 1));
        CU(d_nq.ensure(n));
        CU(d_nsegs.ensure(n));
        CU(d_for.ensure(n));
        CU(cudaMemcpyAsync(d_blocks, blocks.data(), nb * sizeof(SynthSampleCtg), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_frag0, frag0.data(), (nb + 1) * 4, cudaMemcpyHostToDevice, st));
        synth_meta_kernel<<<(unsigned)((nft + 127) / 128), 128, 0, st>>>(m, (int)s, paired, D, overlap, d_blocks, d_frag0, (uint32_t)nb, (uint32_t)nft,
            (int32_t*)(meta + g.pos), d_nsegs, d_nq, (int32_t*)(meta + g.mate), d_for);
        synth_scan2_kernel<<<1, 1024, 0, st>>>(d_nsegs, d_nq, (uint32_t)n, (uint32_t*)(meta + g.seg_off), (uint32_t*)(meta + g.q4_off));
        uint32_t n_seg = 0, n_q4_u = 0;
        CU(cudaMemcpyAsync(&n_seg, meta + g.seg_off + n * 4, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&n_q4_u, meta + g.q4_off + n * 4, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        // ---- phase 2: segment records, bases, qualities
        const size_t n_q4 = n_q4_u;
        const uint32_t q_slots = q4 + 4;          // upper bound of the quads of one read (two segments)
        BlockLayout data_layout;
        const SegmentGroup sg(data_layout, n_seg, n_q4, n_mated != 0);
        uint8_t* data = (uint8_t*)take_block(ctx, w, data_layout.size);
        if (!data) return fail(ctx, MSNV_E_NOMEM, "msnv_shard_synth: out of device memory (sample %u)", s);
        synth_fill_kernel<<<(unsigned)((n * q_slots + 255) / 256), 256, 0, st>>>(m, (int)s, paired, d_blocks, d_frag0, (uint32_t)nb, (uint32_t)n, q_slots,
            (const int32_t*)(meta + g.pos), (const uint32_t*)(meta + g.seg_off), (const uint32_t*)(meta + g.q4_off), d_for,
            (int32_t*)(data + sg.seg_pos), (uint16_t*)(data + sg.seg_len), data + sg.seq2, data + sg.qual);
        unsigned long long* d_sum = reinterpret_cast<unsigned long long*>(d_nq.p);     // d_nq is free again: reuse it for the sum
        CU(cudaMemsetAsync(d_sum, 0, 8, st));
        sum_u16_kernel<<<(unsigned)std::min<size_t>(1024, ((size_t)n_seg + 255) / 256), 256, 0, st>>>((const uint16_t*)(data + sg.seg_len), n_seg, d_sum);
        unsigned long long n_aligned = 0;
        CU(cudaMemcpyAsync(&n_aligned, d_sum, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        CU(cudaGetLastError());
        attach_sample(w, s, meta, g, data, sg, msnv_sample_sizes{(uint32_t)n, (uint32_t)n_mated, L + 3, 0, (uint64_t)n_seg, (uint64_t)n_q4, (uint64_t)n_aligned});
    }
    return MSNV_OK;
}

int msnv_shard_synth(msnv_ctx* ctx, const msnv_synth_desc* d, int64_t* first_column)
{
    if (int rc = msnv_shard_synth_ref(ctx, d, first_column)) return rc;
    return msnv_window_synth(ctx, 0, d, 0, d->n_contigs);
}

int msnv_window_sample_sizes(msnv_ctx* ctx, uint32_t slot, uint32_t sample, msnv_sample_sizes* sizes);
int msnv_shard_sample_sizes(msnv_ctx* ctx, uint32_t sample, msnv_sample_sizes* sizes) { return msnv_window_sample_sizes(ctx, 0, sample, sizes); }

int msnv_window_sample_sizes(msnv_ctx* ctx, uint32_t slot, uint32_t sample, msnv_sample_sizes* sizes)
{
    if (!ctx || !sizes) return MSNV_E_ARG;
    if (!ctx->open || slot >= (uint32_t)N_SLOTS || !ctx->win[slot].open || sample >= ctx->S) return fail(ctx, MSNV_E_ARG, "msnv_window_sample_sizes: no such sample");
    msnv_ctx::Window& w = ctx->win[slot];
    if (w.has_raw && w.sizes[sample].n_reads && w.sizes[sample].n_aligned == 0) {        // expanded on the device: its count is there
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->copy_stream));
        unsigned long long v = 0;
        CU(cudaMemcpy(&v, w.d_aligned + sample, 8, cudaMemcpyDeviceToHost));
        w.sizes[sample].n_aligned = v;
    }
    *sizes = ctx->win[slot].sizes[sample];
    return MSNV_OK;
}

int msnv_shard_export_sample(msnv_ctx* ctx, uint32_t sample, int32_t* pos, uint32_t* seg_off, uint32_t* q4_off, int32_t* mate,
                             int32_t* seg_pos, uint16_t* seg_len, uint8_t* seq2, uint8_t* qual)
{
    if (!ctx) return MSNV_E_ARG;
    if (!ctx->open || sample >= ctx->S) return fail(ctx, MSNV_E_ARG, "msnv_shard_export_sample: no such sample");
    const msnv_sample_sizes z = ctx->win[0].sizes[sample];
    if (z.n_reads == 0) return MSNV_OK;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->copy_stream));
    cudaStream_t st = ctx->stream;
    const SampleDev& d = ctx->win[0].h_samples[sample];
    const size_t n = z.n_reads, n1 = n + 1;
    CU(cudaMemcpyAsync(pos, d.pos, n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(seg_off, d.seg_off, n1 * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(q4_off, d.q4_off, n1 * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(mate, d.mate, n * 4, cudaMemcpyDeviceToHost, st));
    if (z.n_segs) {
        CU(cudaMemcpyAsync(seg_pos, d.seg_pos, (size_t)z.n_segs * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(seg_len, d.seg_len, (size_t)z.n_segs * 2, cudaMemcpyDeviceToHost, st));
    }
    if (z.n_q4) {
        CU(cudaMemcpyAsync(seq2, d.seq2, (size_t)z.n_q4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(qual, d.qual, (size_t)z.n_q4 * 4, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    return MSNV_OK;
}

int msnv_shard_export_ref(msnv_ctx* ctx, uint8_t* ref)
{
    if (!ctx || !ref) return MSNV_E_ARG;
    if (!ctx->open) return fail(ctx, MSNV_E_STATE, "msnv_shard_export_ref: no open shard");
    CU(cudaSetDevice(ctx->device));
    CU(cudaMemcpyAsync(ref, ctx->d_ref, ctx->P, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return MSNV_OK;
}

int msnv_shard_counts(msnv_ctx* ctx, uint32_t sample, uint32_t first, uint32_t n, uint16_t* out)
{
    if (!ctx || !out) return MSNV_E_ARG;
    if (!ctx->has_run) return fail(ctx, MSNV_E_STATE, "msnv_shard_counts: run the shard first");
    if (sample >= ctx->S || (uint64_t)first + n > ctx->P) return fail(ctx, MSNV_E_ARG, "msnv_shard_counts: range out of bounds");
    if (n == 0) return MSNV_OK;
    // the count planes of the last range of the last run are what is still on the device
    const msnv_ctx::Window& w = ctx->win[ctx->last_slot];
    const uint64_t lo = ((uint64_t)w.t0 + ctx->last_ta) * TILE, hi = ((uint64_t)w.t0 + ctx->last_tb) * TILE;
    if (first < lo || (uint64_t)first + n > hi)
        return fail(ctx, MSNV_E_STATE, "msnv_shard_counts: positions %u..%llu are outside the last range of tiles the run kept (%llu..%llu; the tile budget split the run)",
                    first, (unsigned long long)first + n, (unsigned long long)lo, (unsigned long long)hi);
    CU(cudaSetDevice(ctx->device));
    DevBuf<uint16_t> d;                           // 5 counts per position
    CU(d.ensure((uint64_t)n * 5));
    counts_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_tiles, ctx->d_items, ctx->last_item0, ctx->d_tile_begin, w.t0, ctx->d_expect, sample, first, n, d);
    CU(cudaMemcpyAsync(out, d, (size_t)n * 10, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return MSNV_OK;
}

int msnv_get_timings(const msnv_ctx* ctx, msnv_timings* out)
{
    if (!ctx || !out) return MSNV_E_ARG;
    *out = ctx->tm;
    return MSNV_OK;
}

int msnv_cov_run(msnv_ctx* ctx, const msnv_cov_blocks* b, uint32_t max_cov, uint64_t* cov_sum, uint64_t* hist)
{
    if (!ctx || !b || !cov_sum || !hist) return MSNV_E_ARG;
    const uint32_t K = b->n_contigs;
    if (max_cov >= MSNV_COV_MAX_COUNTERS || (uint64_t)K * ((uint64_t)max_cov + 1) > MSNV_COV_MAX_COUNTERS)
        return fail(ctx, MSNV_E_LIMIT, "msnv_cov_run: %u contigs x (max_cov %u + 1) histogram counters exceed the limit of %u",
                    K, max_cov, (unsigned)MSNV_COV_MAX_COUNTERS);
    if (K == 0) return MSNV_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const uint64_t n_blocks = b->blk_off[K];
    std::vector<uint32_t> chunk0(K + 1), chunk_contig;
    uint64_t n_chunks = 0;
    for (uint32_t k = 0; k < K; ++k) {
        chunk0[k] = (uint32_t)n_chunks;
        const uint64_t c = ((uint64_t)b->contig_len[k] + COV_CHUNK - 1) / COV_CHUNK;
        n_chunks += c ? c : 1;
        if (n_chunks > 0x7fffffffull) return fail(ctx, MSNV_E_LIMIT, "msnv_cov_run: too many positions in one call");
    }
    chunk0[K] = (uint32_t)n_chunks;
    chunk_contig.resize(n_chunks);
    for (uint32_t k = 0; k < K; ++k) for (uint32_t c = chunk0[k]; c < chunk0[k + 1]; ++c) chunk_contig[c] = k;

    const size_t hist_n = (size_t)K * (max_cov + 1);
    const uint64_t n_diff = n_chunks * COV_CHUNK, n_meta = ((uint64_t)K + 1) + n_chunks + K + 2 * ((uint64_t)K + 1), n_out = K + hist_n;
    CU(ctx->d_cov_diff.ensure(n_diff, n_diff + n_diff / 8));
    CU(ctx->d_cov_beg.ensure(n_blocks, n_blocks + n_blocks / 8 + 1024));
    CU(ctx->d_cov_end.ensure(n_blocks, n_blocks + n_blocks / 8 + 1024));
    CU(ctx->d_cov_meta.ensure(n_meta, n_meta + 1024));
    CU(ctx->d_cov_out.ensure(n_out, n_out + 1024));
    int32_t* d_diff = ctx->d_cov_diff;
    uint32_t *d_beg = ctx->d_cov_beg, *d_end = ctx->d_cov_end;
    uint32_t *d_chunk0 = ctx->d_cov_meta, *d_cc = d_chunk0 + (K + 1), *d_len = d_cc + n_chunks;
    uint64_t* d_off = reinterpret_cast<uint64_t*>(ctx->d_cov_meta + (((uint64_t)K + 1) + n_chunks + K + 1) / 2 * 2);     // 8-byte aligned
    unsigned long long *d_sum = ctx->d_cov_out, *d_hist = d_sum + K;
    CU(cudaMemsetAsync(d_diff, 0, n_diff * 4, st));
    CU(cudaMemsetAsync(d_sum, 0, n_out * 8, st));
    if (n_blocks) {
        CU(cudaMemcpyAsync(d_beg, b->beg, n_blocks * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_end, b->end, n_blocks * 4, cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemcpyAsync(d_chunk0, chunk0.data(), ((size_t)K + 1) * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_cc, chunk_contig.data(), n_chunks * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_len, b->contig_len, (size_t)K * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_off, b->blk_off, ((size_t)K + 1) * 8, cudaMemcpyHostToDevice, st));
    CU(cudaEventRecord(ctx->ev[0], st));
    if (n_blocks)
        cov_scatter_kernel<<<(unsigned)((n_blocks + 255) / 256), 256, 0, st>>>(d_beg, d_end, d_off, d_chunk0, K, n_blocks, d_diff);
    CU(cudaEventRecord(ctx->ev[1], st));
    cov_scan_kernel<<<(unsigned)n_chunks, COV_THREADS, 0, st>>>(d_diff, d_cc, d_chunk0, d_len, max_cov, d_sum, d_hist);
    CU(cudaEventRecord(ctx->ev[2], st));
    CU(cudaMemcpyAsync(cov_sum, d_sum, (size_t)K * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hist, d_hist, hist_n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    ctx->tm = msnv_timings{};
    cudaEventElapsedTime(&ctx->tm.ms_cov_scatter, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->tm.ms_cov_scan, ctx->ev[1], ctx->ev[2]);
    ctx->tm.cov_blocks = n_blocks; ctx->tm.kernel_launches = n_blocks ? 2u : 1u;
    for (uint32_t k = 0; k < K; ++k) ctx->tm.cov_positions += b->contig_len[k];
    return MSNV_OK;
}

}  // extern "C"

// ---- BGZF inflate: an object of its own, so that every decoding thread can own one next to the context's thread
struct msnv_inflater {
    int device = 0;
    size_t max_bytes = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    PinnedBuf<uint8_t> h_comp, h_out;                 // page-locked staging, max_bytes each
    DevBuf<uint8_t> d_comp, d_out;
    PinnedBuf<msnv_bgzf_member> h_m; DevBuf<msnv_bgzf_member> d_m;
    PinnedBuf<int32_t> h_status; DevBuf<int32_t> d_status;
    cudaEvent_t ev[2] = {};
    float kernel_ms = 0;
};

// (the inflater's functions call it `ctx`, the name CU records an error on)
extern "C" {

uint32_t msnv_inflater_max_members(size_t max_batch_bytes) { return (uint32_t)std::min<uint64_t>(max_batch_bytes / 64 + 1024, 0xffffffffu); }

int msnv_inflater_create(int device, size_t max_batch_bytes, msnv_inflater** out)
{
    if (!out) return MSNV_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device < 0 || device >= n) return MSNV_E_CUDA;
    if (max_batch_bytes == 0) return MSNV_E_ARG;
    msnv_inflater* ctx = new msnv_inflater();
    ctx->device = device;
    ctx->max_bytes = max_batch_bytes;
    *out = ctx;                                   // returned even on failure so the caller can read the error
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (auto& e : ctx->ev) CU(cudaEventCreate(&e));
    CU(ctx->h_comp.ensure(max_batch_bytes));
    CU(ctx->h_out.ensure(max_batch_bytes));
    CU(ctx->d_comp.ensure(max_batch_bytes));
    CU(ctx->d_out.ensure(max_batch_bytes));
    // member arrays sized once for the largest batch: growing them later would free memory, which waits for the whole
    // device, including a context's work on another thread
    const uint64_t cap = msnv_inflater_max_members(max_batch_bytes);
    CU(ctx->h_m.ensure(cap));
    CU(ctx->h_status.ensure(cap));
    CU(ctx->d_m.ensure(cap));
    CU(ctx->d_status.ensure(cap));
    return MSNV_OK;
}

void msnv_inflater_destroy(msnv_inflater* inf)
{
    if (!inf) return;
    cudaSetDevice(inf->device);
    if (inf->stream) cudaStreamSynchronize(inf->stream);
    for (auto& e : inf->ev) if (e) cudaEventDestroy(e);
    if (inf->stream) cudaStreamDestroy(inf->stream);
    delete inf;                                   // (the buffers free themselves)
}

const char* msnv_inflater_last_error(const msnv_inflater* inf) { return inf ? inf->err.c_str() : "no inflater (no CUDA device?)"; }

int msnv_inflater_kernel_ms(const msnv_inflater* inf, float* ms)
{
    if (!inf || !ms) return MSNV_E_ARG;
    *ms = inf->kernel_ms;
    return MSNV_OK;
}

int msnv_inflate(msnv_inflater* ctx, const uint8_t* comp, size_t comp_bytes, const msnv_bgzf_member* m, uint32_t n,
                 uint8_t* out, int32_t* status)
{
    if (!ctx || (n && (!comp || !m || !out || !status))) return MSNV_E_ARG;
    ctx->kernel_ms = 0;
    if (n == 0) return MSNV_OK;
    if (n > ctx->d_m.cap) return fail(ctx, MSNV_E_LIMIT, "msnv_inflate: %u members exceed the inflater's %u", n, (uint32_t)ctx->d_m.cap);
    if (comp_bytes > ctx->max_bytes) return fail(ctx, MSNV_E_ARG, "msnv_inflate: %zu compressed bytes exceed the inflater's batch of %zu", comp_bytes, ctx->max_bytes);
    uint64_t out_bytes = 0;
    for (uint32_t i = 0; i < n; ++i) {
        if (m[i].coff > comp_bytes || m[i].clen > comp_bytes - m[i].coff)
            return fail(ctx, MSNV_E_ARG, "msnv_inflate: member %u lies outside the %zu compressed bytes", i, comp_bytes);
        if (m[i].ooff > ctx->max_bytes || m[i].isize > ctx->max_bytes - m[i].ooff)
            return fail(ctx, MSNV_E_ARG, "msnv_inflate: member %u's output exceeds the inflater's batch of %zu bytes", i, ctx->max_bytes);
        out_bytes = std::max<uint64_t>(out_bytes, m[i].ooff + m[i].isize);
    }
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    memcpy(ctx->h_comp, comp, comp_bytes);
    memcpy(ctx->h_m, m, (size_t)n * sizeof(msnv_bgzf_member));
    CU(cudaMemcpyAsync(ctx->d_comp, ctx->h_comp, comp_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_m, ctx->h_m, (size_t)n * sizeof(msnv_bgzf_member), cudaMemcpyHostToDevice, st));
    CU(cudaEventRecord(ctx->ev[0], st));
    inflate_kernel<<<(n + INFLATE_WARPS - 1) / INFLATE_WARPS, INFLATE_WARPS * 32, 0, st>>>(ctx->d_comp, ctx->d_m, n, ctx->d_out, ctx->d_status);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ctx->ev[1], st));
    CU(cudaMemcpyAsync(ctx->h_out, ctx->d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ctx->h_status, ctx->d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    cudaEventElapsedTime(&ctx->kernel_ms, ctx->ev[0], ctx->ev[1]);
    memcpy(out, ctx->h_out, out_bytes);
    memcpy(status, ctx->h_status, (size_t)n * 4);
    return MSNV_OK;
}

}  // extern "C"
#undef CU
