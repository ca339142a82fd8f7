// snpCall -- drop-in for the reference's src/snpCaller/snpCall (call_vC.cpp), GPU backed.
//
// Command line, exit codes and output formats are those of call_vC.cpp:346-416 (getopt string
// "hdab:f:g:i:c:p:t:"), so the unchanged metaSNV.py:166-176 drives it. Two input modes on stdin:
//   * a one-line job descriptor "#MSNV1\t<ref.fa>\t<bed or ->\t<bam list>" written by this
//     repository's `samtools mpileup` stand-in: BAMs are decoded here and the pileup itself runs on
//     the GPU (no text is ever rendered);
//   * classic `samtools mpileup` text (any real samtools): parsed on the host into count tiles, then
//     the same GPU call / compaction kernels run.
// There is no CPU calling path: without a CUDA device the program fails with a non-zero status.
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <memory>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/msnv.h"
#include "../host/pileup_input.hpp"
#include "../host/sample_layout.hpp"
#include "../host/snp_output.hpp"
#include "../host/text_pileup.hpp"

using namespace msnv;

static int print_usage()
{
    fprintf(stderr, "\n");
    fprintf(stderr, "metaSNV --- metagenomic SNV caller (B200 build)\n\n");
    fprintf(stderr, "Usage:   snpCall [options] <stdin.mpileup> \n");
    fprintf(stderr, "Options: \n");
    fprintf(stderr, "     -f,     faidx indexed reference metagenome \n ");
    fprintf(stderr, "    -g,     gene annotation file [NULL].\n");
    fprintf(stderr, "     -i,     individual SNPs output file [NULL].\n\n");
    fprintf(stderr, "SNP definition: \n");
    fprintf(stderr, "     -c,     minimum coverage (mapped reads) per position [4]\n ");
    fprintf(stderr, "    -p,     minimum non-reference nucleotide allele frequency per position [0.01].\n");
    fprintf(stderr, "     -t,     minimum number of non-reference nucleotides per position [4].\n\n");
    fprintf(stderr, "Note: Expecting samtools mpileup as standard input\n\n");
    return 1;
}

static bool verbose() { static int v = getenv("MSNV_VERBOSE") ? 1 : 0; return v != 0; }
static double g_t0 = 0;
static void stage(const char* what);
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static void stage(const char* what) { if (verbose()) fprintf(stderr, "[msnv %8.3f s] %s\n", now_s() - g_t0, what); }

static int pick_device(const std::string& indiv_path)
{
    const int n = msnv_device_count();
    if (n <= 0) return -1;
    if (const char* e = getenv("MSNV_DEVICE")) return atoi(e) % n;
    // metaSNV.py names the per-split outputs "...best_split_<k>" (metaSNV.py:199-207): split k -> GPU k mod n
    size_t p = indiv_path.rfind("best_split_");
    if (p != std::string::npos) return atoi(indiv_path.c_str() + p + 11) % n;
    return 0;
}

struct Job { std::string ref, bed, list; };

// Pinned bounce buffers between the decoding threads and the device. Page-locking memory costs about a second per
// gigabyte, so the pool is small (a few chunks, locked in the background while the first window decodes) and
// recycled: a decoding thread copies its finished batch into the chunk that is being filled (several batches share a
// chunk), the main thread queues the upload from there (DMA at the host link's rate, it overlaps the decoding) and a
// chunk goes back to the pool once it is full and the copies of all its batches have run.
struct BouncePool {
    static constexpr size_t CHUNK = (size_t)128 << 20;
    struct Chunk { uint8_t* base; size_t used; int pending; bool sealed; };
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Chunk> chunks;
    std::vector<int> free_ids;
    int cur = -1;                                          // the chunk being filled
    bool closed = false;                                   // no more chunks will come (allocation failed or stopped)
    bool aborted = false;                                  // the run failed: no chunk will be handed back, so none is handed out
    void add(uint8_t* p) { { std::lock_guard<std::mutex> lk(mu); chunks.push_back(Chunk{p, 0, 0, false}); free_ids.push_back((int)chunks.size() - 1); } cv.notify_all(); }
    void close() { { std::lock_guard<std::mutex> lk(mu); closed = true; } cv.notify_all(); }
    void abort() { { std::lock_guard<std::mutex> lk(mu); aborted = true; } cv.notify_all(); }
    // room for one batch: (pointer, chunk id), or (nullptr, -1) when the batch is larger than a chunk, there is no pool or
    // the run failed
    uint8_t* acquire(size_t bytes, int& id) {
        const size_t need = (bytes + 255) & ~(size_t)255;
        id = -1;
        if (need > CHUNK) return nullptr;
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            if (aborted) return nullptr;
            if (cur >= 0 && chunks[cur].used + need <= CHUNK) break;
            if (cur >= 0) { chunks[cur].sealed = true; maybe_free(cur); cur = -1; }
            if (!free_ids.empty()) { cur = free_ids.back(); free_ids.pop_back(); chunks[cur].used = 0; chunks[cur].sealed = false; break; }
            if (closed && chunks.empty()) return nullptr;
            cv.wait(lk);
        }
        Chunk& c = chunks[cur];
        uint8_t* p = c.base + c.used;
        c.used += need; ++c.pending;
        id = cur;
        return p;
    }
    // the copies of these batches have run
    void release(const std::vector<int>& ids) {
        { std::lock_guard<std::mutex> lk(mu); for (int id : ids) { --chunks[id].pending; maybe_free(id); } }
        cv.notify_all();
    }
private:
    void maybe_free(int id) { if (chunks[id].sealed && chunks[id].pending == 0) { chunks[id].sealed = false; chunks[id].used = 0; free_ids.push_back(id); } }
};

// one sample's batch as the library wants it: copied into a bounce chunk when it fits one (else the decoder's own arrays),
// packed by the library's block layout so that each group goes up in one copy
static msnv_raw_reads stage_raw(const RawReads& r, BouncePool& pool, int& chunk)
{
    msnv_raw_reads v = r.view();
    chunk = -1;
    if (v.n_reads == 0) return v;
    BlockLayout reads, records;
    const ReadGroup g(reads, r.pos.size());
    const RawGroup x(records, r.pos.size(), r.raw.size());
    uint8_t* p = pool.acquire(reads.size + records.size, chunk);
    if (!p) return v;
    uint8_t* p2 = p + reads.size;
    auto put = [&](uint8_t* base, size_t o, const void* src, size_t bytes) { memcpy(base + o, src, bytes); return base + o; };
    v.pos = (const int32_t*)put(p, g.pos, r.pos.data(), r.pos.size() * 4);
    v.seg_off = (const uint32_t*)put(p, g.seg_off, r.seg_off.data(), r.seg_off.size() * 4);
    v.q4_off = (const uint32_t*)put(p, g.q4_off, r.q4_off.data(), r.q4_off.size() * 4);
    v.mate = (const int32_t*)put(p, g.mate, r.mate.data(), r.mate.size() * 4);
    v.raw_off = (const uint32_t*)put(p2, x.raw_off, r.raw_off.data(), r.raw_off.size() * 4);
    v.raw = put(p2, x.raw, r.raw.data(), r.raw.size() * 4);
    v.n_cigar = (const uint16_t*)put(p2, x.n_cigar, r.n_cigar.data(), r.n_cigar.size() * 2);
    v.l_seq = (const uint16_t*)put(p2, x.l_seq, r.l_seq.data(), r.l_seq.size() * 2);
    return v;
}

static std::string dir_of(const std::string& p) { size_t k = p.rfind('/'); return k == std::string::npos ? std::string(".") : p.substr(0, k); }
static std::string base_of(const std::string& p) { size_t k = p.rfind('/'); return k == std::string::npos ? p : p.substr(k + 1); }

// Direct mode. The shard is cut into position windows (msnv_window_*): while the GPU runs window k the decoding threads
// are already on window k+1, and every finished batch of k+1 is copied to pinned memory and queued for upload at once,
// so inflate / parse, the host link and the kernels overlap and neither the host nor the device holds a whole shard.
static int run_direct(const Job& job, const msnv_call_params& prm, const std::string& fasta_opt, const std::string& genes_opt,
                      FILE* indiv, const std::string& indiv_path)
{
    const double t_start = now_s();
    std::vector<std::string> bams;
    {
        std::ifstream in(job.list);
        if (!in) { fprintf(stderr, "snpCall: cannot open %s\n", job.list.c_str()); return 1; }
        std::string l;
        while (std::getline(in, l)) {
            while (!l.empty() && (l.back() == '\r' || l.back() == ' ')) l.pop_back();
            if (!l.empty()) bams.push_back(l);
        }
    }
    const uint32_t S = (uint32_t)bams.size();
    fprintf(stderr, "Identified %d samples\n", (int)S);
    if (S == 0) return 0;

    // the CUDA context takes half a second to come up: create it while the reference is being read
    const int dev = pick_device(indiv_path);
    msnv_ctx* ctx = nullptr;
    int ctx_rc = MSNV_E_CUDA;
    std::thread ctx_thread([&]() { if (dev >= 0) ctx_rc = msnv_create(dev, &ctx); });

    std::string err;
    BamHeader hdr;
    uint64_t bam_bytes_total = 0;
    { BamReader r; if (!r.open(bams[0])) { fprintf(stderr, "snpCall: %s\n", r.error().c_str()); ctx_thread.join(); return 1; } hdr = r.header(); }
    for (const std::string& b : bams) { FILE* f = fopen(b.c_str(), "rb"); if (f) { fseek(f, 0, SEEK_END); bam_bytes_total += (uint64_t)ftell(f); fclose(f); } }
    Bed bed; bool has_bed = job.bed != "-";
    ShardLayout layout;
    Fasta fa;
    bool ok = (!has_bed || bed.load(job.bed, err)) && layout.build(hdr, has_bed ? &bed : nullptr, err) && fa.load(job.ref, err);
    if (!ok) { fprintf(stderr, "snpCall: %s\n", err.c_str()); ctx_thread.join(); return 1; }
    std::vector<int64_t> ref_len(hdr.names.size(), -1);
    for (size_t t = 0; t < hdr.names.size(); ++t) { int fi = fa.find(hdr.names[t]); if (fi >= 0) ref_len[t] = (int64_t)fa.seqs[fi].size(); }
    if (layout.n_positions == 0) { ctx_thread.join(); return 0; }
    std::vector<uint8_t> ref = shard_reference(layout, hdr, fa);

    Annotation ann;
    if (!fasta_opt.empty() && !genes_opt.empty()) {
        fprintf(stderr, "Found reference genomes and annotation file.\nLoading Genomes...\n");
        if (!ann.load(genes_opt, fasta_opt, err)) { fprintf(stderr, "%s\n", err.c_str()); ctx_thread.join(); return 255; }
        fprintf(stderr, "Genomes loaded!\n");
    }
    stage("reference and annotation loaded");
    // ---- windows: ranges of tiles sized so that one window's decoded reads are about MSNV_WINDOW_MB (default 4096)
    const uint32_t n_tiles = layout.n_positions / MSNV_TILE;
    uint64_t header_len = 0; for (uint32_t l : hdr.lens) header_len += l;
    // decoded batches take ~4x the BAM bytes (1.5 B per aligned base against ~0.4); a split reads its share of the files
    const double share = header_len ? std::min(1.0, (double)layout.n_positions / (double)header_len) : 1.0;
    const double est_bytes = 4.0 * (double)bam_bytes_total * share + 1.0;
    const double win_mb = getenv("MSNV_WINDOW_MB") ? atof(getenv("MSNV_WINDOW_MB")) : 4096.0;
    uint32_t n_windows = (uint32_t)std::ceil(est_bytes / (std::max(1.0, win_mb) * 1048576.0));
    if (getenv("MSNV_WINDOWS")) n_windows = (uint32_t)atoi(getenv("MSNV_WINDOWS"));
    const char* dump = getenv("MSNV_DUMP_COUNTS");               // (test hook below: wants the whole shard in one window)
    if (dump) n_windows = 1;
    if (n_windows < 1) n_windows = 1;
    if (n_windows > n_tiles) n_windows = n_tiles;
    const uint32_t tiles_per_window = (n_tiles + n_windows - 1) / n_windows;
    n_windows = (n_tiles + tiles_per_window - 1) / tiles_per_window;

    // wait for the context before decoding: decoding while it comes up gains nothing on average (21 interleaved runs on four
    // boxes, 2 GB of BAM: 4.1 s against 4.0 s) - it hides a slow context (1 - 3 s) but decodes slower while the driver maps
    // memory (the decoders' page faults and the driver's mappings contend for the address-space lock); BASELINE.md section 4.
    ctx_thread.join();
    stage("CUDA context created");

    // ---- decoders (one per BAM, resumable) and the thread pool
    int n_threads = (int)std::thread::hardware_concurrency();
    if (const char* e = getenv("MSNV_THREADS")) n_threads = atoi(e);
    if (n_threads < 1) n_threads = 1;
    int inflate_threads = 1;
    if ((int)S < n_threads) { inflate_threads = n_threads / (int)S; n_threads = (int)S; }
    // the coverage pass leaves "<project>/cov/<bam>.cov.tidx" (this repository's qaCompute): lets a split seek to its contigs
    const std::string cov_dir = indiv_path.empty() ? std::string() : dir_of(dir_of(indiv_path)) + "/cov/";
    std::vector<std::unique_ptr<SampleDecoder>> dec(S);
    {
        std::atomic<uint32_t> nx(0); std::atomic<bool> bad(false); std::mutex mu; std::string first_err;
        std::vector<std::thread> pool;
        for (int t = 0; t < n_threads; ++t)
            pool.emplace_back([&]() {
                for (;;) {
                    const uint32_t s = nx.fetch_add(1);
                    if (s >= S || bad) break;
                    dec[s].reset(new SampleDecoder());
                    std::string e;
                    const std::string hint = cov_dir.empty() ? std::string() : cov_dir + base_of(bams[s]) + ".cov.tidx";
                    if (!dec[s]->open(bams[s], layout, ref_len, inflate_threads, hint, e)) {
                        std::lock_guard<std::mutex> lk(mu);
                        if (first_err.empty()) first_err = e;
                        bad = true;
                    }
                }
            });
        for (auto& th : pool) th.join();
        if (bad) { fprintf(stderr, "snpCall: %s\n", first_err.c_str()); msnv_destroy(ctx); return 1; }
    }
    stage("decoders open");
    if (dev < 0 || ctx_rc != MSNV_OK) {
        fprintf(stderr, "snpCall: no usable CUDA device (%s); this build has no CPU calling path\n", msnv_last_error(ctx));
        msnv_destroy(ctx);
        return 1;
    }

    // bounce chunks are page-locked (that needs only the context) while the first window decodes; a decoding thread whose batch
    // is ready waits in acquire() for one
    BouncePool pool;
    std::atomic<bool> stop_pinning(false);
    std::thread pinner([&]() {
        size_t n = (size_t)std::min(8.0, std::max(2.0, est_bytes / (double)BouncePool::CHUNK));
        if (const char* e = getenv("MSNV_BOUNCE_CHUNKS")) n = (size_t)std::max(0, atoi(e));
        for (size_t i = 0; i < n && !stop_pinning; ++i) {
            uint8_t* p = (uint8_t*)msnv_pinned_alloc(BouncePool::CHUNK);
            if (!p) break;
            pool.add(p);
        }
        pool.close();
    });
    struct PinJoin { std::atomic<bool>& stop; std::thread& t; ~PinJoin() { stop = true; if (t.joinable()) t.join(); } } pin_join{stop_pinning, pinner};

    std::vector<RawReads> batch[2];
    batch[0].resize(S); batch[1].resize(S);
    struct WindowJob {
        std::vector<std::thread> pool; std::atomic<uint32_t> next{0}; std::atomic<bool> failed{false};
        std::mutex mu; std::vector<uint32_t> ready; std::string err; uint32_t n_done = 0;
        std::vector<msnv_raw_reads> view; std::vector<int> chunk;       // per sample: the staged batch
    };
    auto start_window = [&](WindowJob& J, uint32_t k) {
        const uint32_t lo = k * tiles_per_window * MSNV_TILE, hi = std::min<uint64_t>((uint64_t)(k + 1) * tiles_per_window * MSNV_TILE, layout.n_positions);
        J.next = 0; J.failed = false; J.ready.clear(); J.err.clear(); J.n_done = 0;
        J.view.assign(S, msnv_raw_reads{}); J.chunk.assign(S, -1);
        for (int t = 0; t < n_threads; ++t)
            J.pool.emplace_back([&J, &dec, &batch, &pool, k, lo, hi, S]() {
                for (;;) {
                    const uint32_t s = J.next.fetch_add(1);
                    if (s >= S) break;
                    std::string e;
                    bool good = true;
                    if (!J.failed) good = dec[s]->window(lo, (uint32_t)hi, k ? &batch[(k - 1) & 1][s] : nullptr, batch[k & 1][s], e);
                    if (good && !J.failed) J.view[s] = stage_raw(batch[k & 1][s], pool, J.chunk[s]);
                    std::lock_guard<std::mutex> lk(J.mu);
                    if (!good) { if (J.err.empty()) J.err = e; J.failed = true; }
                    J.ready.push_back(s);
                }
            });
    };

    stage("first window starts");
    const double t_dec0 = now_s();
    std::unique_ptr<WindowJob> cur(new WindowJob()), nxt;
    start_window(*cur, 0);
    if (msnv_shard_begin(ctx, S, layout.n_positions, ref.data()) != MSNV_OK) {
        fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx));
        cur->failed = true; pool.abort();
        for (auto& th : cur->pool) th.join();
        msnv_destroy(ctx); return 1;
    }
    HitWriter w;
    w.pop_out = stdout; w.indiv_out = indiv; w.ann = ann.active() ? &ann : nullptr;
    std::vector<HitWriter::Contig> ctgs;
    for (const auto& c : layout.ctgs) ctgs.push_back(HitWriter::Contig{hdr.names[c.tid], c.offset, c.len});
    const HitWriter::Locator locate = HitWriter::shard_locator(ctgs, ref.data());

    double t_add = 0, t_wait_upload = 0, t_run = 0, t_format = 0, t_decode_wait = 0;
    uint64_t h2d_bytes = 0, pageable_bytes = 0, n_hits_total = 0, items_total = 0, ranges_total = 0;
    msnv_timings tm_sum; memset(&tm_sum, 0, sizeof tm_sum);
    bool masked = false;
    int64_t first_col = -1;
    int rc = 0;
    for (uint32_t k = 0; k < n_windows && !rc; ++k) {
        const uint32_t slot = k & 1u;
        const uint32_t lo = k * tiles_per_window * MSNV_TILE, hi = (uint32_t)std::min<uint64_t>((uint64_t)(k + 1) * tiles_per_window * MSNV_TILE, layout.n_positions);
        if (n_windows > 1 && msnv_window_begin(ctx, slot, lo, hi) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); rc = 1; }
        // drain: queue the upload of every batch of this window as soon as its thread is through, hand bounce chunks back
        uint32_t taken = 0;
        std::vector<int> in_flight;
        auto recycle = [&]() {
            if (in_flight.empty()) return true;
            const double a = now_s();
            if (msnv_shard_sync(ctx) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); return false; }
            t_add += now_s() - a;
            pool.release(in_flight); in_flight.clear();
            return true;
        };
        while (taken < S && !rc) {
            std::vector<uint32_t> got;
            { std::lock_guard<std::mutex> lk(cur->mu); got.assign(cur->ready.begin() + taken, cur->ready.end()); }
            if (got.empty()) {
                if (!recycle()) { rc = 1; break; }                 // (threads may be waiting for a chunk)
                const double a = now_s(); std::this_thread::sleep_for(std::chrono::microseconds(100)); t_decode_wait += now_s() - a;
                continue;
            }
            taken += (uint32_t)got.size();
            if (cur->failed) { for (uint32_t s : got) if (cur->chunk[s] >= 0) in_flight.push_back(cur->chunk[s]); recycle(); continue; }
            for (uint32_t s : got) {
                const double a = now_s();
                const uint32_t lib_slot = n_windows > 1 ? slot : 0u;          // (one window: the whole shard, opened by msnv_shard_begin in slot 0)
                if (msnv_window_add_sample_raw(ctx, lib_slot, s, &cur->view[s]) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); rc = 1; break; }
                if (cur->chunk[s] >= 0) in_flight.push_back(cur->chunk[s]);
                (cur->chunk[s] >= 0 ? h2d_bytes : pageable_bytes) += batch[slot][s].bytes();
                t_add += now_s() - a;
            }
            if (in_flight.size() >= 48 && !recycle()) { rc = 1; break; }
        }
        if (!recycle()) rc = 1;
        if (rc) { cur->failed = true; pool.abort(); }
        for (auto& th : cur->pool) th.join();
        cur->pool.clear();
        if (cur->failed) { fprintf(stderr, "snpCall: %s\n", cur->err.c_str()); rc = 1; }
        if (rc) break;
        // the next window decodes while this one runs
        if (k + 1 < n_windows) { nxt.reset(new WindowJob()); start_window(*nxt, k + 1); }
        // the reference consumes the first pileup line without calling it (call_vC.cpp:423-434): the smallest first column over the samples
        if (!masked) {
            for (uint32_t s = 0; s < S; ++s) { const int64_t c = dec[s]->stats().first_column; if (c >= 0 && (first_col < 0 || c < first_col)) first_col = c; }
            if (first_col >= 0) {
                if (msnv_shard_mask_position(ctx, (uint32_t)first_col) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); rc = 1; break; }
                masked = true;
            }
        }
        double a = now_s();
        if (msnv_shard_sync(ctx) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); rc = 1; break; }     // uploads that the decoding did not hide
        t_wait_upload += now_s() - a;
        a = now_s();
        msnv_hits hits;
        const int rrc = n_windows > 1 ? msnv_window_run(ctx, slot, &prm, &hits) : msnv_shard_run(ctx, &prm, &hits);
        if (rrc != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); rc = 1; break; }
        t_run += now_s() - a;
        if (verbose()) fprintf(stderr, "[msnv %8.3f s] window %u of %u done (%u hits)\n", now_s() - g_t0, k + 1, n_windows, hits.n_hits);
        msnv_timings tm; msnv_get_timings(ctx, &tm);
        tm_sum.ms_index += tm.ms_index; tm_sum.ms_pileup += tm.ms_pileup; tm_sum.ms_call += tm.ms_call; tm_sum.ms_compact += tm.ms_compact;
        tm_sum.ms_gather += tm.ms_gather; tm_sum.kernel_launches += tm.kernel_launches; items_total += tm.n_items;
        ranges_total += tm.n_ranges;            // ranges of tiles the tile budget cut this window into

        // test hook: per-sample, per-position A,C,G,T,N counts of the whole shard (msnv_shard_counts)
        if (dump) {
            FILE* f = fopen(dump, "wb");
            FILE* g = fopen((std::string(dump) + ".layout").c_str(), "w");
            if (f && g) {
                std::vector<uint16_t> buf((size_t)layout.n_positions * 5);
                for (uint32_t s = 0; s < S; ++s) {
                    if (msnv_shard_counts(ctx, s, 0, layout.n_positions, buf.data()) != MSNV_OK) { fprintf(stderr, "snpCall: %s\n", msnv_last_error(ctx)); break; }
                    fwrite(buf.data(), 2, buf.size(), f);
                }
                fprintf(g, "%u\t%u\t%lld\n", S, layout.n_positions, (long long)first_col);
                for (const auto& c : layout.ctgs) fprintf(g, "%s\t%u\t%u\n", hdr.names[c.tid].c_str(), c.offset, c.len);
            }
            if (f) fclose(f);
            if (g) fclose(g);
        }
        a = now_s();
        w.write(hits, locate);
        n_hits_total += hits.n_hits;
        t_format += now_s() - a;
        if (k + 1 < n_windows) cur = std::move(nxt);
    }
    if (nxt) { for (auto& th : nxt->pool) th.join(); }
    if (cur) { for (auto& th : cur->pool) th.join(); }
    const double t_dec1 = now_s();
    if (rc) { msnv_destroy(ctx); return rc; }
    fflush(stdout);
    const double t_end = now_s();
    stage("kernels done, output written");

    uint64_t iupac = 0;
    if (msnv_expand_stats(ctx, &iupac) == MSNV_OK && iupac)
        fprintf(stderr, "[msnv] %llu read bases are neither A/C/G/T nor N; such bases are not counted\n", (unsigned long long)iupac);
    DecodeStats tot;
    uint32_t n_indexed = 0;
    for (uint32_t s = 0; s < S; ++s) {
        const DecodeStats& d = dec[s]->stats();
        tot.records += d.records; tot.accepted += d.accepted; tot.dropped_by_cap += d.dropped_by_cap;
        tot.aligned_bases += d.aligned_bases; tot.pairs += d.pairs; tot.compressed_bytes += d.compressed_bytes;
        tot.seconds += d.seconds; tot.inflate_seconds += d.inflate_seconds;
        n_indexed += dec[s]->used_index() ? 1u : 0u;
    }
    if (const char* pj = getenv("MSNV_PERF_JSON")) {
        FILE* f = fopen(pj, "a");
        if (f) {
            fprintf(f,
                    "{\"tool\": \"snpCall\", \"device\": %d, \"samples\": %u, \"positions\": %u, \"windows\": %u, \"bams_read_through_index\": %u, "
                    "\"records\": %llu, \"reads\": %llu, \"aligned_bases\": %llu, \"pairs\": %llu, \"dropped_by_cap\": %llu, "
                    "\"bam_bytes\": %llu, \"bam_bytes_inflated\": %llu, \"h2d_bytes\": %llu, \"h2d_pageable_bytes\": %llu, \"hits\": %llu, "
                    "\"decode_threads\": %d, \"decode_wall_s\": %.6f, \"decode_cpu_s\": %.6f, \"inflate_cpu_s\": %.6f, "
                    "\"h2d_s\": %.6f, \"h2d_not_hidden_s\": %.6f, \"waiting_for_decode_s\": %.6f, "
                    "\"gpu_run_wall_s\": %.6f, \"format_s\": %.6f, \"total_s\": %.6f, "
                    "\"ms_index\": %.4f, \"ms_pileup\": %.4f, \"ms_call\": %.4f, \"ms_compact\": %.4f, \"ms_gather\": %.4f, "
                    "\"items\": %llu, \"launches\": %u, \"ranges\": %llu}\n",
                    dev, S, layout.n_positions, n_windows, n_indexed, (unsigned long long)tot.records, (unsigned long long)tot.accepted,
                    (unsigned long long)tot.aligned_bases, (unsigned long long)tot.pairs, (unsigned long long)tot.dropped_by_cap,
                    (unsigned long long)bam_bytes_total, (unsigned long long)tot.compressed_bytes, (unsigned long long)h2d_bytes,
                    (unsigned long long)pageable_bytes, (unsigned long long)n_hits_total, n_threads * inflate_threads,
                    t_dec1 - t_dec0, tot.seconds, tot.inflate_seconds, t_add, t_wait_upload, t_decode_wait, t_run, t_format, t_end - t_start,
                    tm_sum.ms_index, tm_sum.ms_pileup, tm_sum.ms_call, tm_sum.ms_compact, tm_sum.ms_gather, (unsigned long long)items_total,
                    tm_sum.kernel_launches, (unsigned long long)ranges_total);
            fclose(f);
        }
    }
    // the process is about to exit: the driver reclaims the device; freeing every block one by one
    // (each cudaFree is a device-wide synchronisation) would only add seconds
    stop_pinning = true;
    if (pinner.joinable()) pinner.join();
    if (getenv("MSNV_CLEAN_EXIT")) { for (auto& c : pool.chunks) msnv_pinned_free(c.base); msnv_destroy(ctx); return 0; }
    // nor are the decoded batches and decoders (gigabytes of vectors) worth freeing one by one: everything is written, leave
    if (indiv) fclose(indiv);
    fflush(stdout); fflush(stderr);
    stage("exit");
    _exit(0);
}

int main(int argc, char** argv)
{
    g_t0 = now_s();
    FILE* individualFile = NULL;
    std::string fasta_opt, genes_opt, indiv_path;
    msnv_call_params prm; prm.min_coverage = 4; prm.calling_threshold = 4; prm.min_fraction = 0.01;
    int c;
    opterr = 0;
    while ((c = getopt(argc, argv, "hdab:f:g:i:c:p:t:")) != -1) switch (c) {
        case 'h': print_usage(); return -1;
        case 'a': break;
        case 'd': break;
        case 'b': break;
        case 'f': { FILE* f = fopen(optarg, "r"); if (!f) { fprintf(stderr, "Cannot open %s\n", optarg); return -1; } fclose(f); fasta_opt = optarg; break; }
        case 'g': { FILE* f = fopen(optarg, "r"); if (!f) { fprintf(stderr, "Cannot open %s\n", optarg); return -1; } fclose(f); genes_opt = optarg; break; }
        case 'i':
            individualFile = fopen(optarg, "w");
            if (!individualFile) { fprintf(stderr, "Cannot open %s\n", optarg); return -1; }
            indiv_path = optarg;
            break;
        case 'c': prm.min_coverage = (int32_t)atol(optarg); break;
        case 'p': prm.min_fraction = atof(optarg); break;
        case 't': prm.calling_threshold = (int32_t)atol(optarg); break;
        case '?':
            if (optopt == 'f') fprintf(stderr, "Option -%c requires a reference file.\n", optopt);
            else if (optopt == 'g') fprintf(stderr, "Option -%c requires an annotation file.\n", optopt);
            else if (optopt == 'i') fprintf(stderr, "Option -%c requires an output filename.\n", optopt);
            else if (isprint(optopt)) fprintf(stderr, "Unknown option `-%c'.\n", optopt);
            else { fprintf(stderr, "Unknown option character `\\x%x'.\n", optopt); return 1; }
            abort();                                   // the reference falls through to abort() (call_vC.cpp:391-409)
        default: abort();
    }
    for (int index = optind; index < argc; index++) { printf("Non-option argument %s\n", argv[index]); return 0; }

    // first line of stdin decides the mode
    std::string first;
    {
        int ch;
        while ((ch = fgetc(stdin)) != EOF) { first.push_back((char)ch); if (ch == '\n') break; }
    }
    int rc;
    if (first.compare(0, 7, "#MSNV1\t") == 0) {
        while (!first.empty() && (first.back() == '\n' || first.back() == '\r')) first.pop_back();
        std::vector<std::string> f; size_t p = 7;
        for (;;) { size_t q = first.find('\t', p); f.push_back(first.substr(p, q == std::string::npos ? q : q - p)); if (q == std::string::npos) break; p = q + 1; }
        if (f.size() != 3) { fprintf(stderr, "snpCall: malformed job descriptor on stdin\n"); return 1; }
        Job job{f[0], f[1], f[2]};
        rc = run_direct(job, prm, fasta_opt, genes_opt, individualFile, indiv_path);
    } else {
        rc = run_text_mode(first, stdin, prm, fasta_opt, genes_opt, individualFile, pick_device(indiv_path));
    }
    if (individualFile) fclose(individualFile);
    fflush(stdout); fflush(stderr);
    stage("exit");
    if (!getenv("MSNV_CLEAN_EXIT")) _exit(rc & 0xff);      // skip static destructors / CUDA runtime teardown
    return rc;
}
