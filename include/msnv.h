/* msnv.h -- C ABI of libmsnv_gpu.so: the B200 (sm_100a) implementation of metaSNV Part I's hot path.
 *
 * The reference has no library API for this path: the boundary is a process boundary
 * (metaSNV.py:63-65 spawns `qaCompute`, metaSNV.py:160-176 pipes `samtools mpileup` into
 * `snpCall`). The host programs that keep those command lines (metasnv_b200/csrc/bin) are thin:
 * they decode BAM into the structure-of-arrays batches declared here and call these entry points,
 * which are what a maintainer of the reference would bind instead of
 *   - the per-line counting / calling loop of src/snpCaller/call_vC.cpp:466-668 together with the
 *     column building that `samtools mpileup` does upstream of it (metaSNV.py:160-165), and
 *   - the scatter / prefix-sum / histogram of src/qaTools/qaCompute.cpp:530-552 and :125-221.
 *
 * Conventions: every function returns 0 on success or a negative msnv_status; nothing throws.
 * A context belongs to one device and one host thread at a time. Host buffers handed to
 * msnv_shard_add_sample() are copied asynchronously on the context's stream (a DMA when they are
 * pinned) and must stay valid until msnv_shard_sync() or msnv_shard_run() returns. Result pointers
 * are owned by the context and stay valid until the next msnv_shard_begin() / msnv_destroy().
 * There is no CPU implementation behind this ABI: without a CUDA device every call fails.
 */
#ifndef MSNV_H
#define MSNV_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSNV_ABI_VERSION 6

/* Positions per tile: contigs of a shard are laid out back to back in a "shard coordinate" space,
 * each starting at a multiple of MSNV_TILE, so a tile never spans two contigs. The kernels are written
 * for 1024 (256 quads per tile: the pileup kernel tags a staged quad with one byte); the library
 * refuses to compile for another value. */
#ifndef MSNV_TILE
#define MSNV_TILE 1024
#endif
/* Limits of the tiled pileup kernel (longer reads are rejected with MSNV_E_LIMIT). The reference span of a read (pos to
 * its last covered position, deletions and skips included) bounds how far back the index looks for a tile's reads: every
 * read starting within the span in front of a tile is a candidate of the tile. */
#define MSNV_MAX_READ_BASES 4096
#define MSNV_MAX_READ_SEGMENTS 128
#define MSNV_MAX_READ_SPAN (8 * MSNV_MAX_READ_BASES)

typedef enum {
    MSNV_OK = 0,
    MSNV_E_CUDA = -1,      /* a CUDA call failed; see msnv_last_error() */
    MSNV_E_ARG = -2,       /* invalid argument */
    MSNV_E_STATE = -3,     /* call out of order */
    MSNV_E_LIMIT = -4,     /* input exceeds a documented limit */
    MSNV_E_NOMEM = -5
} msnv_status;

typedef struct msnv_ctx msnv_ctx;

/* One sample's reads that take part in the pileup, in coordinate order. "Take part" = the read
 * passed `samtools mpileup`'s default read filters and depth cap (SURVEY.md Annex A.1, A.3); that
 * filtering is part of BAM decoding on the host, and so is the CIGAR: the device sees a read as its
 * ALIGNED SEGMENTS (one per M/=/X operation), stored position-aligned. Inserted and clipped bases
 * never reach a pileup column that snpCall counts (call_vC.cpp:503-535 skips "+n..."), so they are
 * not stored. Offsets are prefix sums with n_reads+1 entries.
 *   pos      shard coordinate of the first reference base the read covers
 *   seg_off  first segment of the read in seg_pos / seg_len
 *   q4_off   first 4-position group ("quad") of the read in `seq2` (byte index) / `qual` (byte index * 4)
 *   mate     index of the mate this read is paired with by mpileup's overlap detection (Annex A.2), else -1;
 *            symmetric (mate[mate[i]] == i), a read takes part in at most one pair
 *   seg_pos  shard coordinate of the segment's first base; ascending within a read, segments of a
 *            read do not overlap
 *   seg_len  its length in bases (>= 1)
 *   qual     segment k of a read owns nq(k) = ((seg_pos & 3) + seg_len + 3) / 4 quads, right behind
 *            the quads of segment k-1 (the first segment starts at q4_off). Byte i of those 4*nq(k)
 *            bytes belongs to shard coordinate (seg_pos & ~3) + i: the bytes of a quad are four
 *            consecutive positions starting at a multiple of four. Value: min(phred,127), bit 7 set
 *            when the base is not A/C/G/T (N or IUPAC code); the padding bytes in front of and behind
 *            the segment are 0
 *   seq2     same geometry, 2 bits per position: position k of a quad in bits 2k..2k+1 of the quad's
 *            byte, A=0 C=1 G=2 T=3 (0 for non-ACGT bases and padding)
 *   max_span largest reference span (last covered position - pos + 1) over the reads */
typedef struct {
    uint32_t        n_reads;
    uint32_t        max_span;
    uint32_t        reserved0, reserved1;
    const int32_t*  pos;
    const uint32_t* seg_off;
    const uint32_t* q4_off;
    const int32_t*  mate;
    const int32_t*  seg_pos;
    const uint16_t* seg_len;
    const uint8_t*  seq2;
    const uint8_t*  qual;
} msnv_sample_reads;

/* The same reads as BAM stores them: the device walks the CIGARs, packs the bases and lays the aligned segments out
 * (what `samtools mpileup`'s resolve_cigar2 / pileup_seq do per column upstream of snpCall, metaSNV.py:160-165); the host
 * only supplies what it has after filtering anyway. Per read:
 *   pos       shard coordinate of the first reference base
 *   mate      as in msnv_sample_reads
 *   seg_off, q4_off   prefix sums (n_reads + 1) of the read's aligned segments (M/=/X operations of non-zero length) and of the
 *             quads they occupy in the position-aligned layout (a segment at shard coordinate x of length l: ((x & 3) + l + 3) / 4)
 *   raw_off   prefix sums (n_reads + 1) of the reads' blobs in `raw`, in units of 4 bytes
 *   n_cigar, l_seq   as in the BAM record
 *   raw       per read, 4-byte aligned: n_cigar little-endian u32 CIGAR operations (len << 4 | op), (l_seq + 1) / 2 bytes
 *             of 4-bit bases, l_seq phred qualities - the record's own bytes, BAM section 4.2 */
typedef struct {
    uint32_t        n_reads;
    uint32_t        max_span;
    uint32_t        reserved0, reserved1;
    const int32_t*  pos;
    const int32_t*  mate;
    const uint32_t* seg_off;
    const uint32_t* q4_off;
    const uint32_t* raw_off;
    const uint16_t* n_cigar;
    const uint16_t* l_seq;
    const uint8_t*  raw;
} msnv_raw_reads;

/* snpCall's thresholds (call_vC.cpp:26-36, options -c -t -p). */
typedef struct {
    int32_t min_coverage;       /* -c, default 4 */
    int32_t calling_threshold;  /* -t, default 4 */
    double  min_fraction;       /* -p, default 0.01 */
} msnv_call_params;

/* Called positions of a shard, ascending by position. Allele order in every mask/array is
 * A, C, G, T (bit 0..3 / index 0..3). A position is listed when pop_mask | ind_mask != 0:
 *   pop_mask  alleles passing the population test   (call_vC.cpp:588)  -> called_SNPs line
 *   ind_mask  alleles passing only the individual test (call_vC.cpp:592-600) -> indiv_called line
 *   cov       [n_hits][n_samples] per-sample coverage (the "c1|...|cS" column, call_vC.cpp:316-325)
 *   allele    [n_hits][4][n_samples] per-sample count of each non-reference allele (0 for the
 *             reference's own base, which mpileup renders as '.'/',')
 *   total     [n_hits][5] population totals: coverage, then A, C, G, T */
typedef struct {
    uint32_t        n_hits;
    uint32_t        n_samples;
    const uint32_t* pos;
    const uint8_t*  pop_mask;
    const uint8_t*  ind_mask;
    const uint16_t* cov;
    const uint16_t* allele;
    const uint32_t* total;
} msnv_hits;

/* Device-side timings of the last msnv_shard_run(), milliseconds (CUDA events on the context's
 * stream), plus the work it did. */
typedef struct {
    float    ms_index, ms_d2h /* copy of the hits to the host, not part of ms_total */;
    float    ms_pileup /* mate-overlap pass + pileup kernel */, ms_call, ms_compact, ms_gather;
    float    ms_total;          /* index + pileup + call + compact + gather */
    uint64_t n_items;           /* active (sample, tile) pairs */
    uint64_t n_reads;
    uint64_t n_bases;           /* staged base slots resident for the window (4 x quads, padding included) */
    uint32_t n_tiles;
    uint32_t kernel_launches;
    uint32_t n_ranges;          /* ranges of tiles the run was split into to fit the tile budget (1 = none) */
    float    ms_mate;           /* the mate-overlap pass alone (included in ms_pileup) */
    /* last msnv_cov_run(): device time of its two kernels (difference scatter; prefix sum + histogram), what they processed */
    float    ms_cov_scatter, ms_cov_scan;
    uint32_t reserved;
    uint64_t cov_positions, cov_blocks;
} msnv_timings;

int         msnv_abi_version(void);
int         msnv_tile(void);              /* MSNV_TILE the library was built with */
int         msnv_device_count(void);
int         msnv_create(int device, msnv_ctx** out);
void        msnv_destroy(msnv_ctx* ctx);
const char* msnv_last_error(const msnv_ctx* ctx);

/* Page-locked host memory for the batches handed to msnv_shard_add_sample() (cudaHostAlloc / cudaFreeHost);
 * usable from any thread once a context exists. */
void*       msnv_pinned_alloc(size_t bytes);
void        msnv_pinned_free(void* p);

/* ---- pileup + call (replaces `samtools mpileup ... | snpCall`, metaSNV.py:160-176) ---- */

/* Start a shard of n_positions shard coordinates (a multiple of MSNV_TILE) seen by n_samples
 * samples. `ref` holds one reference character per position exactly as mpileup would print it
 * (FASTA case preserved, 'N' where the FASTA has no base); 0 marks a position that must not be
 * called (padding between contigs, positions outside the -l BED, the first pileup line that
 * call_vC.cpp:423 consumes). */
int msnv_shard_begin(msnv_ctx* ctx, uint32_t n_samples, uint32_t n_positions, const uint8_t* ref);
/* Copy one sample's reads to the device. Samples without reads need not be added. */
int msnv_shard_add_sample(msnv_ctx* ctx, uint32_t sample, const msnv_sample_reads* reads);
/* Mark one shard coordinate as not callable after msnv_shard_begin() (same effect as ref[pos] = 0). */
int msnv_shard_mask_position(msnv_ctx* ctx, uint32_t pos);
/* Wait until every copy queued by msnv_shard_add_sample() has completed. */
int msnv_shard_sync(msnv_ctx* ctx);
/* Run pileup (with mpileup's mate-overlap quality correction), calling and compaction; fills *hits.
 * The uploaded reads are never modified, so it may be called repeatedly, e.g. with other parameters. */
int msnv_shard_run(msnv_ctx* ctx, const msnv_call_params* params, msnv_hits* hits);
/* ---- shards larger than device memory: position windows ----
 * A shard may be processed as a sequence of windows [pos_lo, pos_hi) of shard coordinates (multiples of MSNV_TILE,
 * ascending, disjoint), the way the reference streams through its input with O(samples) memory (call_vC.cpp:466-479).
 * For each window the caller hands in, per sample, the reads that overlap it (pos < pos_hi and last covered position
 * >= pos_lo; a read that straddles a boundary is given to both windows, mate links are window-local) and gets the
 * called positions inside it. The context has two window slots: queue the uploads of window k+1 (slot (k+1) & 1)
 * before calling msnv_window_run() for window k and the copies overlap its kernels. msnv_window_run() returns
 * when the hits are on the host; the slot's host buffers may be reused then.
 * msnv_shard_begin() opens the whole shard as one window in slot 0, which is what msnv_shard_add_sample() and
 * msnv_shard_run() operate on. Whatever the window, count planes are produced for ranges of tiles that fit the
 * free device memory (MSNV_TILE_BUDGET_MB overrides), so neither reads nor counts of a shard must fit the device. */
int msnv_window_begin(msnv_ctx* ctx, uint32_t slot, uint32_t pos_lo, uint32_t pos_hi);
int msnv_window_add_sample(msnv_ctx* ctx, uint32_t slot, uint32_t sample, const msnv_sample_reads* reads);
int msnv_window_run(msnv_ctx* ctx, uint32_t slot, const msnv_call_params* params, msnv_hits* hits);
/* The same as msnv_window_add_sample() from BAM-shaped records: copied to the device and expanded there (expand_kernel:
 * CIGAR walk, 4-bit -> 2-bit bases, quality capping, position alignment). Slot 0 after msnv_shard_begin() is the whole shard.
 * msnv_expand_stats(): bases seen so far that are neither A/C/G/T nor N (IUPAC codes; they are counted as "other"). */
int msnv_window_add_sample_raw(msnv_ctx* ctx, uint32_t slot, uint32_t sample, const msnv_raw_reads* reads);
int msnv_expand_stats(msnv_ctx* ctx, uint64_t* iupac_bases);

/* Test/inspection hook: per-position A,C,G,T,N counts ([n][5], uint16) of one sample after the last
 * run, for shard coordinates [first, first+n). */
int msnv_shard_counts(msnv_ctx* ctx, uint32_t sample, uint32_t first, uint32_t n, uint16_t* out);
int msnv_get_timings(const msnv_ctx* ctx, msnv_timings* out);

/* Classic mode: counts parsed by the host from `samtools mpileup` text (call_vC.cpp:503-535) for a
 * batch of n_positions pileup lines (a multiple of MSNV_TILE; pad with ref = 0). Layout of both
 * arrays: [tile][sample][MSNV_TILE]. acgt packs the letter counts a+A | c+C << 16 | g+G << 32 | t+T << 48,
 * matches holds '.' + ','. Runs the same call / compaction / gather kernels as msnv_shard_run();
 * hit positions index the batch's lines. Replaces any open shard. */
int msnv_call_counts(msnv_ctx* ctx, uint32_t n_samples, uint32_t n_positions, const uint8_t* ref, const uint64_t* acgt,
                     const uint16_t* matches, const msnv_call_params* params, msnv_hits* hits);

/* ---- synthetic shards (benchmark / test input, no reference counterpart) ----
 * Fills a shard on the device from the stateless read model of csrc/host/synth_model.h -- the same
 * model `msnv_synth` writes BAM files from -- so the full BASELINE.json shapes can be benchmarked
 * without materialising hundreds of GB of BAM. Equivalent to msnv_shard_begin() plus one
 * msnv_shard_add_sample() per sample with what decoding those BAMs yields (only reads the mpileup
 * filters accept; the model's filtered "junk" records do not exist here). */
typedef struct {
    uint64_t seed;
    uint32_t n_samples, read_len, depth_x100, presence_ppm, paired_pct, site_ppm, err_ppm, nbase_ppm, refn_ppm;
    uint32_t indel_pct_x10, clip_pct_x10, mapq0_pct_x10;
    uint32_t n_contigs;
    const uint32_t* contig_len;      /* [n_contigs], in header (tid) order */
    const uint32_t* contig_genome;   /* [n_contigs] genome index of each contig */
    uint32_t        n_genomes;
    const uint32_t* genome_n_sub;    /* [n_genomes] number of subspecies clusters */
} msnv_synth_desc;
/* first_column (optional): shard coordinate of the first pileup column, i.e. what the caller would
 * pass to msnv_shard_mask_position(); -1 when the shard has no reads. */
int msnv_shard_synth(msnv_ctx* ctx, const msnv_synth_desc* desc, int64_t* first_column);
/* The same in two steps, for shards that do not fit the device: msnv_shard_synth_ref() begins the shard and generates its
 * reference; msnv_window_synth() then opens the window that covers contigs [ctg_lo, ctg_hi) in `slot` and fills it with
 * their reads (msnv_window_run() processes it). msnv_shard_synth() = the reference + one window with every contig. */
int msnv_shard_synth_ref(msnv_ctx* ctx, const msnv_synth_desc* desc, int64_t* first_column);
int msnv_window_synth(msnv_ctx* ctx, uint32_t slot, const msnv_synth_desc* desc, uint32_t ctg_lo, uint32_t ctg_hi);

/* Copy one sample of the open shard back to host arrays sized from *sizes (as returned by
 * msnv_shard_sample_sizes): used to stage pinned host buffers for end-to-end timing. */
typedef struct { uint32_t n_reads, n_mated, max_span, reserved; uint64_t n_segs, n_q4, n_aligned /* sum of seg_len */; } msnv_sample_sizes;
int msnv_shard_sample_sizes(msnv_ctx* ctx, uint32_t sample, msnv_sample_sizes* sizes);                  /* window slot 0 */
int msnv_window_sample_sizes(msnv_ctx* ctx, uint32_t slot, uint32_t sample, msnv_sample_sizes* sizes);
int msnv_shard_export_sample(msnv_ctx* ctx, uint32_t sample, int32_t* pos, uint32_t* seg_off, uint32_t* q4_off, int32_t* mate,
                             int32_t* seg_pos, uint16_t* seg_len, uint8_t* seq2, uint8_t* qual);
/* Copy the shard's reference characters (n_positions bytes) back to the host. */
int msnv_shard_export_ref(msnv_ctx* ctx, uint8_t* ref);

/* ---- coverage (replaces the reductions of qaCompute, metaSNV.py:63-65) ---- */

/* Coverage blocks of one BAM: for every read qaCompute counts (qaCompute.cpp:461-462,518,524-526)
 * and every 'M' operation, the half-open index range [beg, end) of its contig's coverage array that
 * the reference increments (qaCompute.cpp:530-552, including its 1-based shift and end clamp).
 * Blocks are grouped by contig: blocks of contig k are blk_off[k] .. blk_off[k+1]; within a contig
 * they are in file order (non-decreasing beg up to the span of one read). */
typedef struct {
    uint32_t        n_contigs;
    const uint32_t* contig_len;   /* [n_contigs] chrSize */
    const uint64_t* blk_off;      /* [n_contigs+1] */
    const uint32_t* beg;          /* [blk_off[n_contigs]] */
    const uint32_t* end;
} msnv_cov_blocks;

/* Per contig: cov_sum[k] = sum of coverage over indices [0, chrSize) and hist[k][c] for
 * c = 0..max_cov = number of indices with min(coverage, max_cov) == c (qaCompute.cpp:142-165).
 * Any max_cov is exact; the histograms of one call may hold at most MSNV_COV_MAX_COUNTERS counters
 * (n_contigs x (max_cov + 1), 8 bytes each on the device and in `hist`), more is MSNV_E_LIMIT. */
#define MSNV_COV_MAX_COUNTERS (1u << 27)
int msnv_cov_run(msnv_ctx* ctx, const msnv_cov_blocks* blocks, uint32_t max_cov, uint64_t* cov_sum, uint64_t* hist);

/* ---- BGZF inflate on the device (the decompression in front of every BAM decode) ----
 * An inflater owns a stream, device buffers and page-locked staging buffers on one device. It is separate from the
 * context: one inflater serves one host thread at a time, and different inflaters may be used from different threads
 * at the same time as each other and as a context's calls. */
typedef struct msnv_inflater msnv_inflater;

/* One BGZF member of a batch: its raw-DEFLATE data comp[coff, coff + clen), the ISIZE and CRC32 of its trailer, and
 * where its isize inflated bytes go in the output (out[ooff, ooff + isize)). */
typedef struct { uint64_t coff; uint32_t clen, isize, crc, reserved; uint64_t ooff; } msnv_bgzf_member;

/* Per-member result of msnv_inflate(). */
typedef enum {
    MSNV_INFLATE_OK = 0,
    MSNV_INFLATE_TRUNCATED = 1,     /* the stream ends before its final block does */
    MSNV_INFLATE_BAD_CODE = 2,      /* invalid block type, stored length, code lengths or code */
    MSNV_INFLATE_BAD_DISTANCE = 3,  /* a match reaches in front of the member's first output byte */
    MSNV_INFLATE_TOO_LONG = 4,      /* the stream holds more than isize bytes */
    MSNV_INFLATE_TOO_SHORT = 5,     /* the stream holds fewer than isize bytes */
    MSNV_INFLATE_BAD_CRC = 6        /* the inflated bytes do not have the trailer's CRC32 */
} msnv_inflate_status;

/* max_batch_bytes bounds both comp_bytes and the output span of one msnv_inflate() call, and a call takes at most
 * msnv_inflater_max_members(max_batch_bytes) = max_batch_bytes / 64 + 1024 members (MSNV_E_LIMIT beyond; a BGZF member
 * of real data is far larger than 64 bytes). Every buffer is allocated here, none later. */
uint32_t    msnv_inflater_max_members(size_t max_batch_bytes);
int         msnv_inflater_create(int device, size_t max_batch_bytes, msnv_inflater** out);
/* Inflates n members into out[0, max(ooff + isize)) and returns when out is filled on the host. status[i] is the
 * member's msnv_inflate_status; a malformed member affects no other member. Output bytes that no member covers are
 * unspecified. Returns MSNV_E_ARG for a member outside comp or a batch above max_batch_bytes. */
int         msnv_inflate(msnv_inflater* inf, const uint8_t* comp, size_t comp_bytes, const msnv_bgzf_member* m, uint32_t n,
                         uint8_t* out, int32_t* status);
void        msnv_inflater_destroy(msnv_inflater* inf);
const char* msnv_inflater_last_error(const msnv_inflater* inf);
/* Device time of the last msnv_inflate() call's kernel, milliseconds (CUDA events; copies excluded). */
int         msnv_inflater_kernel_ms(const msnv_inflater* inf, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* MSNV_H */
