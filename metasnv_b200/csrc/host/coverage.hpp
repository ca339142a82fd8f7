// coverage.hpp -- qaCompute's per-BAM logic, shared by bin/qaCompute (one BAM per process) and bin/metaSNV_coverage (a
// whole project in one process):
//   * decode: one pass over a BAM into the coverage blocks the reference would increment, the per-contig bookkeeping,
//     the read statistics and the TidIndex (qaCompute.cpp:441-593);
//   * run: per-contig coverage sums and clamped histograms of those blocks on the GPU (msnv_cov_run);
//   * write: the text of <out> and <out>.detail (qaCompute.cpp:193-263,439,600-654) and the <out>.tidx sidecar.
// The text format is written here and nowhere else.
#pragma once
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>

#include "../../../include/msnv.h"
#include "bam.hpp"

namespace msnv {

class CovBam {
public:
    // Opens the BAM and reads its header. On failure error() holds qaCompute's two-line message, which names the BAM.
    bool open(const std::string& path, int inflate_threads);
    // Reads every record (reads with mapq >= min_qual are counted). Warnings go to stderr as qaCompute prints them,
    // `prog` naming the program. On failure error() holds the message without the program's prefix. The BAM is closed
    // on return either way.
    bool decode(int min_qual, const char* prog);
    const std::string& error() const { return err_; }
    const std::string& path() const { return path_; }

    // Contigs that had a mapped record (K = seen_tid.size()); cov_sum gets K sums, hist K x (max_cov + 1) counters.
    // With K == 0 nothing runs and ctx is not used; write_text then needs neither array.
    int run(msnv_ctx* ctx, int max_cov, std::vector<uint64_t>& cov_sum, std::vector<uint64_t>& hist) const;

    // The coverage table and read statistics into `out`, the per-contig histogram into `detail` (may be null), and with
    // !silent the per-contig lines qaCompute prints on stdout.
    void write_text(FILE* out, FILE* detail, bool silent, int max_cov, const uint64_t* cov_sum, const uint64_t* hist) const;
    // "<out>.tidx" (unless MSNV_NO_TIDX is set); best effort, as a missing sidecar only costs the calling pass a full read.
    void save_tidx(const std::string& out) const;
    // What `qaCompute -c max_cov -d -i <bam> <out>` writes: <out>, <out>.detail and <out>.tidx. False with err set when a
    // file cannot be created.
    bool write_files(const std::string& out, int max_cov, const uint64_t* cov_sum, const uint64_t* hist, std::string& err) const;

    // Frees the coverage blocks (8 bytes per counted M operation), the bulk of a decoded BAM.
    void release_blocks();

    uint64_t bam_bytes() const { return bam_bytes_; }
    double inflate_seconds() const { return inflate_s_; }
    uint64_t n_blocks() const { return beg_.size(); }
    size_t n_contigs_seen() const { return seen_tid_.size(); }

private:
    std::string path_, err_;
    std::unique_ptr<BamReader> rd_;
    BamHeader head_;
    uint64_t bam_bytes_ = 0;
    double inflate_s_ = 0;
    uint32_t unmapped_ = 0, zero_quality_ = 0, total_reads_ = 0, proper_pairs_ = 0, duplicates_ = 0;
    std::vector<int> seen_tid_;             // contigs that had a mapped record, in file order
    std::vector<uint32_t> used_reads_;      // [K] reads the coverage of each is based on
    std::vector<uint64_t> blk_off_;         // [K+1]
    std::vector<uint32_t> beg_, end_;       // coverage blocks: index ranges [beg, end) of the reference's array
    TidIndex tidx_;
};

}  // namespace msnv
