// coverage.cc -- see coverage.hpp.
#include "coverage.hpp"

#include <cstdlib>

namespace msnv {

bool CovBam::open(const std::string& path, int inflate_threads)
{
    path_ = path;
    rd_.reset(new BamReader);
    if (!rd_->open(path, inflate_threads)) {
        err_ = "Failed to open file " + path + "\nNULL pointer error (" + rd_->error() + ")";
        rd_.reset();
        return false;
    }
    head_ = rd_->header();
    bam_bytes_ = rd_->compressed_size();
    return true;
}

bool CovBam::decode(int min_qual, const char* prog)
{
    BamReader& rd = *rd_;
    const int n_targets = (int)head_.names.size();
    blk_off_.assign(1, 0);
    int currentTid = -1;
    bool warned = false;
    BamRecord r;
    int rc;
    // where the records of every contig start (BGZF virtual offsets): written next to the coverage file so that the SNV
    // calling pass can seek to the contigs of its genome bin instead of inflating every BAM once per bin (metaSNV.py:157-165)
    tidx_.first.assign((size_t)n_targets, TidIndex::NONE);
    int idx_tid = -1;
    bool ok = true;
    for (;;) {
        const uint64_t at = rd.tell();
        if ((rc = rd.next(r)) <= 0) break;
        const BamCore& c = r.core;
        if (c.tid != idx_tid && c.tid >= 0 && c.tid < n_targets) { if (tidx_.first[(size_t)c.tid] == TidIndex::NONE) tidx_.first[(size_t)c.tid] = at; idx_tid = c.tid; }
        if (c.flag & FLAG_UNMAP) { ++unmapped_; ++total_reads_; continue; }
        if (c.tid != currentTid) {
            if (c.tid == -1) {
                fprintf(stderr, "Read a read that has mapped flags, but isn't actually mapped: %s\nTrying to recover\n", r.qname);
                ++unmapped_; ++total_reads_;
                continue;
            }
            if (c.tid < currentTid || c.tid >= n_targets) { err_ = path_ + " is not coordinate sorted (or has a bad reference id)"; ok = false; break; }
            if (currentTid != -1) blk_off_.push_back(beg_.size());
            currentTid = c.tid;
            seen_tid_.push_back(c.tid);
            used_reads_.push_back(0);
        }
        if ((int)c.mapq >= min_qual) {
            if (c.flag & FLAG_PROPER_PAIR) ++proper_pairs_;
            if (c.flag & FLAG_DUP) ++duplicates_;
            else {
                const uint32_t chrSize = head_.lens[c.tid];
                uint64_t pp = (uint64_t)(uint32_t)c.pos + 1;
                int i = 0;
                if (c.n_cigar > 0) {
                    const uint32_t op0 = r.cigar_at(0) & 0xf;
                    if (op0 == CIG_S || op0 == CIG_H) i = 1;
                }
                for (; i < c.n_cigar; ++i) {
                    const uint32_t w = r.cigar_at(i), op = w & 0xf, len = w >> 4;
                    if (op != CIG_M) { pp += len; continue; }
                    const uint64_t b = pp;
                    pp += len;
                    const uint64_t e = pp >= chrSize ? (uint64_t)chrSize - 1 : pp;
                    if (b >= chrSize || e < b) {
                        // the reference writes outside its array / drives a counter negative here (undefined behaviour)
                        if (!warned) { fprintf(stderr, "%s: read %s reaches beyond contig %s; the overhang is ignored\n", prog, r.qname, head_.names[c.tid].c_str()); warned = true; }
                        continue;
                    }
                    if (e > b) { beg_.push_back((uint32_t)b); end_.push_back((uint32_t)e); }
                }
                ++used_reads_.back();
            }
        } else ++zero_quality_;
        ++total_reads_;
    }
    if (ok && rc < 0) { err_ = rd.error(); ok = false; }
    inflate_s_ = rd.inflate_seconds();
    rd_.reset();
    if (!ok) return false;
    blk_off_.push_back(beg_.size());
    if (seen_tid_.empty()) blk_off_.assign(1, 0);
    return true;
}

int CovBam::run(msnv_ctx* ctx, int max_cov, std::vector<uint64_t>& cov_sum, std::vector<uint64_t>& hist) const
{
    // per-contig coverage sum and clamped histogram (qaCompute.cpp:142-165)
    const uint32_t K = (uint32_t)seen_tid_.size();
    cov_sum.assign(K, 0);
    hist.assign((size_t)K * ((size_t)max_cov + 1), 0);
    if (!K) return MSNV_OK;
    std::vector<uint32_t> clen(K);
    for (uint32_t k = 0; k < K; ++k) clen[k] = head_.lens[seen_tid_[k]];
    msnv_cov_blocks blocks;
    blocks.n_contigs = K; blocks.contig_len = clen.data(); blocks.blk_off = blk_off_.data();
    blocks.beg = beg_.data(); blocks.end = end_.data();
    return msnv_cov_run(ctx, &blocks, (uint32_t)max_cov, cov_sum.data(), hist.data());
}

void CovBam::write_text(FILE* outputFile, FILE* detailed, bool silent, int maxCoverage, const uint64_t* cov_sum, const uint64_t* hist) const
{
    // ---- text output, in header order (qaCompute.cpp:214-217,226-263,439,600-602)
    const int n_targets = (int)head_.names.size();
    uint64_t totalGenomeLength = 0;
    for (int i = 0; i < n_targets; ++i) totalGenomeLength += head_.lens[i];
    const uint32_t K = (uint32_t)seen_tid_.size(), bins = (uint32_t)maxCoverage + 1;
    fprintf(outputFile, "Chromosome\tSeq_lem\tAvg_Cov\n");
    std::vector<uint64_t> global(bins, 0);
    uint32_t k = 0;
    for (int t = 0; t < n_targets; ++t) {
        const char* name = head_.names[t].c_str();
        const uint32_t chrSize = head_.lens[t];
        if (k < K && seen_tid_[k] == t) {
            if (!silent) {
                printf("Computing %s of size %u... \n", name, chrSize);
                fprintf(stdout, "Basing coverage on %u reads\n", used_reads_[k]);
                fprintf(stdout, "Coverage sum %lu ! \n", (unsigned long)cov_sum[k]);
                fprintf(stdout, "Average coverage over %s : %3.2f\n", name, (double)cov_sum[k] / chrSize);
            }
            if (detailed) {
                fprintf(detailed, "%s\t%d\t", name, chrSize);
                for (int i = 1; i <= maxCoverage; ++i) {
                    uint64_t coverage = 0;
                    for (int x = i; x <= maxCoverage; ++x) coverage += hist[(size_t)k * bins + x];
                    fprintf(detailed, "%d\t", int(coverage));
                }
                fprintf(detailed, "\n");
            }
            fprintf(outputFile, "%s\t%d\t%3.5f\n", name, chrSize, (double)cov_sum[k] / chrSize);
            for (uint32_t x = 0; x < bins; ++x) global[x] += hist[(size_t)k * bins + x];
            ++k;
        } else {
            if (!silent) {
                printf("Computing %s of size %u... \n", name, chrSize);
                printf("Coverage sum %d ! \n", 0);
                printf("Average coverage over %s : %3.5f\n", name, 0.0);
            }
            fprintf(outputFile, "%s\t%d\t%3.5f\n", name, chrSize, 0.0);
            if (detailed) {
                fprintf(detailed, "%s\t%d\t", name, chrSize);
                for (int i = 1; i <= maxCoverage; ++i) fprintf(detailed, "%d\t", 0);
                fprintf(detailed, "\n");
            }
        }
    }

    // ---- global table and read statistics (qaCompute.cpp:623-654)
    fprintf(outputFile, "\nCov*X\tPercentage\tNr. of bases\n");
    for (int i = 1; i <= maxCoverage; ++i) {
        uint64_t coverage = 0;
        for (int x = i; x <= maxCoverage; ++x) coverage += global[x];
        fprintf(outputFile, "%d\t%3.5f\t%lu\n", i, (double)(coverage) / totalGenomeLength * 100, (unsigned long)coverage);
    }
    fprintf(outputFile, "\nOther\n");
    double procentageOfUnmapped = 100 * ((double)unmapped_ / total_reads_);
    double procentageOfZeroQuality = 100 * ((double)zero_quality_ / total_reads_);
    fprintf(outputFile, "Total number of reads: %u\n", total_reads_);
    fprintf(outputFile, "Total number of duplicates found and ignored: %u\n", duplicates_);
    fprintf(outputFile, "Percentage of unmapped reads: %3.5f\n", procentageOfUnmapped);
    fprintf(outputFile, "Percentage of sub-par quality mappings: %3.5f\n", procentageOfZeroQuality);
    int32_t nrOfPaires = total_reads_ / 2;
    double procOfProperPaires = (double)(100 * (double)proper_pairs_ / 2) / nrOfPaires;
    fprintf(outputFile, "Number of proper paired reads: %u\n", proper_pairs_);
    fprintf(outputFile, "Percentage of proper pairs: %3.5f\n", procOfProperPaires);
}

void CovBam::save_tidx(const std::string& out) const
{
    if (!getenv("MSNV_NO_TIDX")) tidx_.save(out + ".tidx", bam_bytes_);
}

bool CovBam::write_files(const std::string& out, int max_cov, const uint64_t* cov_sum, const uint64_t* hist, std::string& err) const
{
    FILE* f = fopen(out.c_str(), "wt");
    if (!f) { err = "cannot create " + out; return false; }
    FILE* d = fopen((out + ".detail").c_str(), "wt");
    if (!d) { fclose(f); err = "cannot create " + out + ".detail"; return false; }
    save_tidx(out);
    write_text(f, d, true, max_cov, cov_sum, hist);
    const bool ok = (fclose(f) == 0) & (fclose(d) == 0);
    if (!ok) err = "cannot write " + out + " or its .detail";
    return ok;
}

void CovBam::release_blocks()
{
    std::vector<uint32_t>().swap(beg_);
    std::vector<uint32_t>().swap(end_);
}

}  // namespace msnv
