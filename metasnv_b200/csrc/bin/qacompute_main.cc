// qaCompute -- drop-in for the reference's src/qaTools/qaCompute (qaCompute.cpp), GPU backed.
//
// Keeps the command line (getopt string "mdip:s:q:c:h:x:a:", qaCompute.cpp:312), the two output
// files and their exact text (qaCompute.cpp:193-217,239-246,439,623-654) for the surface metaSNV.py
// uses: `qaCompute -c 10 -d -i <bam> <out>` (metaSNV.py:63-65). The host streams the BAM once and
// turns every counted 'M' operation into the index range the reference would increment
// (qaCompute.cpp:530-552); prefix sums, per-contig coverage sums and histograms run on the GPU
// (msnv_cov_run). The modes metaSNV never uses (-m median, -p profile, -s span coverage, -x regions,
// -a subsampling, -h alternative header) are parsed and refused.
#include <getopt.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <algorithm>
#include <vector>

#include "../../../include/msnv.h"
#include "../host/bam.hpp"

using namespace msnv;

static int print_usage()
{
    fprintf(stderr, "\n");
    fprintf(stderr, "Usage:   qaCompute [options] <in.bam> <output.out>\n");
    fprintf(stderr, "Options: \n");
    fprintf(stderr, "         -q            Quality threshold. (min quality to consider) [1].\n");
    fprintf(stderr, "         -d            Print per-chromosome histogram [<output.out>.detail]\n");
    fprintf(stderr, "         -i            Silent.Don't print too much stuff!\n");
    fprintf(stderr, "         -c [INT]      Maximum coverage to consider in histogram [30]\n");
    fprintf(stderr, "         -m -p -s -x -a -h are not supported by the B200 build\n");
    fprintf(stderr, "\n");
    fprintf(stderr, "Note: Input file should be sorted\n\n");
    return 1;
}

int main(int argc, char* argv[])
{
    int maxCoverage = 30, minQual = 1;
    bool doDetail = false, silent = false;
    int arg;
    while ((arg = getopt(argc, argv, "mdip:s:q:c:h:x:a:")) >= 0) {
        switch (arg) {
            case 'd': doDetail = true; break;
            case 'i': silent = true; break;
            case 'q': minQual = atoi(optarg); break;
            case 'c': maxCoverage = atoi(optarg); break;
            case 'm': case 'p': case 's': case 'h': case 'x': case 'a':
                fprintf(stderr, "qaCompute: option -%c is not supported by the B200 build (metaSNV.py only uses -c -d -i)\n", arg);
                return -1;
            default:
                fprintf(stderr, "Read wrong argument %d with value %s\n", arg, optarg);
                return -1;
        }
    }
    if (argc - optind != 2) { print_usage(); return 1; }
    if (maxCoverage < 1) { fprintf(stderr, "qaCompute: -c must be at least 1\n"); return -1; }

    // BGZF members are independent: inflate them with a few threads (metaSNV.py runs `--threads` of these processes at once,
    // metaSNV.py:58, so the default stays small; MSNV_THREADS overrides)
    int inflate_threads = std::min(4u, std::max(1u, std::thread::hardware_concurrency() / 4u));
    if (const char* e = getenv("MSNV_THREADS")) inflate_threads = std::max(1, atoi(e));
    // GPU of this process: MSNV_DEVICE, else spread the BAMs over the GPUs by a hash of the path. The CUDA context takes about
    // half a second to come up: create it in the background while the BAM is being read.
    const int nd = msnv_device_count();
    int dev = 0;
    if (const char* e = getenv("MSNV_DEVICE")) dev = atoi(e);
    else if (nd > 1) { uint32_t hsh = 2166136261u; for (const char* c = argv[optind]; *c; ++c) hsh = (hsh ^ (unsigned char)*c) * 16777619u; dev = (int)(hsh % (uint32_t)nd); }
    msnv_ctx* ctx = nullptr;
    int ctx_rc = MSNV_E_CUDA;
    std::thread ctx_thread([&]() { if (nd > 0) ctx_rc = msnv_create(dev % nd, &ctx); });
    struct Joiner { std::thread& t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{ctx_thread};

    BamReader rd;
    if (!rd.open(argv[optind], inflate_threads)) {
        fprintf(stderr, "qaCompute: Failed to open file %s\n", argv[optind]);
        fprintf(stderr, "NULL pointer error (%s)\n", rd.error().c_str());
        return 1;
    }
    const BamHeader& head = rd.header();
    FILE* outputFile = fopen(argv[optind + 1], "wt");
    if (!outputFile) { fprintf(stderr, "qaCompute: Filed to create output file %s\n", argv[optind + 1]); return 1; }
    FILE* detailed = NULL;
    if (doDetail) {
        std::string fName = std::string(argv[optind + 1]) + ".detail";
        detailed = fopen(fName.c_str(), "wt");
        if (!detailed) fprintf(stderr, "qaCompute: Unable to create detailed output file %s. No details will be printed!\n", fName.c_str());
        fprintf(stdout, "Printing details in %s!\n", fName.c_str());
    }

    const int n_targets = (int)head.names.size();
    uint64_t totalGenomeLength = 0;
    for (int i = 0; i < n_targets; ++i) totalGenomeLength += head.lens[i];

    // ---- one pass over the BAM: read statistics and coverage blocks (qaCompute.cpp:441-593)
    uint32_t unmappedReads = 0, zeroQualityReads = 0, totalNumberOfReads = 0, totalProperPaires = 0, duplicates = 0;
    std::vector<int> seen_tid;                 // contigs that had a mapped record, in file order
    std::vector<uint32_t> used_reads;
    std::vector<uint64_t> blk_off(1, 0);
    std::vector<uint32_t> beg, end;
    int currentTid = -1;
    bool warned = false;
    BamRecord r;
    int rc;
    // where the records of every contig start (BGZF virtual offsets): written next to the coverage file so that the SNV
    // calling pass can seek to the contigs of its genome bin instead of inflating every BAM once per bin (metaSNV.py:157-165)
    TidIndex tidx;
    tidx.first.assign((size_t)n_targets, TidIndex::NONE);
    int idx_tid = -1;
    for (;;) {
        const uint64_t at = rd.tell();
        if ((rc = rd.next(r)) <= 0) break;
        const BamCore& c = r.core;
        if (c.tid != idx_tid && c.tid >= 0 && c.tid < n_targets) { if (tidx.first[(size_t)c.tid] == TidIndex::NONE) tidx.first[(size_t)c.tid] = at; idx_tid = c.tid; }
        if (c.flag & FLAG_UNMAP) { ++unmappedReads; ++totalNumberOfReads; continue; }
        if (c.tid != currentTid) {
            if (c.tid == -1) {
                fprintf(stderr, "Read a read that has mapped flags, but isn't actually mapped: %s\nTrying to recover\n", r.qname);
                ++unmappedReads; ++totalNumberOfReads;
                continue;
            }
            if (c.tid < currentTid || c.tid >= n_targets) { fprintf(stderr, "qaCompute: %s is not coordinate sorted (or has a bad reference id)\n", argv[optind]); return 1; }
            if (currentTid != -1) blk_off.push_back(beg.size());
            currentTid = c.tid;
            seen_tid.push_back(c.tid);
            used_reads.push_back(0);
        }
        if ((int)c.mapq >= minQual) {
            if (c.flag & FLAG_PROPER_PAIR) ++totalProperPaires;
            if (c.flag & FLAG_DUP) ++duplicates;
            else {
                const uint32_t chrSize = head.lens[c.tid];
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
                        if (!warned) { fprintf(stderr, "qaCompute: read %s reaches beyond contig %s; the overhang is ignored\n", r.qname, head.names[c.tid].c_str()); warned = true; }
                        continue;
                    }
                    if (e > b) { beg.push_back((uint32_t)b); end.push_back((uint32_t)e); }
                }
                ++used_reads.back();
            }
        } else ++zeroQualityReads;
        ++totalNumberOfReads;
    }
    if (rc < 0) { fprintf(stderr, "qaCompute: %s\n", rd.error().c_str()); return 1; }
    blk_off.push_back(beg.size());
    if (seen_tid.empty()) blk_off.assign(1, 0);

    // ---- GPU: per-contig coverage sum and clamped histogram (qaCompute.cpp:142-165)
    const uint32_t K = (uint32_t)seen_tid.size();
    if ((uint64_t)std::max<uint32_t>(K, 1) * ((uint64_t)maxCoverage + 1) > MSNV_COV_MAX_COUNTERS) {
        fprintf(stderr, "qaCompute: -c %d needs more than %u histogram counters for %u contigs\n", maxCoverage, (unsigned)MSNV_COV_MAX_COUNTERS, K);
        return 1;
    }
    const uint32_t bins = (uint32_t)maxCoverage + 1;
    std::vector<uint64_t> cov_sum(K, 0), hist((size_t)K * bins, 0);
    if (K) {
        std::vector<uint32_t> clen(K);
        for (uint32_t k = 0; k < K; ++k) clen[k] = head.lens[seen_tid[k]];
        ctx_thread.join();
        if (nd <= 0 || ctx_rc != MSNV_OK) {
            fprintf(stderr, "qaCompute: no usable CUDA device (%s); this build has no CPU path\n", msnv_last_error(ctx));
            msnv_destroy(ctx);
            return 1;
        }
        msnv_cov_blocks blocks;
        blocks.n_contigs = K; blocks.contig_len = clen.data(); blocks.blk_off = blk_off.data();
        blocks.beg = beg.data(); blocks.end = end.data();
        if (msnv_cov_run(ctx, &blocks, (uint32_t)maxCoverage, cov_sum.data(), hist.data()) != MSNV_OK) {
            fprintf(stderr, "qaCompute: %s\n", msnv_last_error(ctx));
            msnv_destroy(ctx);
            return 1;
        }
        if (getenv("MSNV_CLEAN_EXIT")) msnv_destroy(ctx);      // otherwise left to process exit (see snpcall_main.cc)
    }

    if (!getenv("MSNV_NO_TIDX")) tidx.save(std::string(argv[optind + 1]) + ".tidx", rd.compressed_size());     // best effort

    // ---- text output, in header order (qaCompute.cpp:214-217,226-263,439,600-602)
    fprintf(outputFile, "Chromosome\tSeq_lem\tAvg_Cov\n");
    std::vector<uint64_t> global(bins, 0);
    uint32_t k = 0;
    for (int t = 0; t < n_targets; ++t) {
        const char* name = head.names[t].c_str();
        const uint32_t chrSize = head.lens[t];
        if (k < K && seen_tid[k] == t) {
            if (!silent) {
                printf("Computing %s of size %u... \n", name, chrSize);
                fprintf(stdout, "Basing coverage on %u reads\n", used_reads[k]);
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
    double procentageOfUnmapped = 100 * ((double)unmappedReads / totalNumberOfReads);
    double procentageOfZeroQuality = 100 * ((double)zeroQualityReads / totalNumberOfReads);
    fprintf(outputFile, "Total number of reads: %u\n", totalNumberOfReads);
    fprintf(outputFile, "Total number of duplicates found and ignored: %u\n", duplicates);
    fprintf(outputFile, "Percentage of unmapped reads: %3.5f\n", procentageOfUnmapped);
    fprintf(outputFile, "Percentage of sub-par quality mappings: %3.5f\n", procentageOfZeroQuality);
    int32_t nrOfPaires = totalNumberOfReads / 2;
    double procOfProperPaires = (double)(100 * (double)totalProperPaires / 2) / nrOfPaires;
    fprintf(outputFile, "Number of proper paired reads: %u\n", totalProperPaires);
    fprintf(outputFile, "Percentage of proper pairs: %3.5f\n", procOfProperPaires);
    fclose(outputFile);
    if (detailed) fclose(detailed);
    fflush(stdout); fflush(stderr);
    if (!getenv("MSNV_CLEAN_EXIT")) _exit(0);
    return 0;
}
