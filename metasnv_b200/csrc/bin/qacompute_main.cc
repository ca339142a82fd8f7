// qaCompute -- drop-in for the reference's src/qaTools/qaCompute (qaCompute.cpp), GPU backed.
//
// Keeps the command line (getopt string "mdip:s:q:c:h:x:a:", qaCompute.cpp:312), the two output
// files and their exact text (qaCompute.cpp:193-217,239-246,439,623-654) for the surface metaSNV.py
// uses: `qaCompute -c 10 -d -i <bam> <out>` (metaSNV.py:63-65). The host streams the BAM once and
// turns every counted 'M' operation into the index range the reference would increment
// (qaCompute.cpp:530-552); prefix sums, per-contig coverage sums and histograms run on the GPU
// (msnv_cov_run). The per-BAM logic and the text format live in host/coverage.cc, which
// bin/metaSNV_coverage shares. The modes metaSNV never uses (-m median, -p profile, -s span coverage, -x regions,
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
#include "../host/coverage.hpp"

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

    CovBam bam;
    if (!bam.open(argv[optind], inflate_threads)) {
        fprintf(stderr, "qaCompute: %s\n", bam.error().c_str());
        return 1;
    }
    FILE* outputFile = fopen(argv[optind + 1], "wt");
    if (!outputFile) { fprintf(stderr, "qaCompute: Filed to create output file %s\n", argv[optind + 1]); return 1; }
    FILE* detailed = NULL;
    if (doDetail) {
        std::string fName = std::string(argv[optind + 1]) + ".detail";
        detailed = fopen(fName.c_str(), "wt");
        if (!detailed) fprintf(stderr, "qaCompute: Unable to create detailed output file %s. No details will be printed!\n", fName.c_str());
        fprintf(stdout, "Printing details in %s!\n", fName.c_str());
    }

    // ---- one pass over the BAM: read statistics and coverage blocks
    if (!bam.decode(minQual, "qaCompute")) { fprintf(stderr, "qaCompute: %s\n", bam.error().c_str()); return 1; }

    // ---- GPU: per-contig coverage sum and clamped histogram
    const uint32_t K = (uint32_t)bam.n_contigs_seen();
    if ((uint64_t)std::max<uint32_t>(K, 1) * ((uint64_t)maxCoverage + 1) > MSNV_COV_MAX_COUNTERS) {
        fprintf(stderr, "qaCompute: -c %d needs more than %u histogram counters for %u contigs\n", maxCoverage, (unsigned)MSNV_COV_MAX_COUNTERS, K);
        return 1;
    }
    std::vector<uint64_t> cov_sum, hist;
    if (K) {
        ctx_thread.join();
        if (nd <= 0 || ctx_rc != MSNV_OK) {
            fprintf(stderr, "qaCompute: no usable CUDA device (%s); this build has no CPU path\n", msnv_last_error(ctx));
            msnv_destroy(ctx);
            return 1;
        }
        if (bam.run(ctx, maxCoverage, cov_sum, hist) != MSNV_OK) {
            fprintf(stderr, "qaCompute: %s\n", msnv_last_error(ctx));
            msnv_destroy(ctx);
            return 1;
        }
        if (getenv("MSNV_CLEAN_EXIT")) msnv_destroy(ctx);      // otherwise left to process exit (see snpcall_main.cc)
    }

    bam.save_tidx(argv[optind + 1]);     // best effort
    bam.write_text(outputFile, detailed, silent, maxCoverage, cov_sum.data(), hist.data());
    fclose(outputFile);
    if (detailed) fclose(detailed);
    fflush(stdout); fflush(stderr);
    if (!getenv("MSNV_CLEAN_EXIT")) _exit(0);
    return 0;
}
