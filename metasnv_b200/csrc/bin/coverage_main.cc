// metaSNV_coverage -- the coverage pass of metaSNV.py:compute_opt (metaSNV.py:58-69) in one process and one CUDA context.
//
//   metaSNV_coverage <project_dir> <all_samples>
//
// For every BAM listed in all_samples (surrounding white space stripped, blank lines skipped) it writes
// <project_dir>/cov/<basename>.cov, .cov.detail and .cov.tidx, byte-identical to what
// `qaCompute -c 10 -d -i <bam> <project_dir>/cov/<basename>.cov` writes: the per-BAM logic is host/coverage.cc, which
// qaCompute runs too. compute_opt starts one qaCompute per BAM, and each of those processes pays 0.5-1 s for its CUDA
// context, which the driver creates one after another; on a project of many small BAMs that is most of the pass.
//
// Structure: W decode threads, each inflating with T threads (W x T = the host's cores, MSNV_THREADS overrides), take the
// BAMs largest first so that one big BAM does not form the tail. The main thread creates the context (MSNV_DEVICE, else
// device 0) while the first BAMs decode, and is the only thread that uses it: msnv_cov_run on each BAM as it becomes
// ready, then its files, then its blocks are freed. At most W + 1 decoded BAMs are alive at any time.
//
// A BAM that cannot be opened, is unsorted or is truncated gets one message on stderr naming it; every other BAM is still
// written, and the exit code is 1. Two lines with the same basename would write the same files and are refused before any
// work starts. With MSNV_PERF_JSON set, one JSON record is appended to that file.
#include <sys/resource.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../host/coverage.hpp"

using namespace msnv;

namespace {

constexpr int kMaxCov = 10;           // metaSNV.py:63-65 always runs `qaCompute -c 10 -d -i`
constexpr int kMinQual = 1;           // qaCompute's default -q

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

double process_cpu_s()
{
    rusage u;
    getrusage(RUSAGE_SELF, &u);
    return u.ru_utime.tv_sec + u.ru_stime.tv_sec + 1e-6 * (u.ru_utime.tv_usec + u.ru_stime.tv_usec);
}

std::string strip(const std::string& s)
{
    size_t b = 0, e = s.size();
    while (b < e && isspace((unsigned char)s[b])) ++b;
    while (e > b && isspace((unsigned char)s[e - 1])) --e;
    return s.substr(b, e - b);
}

std::string base_name(const std::string& p)           // os.path.basename
{
    const size_t s = p.rfind('/');
    return s == std::string::npos ? p : p.substr(s + 1);
}

// CovBam's messages are qaCompute's; on one line, naming the BAM when the message does not already
std::string one_line(const std::string& bam, std::string msg)
{
    std::replace(msg.begin(), msg.end(), '\n', ' ');
    return msg.find(bam) == std::string::npos ? bam + ": " + msg : msg;
}

bool make_dir(const std::string& d)
{
    return mkdir(d.c_str(), 0777) == 0 || errno == EEXIST;
}

struct Job { std::string bam, out; uint64_t bytes; };

struct Decoded {
    size_t job;
    CovBam bam;
    bool ok = false;
    double seconds = 0;
};

}  // namespace

int main(int argc, char** argv)
{
    const double t_start = now_s();
    if (argc != 3) { fprintf(stderr, "usage: metaSNV_coverage <project_dir> <all_samples>\n"); return 1; }
    const std::string project = argv[1];

    std::vector<Job> jobs;
    {
        FILE* f = fopen(argv[2], "r");
        if (!f) { fprintf(stderr, "metaSNV_coverage: cannot read %s\n", argv[2]); return 1; }
        std::string line;
        int c;
        std::map<std::string, std::string> by_base;
        for (;;) {
            c = fgetc(f);
            if (c != EOF && c != '\n') { line.push_back((char)c); continue; }
            const std::string bam = strip(line);
            line.clear();
            if (!bam.empty()) {
                const std::string b = base_name(bam);
                auto it = by_base.emplace(b, bam);
                if (!it.second) {
                    fprintf(stderr, "metaSNV_coverage: %s and %s would both write cov/%s.cov\n", it.first->second.c_str(), bam.c_str(), b.c_str());
                    fclose(f);
                    return 1;
                }
                struct stat st;
                jobs.push_back(Job{bam, project + "/cov/" + b + ".cov", stat(bam.c_str(), &st) == 0 ? (uint64_t)st.st_size : 0});
            }
            if (c == EOF) break;
        }
        const bool read_error = ferror(f);
        fclose(f);
        if (read_error) { fprintf(stderr, "metaSNV_coverage: cannot read %s\n", argv[2]); return 1; }
        if (jobs.empty()) { fprintf(stderr, "metaSNV_coverage: %s lists no BAM\n", argv[2]); return 1; }
    }

    const int nd = msnv_device_count();
    if (nd <= 0) { fprintf(stderr, "metaSNV_coverage: no usable CUDA device (%s); this build has no CPU path\n", msnv_last_error(nullptr)); return 1; }
    if (!make_dir(project) || !make_dir(project + "/cov")) { fprintf(stderr, "metaSNV_coverage: cannot create %s/cov\n", project.c_str()); return 1; }

    // largest first; ties keep the order of all_samples
    std::vector<size_t> order(jobs.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return jobs[a].bytes > jobs[b].bytes; });
    uint64_t bam_bytes = 0;
    for (const Job& j : jobs) bam_bytes += j.bytes;

    // BGZF inflate bounds the pass: W BAMs at a time with T inflate threads each, W x T = the host's cores
    int cores = (int)std::max(1u, std::thread::hardware_concurrency());
    if (const char* e = getenv("MSNV_THREADS")) cores = std::max(1, atoi(e));
    const int W = (int)std::min<size_t>((size_t)cores, jobs.size()), T = std::max(1, cores / W);
    const size_t max_alive = (size_t)W + 1;

    std::mutex mu;
    std::condition_variable cv;
    size_t next = 0, alive = 0, peak_alive = 0;
    bool stop = false;
    std::deque<std::unique_ptr<Decoded>> ready;
    double t_dec_end = 0;
    auto worker = [&]() {
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return stop || next >= jobs.size() || alive < max_alive; });
            if (stop || next >= jobs.size()) return;
            std::unique_ptr<Decoded> d(new Decoded);
            d->job = order[next++];
            peak_alive = std::max(peak_alive, ++alive);
            lk.unlock();
            const double t0 = now_s();
            d->ok = d->bam.open(jobs[d->job].bam, T) && d->bam.decode(kMinQual, "metaSNV_coverage");
            const double t1 = now_s();
            d->seconds = t1 - t0;
            lk.lock();
            t_dec_end = std::max(t_dec_end, t1);
            ready.push_back(std::move(d));
            cv.notify_all();
        }
    };
    const double t_dec0 = now_s();
    std::vector<std::thread> workers;
    for (int w = 0; w < W; ++w) workers.emplace_back(worker);
    auto join_workers = [&]() { for (auto& t : workers) if (t.joinable()) t.join(); };

    // the context comes up while the first BAMs decode; this thread is the only one that uses it
    int dev = 0;
    if (const char* e = getenv("MSNV_DEVICE")) dev = atoi(e);
    msnv_ctx* ctx = nullptr;
    if (msnv_create(dev % nd, &ctx) != MSNV_OK) {
        fprintf(stderr, "metaSNV_coverage: no usable CUDA device (%s); this build has no CPU path\n", msnv_last_error(ctx));
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv.notify_all();
        join_workers();
        return 1;
    }
    const double t_ctx = now_s() - t_start;

    int failed = 0;
    float ms_scatter = 0, ms_scan = 0;
    uint64_t n_blocks = 0;
    // decode_cpu_s / inflate_cpu_s in the perf record: the decode threads' busy time per BAM and, of it, BGZF inflate, summed
    // over the BAMs (as snpCall reports them); process_cpu_s is the process's CPU time
    double t_wait = 0, t_gpu = 0, t_write = 0, t_decode = 0, t_inflate = 0;
    std::vector<uint64_t> cov_sum, hist;
    for (size_t got = 0; got < jobs.size(); ++got) {
        std::unique_ptr<Decoded> d;
        {
            const double a = now_s();
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return !ready.empty(); });
            d = std::move(ready.front());
            ready.pop_front();
            t_wait += now_s() - a;
        }
        const Job& j = jobs[d->job];
        if (!d->ok) {
            fprintf(stderr, "metaSNV_coverage: %s\n", one_line(j.bam, d->bam.error()).c_str());
            ++failed;
        } else {
            double a = now_s();
            if (d->bam.run(ctx, kMaxCov, cov_sum, hist) != MSNV_OK) {
                // a CUDA error (the context is then unusable) or a limit of msnv_cov_run: report it and stop
                fprintf(stderr, "metaSNV_coverage: %s: %s\n", j.bam.c_str(), msnv_last_error(ctx));
                { std::lock_guard<std::mutex> lk(mu); stop = true; }
                cv.notify_all();
                join_workers();
                return 1;
            }
            if (d->bam.n_contigs_seen()) {
                msnv_timings tm;
                msnv_get_timings(ctx, &tm);
                ms_scatter += tm.ms_cov_scatter; ms_scan += tm.ms_cov_scan;
            }
            n_blocks += d->bam.n_blocks();
            d->bam.release_blocks();
            const double b = now_s();
            t_gpu += b - a;
            std::string err;
            if (!d->bam.write_files(j.out, kMaxCov, cov_sum.data(), hist.data(), err)) {
                fprintf(stderr, "metaSNV_coverage: %s\n", err.c_str());
                ++failed;
            }
            t_write += now_s() - b;
        }
        t_decode += d->seconds;
        t_inflate += d->bam.inflate_seconds();
        std::lock_guard<std::mutex> lk(mu);
        --alive;
        cv.notify_all();
    }
    join_workers();
    const double t_end = now_s();

    if (const char* pj = getenv("MSNV_PERF_JSON")) {
        if (FILE* f = fopen(pj, "a")) {
            fprintf(f,
                    "{\"tool\": \"metaSNV_coverage\", \"device\": %d, \"bams\": %zu, \"bams_failed\": %d, \"bam_bytes\": %llu, "
                    "\"decode_workers\": %d, \"inflate_threads\": %d, \"peak_decoded_bams\": %zu, \"cov_blocks\": %llu, "
                    "\"decode_wall_s\": %.6f, \"decode_cpu_s\": %.6f, \"inflate_cpu_s\": %.6f, \"process_cpu_s\": %.6f, "
                    "\"ctx_ready_s\": %.6f, \"waiting_for_decode_s\": %.6f, \"gpu_s\": %.6f, \"write_s\": %.6f, "
                    "\"ms_cov_scatter\": %.4f, \"ms_cov_scan\": %.4f, \"total_s\": %.6f}\n",
                    dev % nd, jobs.size(), failed, (unsigned long long)bam_bytes, W, T, peak_alive, (unsigned long long)n_blocks,
                    t_dec_end - t_dec0, t_decode, t_inflate, process_cpu_s(), t_ctx, t_wait, t_gpu, t_write, ms_scatter, ms_scan, t_end - t_start);
            fclose(f);
        }
    }
    fflush(stdout); fflush(stderr);
    if (getenv("MSNV_CLEAN_EXIT")) { msnv_destroy(ctx); return failed ? 1 : 0; }
    _exit(failed ? 1 : 0);     // the driver reclaims the device at exit; tearing the context down only adds time
}
