// msnv_decode_dump -- host-only inspection tool: runs the BAM decoder of the direct pileup path
// (host/pileup_input.cc: mpileup's read filters, depth cap, overlap pairing) and writes the batches it hands to `snpCall`,
// expanded on the host into the position-aligned structure of arrays of msnv_sample_reads, as raw little-endian files,
// so that the CPU test suite can check the decoder and the layout of include/msnv.h against the oracle without a GPU
// (tests/test_decode_cpu.py), and the GPU suite can check expand_kernel against the expansion here.
//   msnv_decode_dump <ref.fa> <list of BAMs> <out dir> [bed]
// MSNV_DUMP_RAW=1 also writes each sample as the BAM-shaped records the decoder emits (raw_*.bin). MSNV_DUMP_WINDOWS=N also
// cuts the shard into N position windows the way snpCall does and writes, per window k, the batch SampleDecoder::window
// hands on for it, the reads carried over from window k-1 included: w<k>.s<sample>.<array>.bin; layout.json lists the
// windows' bounds and batch sizes under "windows".
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "../host/pileup_input.hpp"

using namespace msnv;

// Growable host-side arrays of one sample, in the layout of msnv_sample_reads.
struct SampleReads {
    std::vector<int32_t>  pos;
    std::vector<uint32_t> seg_off, q4_off;
    std::vector<int32_t>  mate;
    std::vector<int32_t>  seg_pos;
    std::vector<uint16_t> seg_len;
    std::vector<uint8_t>  seq2, qual;
    uint32_t max_span = 0;
};

// The position-aligned layout of a BAM-shaped batch, as expand_kernel (gpu/kernels.cuh) builds it on the device, written
// separately and one base at a time: the tests compare the two. Every M/=/X operation of non-zero length becomes a segment;
// byte i of its quads belongs to shard coordinate (seg_pos & ~3) + i; a base is its 2-bit code (A=0 C=1 G=2 T=3), or bit 7
// of its quality for anything else; qualities are capped at 127; padding stays 0. The decoder has already checked that no
// CIGAR is longer than its sequence.
static SampleReads expand_on_host(const RawReads& r)
{
    SampleReads x;
    x.pos = r.pos; x.seg_off = r.seg_off; x.q4_off = r.q4_off; x.mate = r.mate; x.max_span = r.max_span;
    x.seg_pos.assign(r.seg_off.back(), 0);
    x.seg_len.assign(r.seg_off.back(), 0);
    x.seq2.assign(r.q4_off.back(), 0);
    x.qual.assign(4 * (size_t)r.q4_off.back(), 0);
    const uint8_t* raw = reinterpret_cast<const uint8_t*>(r.raw.data());
    for (size_t i = 0; i < r.pos.size(); ++i) {
        const uint8_t* cigar = raw + 4 * (size_t)r.raw_off[i];
        const uint8_t* seq4 = cigar + 4 * (size_t)r.n_cigar[i];
        const uint8_t* ql = seq4 + (r.l_seq[i] + 1) / 2;
        uint32_t rx = (uint32_t)r.pos[i], qy = 0, k = r.seg_off[i];
        size_t Q = r.q4_off[i];
        for (uint32_t c = 0; c < r.n_cigar[i]; ++c) {
            uint32_t w;
            memcpy(&w, cigar + 4 * (size_t)c, 4);
            const uint32_t op = w & 0xf, len = w >> 4;
            if (op == CIG_M || op == CIG_EQ || op == CIG_X) {
                if (len) {
                    x.seg_pos[k] = (int32_t)rx; x.seg_len[k] = (uint16_t)len; ++k;
                    for (uint32_t o = 0; o < len; ++o) {
                        const uint32_t q = qy + o;
                        const uint8_t b4 = (q & 1) ? (seq4[q >> 1] & 0xf) : (seq4[q >> 1] >> 4);     // "=ACMGRSVTWYHKDBN"
                        const int code = b4 == 1 ? 0 : b4 == 2 ? 1 : b4 == 4 ? 2 : b4 == 8 ? 3 : -1;
                        const size_t at = 4 * Q + (rx & 3u) + o;
                        x.qual[at] = (uint8_t)(std::min<uint8_t>(ql[q], 127) | (code < 0 ? 0x80 : 0));
                        if (code >= 0) x.seq2[at / 4] |= (uint8_t)(code << (2 * (at % 4)));
                    }
                    Q += ((rx & 3u) + len + 3u) / 4;
                }
                rx += len; qy += len;
            } else if (op == CIG_D || op == CIG_N) rx += len;
            else if (op == CIG_I || op == CIG_S) qy += len;
        }
    }
    return x;
}

template <class T> static bool dump(const std::string& path, const std::vector<T>& v)
{
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = v.empty() || fwrite(v.data(), sizeof(T), v.size(), f) == v.size();
    return fclose(f) == 0 && ok;
}

// one batch under `p`: the aligned layout, and with `raw` the BAM-shaped records it was expanded from
static bool dump_batch(const std::string& p, const SampleReads& x, const RawReads& r, bool raw)
{
    return dump(p + "pos.bin", x.pos) && dump(p + "seg_off.bin", x.seg_off) && dump(p + "q4_off.bin", x.q4_off) && dump(p + "mate.bin", x.mate) &&
           dump(p + "seg_pos.bin", x.seg_pos) && dump(p + "seg_len.bin", x.seg_len) && dump(p + "seq2.bin", x.seq2) && dump(p + "qual.bin", x.qual) &&
           (!raw || (dump(p + "raw_pos.bin", r.pos) && dump(p + "raw_mate.bin", r.mate) && dump(p + "raw_seg_off.bin", r.seg_off) &&
                     dump(p + "raw_q4_off.bin", r.q4_off) && dump(p + "raw_off.bin", r.raw_off) && dump(p + "raw_n_cigar.bin", r.n_cigar) &&
                     dump(p + "raw_l_seq.bin", r.l_seq) && dump(p + "raw.bin", r.raw)));
}

int main(int argc, char** argv)
{
    if (argc < 4) { fprintf(stderr, "usage: msnv_decode_dump <ref.fa> <list of BAMs> <out dir> [bed]\n"); return 2; }
    const std::string ref_path = argv[1], list = argv[2], out = argv[3], bed_path = argc > 4 ? argv[4] : "-";
    std::vector<std::string> bams;
    { std::ifstream in(list); std::string l; while (std::getline(in, l)) if (!l.empty()) bams.push_back(l); }
    if (bams.empty()) { fprintf(stderr, "msnv_decode_dump: no BAM files in %s\n", list.c_str()); return 1; }
    std::string err;
    BamHeader hdr;
    { BamReader r; if (!r.open(bams[0])) { fprintf(stderr, "msnv_decode_dump: %s\n", r.error().c_str()); return 1; } hdr = r.header(); }
    Bed bed; const bool has_bed = bed_path != "-";
    if (has_bed && !bed.load(bed_path, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
    ShardLayout layout;
    if (!layout.build(hdr, has_bed ? &bed : nullptr, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
    Fasta fa;
    if (!fa.load(ref_path, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
    std::vector<int64_t> ref_len(hdr.names.size(), -1);
    for (size_t t = 0; t < hdr.names.size(); ++t) { int fi = fa.find(hdr.names[t]); if (fi >= 0) ref_len[t] = (int64_t)fa.seqs[fi].size(); }
    if (!dump(out + "/ref.bin", shard_reference(layout, hdr, fa))) { fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1; }

    FILE* js = fopen((out + "/layout.json").c_str(), "w");
    if (!js) { fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1; }
    fprintf(js, "{\"tile\": %d, \"n_positions\": %u, \"contigs\": [", MSNV_TILE, layout.n_positions);
    for (size_t i = 0; i < layout.ctgs.size(); ++i)
        fprintf(js, "%s{\"name\": \"%s\", \"offset\": %u, \"len\": %u}", i ? ", " : "", hdr.names[layout.ctgs[i].tid].c_str(), layout.ctgs[i].offset, layout.ctgs[i].len);
    const uint32_t n_tiles = layout.n_positions / MSNV_TILE;
    uint32_t n_windows = getenv("MSNV_DUMP_WINDOWS") ? (uint32_t)atoi(getenv("MSNV_DUMP_WINDOWS")) : 0, tiles_per_window = 0;
    if (n_tiles == 0) n_windows = 0;                  // (a BED that selects no contig: nothing to cut)
    if (n_windows) {
        // snpCall's rule (bin/snpcall_main.cc): equal windows of whole tiles, the last one shorter
        if (n_windows > n_tiles) n_windows = n_tiles;
        tiles_per_window = (n_tiles + n_windows - 1) / n_windows;
        n_windows = (n_tiles + tiles_per_window - 1) / tiles_per_window;
    }
    const bool raw = getenv("MSNV_DUMP_RAW") != nullptr;
    std::vector<std::string> win_json(n_windows);
    fprintf(js, "], \"samples\": [");
    for (size_t s = 0; s < bams.size(); ++s) {
        SampleDecoder d; RawReads rr;
        if (!d.open(bams[s], layout, ref_len, 1, std::string(), err) || !d.window(0, layout.n_positions, nullptr, rr, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
        const DecodeStats& st = d.stats();
        const SampleReads r = expand_on_host(rr);
        if (!dump_batch(out + "/s" + std::to_string(s) + ".", r, rr, raw)) { fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1; }
        fprintf(js, "%s{\"n_reads\": %zu, \"n_segs\": %zu, \"n_q4\": %zu, \"max_span\": %u, \"first_column\": %lld, \"records\": %llu, \"accepted\": %llu, "
                    "\"dropped_by_cap\": %llu, \"aligned_bases\": %llu, \"pairs\": %llu, \"decode_s\": %.6f, \"inflate_s\": %.6f}",
                s ? ", " : "", r.pos.size(), r.seg_pos.size(), r.seq2.size(), r.max_span, (long long)st.first_column, (unsigned long long)st.records,
                (unsigned long long)st.accepted, (unsigned long long)st.dropped_by_cap, (unsigned long long)st.aligned_bases, (unsigned long long)st.pairs,
                st.seconds, st.inflate_seconds);
        if (n_windows) {
            SampleDecoder dw; RawReads rb[2];
            if (!dw.open(bams[s], layout, ref_len, 1, std::string(), err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
            for (uint32_t k = 0; k < n_windows; ++k) {
                const uint32_t lo = k * tiles_per_window * MSNV_TILE, hi = std::min(lo + tiles_per_window * MSNV_TILE, layout.n_positions);
                RawReads& rw = rb[k & 1];
                if (!dw.window(lo, hi, k ? &rb[(k - 1) & 1] : nullptr, rw, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
                const SampleReads w = expand_on_host(rw);
                if (!dump_batch(out + "/w" + std::to_string(k) + ".s" + std::to_string(s) + ".", w, rw, raw)) {
                    fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1;
                }
                if (!s) win_json[k] = "{\"lo\": " + std::to_string(lo) + ", \"hi\": " + std::to_string(hi) + ", \"samples\": [";
                win_json[k] += std::string(s ? ", " : "") + "{\"n_reads\": " + std::to_string(w.pos.size()) + ", \"n_segs\": " + std::to_string(w.seg_pos.size()) +
                               ", \"n_q4\": " + std::to_string(w.seq2.size()) + ", \"max_span\": " + std::to_string(w.max_span) +
                               ", \"raw_n_reads\": " + std::to_string(rw.pos.size()) + ", \"raw_max_span\": " + std::to_string(rw.max_span) + "}";
            }
        }
    }
    fprintf(js, "], \"windows\": [");
    for (uint32_t k = 0; k < n_windows; ++k) fprintf(js, "%s%s]}", k ? ", " : "", win_json[k].c_str());
    fprintf(js, "]}\n");
    fclose(js);
    return 0;
}
