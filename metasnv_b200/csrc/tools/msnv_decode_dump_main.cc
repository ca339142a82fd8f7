// msnv_decode_dump -- host-only inspection tool: runs the BAM decoder of the direct pileup path
// (host/pileup_input.cc: mpileup's read filters, depth cap, overlap pairing, position-aligned segments)
// and writes the structure-of-arrays batches that `snpCall` would hand to msnv_shard_add_sample() as raw
// little-endian files, so that the CPU test suite can check the decoder and the layout of include/msnv.h
// against the oracle without a GPU (tests/test_decode_cpu.py).
//   msnv_decode_dump <ref.fa> <list of BAMs> <out dir> [bed]
// MSNV_DUMP_RAW=1 adds each sample as BAM-shaped records (raw_*.bin). MSNV_DUMP_WINDOWS=N also cuts the shard into N
// position windows the way snpCall does and writes, per window k, the batch SampleDecoder::window (and with MSNV_DUMP_RAW,
// window_raw) hands on for it, the reads carried over from window k-1 included: w<k>.s<sample>.<array>.bin; layout.json
// lists the windows' bounds and batch sizes under "windows".
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <string>
#include <vector>

#include "../host/pileup_input.hpp"

using namespace msnv;

template <class T> static bool dump(const std::string& path, const std::vector<T>& v)
{
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = v.empty() || fwrite(v.data(), sizeof(T), v.size(), f) == v.size();
    return fclose(f) == 0 && ok;
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
        SampleReads r; DecodeStats st;
        if (!decode_sample_for_pileup(bams[s], layout, ref_len, 1, r, st, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
        const std::string p = out + "/s" + std::to_string(s) + ".";
        if (!dump(p + "pos.bin", r.pos) || !dump(p + "seg_off.bin", r.seg_off) || !dump(p + "q4_off.bin", r.q4_off) || !dump(p + "mate.bin", r.mate) ||
            !dump(p + "seg_pos.bin", r.seg_pos) || !dump(p + "seg_len.bin", r.seg_len) || !dump(p + "seq2.bin", r.seq2) || !dump(p + "qual.bin", r.qual)) {
            fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1;
        }
        if (raw) {
            // the same sample as BAM-shaped records (what snpCall uploads when the device expands them)
            SampleDecoder d2; RawReads rr;
            if (!d2.open(bams[s], layout, ref_len, 1, std::string(), err) || !d2.window_raw(0, layout.n_positions, nullptr, rr, err)) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
            if (!dump(p + "raw_pos.bin", rr.pos) || !dump(p + "raw_mate.bin", rr.mate) || !dump(p + "raw_seg_off.bin", rr.seg_off) || !dump(p + "raw_q4_off.bin", rr.q4_off) ||
                !dump(p + "raw_off.bin", rr.raw_off) || !dump(p + "raw_n_cigar.bin", rr.n_cigar) || !dump(p + "raw_l_seq.bin", rr.l_seq) || !dump(p + "raw.bin", rr.raw)) {
                fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1;
            }
        }
        fprintf(js, "%s{\"n_reads\": %zu, \"n_segs\": %zu, \"n_q4\": %zu, \"max_span\": %u, \"first_column\": %lld, \"records\": %llu, \"accepted\": %llu, "
                    "\"dropped_by_cap\": %llu, \"aligned_bases\": %llu, \"pairs\": %llu, \"decode_s\": %.6f, \"inflate_s\": %.6f}",
                s ? ", " : "", r.pos.size(), r.seg_pos.size(), r.seq2.size(), r.max_span, (long long)st.first_column, (unsigned long long)st.records,
                (unsigned long long)st.accepted, (unsigned long long)st.dropped_by_cap, (unsigned long long)st.aligned_bases, (unsigned long long)st.pairs,
                st.seconds, st.inflate_seconds);
        if (n_windows) {
            SampleDecoder d, dr; SampleReads wb[2]; RawReads rb[2];
            if (!d.open(bams[s], layout, ref_len, 1, std::string(), err) || (raw && !dr.open(bams[s], layout, ref_len, 1, std::string(), err))) {
                fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1;
            }
            for (uint32_t k = 0; k < n_windows; ++k) {
                const uint32_t lo = k * tiles_per_window * MSNV_TILE, hi = std::min(lo + tiles_per_window * MSNV_TILE, layout.n_positions);
                SampleReads& w = wb[k & 1]; RawReads& rw = rb[k & 1];
                if (!d.window(lo, hi, k ? &wb[(k - 1) & 1] : nullptr, w, err) ||
                    (raw && !dr.window_raw(lo, hi, k ? &rb[(k - 1) & 1] : nullptr, rw, err))) { fprintf(stderr, "msnv_decode_dump: %s\n", err.c_str()); return 1; }
                const std::string q = out + "/w" + std::to_string(k) + ".s" + std::to_string(s) + ".";
                bool ok = dump(q + "pos.bin", w.pos) && dump(q + "seg_off.bin", w.seg_off) && dump(q + "q4_off.bin", w.q4_off) && dump(q + "mate.bin", w.mate) &&
                          dump(q + "seg_pos.bin", w.seg_pos) && dump(q + "seg_len.bin", w.seg_len) && dump(q + "seq2.bin", w.seq2) && dump(q + "qual.bin", w.qual);
                if (raw)
                    ok = ok && dump(q + "raw_pos.bin", rw.pos) && dump(q + "raw_mate.bin", rw.mate) && dump(q + "raw_seg_off.bin", rw.seg_off) &&
                         dump(q + "raw_q4_off.bin", rw.q4_off) && dump(q + "raw_off.bin", rw.raw_off) && dump(q + "raw_n_cigar.bin", rw.n_cigar) &&
                         dump(q + "raw_l_seq.bin", rw.l_seq) && dump(q + "raw.bin", rw.raw);
                if (!ok) { fprintf(stderr, "msnv_decode_dump: cannot write to %s\n", out.c_str()); return 1; }
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
