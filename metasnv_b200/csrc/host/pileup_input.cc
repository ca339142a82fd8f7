// pileup_input.cc -- see pileup_input.hpp.
#include "pileup_input.hpp"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <queue>

namespace msnv {

// ------------------------------------------------------------------ FASTA / BED
bool Fasta::load(const std::string& path, std::string& err)
{
    FILE* f = fopen(path.c_str(), "r");
    if (!f) { err = "cannot open reference " + path; return false; }
    char* line = nullptr; size_t cap = 0; ssize_t n;
    int cur = -1;
    while ((n = getline(&line, &cap, f)) > 0) {
        while (n > 0 && (line[n - 1] == '\n' || line[n - 1] == '\r')) line[--n] = 0;
        if (line[0] == '>') {
            char* e = line + 1;
            while (*e && !isspace((unsigned char)*e)) ++e;
            std::string nm(line + 1, e);
            cur = (int)names.size();
            names.push_back(nm); seqs.emplace_back();
            index.emplace(nm, cur);                 // keeps the first record of a duplicated name
        } else if (cur >= 0) {
            seqs[cur].append(line, (size_t)n);
        }
    }
    free(line);
    fclose(f);
    return true;
}

bool Bed::load(const std::string& path, std::string& err)
{
    std::ifstream in(path);
    if (!in) { err = "cannot open " + path; return false; }
    std::string line;
    while (std::getline(in, line)) {
        if (line.empty() || line[0] == '#') continue;
        char name[4096]; long long a = 0, b = 0;
        int k = sscanf(line.c_str(), "%4095s %lld %lld", name, &a, &b);
        if (k < 2) continue;
        Iv iv;
        if (k == 2) { iv.beg = a - 1; iv.end = a; } else { iv.beg = a; iv.end = b; }
        by_name[name].push_back(iv);
    }
    return true;
}

// ------------------------------------------------------------------ shard layout
bool ShardLayout::build(const BamHeader& hdr, const Bed* b, std::string& err)
{
    ctgs.clear(); bed.clear();
    slot_of_tid.assign(hdr.names.size(), -1);
    has_bed = b != nullptr;
    uint64_t off = 0;
    for (size_t t = 0; t < hdr.names.size(); ++t) {
        std::vector<Bed::Iv> ivs;
        if (b) {
            auto it = b->by_name.find(hdr.names[t]);
            if (it == b->by_name.end()) continue;
            ivs = it->second;
            std::sort(ivs.begin(), ivs.end(), [](const Bed::Iv& x, const Bed::Iv& y) { return x.beg < y.beg; });
            std::vector<Bed::Iv> merged;
            for (const Bed::Iv& iv : ivs) {
                if (iv.end <= iv.beg) continue;
                if (!merged.empty() && iv.beg <= merged.back().end) merged.back().end = std::max(merged.back().end, iv.end);
                else merged.push_back(iv);
            }
            ivs.swap(merged);
            if (ivs.empty()) continue;
        } else {
            ivs.push_back(Bed::Iv{0, (int64_t)hdr.lens[t]});
        }
        Ctg c; c.tid = (int)t; c.len = hdr.lens[t]; c.offset = (uint32_t)off;
        slot_of_tid[t] = (int)ctgs.size();
        ctgs.push_back(c); bed.push_back(ivs);
        off += ((uint64_t)hdr.lens[t] + MSNV_TILE - 1) / MSNV_TILE * MSNV_TILE;
        if (hdr.lens[t] == 0) off += MSNV_TILE;
        if (off > 0x7ff00000ull) { err = "shard larger than 2^31 positions; use more splits"; return false; }
    }
    n_positions = (uint32_t)off;
    return true;
}

bool ShardLayout::overlaps(int slot, int64_t beg, int64_t end) const
{
    for (const Bed::Iv& iv : bed[slot]) if (iv.beg < end && beg < iv.end) return true;
    return false;
}

int64_t ShardLayout::first_inside(int slot, int64_t beg, int64_t end) const
{
    for (const Bed::Iv& iv : bed[slot]) {                 // sorted, disjoint
        if (iv.end <= beg) continue;
        int64_t p = std::max(beg, iv.beg);
        return p < end ? p : -1;
    }
    return -1;
}

std::vector<uint8_t> shard_reference(const ShardLayout& layout, const BamHeader& hdr, const Fasta& fa)
{
    std::vector<uint8_t> ref(layout.n_positions, 0);
    for (size_t k = 0; k < layout.ctgs.size(); ++k) {
        const ShardLayout::Ctg& c = layout.ctgs[k];
        int fi = fa.find(hdr.names[c.tid]);
        const std::string* seq = fi >= 0 ? &fa.seqs[fi] : nullptr;
        for (const Bed::Iv& iv : layout.bed[k]) {
            int64_t e = std::min<int64_t>(iv.end, c.len);
            for (int64_t p = std::max<int64_t>(iv.beg, 0); p < e; ++p)
                ref[c.offset + p] = (seq && p < (int64_t)seq->size()) ? (uint8_t)(*seq)[p] : (uint8_t)'N';
        }
    }
    return ref;
}

// ------------------------------------------------------------------ SoA helpers
msnv_raw_reads RawReads::view() const
{
    msnv_raw_reads v;
    memset(&v, 0, sizeof v);
    v.n_reads = (uint32_t)pos.size();
    v.max_span = max_span;
    v.pos = pos.data(); v.mate = mate.data(); v.seg_off = seg_off.data(); v.q4_off = q4_off.data(); v.raw_off = raw_off.data();
    v.n_cigar = n_cigar.data(); v.l_seq = l_seq.data(); v.raw = reinterpret_cast<const uint8_t*>(raw.data());
    return v;
}

size_t RawReads::bytes() const
{
    return pos.size() * 8 + seg_off.size() * 4 + q4_off.size() * 4 + raw_off.size() * 4 + n_cigar.size() * 2 + l_seq.size() * 2 + raw.size() * 4;
}

namespace {

inline uint64_t hash_qname(const char* s)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (; *s; ++s) { h ^= (unsigned char)*s; h *= 0x100000001b3ull; }
    h ^= h >> 29; h *= 0xbf58476d1ce4e5b9ull; h ^= h >> 32;
    return h;
}

struct Buffered { int32_t end; uint64_t qh; };
struct ByEnd { bool operator()(const Buffered& a, const Buffered& b) const { return a.end > b.end; } };
struct Stored { uint64_t ordinal; int32_t end; };

}  // namespace

// ------------------------------------------------------------------ resumable decoder
struct SampleDecoderState {
    std::string path;
    const ShardLayout* layout = nullptr;
    const std::vector<int64_t>* ref_len = nullptr;
    BamReader rd;
    DecodeStats st;
    bool eof = false;
    // one record read ahead (it belongs to a later window): kept as a private copy of its bytes
    bool have_pending = false;
    BamRecord pending; std::vector<uint8_t> pending_bytes;
    // state of htslib's pileup iterator that the depth cap and the overlap hash depend on
    int cur_tid = -1; int32_t last_pos = -1;
    std::priority_queue<Buffered, std::vector<Buffered>, ByEnd> buffered;    // reads the iterator still holds
    std::unordered_map<uint64_t, Stored> olap;                               // qname -> earlier mate waiting for its partner (index = ordinal)
    bool warned_overhang = false;
    uint64_t n_emitted = 0;                      // ordinal of the next accepted read over the whole file
    uint64_t base = 0;                           // ordinal of the first read of the window batch being built
    // index-driven reading: runs of consecutive tids of the shard, visited in order
    TidIndex index;
    std::vector<std::pair<int, int>> runs;       // [first tid, last tid]
    size_t run_i = 0; bool in_run = false;
    std::chrono::steady_clock::time_point t_open;
};

SampleDecoder::SampleDecoder() : st_(new SampleDecoderState()) {}
SampleDecoder::~SampleDecoder() { delete st_; }
const DecodeStats& SampleDecoder::stats() const { return st_->st; }
bool SampleDecoder::used_index() const { return st_->index.valid() && !st_->runs.empty(); }

bool SampleDecoder::open(const std::string& bam_path, const ShardLayout& layout, const std::vector<int64_t>& ref_len_of_tid, int inflate_threads,
                         const std::string& index_hint, std::string& err)
{
    SampleDecoderState& S = *st_;
    S.path = bam_path; S.layout = &layout; S.ref_len = &ref_len_of_tid;
    if (!S.rd.open(bam_path, inflate_threads)) { err = S.rd.error(); return false; }
    // mpileup takes the contigs from the first file's header and trusts the others to agree; a file whose header
    // differs would be piled up against the wrong coordinates, so it is refused here instead
    const BamHeader& h = S.rd.header();
    if (h.lens.size() != layout.slot_of_tid.size()) { err = bam_path + ": its header lists " + std::to_string(h.lens.size()) + " contigs, the first file's " + std::to_string(layout.slot_of_tid.size()); return false; }
    for (const ShardLayout::Ctg& c : layout.ctgs)
        if (h.lens[c.tid] != c.len) { err = bam_path + ": contig " + h.names[c.tid] + " has another length than in the first file's header"; return false; }
    // a split (-l) names a few contigs: with an index, read only the runs of the file that hold them
    if (layout.has_bed && !getenv("MSNV_NO_INDEX") && S.index.find_for(bam_path, index_hint, S.rd.compressed_size(), h.lens.size())) {
        for (const ShardLayout::Ctg& c : layout.ctgs) {
            if (!S.runs.empty() && S.runs.back().second + 1 == c.tid) S.runs.back().second = c.tid;
            else S.runs.emplace_back(c.tid, c.tid);
        }
    }
    return true;
}

// next record of the shard's part of the file: 1 = delivered, 0 = no more, -1 = error
static int next_record(SampleDecoderState& S, BamRecord& r)
{
    if (S.runs.empty()) return S.rd.next(r);
    for (;;) {
        if (!S.in_run) {
            // start of the next run: the first of its tids that has records
            uint64_t off = TidIndex::NONE;
            while (S.run_i < S.runs.size() && off == TidIndex::NONE) {
                for (int t = S.runs[S.run_i].first; t <= S.runs[S.run_i].second && off == TidIndex::NONE; ++t) off = S.index.first[(size_t)t];
                if (off == TidIndex::NONE) ++S.run_i;
            }
            if (S.run_i >= S.runs.size()) return 0;
            if (!S.rd.seek(off)) return -1;
            S.in_run = true;
        }
        const int rc = S.rd.next(r);
        if (rc <= 0) return rc;
        if (r.core.tid >= 0 && r.core.tid <= S.runs[S.run_i].second) return 1;     // (an index entry may point a little before the tid: earlier tids are filtered by the caller)
        S.in_run = false; ++S.run_i;                                                // past the run: on to the next one
    }
}

bool SampleDecoder::window(uint32_t pos_lo, uint32_t pos_hi, const RawReads* prev, RawReads& o, std::string& err)
{
    SampleDecoderState& S = *st_;
    const ShardLayout& layout = *S.layout;
    const std::vector<int64_t>& ref_len_of_tid = *S.ref_len;
    DecodeStats& st = S.st;
    const std::string& bam_path = S.path;
    auto t0 = std::chrono::steady_clock::now();
    const int MAXCNT = 8000;                         // samtools mpileup -d default (>= 1.9), per file

    // ---- the previous window's reads that reach this one: a contiguous tail of its batch
    o = RawReads();
    if (prev && !prev->pos.empty()) {
        const RawReads& p = *prev;
        const size_t n = p.pos.size();
        size_t first = n;
        for (size_t i = n; i-- > 0;) {
            if ((int64_t)p.pos[i] + (int64_t)p.max_span <= (int64_t)pos_lo) break;          // no earlier read can reach the window either
            if ((int64_t)p.end[i] > (int64_t)pos_lo) first = i;
        }
        if (first < n) {
            const uint32_t s0 = p.seg_off[first], q0 = p.q4_off[first], r0 = p.raw_off[first];
            o.pos.assign(p.pos.begin() + first, p.pos.end());
            o.end.assign(p.end.begin() + first, p.end.end());
            o.n_cigar.assign(p.n_cigar.begin() + first, p.n_cigar.end());
            o.l_seq.assign(p.l_seq.begin() + first, p.l_seq.end());
            o.seg_off.resize(n - first + 1); o.q4_off.resize(n - first + 1); o.raw_off.resize(n - first + 1); o.mate.resize(n - first);
            for (size_t i = first; i <= n; ++i) { o.seg_off[i - first] = p.seg_off[i] - s0; o.q4_off[i - first] = p.q4_off[i] - q0; o.raw_off[i - first] = p.raw_off[i] - r0; }
            for (size_t i = first; i < n; ++i) { const int64_t m = (int64_t)p.mate[i] - (int64_t)first; o.mate[i - first] = m >= 0 ? (int32_t)m : -1; }
            o.raw.assign(p.raw.begin() + r0, p.raw.end());
            o.max_span = p.max_span;
        }
        S.base = S.n_emitted - (n - first);
    } else {
        S.base = S.n_emitted;
    }

    BamRecord r;
    for (;;) {
        if (S.have_pending) { r = S.pending; S.have_pending = false; }
        else {
            if (S.eof) break;
            const int rc = next_record(S, r);
            if (rc < 0) { err = bam_path + ": " + S.rd.error(); return false; }
            if (rc == 0) { S.eof = true; break; }
            ++st.records;
        }
        const BamCore& c = r.core;
        // ---- mplp_func (SURVEY.md Annex A.1)
        if (c.tid < 0 || (c.flag & FLAG_UNMAP)) continue;
        if (c.flag & (FLAG_UNMAP | FLAG_SECONDARY | FLAG_QCFAIL | FLAG_DUP)) continue;
        if ((size_t)c.tid >= layout.slot_of_tid.size()) continue;
        int32_t rlen = 0; uint32_t n_seg = 0;
        for (int i = 0; i < c.n_cigar; ++i) {
            const uint32_t w = r.cigar_at(i), op = w & 0xf;
            if (op == CIG_M || op == CIG_EQ || op == CIG_X) { rlen += (int32_t)(w >> 4); n_seg += (w >> 4) != 0; }
            else if (op == CIG_D || op == CIG_N) rlen += (int32_t)(w >> 4);
        }
        const int slot = layout.slot_of_tid[c.tid];
        const int32_t end = c.pos + rlen;
        if (layout.has_bed) {
            if (slot < 0 || !layout.overlaps(slot, c.pos, c.pos + (rlen ? rlen : 1))) continue;
        }
        if (ref_len_of_tid[c.tid] >= 0 && ref_len_of_tid[c.tid] <= c.pos) continue;
        if ((c.flag & FLAG_PAIRED) && !(c.flag & FLAG_PROPER_PAIR)) continue;
        if (slot < 0) continue;
        // ---- outside the contract of this implementation (documented in DESIGN.md)
        if (rlen == 0) continue;                                   // no reference base: builds no column
        if (c.pos < 0 || (uint32_t)end > layout.ctgs[slot].len) {
            if (!S.warned_overhang) { fprintf(stderr, "[msnv] %s: read %s extends beyond its contig; such reads are skipped\n", bam_path.c_str(), r.qname); S.warned_overhang = true; }
            continue;
        }
        if (c.l_seq > MSNV_MAX_READ_BASES || n_seg > MSNV_MAX_READ_SEGMENTS) {
            err = bam_path + ": read " + r.qname + " exceeds the supported length (" + std::to_string(MSNV_MAX_READ_BASES) +
                  " bases / " + std::to_string(MSNV_MAX_READ_SEGMENTS) + " aligned segments)";
            return false;
        }
        if (rlen > MSNV_MAX_READ_SPAN) {
            err = bam_path + ": read " + r.qname + " spans " + std::to_string(rlen) + " reference positions, more than the supported " +
                  std::to_string(MSNV_MAX_READ_SPAN) + " (deletions and skips included)";
            return false;
        }
        const ShardLayout::Ctg& ctg = layout.ctgs[slot];
        // ---- a read of a later window: keep it for the next call (its bytes live in the reader's buffer only until the next record)
        if ((uint64_t)ctg.offset + (uint32_t)c.pos >= pos_hi) {
            const size_t nb = 32 + (size_t)c.l_read_name + 4 * (size_t)c.n_cigar + (size_t)((c.l_seq + 1) / 2) + (size_t)c.l_seq;
            const uint8_t* src = (const uint8_t*)r.qname - 32;
            if (!S.pending_bytes.empty() && src == S.pending_bytes.data()) { S.pending = r; S.have_pending = true; break; }   // it was the pending one already
            std::vector<uint8_t> copy(nb);
            memcpy(copy.data() + 32, src + 32, nb - 32);
            S.pending_bytes.swap(copy);
            S.pending = r;
            const uint8_t* p = S.pending_bytes.data();
            S.pending.qname = (const char*)(p + 32);
            S.pending.cigar = p + 32 + c.l_read_name;
            S.pending.seq = S.pending.cigar + 4 * (size_t)c.n_cigar;
            S.pending.qual = S.pending.seq + (c.l_seq + 1) / 2;
            S.have_pending = true;
            break;
        }

        // ---- bam_plp_push: the input must be coordinate sorted (htslib stops with "the input is not sorted"); the
        // device-side index searches the positions and relies on it
        if (c.tid < S.cur_tid || (c.tid == S.cur_tid && c.pos < S.last_pos)) {
            err = bam_path + " is not coordinate sorted (read " + r.qname + ")";
            return false;
        }
        // ---- expiry of buffered reads, depth cap (Annex A.3)
        if (c.tid != S.cur_tid) {
            while (!S.buffered.empty()) S.buffered.pop();
            S.olap.clear();
            S.cur_tid = c.tid; S.last_pos = -1;
        } else {
            // columns < last_pos have been produced; they released every read ending at or before last_pos-1
            while (!S.buffered.empty() && S.buffered.top().end <= S.last_pos - 1) {
                S.olap.erase(S.buffered.top().qh);
                S.buffered.pop();
            }
        }
        const uint64_t qh = hash_qname(r.qname);
        if (c.pos == S.last_pos && (int)S.buffered.size() + 1 > MAXCNT) {
            S.olap.erase(qh);
            ++st.dropped_by_cap;
            continue;
        }
        S.last_pos = c.pos;
        S.buffered.push(Buffered{end, qh});
        if (S.buffered.size() > st.max_buffered) st.max_buffered = (uint32_t)S.buffered.size();

        const uint64_t ordinal = S.n_emitted++;
        const uint32_t idx = (uint32_t)(ordinal - S.base);          // index in this window's batch
        // ---- overlap_push (Annex A.2)
        int32_t mate_idx = -1;
        if (!(c.flag & FLAG_MUNMAP) && (c.flag & FLAG_PROPER_PAIR) &&
            !((c.mtid >= 0 && c.tid != c.mtid) ||
              ((c.tlen < 0 ? -(int64_t)c.tlen : (int64_t)c.tlen) >= 2 * (int64_t)c.l_seq && c.mpos >= end))) {
            auto it = S.olap.find(qh);
            if (it == S.olap.end()) {
                if (c.mpos >= c.pos) S.olap.emplace(qh, Stored{ordinal, end});
            } else {
                // (a partner that is not part of this batch ended before the window: no common position inside it)
                if (it->second.end > c.pos && it->second.ordinal >= S.base) mate_idx = (int32_t)(it->second.ordinal - S.base);
                S.olap.erase(it);
            }
        }
        // ---- offsets of the aligned layout (the device fills it) and the record's own bytes
        size_t quads = 0, q_len = 0;
        {
            uint32_t rx = ctg.offset + (uint32_t)c.pos;
            for (int i = 0; i < c.n_cigar; ++i) {
                const uint32_t w = r.cigar_at(i), op = w & 0xf, len = w >> 4;
                if (op == CIG_M || op == CIG_EQ || op == CIG_X) { if (len) { quads += ((rx & 3u) + len + 3u) >> 2; st.aligned_bases += len; } rx += len; q_len += len; }
                else if (op == CIG_D || op == CIG_N) rx += len;
                else if (op == CIG_I || op == CIG_S) q_len += len;
            }
        }
        if (q_len > (size_t)c.l_seq) { err = bam_path + ": read " + r.qname + ": CIGAR longer than the sequence"; return false; }
        if (o.q4_off.back() + quads > 0xffffffffull) { err = bam_path + ": more than 2^34 bases in one shard of one sample"; return false; }
        o.pos.push_back((int32_t)(ctg.offset + (uint32_t)c.pos));
        o.end.push_back((int32_t)(ctg.offset + (uint32_t)end));
        o.mate.push_back(mate_idx);
        if (mate_idx >= 0) { o.mate[(size_t)mate_idx] = (int32_t)idx; ++st.pairs; }
        o.seg_off.push_back(o.seg_off.back() + n_seg);
        o.q4_off.push_back((uint32_t)(o.q4_off.back() + quads));
        o.n_cigar.push_back((uint16_t)c.n_cigar);
        o.l_seq.push_back((uint16_t)c.l_seq);
        const size_t nb = 4 * (size_t)c.n_cigar + (size_t)((c.l_seq + 1) / 2) + (size_t)c.l_seq, nw = (nb + 3) / 4;
        const size_t w0 = o.raw.size();
        o.raw.resize(w0 + nw, 0);
        memcpy(o.raw.data() + w0, r.cigar, nb);                      // CIGAR, bases and qualities are contiguous in the record
        o.raw_off.push_back((uint32_t)(w0 + nw));
        if ((uint32_t)rlen > o.max_span) o.max_span = (uint32_t)rlen;
        if (st.first_column < 0) {
            int64_t p = layout.first_inside(slot, c.pos, end);
            if (p >= 0) st.first_column = (int64_t)ctg.offset + p;
        }
        ++st.accepted;
    }
    if (st.max_buffered + 64u > 65535u) { err = bam_path + ": pileup depth above 65535 is not supported"; return false; }
    st.compressed_bytes = S.rd.compressed_bytes_read();
    st.inflate_seconds = S.rd.inflate_seconds();
    st.seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return true;
}

}  // namespace msnv
