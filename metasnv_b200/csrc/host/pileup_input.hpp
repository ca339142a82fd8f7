// pileup_input.hpp -- BAM -> structure-of-arrays read batches for the GPU pileup (include/msnv.h),
// including everything `samtools mpileup` decides per read before it builds columns: the default
// flag / orphan / BED / reference-length filters, the per-file depth cap and the mate-overlap
// pairing (SURVEY.md Annex A.1-A.3; the reference reaches this code through metaSNV.py:160-165).
// These are sequential, order-dependent per-file rules, so they run in the decoding thread; the
// per-base work (overlap quality correction, CIGAR walk, counting) is done on the device.
#pragma once
#include <cstdint>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../../include/msnv.h"
#include "bam.hpp"

namespace msnv {

// Reference sequences by name (name = first word of the FASTA header, as faidx does).
struct Fasta {
    std::vector<std::string> names;
    std::vector<std::string> seqs;
    std::unordered_map<std::string, int> index;      // first record of a name wins
    bool load(const std::string& path, std::string& err);
    int find(const std::string& name) const { auto it = index.find(name); return it == index.end() ? -1 : it->second; }
};

// -l file: 3 columns = BED (0-based half open), 2 columns = 1-based position.
struct Bed {
    struct Iv { int64_t beg, end; };
    std::unordered_map<std::string, std::vector<Iv>> by_name;
    bool load(const std::string& path, std::string& err);
};

// Contigs of one shard in shard coordinates (each contig starts at a multiple of MSNV_TILE).
struct ShardLayout {
    struct Ctg { int tid; uint32_t len; uint32_t offset; };
    std::vector<Ctg> ctgs;                    // ascending tid
    std::vector<int> slot_of_tid;             // tid -> index into ctgs, or -1
    std::vector<std::vector<Bed::Iv>> bed;    // per ctg: sorted intervals the shard covers ([0,len) without -l)
    uint32_t n_positions = 0;
    bool has_bed = false;
    // All contigs of the header (no -l), or those named in the BED.
    bool build(const BamHeader& hdr, const Bed* bed_or_null, std::string& err);
    bool overlaps(int slot, int64_t beg, int64_t end) const;
    // smallest position in [beg,end) covered by the shard's intervals, or -1
    int64_t first_inside(int slot, int64_t beg, int64_t end) const;
};

// One sample's batch as BAM stores it (msnv_raw_reads): the device walks the CIGARs and packs the bases (expand_kernel),
// the decoding thread only copies the record's own bytes. `end` (one past the last reference base, shard coordinate) is
// the host's: it decides which reads a later window still needs.
struct RawReads {
    std::vector<int32_t>  pos, end, mate;
    std::vector<uint32_t> seg_off{0}, q4_off{0}, raw_off{0};
    std::vector<uint16_t> n_cigar, l_seq;
    std::vector<uint32_t> raw;
    uint32_t max_span = 0;
    msnv_raw_reads view() const;
    size_t bytes() const;
};

struct SampleDecoderState;

struct DecodeStats {
    uint64_t records = 0, accepted = 0, dropped_by_cap = 0, aligned_bases = 0, pairs = 0;
    uint64_t compressed_bytes = 0;
    double seconds = 0, inflate_seconds = 0;
    // first pileup column this sample would emit (shard coordinate), or -1
    int64_t first_column = -1;
    uint32_t max_buffered = 0;
};

// Resumable decoder of one BAM: the shard is handed out window by window (ascending, disjoint ranges of shard
// coordinates), so neither the host nor the device has to hold a whole shard - the reference's pipe streams the same
// way (call_vC.cpp:466-479 reads one pileup line at a time). Everything mpileup decides per read in file order
// (filters, depth cap, mate pairing) carries over from window to window.
//   window(lo, hi, prev, out): `out` = every accepted read that starts before `hi` and ends after `lo`: first the tail
//   of the previous window's batch `prev` (from its first read whose `end` is past `lo` on; pass nullptr for the first
//   window), then the reads decoded now. Mate links are indices into `out`; a link whose partner is not in `out` is
//   dropped (the two then share no position inside the window).
// `ref_len_of_tid[tid]` is the FASTA length of the contig or -1 when the FASTA lacks it (mpileup then keeps every read).
// With a TidIndex and a -l split the decoder seeks to the runs of contigs the split names instead of inflating the
// whole file.
class SampleDecoder {
public:
    SampleDecoder();
    ~SampleDecoder();
    SampleDecoder(const SampleDecoder&) = delete;
    SampleDecoder& operator=(const SampleDecoder&) = delete;
    bool open(const std::string& bam_path, const ShardLayout& layout, const std::vector<int64_t>& ref_len_of_tid, int inflate_threads,
              const std::string& index_hint, std::string& err);
    bool window(uint32_t pos_lo, uint32_t pos_hi, const RawReads* prev, RawReads& out, std::string& err);
    const DecodeStats& stats() const;
    bool used_index() const;
private:
    SampleDecoderState* st_;
};

// Reference characters of the shard, one byte per shard coordinate: the FASTA character where the
// contig has one and the position is inside the shard's intervals, 'N' inside the intervals but
// beyond the FASTA, 0 elsewhere (padding, outside -l).
std::vector<uint8_t> shard_reference(const ShardLayout& layout, const BamHeader& hdr, const Fasta& fa);

}  // namespace msnv
