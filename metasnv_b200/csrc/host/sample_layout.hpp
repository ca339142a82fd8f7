// sample_layout.hpp -- where the arrays of one sample's reads sit inside a block of memory.
//
// libmsnv_gpu lays its device blocks out by this rule. snpCall packs its pinned batches by the same rule, so that
// msnv_window_add_sample_raw finds each group of arrays contiguous and uploads it in one copy instead of one per array.
#pragma once

#include <cstddef>

namespace msnv {

// Consecutive arrays in one block: each starts 256-byte aligned and is followed by at least 32 spare bytes, because the
// pileup kernel's bulk copies read whole 16-byte units. `size` is the block's size so far.
struct BlockLayout {
    size_t size = 0;
    size_t take(size_t bytes) { const size_t o = size; size = (size + bytes + 32 + 255) / 256 * 256; return o; }
};

// The per-read arrays of n reads. `end` is one past the last byte of `mate`.
struct ReadGroup {
    size_t pos, seg_off, q4_off, mate, end;
    ReadGroup(BlockLayout& b, size_t n)
        : pos(b.take(n * 4)), seg_off(b.take((n + 1) * 4)), q4_off(b.take((n + 1) * 4)), mate(b.take(n * 4)), end(mate + n * 4) {}
};

// The aligned segments and bases: n_seg segments and n_q4 quads. `end` is one past the last byte of `qual`. `fix` holds
// the verdicts of the mate-overlap rule, one per quad, and exists only for a sample with mates (else it is 0).
struct SegmentGroup {
    size_t seg_pos, seg_len, seq2, qual, end, fix;
    SegmentGroup(BlockLayout& b, size_t n_seg, size_t n_q4, bool has_mates)
        : seg_pos(b.take(n_seg * 4)), seg_len(b.take(n_seg * 2)), seq2(b.take(n_q4)), qual(b.take(n_q4 * 4)), end(qual + n_q4 * 4),
          fix(has_mates ? b.take(n_q4) : 0) {}
};

// The BAM-shaped records of n reads that expand_kernel reads: offsets, raw_words 32-bit words of records, CIGAR and
// sequence lengths. `end` is one past the last byte of `l_seq`.
struct RawGroup {
    size_t raw_off, raw, n_cigar, l_seq, end;
    RawGroup(BlockLayout& b, size_t n, size_t raw_words)
        : raw_off(b.take((n + 1) * 4)), raw(b.take(raw_words * 4)), n_cigar(b.take(n * 2)), l_seq(b.take(n * 2)), end(l_seq + n * 2) {}
};

}  // namespace msnv
