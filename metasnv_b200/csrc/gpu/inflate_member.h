// inflate_member.h -- one raw-DEFLATE member (RFC 1951: stored, fixed- and dynamic-Huffman blocks) into a buffer of
// exactly `isize` bytes, and the CRC-32 pieces a warp combines. Host + device: the device inflater (msnv_gpu.cu,
// inflate_kernel) runs the symbol decode (msnv_inflate_step) on one lane per member with the tables in the warp's slice
// of shared memory and copies the matches it queues with the whole warp (msnv_inf_match_byte); msnv_inflate_member is
// the same on one thread, which tests/test_inflate_cpu.py compiles with gcc under AddressSanitizer and UBSan against zlib.
//
// Every input byte is fetched through a bounds test (past the end the bit buffer is padded with zeros and the
// decoder reports MSNV_INFLATE_TRUNCATED once it consumes one of them), and every output write is tested against
// `isize`. Nothing faults on malformed input: the result is a status (msnv_inflate_status in include/msnv.h).
// The table layout is csrc/host/fast_inflate.cc's, without its two-literal entries.
#pragma once
#include <stdint.h>

#include "../../../include/msnv.h"

#ifdef __CUDACC__
#define MSNV_INF_HD __host__ __device__ __forceinline__
#else
#define MSNV_INF_HD static inline
#endif

// ---- table entries (as in fast_inflate.cc)
// bits 0..4 code bits to consume (a link: the primary width), bits 5..8 extra bits (a link: subtable index bits),
// bits 9..10 kind, bits 16..31 literal | length or distance base | 0 = end of block, 1 = invalid | subtable offset
enum : uint32_t { MSNV_INF_LITERAL = 0, MSNV_INF_BASE = 1, MSNV_INF_SPECIAL = 2, MSNV_INF_LINK = 3 };
enum : int { MSNV_INF_LL_PRIMARY = 10, MSNV_INF_D_PRIMARY = 8, MSNV_INF_CL_PRIMARY = 7 };
// zlib's bound for a 10-bit root over 286 symbols of up to 15 bits is 1334 entries; distances get a generous 512.
// A code that would need more is refused (MSNV_INFLATE_BAD_CODE), never written past.
enum : int { MSNV_INF_LL_SIZE = 1334, MSNV_INF_D_SIZE = 512, MSNV_INF_CL_SIZE = 1 << MSNV_INF_CL_PRIMARY };

// The decoder's working set: one per member being decoded (about 8.4 KB; in shared memory on the device).
struct MsnvInflateScratch {
    uint32_t ll[MSNV_INF_LL_SIZE];
    uint32_t d[MSNV_INF_D_SIZE];
    uint32_t cl[MSNV_INF_CL_SIZE];
    uint8_t lens[320];                  // 286 + 30 code lengths (hlit + hdist <= 316)
};

MSNV_INF_HD uint32_t msnv_inf_entry(uint32_t nbits, uint32_t extra, uint32_t kind, uint32_t value) { return nbits | extra << 5 | kind << 9 | value << 16; }
MSNV_INF_HD uint32_t msnv_inf_bits(uint32_t e) { return e & 31u; }
MSNV_INF_HD uint32_t msnv_inf_extra(uint32_t e) { return (e >> 5) & 15u; }
MSNV_INF_HD uint32_t msnv_inf_kind(uint32_t e) { return (e >> 9) & 3u; }
MSNV_INF_HD uint32_t msnv_inf_value(uint32_t e) { return e >> 16; }
#define MSNV_INF_INVALID msnv_inf_entry(1, 0, MSNV_INF_SPECIAL, 1)

// the low n (1..15) bits of v in reverse order
MSNV_INF_HD uint32_t msnv_inf_reverse(uint32_t v, int n)
{
#ifdef __CUDA_ARCH__
    return __brev(v) >> (32 - n);
#else
    uint32_t r = 0;
    for (int i = 0; i < n; ++i) r |= ((v >> i) & 1u) << (n - 1 - i);
    return r;
#endif
}

// Order in which a dynamic block sends the code-length code lengths (RFC 1951 3.2.7), 5 bits per entry.
MSNV_INF_HD uint32_t msnv_inf_cl_order(uint32_t i)
{
    // 16 17 18 0 8 7 9 6 10 5 11 4 | 12 3 13 2 14 1 15
    const uint64_t lo = 16ull | 17ull << 5 | 18ull << 10 | 0ull << 15 | 8ull << 20 | 7ull << 25 | 9ull << 30 | 6ull << 35 |
                        10ull << 40 | 5ull << 45 | 11ull << 50 | 4ull << 55;
    const uint64_t hi = 12ull | 3ull << 5 | 13ull << 10 | 2ull << 15 | 14ull << 20 | 1ull << 25 | 15ull << 30;
    return i < 12 ? (uint32_t)(lo >> (5 * i)) & 31u : (uint32_t)(hi >> (5 * (i - 12))) & 31u;
}

enum { MSNV_INF_LITLEN = 0, MSNV_INF_DIST = 1, MSNV_INF_CODELEN = 2 };

MSNV_INF_HD uint32_t msnv_inf_symbol(int alphabet, uint32_t sym, uint32_t nbits)
{
    if (alphabet == MSNV_INF_LITLEN) {
        if (sym < 256) return msnv_inf_entry(nbits, 0, MSNV_INF_LITERAL, sym);
        if (sym == 256) return msnv_inf_entry(nbits, 0, MSNV_INF_SPECIAL, 0);
        if (sym >= 286) return msnv_inf_entry(nbits, 0, MSNV_INF_SPECIAL, 1);
        const uint32_t i = sym - 257;               // lengths 3..258: RFC 1951 3.2.5
        if (i < 8) return msnv_inf_entry(nbits, 0, MSNV_INF_BASE, 3 + i);
        if (i == 28) return msnv_inf_entry(nbits, 0, MSNV_INF_BASE, 258);
        const uint32_t x = (i >> 2) - 1;
        return msnv_inf_entry(nbits, x, MSNV_INF_BASE, ((4u + (i & 3u)) << x) + 3u);
    }
    if (alphabet == MSNV_INF_DIST) {
        if (sym >= 30) return msnv_inf_entry(nbits, 0, MSNV_INF_SPECIAL, 1);
        if (sym < 4) return msnv_inf_entry(nbits, 0, MSNV_INF_BASE, sym + 1);
        const uint32_t x = (sym >> 1) - 1;
        return msnv_inf_entry(nbits, x, MSNV_INF_BASE, ((2u + (sym & 1u)) << x) + 1u);
    }
    return msnv_inf_entry(nbits, 0, MSNV_INF_LITERAL, sym);
}

// Canonical Huffman code of lens[0..n) -> table indexed by the next `primary` input bits (LSB first). Over-subscribed
// codes and codes whose subtables do not fit `capacity` are refused; incomplete ones are accepted (unused patterns
// stay invalid). Before the links are laid out, a primary slot that prefixes long codes holds their widest excess.
MSNV_INF_HD bool msnv_inf_build(int alphabet, const uint8_t* lens, int n, int primary, uint32_t* table, int capacity)
{
    int count[16];
    for (int l = 0; l < 16; ++l) count[l] = 0;
    for (int i = 0; i < n; ++i) ++count[lens[i]];
    count[0] = 0;
    int left = 1;
    for (int l = 1; l <= 15; ++l) { left = left * 2 - count[l]; if (left < 0) return false; }
    uint32_t next[16]; uint32_t code = 0;
    next[0] = 0;
    for (int l = 1; l <= 15; ++l) { code = (code + (uint32_t)count[l - 1]) << 1; next[l] = code; }
    uint32_t first[16];
    for (int l = 0; l < 16; ++l) first[l] = next[l];

    const uint32_t psize = 1u << primary;
    for (uint32_t i = 0; i < psize; ++i) table[i] = 0;
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        if (l <= primary) continue;
        const uint32_t p = msnv_inf_reverse(next[l]++, l) & (psize - 1);
        if ((uint32_t)(l - primary) > table[p]) table[p] = (uint32_t)(l - primary);
    }
    uint32_t used = psize;
    for (uint32_t p = 0; p < psize; ++p) {
        const uint32_t w = table[p];
        if (!w) { table[p] = MSNV_INF_INVALID; continue; }
        const uint32_t size = 1u << w;
        if (used + size > (uint32_t)capacity) return false;
        table[p] = msnv_inf_entry((uint32_t)primary, w, MSNV_INF_LINK, used);
        for (uint32_t i = 0; i < size; ++i) table[used + i] = MSNV_INF_INVALID;
        used += size;
    }
    for (int l = 0; l < 16; ++l) next[l] = first[l];
    for (int s = 0; s < n; ++s) {
        const int l = lens[s];
        if (!l) continue;
        const uint32_t c = msnv_inf_reverse(next[l]++, l);
        if (l <= primary) {
            const uint32_t e = msnv_inf_symbol(alphabet, (uint32_t)s, (uint32_t)l);
            for (uint32_t i = c; i < psize; i += 1u << l) table[i] = e;
        } else {
            const uint32_t link = table[c & (psize - 1)];
            const uint32_t e = msnv_inf_symbol(alphabet, (uint32_t)s, (uint32_t)(l - primary));
            const uint32_t size = 1u << msnv_inf_extra(link);
            for (uint32_t i = c >> primary; i < size; i += 1u << (l - primary)) table[msnv_inf_value(link) + i] = e;
        }
    }
    return true;
}

// LSB-first bit reader; every byte fetch is bounds-tested, zero bytes are invented past the end and counted.
struct MsnvInfBits {
    const uint8_t* in; const uint8_t* end;
    uint64_t buf; int cnt, padded;
};
MSNV_INF_HD void msnv_inf_refill(MsnvInfBits& b)
{
    if (b.end - b.in >= 8) {
        // eight independent byte loads (one memory latency instead of up to seven in a row); bytes beyond the
        // new count land above it and are loaded again, identically, by the next refill
        uint64_t w = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) w |= (uint64_t)b.in[k] << (8 * k);
        b.buf |= w << b.cnt;
        b.in += (63 - b.cnt) >> 3;
        b.cnt |= 56;
        return;
    }
    while (b.cnt <= 56) {
        if (b.in < b.end) b.buf |= (uint64_t)*b.in++ << b.cnt; else b.padded += 8;
        b.cnt += 8;
    }
}
MSNV_INF_HD uint32_t msnv_inf_peek(const MsnvInfBits& b, int n) { return (uint32_t)(b.buf & ((1ull << n) - 1)); }
MSNV_INF_HD void msnv_inf_consume(MsnvInfBits& b, int n) { b.buf >>= n; b.cnt -= n; }
MSNV_INF_HD uint32_t msnv_inf_take(MsnvInfBits& b, int n) { const uint32_t v = msnv_inf_peek(b, n); msnv_inf_consume(b, n); return v; }
// an invented bit was consumed <=> fewer bits remain than were invented
MSNV_INF_HD bool msnv_inf_past_end(const MsnvInfBits& b) { return b.cnt < b.padded; }

// Where a member's decode stands between two calls of msnv_inflate_step.
struct MsnvInfState {
    MsnvInfBits b;
    uint32_t o;                 // output bytes produced (literals written, matches queued)
    bool last, in_block;
};
// A match the decoder has checked and queued: out[o, o + len) repeats the dist bytes in front of o.
struct MsnvInfMatch { uint32_t o, len, dist; };
// Statuses beyond msnv_inflate_status for the step protocol
enum : int { MSNV_INF_RUNNING = -1 };

MSNV_INF_HD void msnv_inflate_begin(MsnvInfState& st, const uint8_t* in, uint32_t in_len)
{
    st.b.in = in; st.b.end = in + in_len; st.b.buf = 0; st.b.cnt = 0; st.b.padded = 0;
    st.o = 0; st.last = false; st.in_block = false;
}

// Out-of-place copy of one queued match, byte j by any thread (the matched bytes repeat with period dist, so every byte
// reads only output that existed before the match).
MSNV_INF_HD void msnv_inf_match_byte(uint8_t* out, const MsnvInfMatch& m, uint32_t j) { out[m.o + j] = out[m.o - m.dist + j % m.dist]; }

// Decodes the member in[0..in_len) into out[0..isize) until it has queued `max_matches` matches, or the member ends, or it
// fails. Literals and stored bytes are written at once; matches are checked (distance, length) and queued in q, to be
// copied in order by msnv_inf_match_byte before the next call. Returns MSNV_INF_RUNNING while there is more, else the
// member's msnv_inflate_status (MSNV_INFLATE_OK only when the final block ends with exactly isize bytes; the CRC is not
// checked here). *n_matches gets the number queued, also when the member ended or failed.
MSNV_INF_HD int msnv_inflate_step(MsnvInfState& st, uint8_t* out, uint32_t isize, MsnvInflateScratch* s, MsnvInfMatch* q,
                                  uint32_t max_matches, uint32_t* n_matches)
{
    MsnvInfBits& b = st.b;
    uint32_t o = st.o, nq = 0;
    *n_matches = 0;
    // a malformed stream read past its end is reported as truncated, whatever the invented zero bits then decode to
#define MSNV_INF_RETURN(x) do { st.o = o; *n_matches = nq; return (x); } while (0)
#define MSNV_INF_FAIL(x) MSNV_INF_RETURN(msnv_inf_past_end(b) ? (int)MSNV_INFLATE_TRUNCATED : (int)(x))
    for (;;) {
        if (!st.in_block) {
            if (st.last) MSNV_INF_RETURN(o == isize ? (int)MSNV_INFLATE_OK : (int)MSNV_INFLATE_TOO_SHORT);
            msnv_inf_refill(b);
            st.last = msnv_inf_take(b, 1) != 0;
            const uint32_t type = msnv_inf_take(b, 2);
            if (msnv_inf_past_end(b)) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
            if (type == 0) {                                    // stored: byte boundary, LEN, NLEN, LEN bytes
                msnv_inf_consume(b, b.cnt & 7);
                msnv_inf_refill(b);
                if (b.cnt - b.padded < 32) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
                const uint32_t len = msnv_inf_take(b, 16), nlen = msnv_inf_take(b, 16);
                if ((len ^ nlen) != 0xffffu) MSNV_INF_RETURN(MSNV_INFLATE_BAD_CODE);
                const uint8_t* src = b.in - (b.cnt - b.padded) / 8;   // the whole bytes still in the buffer go back to the input
                if ((uint32_t)(b.end - src) < len) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
                if (isize - o < len) MSNV_INF_RETURN(MSNV_INFLATE_TOO_LONG);
                for (uint32_t i = 0; i < len; ++i) out[o + i] = src[i];
                o += len;
                b.in = src + len; b.buf = 0; b.cnt = 0; b.padded = 0;
                continue;
            }
            if (type == 1) {
                uint8_t* lens = s->lens;
                for (int i = 0; i < 144; ++i) lens[i] = 8;
                for (int i = 144; i < 256; ++i) lens[i] = 9;
                for (int i = 256; i < 280; ++i) lens[i] = 7;
                for (int i = 280; i < 288; ++i) lens[i] = 8;
                for (int i = 288; i < 288 + 32; ++i) lens[i] = 5;
                if (!msnv_inf_build(MSNV_INF_LITLEN, lens, 288, MSNV_INF_LL_PRIMARY, s->ll, MSNV_INF_LL_SIZE) ||
                    !msnv_inf_build(MSNV_INF_DIST, lens + 288, 32, MSNV_INF_D_PRIMARY, s->d, MSNV_INF_D_SIZE))
                    MSNV_INF_RETURN(MSNV_INFLATE_BAD_CODE);
            } else if (type == 2) {
                const uint32_t hlit = msnv_inf_take(b, 5) + 257, hdist = msnv_inf_take(b, 5) + 1, hclen = msnv_inf_take(b, 4) + 4;
                if (hlit > 286 || hdist > 30) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
                uint8_t* lens = s->lens;
                for (int i = 0; i < 19; ++i) lens[i] = 0;
                for (uint32_t i = 0; i < hclen; ++i) { msnv_inf_refill(b); lens[msnv_inf_cl_order(i)] = (uint8_t)msnv_inf_take(b, 3); }
                if (!msnv_inf_build(MSNV_INF_CODELEN, lens, 19, MSNV_INF_CL_PRIMARY, s->cl, MSNV_INF_CL_SIZE)) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
                uint32_t n = 0;
                while (n < hlit + hdist) {
                    msnv_inf_refill(b);
                    const uint32_t e = s->cl[msnv_inf_peek(b, MSNV_INF_CL_PRIMARY)];
                    if (msnv_inf_kind(e) != MSNV_INF_LITERAL) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
                    msnv_inf_consume(b, (int)msnv_inf_bits(e));
                    const uint32_t sym = msnv_inf_value(e);
                    if (sym < 16) { lens[n++] = (uint8_t)sym; continue; }
                    uint32_t rep, val = 0;
                    if (sym == 16) { if (!n) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE); val = lens[n - 1]; rep = 3 + msnv_inf_take(b, 2); }
                    else if (sym == 17) rep = 3 + msnv_inf_take(b, 3);
                    else rep = 11 + msnv_inf_take(b, 7);
                    if (n + rep > hlit + hdist) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
                    for (uint32_t i = 0; i < rep; ++i) lens[n + i] = (uint8_t)val;
                    n += rep;
                }
                if (msnv_inf_past_end(b)) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
                if (lens[256] == 0) MSNV_INF_RETURN(MSNV_INFLATE_BAD_CODE);
                if (!msnv_inf_build(MSNV_INF_LITLEN, lens, (int)hlit, MSNV_INF_LL_PRIMARY, s->ll, MSNV_INF_LL_SIZE) ||
                    !msnv_inf_build(MSNV_INF_DIST, lens + hlit, (int)hdist, MSNV_INF_D_PRIMARY, s->d, MSNV_INF_D_SIZE))
                    MSNV_INF_RETURN(MSNV_INFLATE_BAD_CODE);
            } else {
                MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
            }
            st.in_block = true;
        }
        const uint32_t* ll = s->ll;
        const uint32_t* dt = s->d;
        for (;;) {
            if (nq == max_matches) MSNV_INF_RETURN(MSNV_INF_RUNNING);
            msnv_inf_refill(b);                                 // >= 56 bits: code 15 + extra 5 + code 15 + extra 13 = 48
            uint32_t e = ll[msnv_inf_peek(b, MSNV_INF_LL_PRIMARY)];
            if (msnv_inf_kind(e) == MSNV_INF_LINK) { msnv_inf_consume(b, MSNV_INF_LL_PRIMARY); e = ll[msnv_inf_value(e) + msnv_inf_peek(b, (int)msnv_inf_extra(e))]; }
            msnv_inf_consume(b, (int)msnv_inf_bits(e));
            if (msnv_inf_past_end(b)) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
            if (msnv_inf_kind(e) == MSNV_INF_LITERAL) {
                if (o >= isize) MSNV_INF_RETURN(MSNV_INFLATE_TOO_LONG);
                out[o++] = (uint8_t)msnv_inf_value(e);
                continue;
            }
            if (msnv_inf_kind(e) == MSNV_INF_SPECIAL) {
                if (msnv_inf_value(e) != 0) MSNV_INF_RETURN(MSNV_INFLATE_BAD_CODE);
                st.in_block = false;                            // end of block
                break;
            }
            const uint32_t len = msnv_inf_value(e) + msnv_inf_take(b, (int)msnv_inf_extra(e));
            uint32_t f = dt[msnv_inf_peek(b, MSNV_INF_D_PRIMARY)];
            if (msnv_inf_kind(f) == MSNV_INF_LINK) { msnv_inf_consume(b, MSNV_INF_D_PRIMARY); f = dt[msnv_inf_value(f) + msnv_inf_peek(b, (int)msnv_inf_extra(f))]; }
            if (msnv_inf_kind(f) != MSNV_INF_BASE) MSNV_INF_FAIL(MSNV_INFLATE_BAD_CODE);
            msnv_inf_consume(b, (int)msnv_inf_bits(f));
            const uint32_t dist = msnv_inf_value(f) + msnv_inf_take(b, (int)msnv_inf_extra(f));
            if (msnv_inf_past_end(b)) MSNV_INF_RETURN(MSNV_INFLATE_TRUNCATED);
            if (dist > o) MSNV_INF_RETURN(MSNV_INFLATE_BAD_DISTANCE);
            if (len > isize - o) MSNV_INF_RETURN(MSNV_INFLATE_TOO_LONG);
            q[nq].o = o; q[nq].len = len; q[nq].dist = dist;
            ++nq;
            o += len;
        }
    }
#undef MSNV_INF_FAIL
#undef MSNV_INF_RETURN
}

// The whole member on one thread: steps, each followed by its queued matches in order.
MSNV_INF_HD int msnv_inflate_member(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t isize, MsnvInflateScratch* s)
{
    MsnvInfState st;
    msnv_inflate_begin(st, in, in_len);
    MsnvInfMatch q[32];
    for (;;) {
        uint32_t n = 0;
        const int r = msnv_inflate_step(st, out, isize, s, q, 32, &n);
        for (uint32_t k = 0; k < n; ++k)
            for (uint32_t j = 0; j < q[k].len; ++j) msnv_inf_match_byte(out, q[k], j);
        if (r != MSNV_INF_RUNNING) return r;
    }
}

// ---- CRC-32 (gzip's, reflected polynomial 0xEDB88320) in pieces
// crc32(0, p, n) as zlib computes it, one bit at a time (no table: the device runs it on every lane of a warp)
MSNV_INF_HD uint32_t msnv_crc32_piece(const uint8_t* p, uint32_t n)
{
    uint32_t c = 0xffffffffu;
    for (uint32_t i = 0; i < n; ++i) {
        c ^= p[i];
        for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (0xedb88320u & (0u - (c & 1u)));
    }
    return ~c;
}
// a * b mod P for reflected polynomials (bit 31 = x^0)
MSNV_INF_HD uint32_t msnv_crc32_mulmod(uint32_t a, uint32_t b)
{
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
// The CRC of a piece that is followed by `after` more bytes, moved to the end of the message: x^(8 * after) * crc mod P.
// The CRC of a message cut into pieces is the XOR of every piece's zlib CRC shifted this way (zlib's crc32_combine,
// applied to all pieces at once), so the lanes of a warp can each take one piece.
MSNV_INF_HD uint32_t msnv_crc32_shift(uint32_t crc, uint32_t after)
{
    uint32_t p = 1u << 31, sq = 1u << 23;                       // x^0, x^8
    while (after) {
        if (after & 1u) p = msnv_crc32_mulmod(sq, p);
        after >>= 1;
        if (after) sq = msnv_crc32_mulmod(sq, sq);
    }
    return msnv_crc32_mulmod(p, crc);
}
