// inflate_member_check -- csrc/gpu/inflate_member.h (the DEFLATE member decoder and CRC pieces the device inflater runs)
// against zlib, compiled for the host: every block type (stored, fixed, dynamic) from zlib's levels 0/1/6/9 and its
// Z_FIXED, Z_HUFFMAN_ONLY and Z_RLE strategies, sizes 0..65536, hand-made streams with matches at distance 1 and 32768,
// the BGZF EOF member, and malformed members, each of which must give its own status. Guard bytes around every output.
// The CRC is checked the way inflate_kernel computes it: 32 pieces (and other counts), shifted and XORed.
#include <zlib.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "inflate_member.h"

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)(rng_state >> 16); }
static long cases = 0, bad = 0;
static MsnvInflateScratch scratch;

static std::vector<uint8_t> make_data(int kind, size_t n)
{
    std::vector<uint8_t> d(n);
    switch (kind) {
        case 0: for (auto& x : d) x = (uint8_t)rnd(); break;                                  // incompressible
        case 1: for (auto& x : d) x = "ACGT"[rnd() & 3]; break;
        case 2: for (auto& x : d) x = (uint8_t)("IIIIIIIIFFFF<<<7"[rnd() & 15]); break;       // quality-like
        case 3: for (size_t i = 0; i < n; ++i) d[i] = (uint8_t)(i % 7 == 0 ? rnd() : 'x'); break;
        case 4: for (auto& x : d) x = 0; break;                                                // one symbol: distance-1 runs
        default: {                                                                            // BAM-like records
            size_t i = 0;
            while (i < n) {
                const size_t l = 40 + rnd() % 200;
                for (size_t k = 0; k < l && i < n; ++k, ++i) d[i] = (uint8_t)(k < 36 ? (k * 37 + (rnd() & 1)) : (k & 1 ? "ACGT"[rnd() & 3] : 'I' - (rnd() % 5 == 0)));
            }
        }
    }
    return d;
}

static std::vector<uint8_t> deflate_raw(const std::vector<uint8_t>& d, int level, int strategy)
{
    z_stream zs; memset(&zs, 0, sizeof zs);
    deflateInit2(&zs, level, Z_DEFLATED, -15, 8, strategy);
    std::vector<uint8_t> out(deflateBound(&zs, (uLong)d.size()) + 64);
    zs.next_in = (Bytef*)d.data(); zs.avail_in = (uInt)d.size();
    zs.next_out = out.data(); zs.avail_out = (uInt)out.size();
    deflate(&zs, Z_FINISH);
    out.resize(zs.total_out);
    deflateEnd(&zs);
    return out;
}

static uint32_t zcrc(const uint8_t* p, size_t n) { return (uint32_t)crc32(crc32(0L, nullptr, 0), p, (uInt)n); }

// the kernel's CRC: `lanes` pieces of ceil(n / lanes) bytes, each shifted to the end and XORed
static uint32_t pieces_crc(const uint8_t* p, uint32_t n, uint32_t lanes)
{
    if (n == 0) return 0;
    const uint32_t piece = (n + lanes - 1) / lanes;
    uint32_t c = 0;
    for (uint32_t l = 0; l < lanes; ++l) {
        const uint32_t lo = l * piece < n ? l * piece : n, hi = lo + piece < n ? lo + piece : n;
        c ^= msnv_crc32_shift(msnv_crc32_piece(p + lo, hi - lo), n - hi);
    }
    return c;
}

// decode + CRC as the device does it, output between guard bytes; returns the status
static int run_member(const std::vector<uint8_t>& c, uint32_t isize, uint32_t crc, std::vector<uint8_t>& out)
{
    std::vector<uint8_t> g((size_t)isize + 64, 0xA5);
    // the input is copied to an exactly sized heap block so that AddressSanitizer sees any read past it
    uint8_t* in = (uint8_t*)malloc(c.size() ? c.size() : 1);
    if (!c.empty()) memcpy(in, c.data(), c.size());
    int st = msnv_inflate_member(in, (uint32_t)c.size(), g.data() + 32, isize, &scratch);
    free(in);
    for (int k = 0; k < 32; ++k)
        if (g[k] != 0xA5 || g[(size_t)isize + 32 + k] != 0xA5) { ++bad; fprintf(stderr, "WROTE OUT OF BOUNDS isize %u\n", isize); break; }
    if (st == MSNV_INFLATE_OK && pieces_crc(g.data() + 32, isize, 32) != crc) st = MSNV_INFLATE_BAD_CRC;
    out.assign(g.begin() + 32, g.begin() + 32 + isize);
    return st;
}

static void expect(const char* what, int got, int want)
{
    ++cases;
    if (got != want) { ++bad; fprintf(stderr, "%s: status %d, expected %d\n", what, got, want); }
}

// LSB-first bit writer; Huffman codes go in most significant bit first (RFC 1951 3.1.1)
struct BitWriter {
    std::vector<uint8_t> b; uint32_t acc = 0; int n = 0;
    void put(uint32_t v, int bits) { for (int i = 0; i < bits; ++i) { acc |= ((v >> i) & 1u) << n; if (++n == 8) { b.push_back((uint8_t)acc); acc = 0; n = 0; } } }
    void huff(uint32_t code, int len) { for (int i = len - 1; i >= 0; --i) put((code >> i) & 1u, 1); }
    void fixed_sym(uint32_t s)
    {
        if (s < 144) huff(0x30 + s, 8); else if (s < 256) huff(0x190 + s - 144, 9); else if (s < 280) huff(s - 256, 7); else huff(0xC0 + s - 280, 8);
    }
    void align() { if (n) { b.push_back((uint8_t)acc); acc = 0; n = 0; } }
};

int main()
{
    // ---- zlib streams: every block type and size, the kernel's CRC pieces against zlib's crc32
    const size_t sizes[] = {0, 1, 2, 3, 7, 8, 31, 32, 33, 63, 64, 257, 258, 259, 1000, 4096, 30000, 32768, 32769, 65279, 65280, 65535, 65536};
    const int strategies[] = {Z_DEFAULT_STRATEGY, Z_FIXED, Z_HUFFMAN_ONLY, Z_RLE};
    for (int kind = 0; kind < 6; ++kind)
        for (size_t n : sizes)
            for (int level : {0, 1, 6, 9})
                for (int st : strategies) {
                    const std::vector<uint8_t> d = make_data(kind, n), c = deflate_raw(d, level, st);
                    std::vector<uint8_t> o;
                    const uint32_t crc = zcrc(d.data(), n);
                    ++cases;
                    const int s = run_member(c, (uint32_t)n, crc, o);
                    if (s != MSNV_INFLATE_OK || o != d) { ++bad; fprintf(stderr, "MISMATCH kind %d n %zu level %d strategy %d status %d\n", kind, n, level, st, s); }
                    if (n) expect("isize one short", run_member(c, (uint32_t)n - 1, crc, o), MSNV_INFLATE_TOO_LONG);
                    expect("isize one long", run_member(c, (uint32_t)n + 1, crc, o), MSNV_INFLATE_TOO_SHORT);
                    expect("wrong CRC", run_member(c, (uint32_t)n, crc ^ 0x10u, o), MSNV_INFLATE_BAD_CRC);
                    if (c.size() > 2) {
                        std::vector<uint8_t> t(c.begin(), c.begin() + (long)(c.size() / 2));
                        expect("truncated", run_member(t, (uint32_t)n, crc, o), MSNV_INFLATE_TRUNCATED);
                    }
                    // bit flips: any status, no out-of-bounds access; accepted output must be zlib's
                    if (n >= 64 && level && (cases & 3) == 0) {
                        std::vector<uint8_t> f = c;
                        f[rnd() % f.size()] ^= (uint8_t)(1u << (rnd() & 7));
                        if (run_member(f, (uint32_t)n, crc, o) == MSNV_INFLATE_OK && o != d) { ++bad; fprintf(stderr, "ACCEPTED CORRUPT STREAM kind %d n %zu\n", kind, n); }
                    }
                }
    // every size up to 600, then sizes in steps of up to 1 KB to 65536 (level 6); 64 KiB of incompressible data at every level
    for (size_t n = 0; n <= 65536; n += 1 + (n < 600 ? 0 : rnd() % 997)) {
        const std::vector<uint8_t> d = make_data((int)(n % 6), n), c = deflate_raw(d, 6, Z_DEFAULT_STRATEGY);
        std::vector<uint8_t> o;
        ++cases;
        if (run_member(c, (uint32_t)n, zcrc(d.data(), n), o) != MSNV_INFLATE_OK || o != d) { ++bad; fprintf(stderr, "MISMATCH size %zu\n", n); }
    }
    for (int level : {0, 1, 6, 9}) {
        const std::vector<uint8_t> d = make_data(0, 65536), c = deflate_raw(d, level, Z_DEFAULT_STRATEGY);
        std::vector<uint8_t> o;
        ++cases;
        if (run_member(c, 65536, zcrc(d.data(), 65536), o) != MSNV_INFLATE_OK || o != d) { ++bad; fprintf(stderr, "MISMATCH incompressible 64 KiB level %d\n", level); }
    }
    // ---- the BGZF EOF member: an empty fixed block, ISIZE 0, CRC 0
    {
        std::vector<uint8_t> o;
        expect("EOF member", run_member({0x03, 0x00}, 0, 0, o), MSNV_INFLATE_OK);
    }
    // ---- hand-made: a literal and a 258-byte match at distance 1; 32768 stored bytes and a match at distance 32768
    {
        BitWriter w;
        w.put(1, 1); w.put(1, 2);
        w.fixed_sym('A'); w.fixed_sym(285); w.put(0, 5);               // length 258, distance code 0 = 1
        w.fixed_sym(256); w.align();
        std::vector<uint8_t> d(259, 'A'), o;
        ++cases;
        if (run_member(w.b, 259, zcrc(d.data(), 259), o) != MSNV_INFLATE_OK || o != d) { ++bad; fprintf(stderr, "MISMATCH distance 1\n"); }
    }
    {
        const std::vector<uint8_t> head = make_data(0, 32768);
        BitWriter w;
        w.put(0, 1); w.put(0, 2); w.align();                           // stored, not final
        w.put(32768, 16); w.put(32768 ^ 0xffff, 16);
        w.b.insert(w.b.end(), head.begin(), head.end());
        w.put(1, 1); w.put(1, 2);
        w.fixed_sym(285); w.huff(29, 5); w.put(32768 - 24577, 13);      // length 258, distance 32768
        w.fixed_sym(256); w.align();
        std::vector<uint8_t> d = head, o;
        d.insert(d.end(), head.begin(), head.begin() + 258);
        ++cases;
        if (run_member(w.b, (uint32_t)d.size(), zcrc(d.data(), d.size()), o) != MSNV_INFLATE_OK || o != d) { ++bad; fprintf(stderr, "MISMATCH distance 32768\n"); }
        // the same match one byte earlier in the stream reaches in front of the output
        BitWriter v;
        v.put(0, 1); v.put(0, 2); v.align();
        v.put(32767, 16); v.put(32767 ^ 0xffff, 16);
        v.b.insert(v.b.end(), head.begin(), head.begin() + 32767);
        v.put(1, 1); v.put(1, 2);
        v.fixed_sym(285); v.huff(29, 5); v.put(32768 - 24577, 13);
        v.fixed_sym(256); v.align();
        expect("distance 32768 after 32767 bytes", run_member(v.b, 32767 + 258, 0, o), MSNV_INFLATE_BAD_DISTANCE);
    }
    // ---- malformed members
    {
        std::vector<uint8_t> o;
        BitWriter w;                                                    // a match as the first symbol
        w.put(1, 1); w.put(1, 2); w.fixed_sym(257); w.put(0, 5); w.fixed_sym(256); w.align();
        expect("distance past the start", run_member(w.b, 3, 0, o), MSNV_INFLATE_BAD_DISTANCE);
        BitWriter u;                                                    // 19 code-length codes of length 1
        u.put(1, 1); u.put(2, 2); u.put(0, 5); u.put(0, 5); u.put(15, 4);
        for (int i = 0; i < 19; ++i) u.put(1, 3);
        u.put(0, 16); u.align();
        expect("over-subscribed code lengths", run_member(u.b, 10, 0, o), MSNV_INFLATE_BAD_CODE);
        BitWriter x;                                                    // block type 3
        x.put(1, 1); x.put(3, 2); x.put(0, 16); x.align();
        expect("reserved block type", run_member(x.b, 10, 0, o), MSNV_INFLATE_BAD_CODE);
        BitWriter y;                                                    // stored block whose NLEN does not match
        y.put(1, 1); y.put(0, 2); y.align(); y.put(5, 16); y.put(5, 16); y.put(0, 32); y.put(0, 8);
        expect("stored length check", run_member(y.b, 5, 0, o), MSNV_INFLATE_BAD_CODE);
        expect("empty input", run_member({}, 0, 0, o), MSNV_INFLATE_TRUNCATED);
    }
    // ---- the CRC pieces against zlib for every piece count a warp could use, on lengths around the piece bounds
    for (uint32_t n : {0u, 1u, 2u, 31u, 32u, 33u, 63u, 64u, 65u, 1000u, 65535u, 65536u})
        for (uint32_t lanes : {1u, 2u, 3u, 7u, 32u}) {
            const std::vector<uint8_t> d = make_data(0, n);
            ++cases;
            if (pieces_crc(d.data(), n, lanes) != zcrc(d.data(), n)) { ++bad; fprintf(stderr, "CRC MISMATCH n %u lanes %u\n", n, lanes); }
        }
    for (int rep = 0; rep < 200; ++rep) {                               // zlib's crc32_combine
        const uint32_t a = rnd(), b = rnd(), len = rnd() % 70000;
        ++cases;
        if ((msnv_crc32_shift(a, len) ^ b) != (uint32_t)crc32_combine(a, b, (z_off_t)len)) { ++bad; fprintf(stderr, "COMBINE MISMATCH len %u\n", len); }
    }
    printf("cases: %ld mismatches: %ld\n", cases, bad);
    return bad != 0;
}
