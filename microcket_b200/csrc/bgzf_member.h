// bgzf_member.h — one BGZF member (SAMv1 §4.1): the header rule, a raw-deflate decoder (RFC 1951) and the trailer check.
// The decoder's control logic (bit reader, Huffman tables, symbol decode, every bound) is written once and compiled twice:
// as CUDA in bgzf.cu, where one warp decodes one member, and as plain C++ in the host form tests/test_bgzf.py runs under
// AddressSanitizer on damaged members.  Only the output side differs: a "writer" W (BgWarp in bgzf.cu, the host harness's
// own) provides lane / nl / sync() for the table builds, the copies (lit, match, stored) and the CRC of the output.
// Bounds, for ANY input bytes: the reader never loads past the member's deflate bytes (it feeds zeros behind them and the
// decoder fails once it has consumed a bit it did not load); W refuses every write past ISIZE and every distance reaching
// back past the start of the member's output.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#ifdef __CUDACC__
#define BG_FN __device__ __forceinline__
#define BG_TABLE __constant__ static const
#else
#define BG_FN inline
#define BG_TABLE static const
#endif

// a member's outcome; the reasons name the first check that failed
enum {
    BG_OK = 0, BG_HEADER, BG_ISIZE, BG_BTYPE, BG_STORED_LEN, BG_CODES, BG_BAD_CODE, BG_SYMBOL, BG_DIST_CODE, BG_TOO_FAR,
    BG_OVERFLOW, BG_OVERRUN, BG_TRAILING, BG_SHORT, BG_CRC, BG_N_REASONS
};
static inline const char *bg_reason(int r) {
    static const char *const t[BG_N_REASONS] = {
        "ok", "header does not fit the member", "ISIZE differs from the member table", "block type 3",
        "stored block LEN != ~NLEN", "bad code lengths (over-subscribed, incomplete, bad repeat or no end-of-block code)",
        "a bit sequence that is no code", "literal/length symbol 286 or 287", "distance code 30 or 31",
        "distance reaches back past the start of the member", "output past ISIZE", "deflate data runs past the member",
        "deflate data does not end right before the trailer", "output shorter than ISIZE", "CRC-32 mismatch"};
    return r >= 0 && r < BG_N_REASONS ? t[r] : "unknown";
}

#define BG_MAX_ISIZE 65536u
#define BG_FAST 9                                            // direct-table bits; longer codes take the canonical walk

static inline uint32_t bg_rd16(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }
static inline uint32_t bg_rd32(const uint8_t *p) { return bg_rd16(p) | bg_rd16(p + 2) << 16; }

// ---------------------------------------------------------------- host member walk
// One BGZF member header at p (avail bytes there): 1 = incomplete (more bytes needed), 0 = whole member of *len bytes
// (BSIZE + 1) and *isize output bytes, -1 = not a BGZF member (*why says how).  The rule of bam_input.hpp: 1f 8b 08 with
// FLG.FEXTRA, a BC subfield with SLEN 2 among any others, room for the header and the 8 trailer bytes, ISIZE <= 64 KiB.
static inline int bg_header(const uint8_t *p, size_t avail, uint32_t *len, uint32_t *isize, const char **why) {
    static const uint8_t magic[4] = {0x1f, 0x8b, 8, 4};
    for (size_t k = 0; k < 4 && k < avail; ++k)
        if (k < 3 ? p[k] != magic[k] : !(p[k] & 4)) { *why = k < 2 ? "not a gzip member" : k == 2 ? "gzip member with a compression method other than deflate" : "gzip but not BGZF: no extra field"; return -1; }
    if (avail < 12) return 1;
    const size_t xlen = bg_rd16(p + 10);
    if (avail < 12 + xlen) return 1;
    long bsize = -1;
    for (size_t x = 0; x + 4 <= xlen;) {
        const uint8_t *s = p + 12 + x; const size_t sl = bg_rd16(s + 2);
        if (s[0] == 'B' && s[1] == 'C' && sl == 2 && x + 6 <= xlen) bsize = (long)bg_rd16(s + 4);
        x += 4 + sl;
    }
    if (bsize < 0) { *why = "gzip but not BGZF: no BC subfield"; return -1; }
    if ((size_t)bsize + 1 < 12 + xlen + 8) { *why = "BSIZE smaller than the header and trailer"; return -1; }
    if (avail < (size_t)bsize + 1) return 1;
    *len = (uint32_t)bsize + 1;
    *isize = bg_rd32(p + bsize + 1 - 4);
    if (*isize > BG_MAX_ISIZE) { *why = "ISIZE larger than 64 KiB"; return -1; }
    return 0;
}

// ---------------------------------------------------------------- decoder
BG_TABLE uint16_t BG_LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
BG_TABLE uint8_t BG_LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
BG_TABLE uint16_t BG_DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
                                  4097, 6145, 8193, 12289, 16385, 24577};
BG_TABLE uint8_t BG_DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
BG_TABLE uint8_t BG_CLORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// LSB-first bit reader over n bytes; zeros behind them, so that a damaged stream reads no byte it does not own
struct BgBits {
    const uint8_t *p; uint32_t n, pos, cnt; uint64_t buf;
    BG_FN void refill() { while (cnt <= 56) { buf |= (uint64_t)(pos < n ? p[pos] : 0) << cnt; ++pos; cnt += 8; } }
    BG_FN uint32_t used() const { return pos * 8 - cnt; }                   // bits consumed
    BG_FN bool over() const { return used() > n * 8; }                    // consumed a bit past the data
    BG_FN uint32_t peek(int k) const { return (uint32_t)(buf & ((1ull << k) - 1)); }
    BG_FN void drop(int k) { buf >>= k; cnt -= k; }
    BG_FN uint32_t take(int k) { const uint32_t v = peek(k); drop(k); return v; }   // caller has refilled
};

// canonical Huffman code (puff.c's layout) plus a direct table of the codes up to BG_FAST bits: fast[bits] = len << 9 | sym, 0 = longer
struct BgHuff { uint16_t count[16], offs[16], sym[288], fast[1 << BG_FAST]; };
struct BgTables { BgHuff lit, dist; uint8_t lens[320]; };   // one per member in flight (a warp's shared memory)

// the canonical walk over the low bits of `bits`, at most maxlen of them: symbol | len << 16, or -1 when no code matches
BG_FN int bg_walk(const BgHuff *h, uint32_t bits, int maxlen) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; ++len) {
        code |= (int)(bits & 1); bits >>= 1;
        const int count = h->count[len];
        if (code - count < first) return h->sym[index + (code - first)] | len << 16;
        index += count; first += count; first <<= 1; code <<= 1;
    }
    return -1;
}

// zlib's inflate_table rules: over-subscribed is an error; incomplete is an error for the code-length code, and for the
// others unless the code is one code of one bit; no code at all builds (any symbol decoded from it is an error)
template <class W> BG_FN bool bg_build(W &w, BgHuff *h, const uint8_t *len, int n, bool clcode) {
    if (w.lane == 0) {
        for (int l = 0; l < 16; ++l) h->count[l] = 0;
        for (int s = 0; s < n; ++s) h->count[len[s]]++;
    }
    w.sync();
    int left = 1, max = 0;
    for (int l = 1; l < 16; ++l) { left = (left << 1) - h->count[l]; if (h->count[l]) max = l; if (left < 0) return false; }
    if (max && left > 0 && (clcode || max != 1)) return false;
    if (w.lane == 0) {
        h->offs[1] = 0;
        for (int l = 1; l < 15; ++l) h->offs[l + 1] = h->offs[l] + h->count[l];
        for (int s = 0; s < n; ++s) if (len[s]) h->sym[h->offs[len[s]]++] = (uint16_t)s;
    }
    w.sync();
    for (int i = w.lane; i < (1 << BG_FAST); i += w.nl) {
        const int e = bg_walk(h, (uint32_t)i, BG_FAST);
        h->fast[i] = (uint16_t)(e < 0 ? 0 : (e >> 16) << 9 | (e & 0xffff));
    }
    w.sync();
    return true;
}

// one symbol; the caller has refilled (>= 57 bits buffered, a code is at most 15)
BG_FN int bg_decode(BgBits &b, const BgHuff *h) {
    const uint32_t e = h->fast[b.peek(BG_FAST)];
    if (e) { b.drop(e >> 9); return e & 511; }
    const int r = bg_walk(h, b.peek(15), 15);
    if (r < 0) return -1;
    b.drop(r >> 16);
    return r & 0xffff;
}

// the raw-deflate stream of b into w (w.pos counts the output so far)
template <class W> BG_FN int bg_inflate(W &w, BgBits &b, BgTables *t) {
    uint32_t last = 0;
    do {
        b.refill();
        if (b.over()) return BG_OVERRUN;
        last = b.take(1);
        const uint32_t type = b.take(2);
        if (type == 3) return BG_BTYPE;
        if (type == 0) {                                                  // stored: byte-aligned LEN, NLEN, LEN bytes
            b.drop(b.cnt & 7);
            const uint32_t len = b.take(16), nlen = b.take(16);
            if (b.over()) return BG_OVERRUN;
            if (len != (~nlen & 0xffff)) return BG_STORED_LEN;
            const uint32_t at = b.used() / 8;
            if (at + len > b.n) return BG_OVERRUN;
            if (int r = w.stored(b.p + at, len)) return r;
            b.pos = at + len; b.cnt = 0; b.buf = 0;
            continue;
        }
        if (type == 1) {                                                  // fixed codes (RFC 1951 §3.2.6)
            if (w.lane == 0) {
                for (int s = 0; s < 288; ++s) t->lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
                for (int s = 0; s < 32; ++s) t->lens[288 + s] = 5;
            }
            w.sync();
            bg_build(w, &t->lit, t->lens, 288, false);
            bg_build(w, &t->dist, t->lens + 288, 32, false);
        } else {                                                          // dynamic codes (§3.2.7)
            const int nlen = (int)b.take(5) + 257, ndist = (int)b.take(5) + 1, ncode = (int)b.take(4) + 4;
            if (nlen > 286 || ndist > 30) return BG_CODES;
            b.refill();
            if (w.lane == 0) for (int i = 0; i < 19; ++i) t->lens[BG_CLORDER[i]] = 0;
            w.sync();
            for (int i = 0; i < ncode; ++i) {                             // at most 57 bits: refill half way
                if (i == 10) b.refill();
                const uint32_t v = b.take(3);
                if (w.lane == 0) t->lens[BG_CLORDER[i]] = (uint8_t)v;
            }
            w.sync();
            if (!bg_build(w, &t->dist, t->lens, 19, true)) return BG_CODES;   // the code-length code, in the distance slot
            int i = 0, prev = -1;
            while (i < nlen + ndist) {
                b.refill();
                if (b.over()) return BG_OVERRUN;
                const int s = bg_decode(b, &t->dist);
                if (s < 0) return BG_BAD_CODE;
                int v = s, rep = 1;
                if (s == 16) { if (prev < 0) return BG_CODES; v = prev; rep = 3 + (int)b.take(2); }
                else if (s == 17) { v = 0; rep = 3 + (int)b.take(3); }
                else if (s == 18) { v = 0; rep = 11 + (int)b.take(7); }
                if (i + rep > nlen + ndist) return BG_CODES;
                if (w.lane == 0) for (int k = 0; k < rep; ++k) t->lens[i + k] = (uint8_t)v;
                i += rep; prev = v;
            }
            w.sync();
            if (t->lens[256] == 0) return BG_CODES;
            if (!bg_build(w, &t->lit, t->lens, nlen, false) || !bg_build(w, &t->dist, t->lens + nlen, ndist, false)) return BG_CODES;
        }
        while (true) {                                                    // symbols: at most 15 + 5 + 15 + 13 bits each
            b.refill();
            if (b.over()) return BG_OVERRUN;
            const int s = bg_decode(b, &t->lit);
            if (s < 0) return BG_BAD_CODE;
            if (s < 256) { if (int r = w.lit((uint32_t)s)) return r; continue; }
            if (s == 256) break;
            if (s > 285) return BG_SYMBOL;
            const uint32_t len = BG_LBASE[s - 257] + b.take(BG_LEXT[s - 257]);
            const int d = bg_decode(b, &t->dist);
            if (d < 0) return BG_BAD_CODE;
            if (d > 29) return BG_DIST_CODE;
            const uint32_t dist = BG_DBASE[d] + b.take(BG_DEXT[d]);
            if (int r = w.match(len, dist)) return r;
        }
    } while (!last);
    if (b.over()) return BG_OVERRUN;
    if ((b.used() + 7) / 8 != b.n) return BG_TRAILING;
    return BG_OK;
}

// a whole member (len bytes at m, the table's isize): header, deflate data, ISIZE and CRC-32 of the output
template <class W> BG_FN int bg_member(W &w, BgTables *t, const uint8_t *m, uint32_t len, uint32_t isize) {
    if (len < 20) return BG_HEADER;
    const uint32_t d0 = 12 + ((uint32_t)m[10] | (uint32_t)m[11] << 8);
    if (d0 + 8 > len) return BG_HEADER;
    const uint8_t *tr = m + len - 8;                                  // CRC-32, ISIZE
    if (((uint32_t)tr[4] | (uint32_t)tr[5] << 8 | (uint32_t)tr[6] << 16 | (uint32_t)tr[7] << 24) != isize) return BG_ISIZE;
    BgBits b; b.p = m + d0; b.n = len - d0 - 8; b.pos = 0; b.cnt = 0; b.buf = 0;
    if (int r = bg_inflate(w, b, t)) return r;
    w.flush();
    if (w.pos != isize) return BG_SHORT;
    const uint32_t crc = w.crc();
    return crc == ((uint32_t)tr[0] | (uint32_t)tr[1] << 8 | (uint32_t)tr[2] << 16 | (uint32_t)tr[3] << 24) ? BG_OK : BG_CRC;
}

// ---------------------------------------------------------------- CRC-32 (reflected, polynomial 0xEDB88320), zlib's combine
BG_FN uint32_t bg_crc_entry(uint32_t i) { for (int k = 0; k < 8; ++k) i = i & 1 ? (i >> 1) ^ 0xEDB88320u : i >> 1; return i; }
BG_FN uint32_t bg_multmodp(uint32_t a, uint32_t b) {                    // a * b mod P (zlib crc32.c)
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// x^(8 n) mod P from x2n[k] = x^(2^k) mod P: crc(A B) = multmodp(x^(8 |B|), crc(A)) ^ crc(B)
BG_FN uint32_t bg_x8nmodp(uint32_t n, const uint32_t *x2n) {
    uint32_t p = 1u << 31; int k = 3;
    while (n) { if (n & 1) p = bg_multmodp(x2n[k & 31], p); n >>= 1; ++k; }
    return p;
}
