// bam_encode.h — one SAM line to one BAM record (SAMv1 §1.4, §4.2): the field tokeniser, the checks, the record bytes and the
// sort key.  Written once and compiled twice: as CUDA in bam_out.cu, where one thread encodes one line (a size pass and a
// write pass over the same code), and as plain C++ in the host form tests/test_bam_encode.py runs under AddressSanitizer.
//
// The bytes are those of tests/bam_writer.encode_records, except that a flag-4 record with a CIGAR gets
// bin = reg2bin(pos, pos + 1) (the SAMv1 rule for unmapped records).  Float values (`f` tags, `B:f` items) are converted
// exactly on the device only on the fast path (an integer mantissa of at most 2^24 and a decimal exponent of at most 10 in
// magnitude: one correctly rounded float multiply or divide, so the result equals strtof); any other value is marked, and
// the library re-encodes the marked lines on the host with strtof.  The record length does not depend on the values.
#pragma once
#include <stdint.h>
#ifdef __CUDACC__
#define BE_FN __host__ __device__ inline
#else
#define BE_FN inline
#endif
#ifndef __CUDA_ARCH__
#include <stdlib.h>
#include <string.h>
#include <string>
#endif

#define BE_REC_FIXED 36u                 // block_size .. tlen
#define BE_MAX_QNAME 254u
#define BE_MAX_CIGAR 65535u
#define BE_MIN_LINE 21u                  // 11 non-empty fields and 10 tabs: a shorter line is refused

// per-line refusals; the codes index be_errstr
enum {
    BE_OK = 0, BE_EFIELDS, BE_EQNAME, BE_EFLAG, BE_ERNAME, BE_EPOS, BE_EMAPQ, BE_ECIGAR, BE_ENCIGAR, BE_ERNEXT, BE_EPNEXT,
    BE_ETLEN, BE_EQUAL, BE_ETAG, BE_ETAGTYPE, BE_EBSUB, BE_EINT, BE_EFLOAT, BE_EPOS0, BE_EHEADER, BE_NERR
};
static const char *const be_errstr[BE_NERR] = {
    "ok", "fewer than 11 fields", "QNAME empty or longer than 254", "bad FLAG", "RNAME not in @SQ", "bad POS", "bad MAPQ",
    "bad CIGAR", "more than 65535 CIGAR operations", "RNEXT not in @SQ", "bad PNEXT", "bad TLEN",
    "QUAL length differs from SEQ or a bad QUAL character", "malformed tag", "unknown tag type", "unknown B subtype",
    "integer tag value out of range", "bad float value", "RNAME set with POS 0", "header line after the first record"};

// the reference dictionary: names back to back (name k = names[off[k], off[k+1])), an open-addressing table of 2^bits slots
// holding tid + 1 (0 = empty), probed linearly from the name's FNV-1a hash
struct BeDict {
    const char *names;
    const uint32_t *off;
    const int32_t *slot;
    uint32_t mask;
    int32_t n_refs;
};

BE_FN uint32_t be_hash(const char *s, uint32_t n) {
    uint32_t h = 2166136261u;
    for (uint32_t i = 0; i < n; ++i) h = (h ^ (uint8_t)s[i]) * 16777619u;
    return h;
}

BE_FN int32_t be_lookup(const BeDict &d, const char *s, uint32_t n) {       // -1 when absent
    for (uint32_t h = be_hash(s, n) & d.mask;; h = (h + 1) & d.mask) {
        const int32_t v = d.slot[h];
        if (!v) return -1;
        const uint32_t a = d.off[v - 1], b = d.off[v];
        if (b - a == n) {
            uint32_t i = 0;
            while (i < n && d.names[a + i] == s[i]) ++i;
            if (i == n) return v - 1;
        }
    }
}

// UCSC binning scheme (SAMv1 §5.3): the smallest bin holding [beg, end)
BE_FN uint32_t be_reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (uint32_t)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (uint32_t)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (uint32_t)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (uint32_t)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (uint32_t)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

// htslib's seq_nt16_table: "=ACMGRSVTWYHKDBN" in either case, anything else 15 (N)
BE_FN uint32_t be_nt16(uint8_t c) {
    if (c >= 'a' && c <= 'z') c -= 32;
    switch (c) {
    case '=': return 0; case 'A': return 1; case 'C': return 2; case 'M': return 3; case 'G': return 4; case 'R': return 5;
    case 'S': return 6; case 'V': return 7; case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11;
    case 'K': return 12; case 'D': return 13; case 'B': return 14; default: return 15;
    }
}

BE_FN int be_cigar_op(uint8_t c) {
    switch (c) {
    case 'M': return 0; case 'I': return 1; case 'D': return 2; case 'N': return 3; case 'S': return 4; case 'H': return 5;
    case 'P': return 6; case '=': return 7; case 'X': return 8; default: return -1;
    }
}

// decimal integer over [s, e): optional '-' when neg_ok, at least one digit, nothing else; false past |v| > 2^40
BE_FN bool be_int(const char *s, const char *e, bool neg_ok, int64_t &v) {
    bool neg = false;
    if (s < e && *s == '-' && neg_ok) { neg = true; ++s; }
    if (s == e) return false;
    int64_t x = 0;
    for (; s < e; ++s) {
        const uint32_t d = (uint32_t)(uint8_t)*s - '0';
        if (d > 9 || x > (1ll << 40)) return false;
        x = x * 10 + d;
    }
    v = neg ? -x : x;
    return true;
}

// 0 = the exact fast path gave *f; 1 = a value strtof takes that is off the fast path (nan, inf, long mantissa, large
// exponent); 2 = not a float
BE_FN int be_float_fast(const char *s, const char *e, float &f) {
    const char *p = s;
    bool neg = false;
    if (p < e && (*p == '+' || *p == '-')) neg = *p++ == '-';
    uint64_t m = 0;
    int nd = 0, sig = 0, ex = 0;
    bool big = false;
    for (; p < e && (uint32_t)(uint8_t)*p - '0' <= 9; ++p, ++nd) {
        if (sig < 19) { m = m * 10 + (*p - '0'); if (m) ++sig; } else { big = true; ++ex; }
    }
    if (p < e && *p == '.') {
        for (++p; p < e && (uint32_t)(uint8_t)*p - '0' <= 9; ++p, ++nd) {
            if (sig < 19) { m = m * 10 + (*p - '0'); if (m) ++sig; --ex; } else big = true;
        }
    }
    if (nd == 0) {                                                  // nan, inf, infinity in any case
        uint32_t n = (uint32_t)(e - p);
        char w[8];
        if (n != 3 && n != 8) return 2;
        for (uint32_t i = 0; i < n; ++i) w[i] = (char)(p[i] | 32);
        const bool nan = n == 3 && w[0] == 'n' && w[1] == 'a' && w[2] == 'n', inf = w[0] == 'i' && w[1] == 'n' && w[2] == 'f';
        if (nan || (inf && n == 3)) return 1;
        if (inf && w[3] == 'i' && w[4] == 'n' && w[5] == 'i' && w[6] == 't' && w[7] == 'y') return 1;
        return 2;
    }
    if (p < e && (*p == 'e' || *p == 'E')) {
        ++p;
        bool eneg = false;
        if (p < e && (*p == '+' || *p == '-')) eneg = *p++ == '-';
        if (p == e) return 2;
        int x = 0;
        for (; p < e; ++p) {
            const uint32_t d = (uint32_t)(uint8_t)*p - '0';
            if (d > 9) return 2;
            if (x < 100000) x = x * 10 + (int)d;
        }
        ex += eneg ? -x : x;
    }
    if (p != e) return 2;
    if (m == 0) { f = neg ? -0.0f : 0.0f; return 0; }
    if (big) return 1;
    while (m % 10 == 0) { m /= 10; ++ex; }
    if (m > (1u << 24) || ex > 10 || ex < -10) return 1;
    const float p10[11] = {1e0f, 1e1f, 1e2f, 1e3f, 1e4f, 1e5f, 1e6f, 1e7f, 1e8f, 1e9f, 1e10f};
    float v = (float)m;
    v = ex >= 0 ? v * p10[ex] : v / p10[-ex];
    f = neg ? -v : v;
    return 0;
}

// where the bytes go: W = false only counts them (the size pass), W = true stores them
template <bool W> struct BeOut {
    uint8_t *p;
    uint32_t at;
    BE_FN void u8(uint32_t v) { if (W) p[at] = (uint8_t)v; at += 1; }
    BE_FN void u16(uint32_t v) { if (W) { p[at] = (uint8_t)v; p[at + 1] = (uint8_t)(v >> 8); } at += 2; }
    BE_FN void u32(uint32_t v) { if (W) { p[at] = (uint8_t)v; p[at + 1] = (uint8_t)(v >> 8); p[at + 2] = (uint8_t)(v >> 16); p[at + 3] = (uint8_t)(v >> 24); } at += 4; }
    BE_FN void put32(uint32_t o, uint32_t v) { if (W) { p[o] = (uint8_t)v; p[o + 1] = (uint8_t)(v >> 8); p[o + 2] = (uint8_t)(v >> 16); p[o + 3] = (uint8_t)(v >> 24); } }
    BE_FN void put16(uint32_t o, uint32_t v) { if (W) { p[o] = (uint8_t)v; p[o + 1] = (uint8_t)(v >> 8); } }
};

// one float value: the fast path, or (exact) strtof on the host, or a mark (*patch) and 0 in its place
template <bool W> BE_FN int be_put_float(BeOut<W> &o, const char *s, const char *e, bool exact, bool *patch) {
    float f = 0;
    const int r = be_float_fast(s, e, f);
    if (r == 2) return BE_EFLOAT;
    if (r == 1) {
#ifndef __CUDA_ARCH__
        if (exact) {
            std::string t(s, e);
            char *end = NULL;
            f = strtof(t.c_str(), &end);
            if (end != t.c_str() + t.size()) return BE_EFLOAT;
        } else *patch = true;
#else
        *patch = true;
#endif
    }
    uint32_t u;
    memcpy(&u, &f, 4);
    o.u32(u);
    return BE_OK;
}

// the next field of the line [*p, e): its bounds, *p past its tab; false when the line has no more fields
BE_FN bool be_field(const char *&p, const char *e, const char *&fb, const char *&fe, bool &more) {
    if (!more) return false;
    fb = p;
    while (p < e && *p != '\t') ++p;
    fe = p;
    more = p < e;
    if (more) ++p;
    return true;
}

// One SAM line (without its newline) -> one BAM record at o (block_size included).  Returns BE_OK or the refusal code.
// exact: convert every float on the host with strtof (host only); otherwise a float off the fast path sets *patch.
template <bool W> BE_FN int be_line(const char *s, uint32_t n, const BeDict &d, bool exact, BeOut<W> &o, bool *patch) {
    if (n && s[0] == '@') return BE_EHEADER;
    if (n < BE_MIN_LINE) return BE_EFIELDS;
    const char *p = s, *e = s + n;
    const char *fb[11], *fe[11];
    bool more = true;
    for (int k = 0; k < 11; ++k)
        if (!be_field(p, e, fb[k], fe[k], more)) return BE_EFIELDS;
    for (int k = 0; k < 11; ++k)
        if (fb[k] == fe[k]) return BE_EFIELDS;
    const uint32_t l_name = (uint32_t)(fe[0] - fb[0]);
    if (l_name > BE_MAX_QNAME) return BE_EQNAME;
    int64_t flag, pos, mapq, pnext, tlen;
    if (!be_int(fb[1], fe[1], false, flag) || flag > 65535) return BE_EFLAG;
    int32_t tid = -1;
    if (!(fe[2] - fb[2] == 1 && *fb[2] == '*')) { tid = be_lookup(d, fb[2], (uint32_t)(fe[2] - fb[2])); if (tid < 0) return BE_ERNAME; }
    if (!be_int(fb[3], fe[3], false, pos) || pos > 2147483647ll) return BE_EPOS;
    if (tid >= 0 && pos == 0) return BE_EPOS0;
    if (!be_int(fb[4], fe[4], false, mapq) || mapq > 255) return BE_EMAPQ;
    int32_t ntid = -1;
    if (fe[6] - fb[6] == 1 && *fb[6] == '=') ntid = tid;
    else if (!(fe[6] - fb[6] == 1 && *fb[6] == '*')) { ntid = be_lookup(d, fb[6], (uint32_t)(fe[6] - fb[6])); if (ntid < 0) return BE_ERNEXT; }
    if (!be_int(fb[7], fe[7], false, pnext) || pnext > 2147483647ll) return BE_EPNEXT;
    if (!be_int(fb[8], fe[8], true, tlen) || tlen > 2147483647ll || tlen < -2147483647ll - 1) return BE_ETLEN;
    const uint32_t r0 = o.at;
    o.at += BE_REC_FIXED;
    for (uint32_t i = 0; i < l_name; ++i) o.u8((uint8_t)fb[0][i]);
    o.u8(0);
    // CIGAR
    uint32_t n_cig = 0;
    int64_t reflen = 0;
    if (!(fe[5] - fb[5] == 1 && *fb[5] == '*')) {
        for (const char *c = fb[5]; c < fe[5];) {
            int64_t len = 0;
            const char *c0 = c;
            while (c < fe[5] && (uint32_t)(uint8_t)*c - '0' <= 9) { len = len * 10 + (*c - '0'); if (len >= (1 << 28)) return BE_ECIGAR; ++c; }
            if (c == c0 || c == fe[5]) return BE_ECIGAR;
            const int op = be_cigar_op((uint8_t)*c++);
            if (op < 0) return BE_ECIGAR;
            if (++n_cig > BE_MAX_CIGAR) return BE_ENCIGAR;
            if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) reflen += len;
            o.u32((uint32_t)len << 4 | (uint32_t)op);
        }
    }
    // SEQ, QUAL
    const bool no_seq = fe[9] - fb[9] == 1 && *fb[9] == '*';
    const uint32_t l_seq = no_seq ? 0 : (uint32_t)(fe[9] - fb[9]);
    for (uint32_t i = 0; i < l_seq; i += 2) {
        const uint32_t hi = be_nt16((uint8_t)fb[9][i]), lo = i + 1 < l_seq ? be_nt16((uint8_t)fb[9][i + 1]) : 0;
        o.u8(hi << 4 | lo);
    }
    if (fe[10] - fb[10] == 1 && *fb[10] == '*') {
        for (uint32_t i = 0; i < l_seq; ++i) o.u8(0xff);
    } else {
        if ((uint32_t)(fe[10] - fb[10]) != l_seq) return BE_EQUAL;
        for (uint32_t i = 0; i < l_seq; ++i) {
            const uint8_t q = (uint8_t)fb[10][i];
            if (q < 33 || q > 126) return BE_EQUAL;
            o.u8(q - 33);
        }
    }
    // tags
    const char *tb, *te;
    while (be_field(p, e, tb, te, more)) {
        if (te - tb < 5 || tb[2] != ':' || tb[4] != ':') return BE_ETAG;
        const char typ = tb[3], *v = tb + 5;
        o.u8((uint8_t)tb[0]); o.u8((uint8_t)tb[1]);
        if (typ == 'i') {
            int64_t x;
            if (!be_int(v, te, true, x) && !(v < te && *v == '+' && be_int(v + 1, te, false, x))) return BE_ETAG;
            if (x < -2147483648ll || x > 4294967295ll) return BE_EINT;
            if (x < 0) {
                if (x >= -128) { o.u8('c'); o.u8((uint32_t)x); }
                else if (x >= -32768) { o.u8('s'); o.u16((uint32_t)x); }
                else { o.u8('i'); o.u32((uint32_t)x); }
            } else if (x < 256) { o.u8('C'); o.u8((uint32_t)x); }
            else if (x < 65536) { o.u8('S'); o.u16((uint32_t)x); }
            else { o.u8('I'); o.u32((uint32_t)x); }
        } else if (typ == 'A') {
            if (te - v != 1) return BE_ETAG;
            o.u8('A'); o.u8((uint8_t)*v);
        } else if (typ == 'f') {
            o.u8('f');
            const int r = be_put_float(o, v, te, exact, patch);
            if (r) return r;
        } else if (typ == 'Z' || typ == 'H') {
            o.u8((uint8_t)typ);
            for (const char *c = v; c < te; ++c) o.u8((uint8_t)*c);
            o.u8(0);
        } else if (typ == 'B') {
            if (v == te) return BE_ETAG;
            const char sub = *v;
            int64_t lo = 0, hi = 0;
            uint32_t w = 0;
            switch (sub) {
            case 'c': lo = -128; hi = 127; w = 1; break;
            case 'C': lo = 0; hi = 255; w = 1; break;
            case 's': lo = -32768; hi = 32767; w = 2; break;
            case 'S': lo = 0; hi = 65535; w = 2; break;
            case 'i': lo = -2147483648ll; hi = 2147483647ll; w = 4; break;
            case 'I': lo = 0; hi = 4294967295ll; w = 4; break;
            case 'f': w = 4; break;
            default: return BE_EBSUB;
            }
            o.u8('B'); o.u8((uint8_t)sub);
            const uint32_t at_n = o.at;
            o.at += 4;
            uint32_t cnt = 0;
            const char *c = v + 1;
            if (c < te && *c != ',') return BE_ETAG;
            while (c < te) {
                const char *ib = ++c;
                while (c < te && *c != ',') ++c;
                ++cnt;
                if (sub == 'f') {
                    const int r = be_put_float(o, ib, c, exact, patch);
                    if (r) return r;
                } else {
                    int64_t x;
                    if (!be_int(ib, c, true, x) && !(ib < c && *ib == '+' && be_int(ib + 1, c, false, x))) return BE_ETAG;
                    if (x < lo || x > hi) return BE_EINT;
                    if (w == 1) o.u8((uint32_t)x); else if (w == 2) o.u16((uint32_t)x); else o.u32((uint32_t)x);
                }
            }
            o.put32(at_n, cnt);
        } else return BE_ETAGTYPE;
    }
    // the fixed part
    const int64_t p0 = pos - 1;
    const uint32_t bin = p0 < 0 ? 4680u : be_reg2bin(p0, p0 + ((flag & 4) || reflen == 0 ? 1 : reflen));
    o.put32(r0, o.at - r0 - 4);
    o.put32(r0 + 4, (uint32_t)tid);
    o.put32(r0 + 8, (uint32_t)p0);
    if (W) { o.p[r0 + 12] = (uint8_t)(l_name + 1); o.p[r0 + 13] = (uint8_t)mapq; }
    o.put16(r0 + 14, bin);
    o.put16(r0 + 16, n_cig);
    o.put16(r0 + 18, (uint32_t)flag);
    o.put32(r0 + 20, l_seq);
    o.put32(r0 + 24, (uint32_t)ntid);
    o.put32(r0 + 28, (uint32_t)(pnext - 1));
    o.put32(r0 + 32, (uint32_t)tlen);
    return BE_OK;
}

BE_FN uint32_t be_rd32(const uint8_t *r) { return (uint32_t)r[0] | (uint32_t)r[1] << 8 | (uint32_t)r[2] << 16 | (uint32_t)r[3] << 24; }

// the coordinate sort key of a record (samtools' comparator): tid with -1 after every reference, pos + 1, the reverse flag.
// key_hi = tid', key_lo = (pos + 1) << 1 | rev
BE_FN void be_key(const uint8_t *r, int32_t n_refs, uint32_t &key_hi, uint32_t &key_lo) {
    const int32_t tid = (int32_t)be_rd32(r + 4), pos = (int32_t)be_rd32(r + 8);
    const uint32_t flag = (uint32_t)r[18] | (uint32_t)r[19] << 8;
    key_hi = tid < 0 ? (uint32_t)n_refs : (uint32_t)tid;
    key_lo = (uint32_t)(pos + 1) << 1 | (flag >> 4 & 1);
}

// the record's end for the index: pos + reference length, or pos + 1 when that length is 0 or flag 4 is set
BE_FN int64_t be_end(const uint8_t *r) {
    const int64_t pos = (int32_t)be_rd32(r + 8);
    const uint32_t l_name = r[12], n_cig = (uint32_t)r[16] | (uint32_t)r[17] << 8, flag = (uint32_t)r[18] | (uint32_t)r[19] << 8;
    int64_t len = 0;
    const uint8_t *c = r + BE_REC_FIXED + l_name;
    for (uint32_t k = 0; k < n_cig; ++k) {
        const uint32_t v = be_rd32(c + 4 * k), op = v & 15;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) len += v >> 4;
    }
    return pos + ((flag & 4) || len == 0 ? 1 : len);
}
