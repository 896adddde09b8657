// bgzf_deflate.h — one BGZF member written (SAMv1 §4.1, RFC 1951): the parse, the per-member Huffman codes, the block-type
// choice, the dynamic header and the bit writer.  Written once and compiled twice: as CUDA in bgzf_deflate.cu, where one CTA
// writes one member, and as plain C++ in the host form tests/test_bgzf_deflate.py runs under AddressSanitizer.  A "team" T
// (the CTA on the device, one thread on the host) provides lane / nl / sync() for the steps that run on every thread.
//
// The compressed bytes are a function of the member's input bytes and of "stored only or not", nothing else:
//   parse     greedy.  The candidate of position i is the latest earlier position of the member whose 4 bytes hash like
//             those at i (head table of 2^BGD_HBITS entries, every position inserted in order), used when it lies within
//             32 768 bytes and its first 4 bytes equal those at i.  Its length is the common prefix, at most 258 bytes and
//             no further than the member's end.  Tokens start at 0 and at i + (match at i ? length : 1).
//   codes     Huffman code lengths per member (Moffat-Katajainen on the symbols sorted by (count, symbol)), limited to 15
//             bits (7 for the code-length code) by moving codes down from the longest lengths; every code has at least two
//             symbols, so every code is complete.
//   block     one block per member: stored, fixed or dynamic, whichever has the fewest bytes (ties in that order).  A stored
//             member is 65 311 bytes at most, under BGZF's 65 536.
// There is no lazy matching and no level knob: levels 1-9 all write these bytes, level 0 writes stored members.
#pragma once
#include "bgzf_member.h"

#define BGD_BLOCK  65280u                          // bgzip's member payload
#define BGD_STORED_MAX (BGD_BLOCK + 31u)           // 18-byte header, 5 bytes of stored-block framing, payload, 8-byte trailer
#define BGD_HBITS  14
#define BGD_NONE   0xffffu                         // an empty head-table slot (positions are < 65 280)
#define BGD_NL     286                             // literal/length symbols that may appear (0-285)
#define BGD_ND     30
#define BGD_NC     19

#ifdef __CUDACC__
BG_FN int bgd_log2(uint32_t x) { return 31 - __clz(x); }
#else
BG_FN int bgd_log2(uint32_t x) { return 31 - __builtin_clz(x); }
#endif

BG_FN uint32_t bgd_hash(const uint8_t *p) {
    const uint32_t x = (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24;
    return (x * 2654435761u) >> (32 - BGD_HBITS);
}

// length 3..258 -> symbol 257..285 and its extra bits (RFC 1951 §3.2.5), distance 1..32768 -> code 0..29
BG_FN void bgd_len_sym(uint32_t len, uint32_t &sym, uint32_t &ext, uint32_t &nb) {
    const uint32_t l = len - 3;
    if (len == 258) { sym = 285; ext = 0; nb = 0; }
    else if (l < 8) { sym = 257 + l; ext = 0; nb = 0; }
    else { nb = (uint32_t)bgd_log2(l) - 2; sym = 257 + 4 * nb + 4 + ((l >> nb) - 4); ext = l & ((1u << nb) - 1); }
}
BG_FN void bgd_dist_sym(uint32_t dist, uint32_t &sym, uint32_t &ext, uint32_t &nb) {
    const uint32_t d = dist - 1;
    if (d < 4) { sym = d; ext = 0; nb = 0; }
    else { nb = (uint32_t)bgd_log2(d) - 1; sym = 2 * nb + 2 + ((d >> nb) & 1); ext = d & ((1u << nb) - 1); }
}
BG_FN uint32_t bgd_fixed_len(int s) { return s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8; }
// the fixed literal/length code of RFC 1951 §3.2.6, bit-reversed.  Not the canonical code of the 286 lengths above: the fixed
// code also gives 8-bit codes to symbols 286 and 287, which shifts every 9-bit code (literals 144-255) by 4
BG_FN uint32_t bgd_fixed_code(int s) {
    uint32_t v = s < 144 ? 0x30 + s : s < 256 ? 0x190 + (s - 144) : s < 280 ? s - 256 : 0xc0 + (s - 280), r = 0;
    for (uint32_t b = 0; b < bgd_fixed_len(s); ++b) { r = r << 1 | (v & 1); v >>= 1; }
    return r;
}

// ---------------------------------------------------------------- the member's codes and block plan
struct BgdPlan {
    uint32_t fl[BGD_NL], fd[BGD_ND], fc[BGD_NC];   // symbol counts (fl[256] = 1: the end-of-block code)
    uint8_t ll[BGD_NL], ld[BGD_ND], lc[BGD_NC];    // code lengths of the chosen block type
    uint16_t cl[BGD_NL], cd[BGD_ND], cc[BGD_NC];   // their codes, bit-reversed for the LSB-first stream
    uint16_t rle[BGD_NL + BGD_ND];                 // the dynamic header's code-length symbols: symbol | extra << 5
    uint32_t key[BGD_NL]; uint16_t sym[BGD_NL];    // scratch of the length construction
    uint16_t cnt[16], next[16];
    uint32_t nrle, hlit, hdist, hclen;
    uint32_t btype;                                // 0 stored, 1 fixed, 2 dynamic
    uint32_t hdr_bits;                             // BFINAL + BTYPE + the dynamic header
    uint64_t bits;                                 // the whole deflate stream (not stored)
};

// Code lengths (at most maxlen bits) of the n symbols with counts f.  All threads of t call it; p->key / p->sym are scratch.
template <class T> BG_FN void bgd_lengths(T &t, BgdPlan *p, const uint32_t *f, int n, int maxlen, uint8_t *len) {
    // symbols in use, at least two (the lowest unused ones join with count 0), ranked by (count, symbol)
    if (t.lane == 0) {                                                 // len[s] = 1 marks "in use" until the lengths are known
        int used = 0;
        for (int s = 0; s < n; ++s) { len[s] = f[s] != 0; used += len[s]; }
        for (int s = 0; s < n && used < 2; ++s) if (!len[s]) { len[s] = 1; ++used; }
    }
    t.sync();
    int m = 0;
    for (int s = 0; s < n; ++s) m += len[s];
    for (int s = t.lane; s < n; s += t.nl) {
        if (!len[s]) continue;
        int r = 0;
        for (int q = 0; q < n; ++q) r += len[q] && (f[q] < f[s] || (f[q] == f[s] && q < s));
        p->key[r] = f[s]; p->sym[r] = (uint16_t)s;
    }
    t.sync();
    if (t.lane == 0) {
        uint32_t *A = p->key;
        // Moffat & Katajainen, in place: A ascending -> code length of each entry
        A[0] += A[1];
        int root = 0, leaf = 2;
        for (int nx = 1; nx < m - 1; ++nx) {
            if (leaf >= m || A[root] < A[leaf]) { A[nx] = A[root]; A[root++] = (uint32_t)nx; }
            else A[nx] = A[leaf++];
            if (leaf >= m || (root < nx && A[root] < A[leaf])) { A[nx] += A[root]; A[root++] = (uint32_t)nx; }
            else A[nx] += A[leaf++];
        }
        A[m - 2] = 0;
        for (int nx = m - 3; nx >= 0; --nx) A[nx] = A[A[nx]] + 1;
        int avbl = 1, used = 0, dpth = 0; root = m - 2; int nx = m - 1;
        while (avbl > 0) {
            while (root >= 0 && (int)A[root] == dpth) { ++used; --root; }
            while (avbl > used) { A[nx--] = (uint32_t)dpth; --avbl; }
            avbl = 2 * used; ++dpth; used = 0;
        }
        // lengths past maxlen clamp to maxlen; then codes move down one level at a time until the Kraft sum is exactly 1
        for (int l = 0; l < 16; ++l) p->cnt[l] = 0;
        for (int k = 0; k < m; ++k) p->cnt[A[k] < (uint32_t)maxlen ? A[k] : (uint32_t)maxlen]++;
        uint32_t total = 0;
        for (int l = maxlen; l > 0; --l) total += (uint32_t)p->cnt[l] << (maxlen - l);
        while (total != (1u << maxlen)) {
            p->cnt[maxlen]--;
            for (int l = maxlen - 1; l > 0; --l) if (p->cnt[l]) { p->cnt[l]--; p->cnt[l + 1] += 2; break; }
            --total;
        }
        for (int s = 0; s < n; ++s) len[s] = 0;
        for (int l = 1, j = m; l <= maxlen; ++l)                        // the most frequent symbols get the shortest codes
            for (int c = p->cnt[l]; c > 0; --c) len[p->sym[--j]] = (uint8_t)l;
    }
    t.sync();
}

// canonical codes of the lengths, bit-reversed (one thread)
BG_FN void bgd_codes(BgdPlan *p, const uint8_t *len, int n, uint16_t *code) {
    for (int l = 0; l < 16; ++l) p->cnt[l] = 0;
    for (int s = 0; s < n; ++s) p->cnt[len[s]]++;
    p->cnt[0] = 0;
    uint32_t c = 0;
    for (int l = 1; l < 16; ++l) { c = (c + p->cnt[l - 1]) << 1; p->next[l] = (uint16_t)c; }
    for (int s = 0; s < n; ++s) {
        const int l = len[s];
        if (!l) { code[s] = 0; continue; }
        uint32_t v = p->next[l]++, r = 0;
        for (int b = 0; b < l; ++b) { r = r << 1 | (v & 1); v >>= 1; }
        code[s] = (uint16_t)r;
    }
}

// The block for a member of n input bytes whose counts p->fl / p->fd are final.  All threads call it.
template <class T> BG_FN void bgd_plan(T &t, BgdPlan *p, uint32_t n) {
    bgd_lengths(t, p, p->fl, BGD_NL, 15, p->ll);
    bgd_lengths(t, p, p->fd, BGD_ND, 15, p->ld);
    if (t.lane == 0) {
        uint32_t hl = BGD_NL, hd = BGD_ND;
        while (hl > 257 && !p->ll[hl - 1]) --hl;
        while (hd > 1 && !p->ld[hd - 1]) --hd;
        p->hlit = hl; p->hdist = hd;
        // run-length code of the hl + hd lengths (one sequence: runs cross from the literal/length into the distance lengths)
        for (int s = 0; s < BGD_NC; ++s) p->fc[s] = 0;
        uint32_t nr = 0, i = 0;
        const uint32_t tot = hl + hd;
        while (i < tot) {
            const uint32_t v = i < hl ? p->ll[i] : p->ld[i - hl];
            uint32_t r = 1;
            while (i + r < tot && (i + r < hl ? p->ll[i + r] : p->ld[i + r - hl]) == v) ++r;
            uint32_t rem = r;
            if (v == 0) {
                while (rem >= 11) { const uint32_t k = rem < 138 ? rem : 138; p->rle[nr++] = (uint16_t)(18 | (k - 11) << 5); p->fc[18]++; rem -= k; }
                if (rem >= 3) { p->rle[nr++] = (uint16_t)(17 | (rem - 3) << 5); p->fc[17]++; rem = 0; }
            } else {
                p->rle[nr++] = (uint16_t)v; p->fc[v]++; --rem;
                while (rem >= 3) { const uint32_t k = rem < 6 ? rem : 6; p->rle[nr++] = (uint16_t)(16 | (k - 3) << 5); p->fc[16]++; rem -= k; }
            }
            while (rem) { p->rle[nr++] = (uint16_t)v; p->fc[v]++; --rem; }
            i += r;
        }
        p->nrle = nr;
    }
    t.sync();
    bgd_lengths(t, p, p->fc, BGD_NC, 7, p->lc);
    if (t.lane == 0) {
        uint32_t hc = BGD_NC;
        while (hc > 4 && !p->lc[BG_CLORDER[hc - 1]]) --hc;
        p->hclen = hc;
        uint64_t extra = 0, dyn = 0, fix = 0;
        for (int s = 0; s < BGD_NL; ++s) {
            dyn += (uint64_t)p->fl[s] * p->ll[s]; fix += (uint64_t)p->fl[s] * bgd_fixed_len(s);
            if (s > 256) extra += (uint64_t)p->fl[s] * BG_LEXT[s - 257];
        }
        for (int s = 0; s < BGD_ND; ++s) { dyn += (uint64_t)p->fd[s] * p->ld[s]; fix += (uint64_t)p->fd[s] * 5; extra += (uint64_t)p->fd[s] * BG_DEXT[s]; }
        uint32_t hdr = 3 + 14 + 3 * hc;
        for (uint32_t k = 0; k < p->nrle; ++k) {
            const uint32_t s = p->rle[k] & 31;
            hdr += p->lc[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        dyn += extra + hdr; fix += extra + 3;
        const uint64_t stored = 8ull * (n + 5);
        if (stored <= (fix + 7) / 8 * 8 && stored <= (dyn + 7) / 8 * 8) { p->btype = 0; p->bits = stored; p->hdr_bits = 0; }
        else if ((fix + 7) / 8 <= (dyn + 7) / 8) {
            p->btype = 1; p->bits = fix; p->hdr_bits = 3;
            for (int s = 0; s < BGD_NL; ++s) p->ll[s] = (uint8_t)bgd_fixed_len(s);
            for (int s = 0; s < BGD_ND; ++s) p->ld[s] = 5;
        } else { p->btype = 2; p->bits = dyn; p->hdr_bits = hdr; }
        if (p->btype == 1) for (int s = 0; s < BGD_NL; ++s) p->cl[s] = (uint16_t)bgd_fixed_code(s);
        if (p->btype == 2) bgd_codes(p, p->ll, BGD_NL, p->cl);
        if (p->btype) { bgd_codes(p, p->ld, BGD_ND, p->cd); bgd_codes(p, p->lc, BGD_NC, p->cc); }
    }
    t.sync();
}

// ---------------------------------------------------------------- bit writer
// LSB-first bits from bit offset `at` of a word array.  S::word(i, v, shared) receives every word the writer touches, with
// shared = the word may also hold another writer's bits (the first word when `at` is not word-aligned, and the last one):
// the device ORs those in (the result does not depend on which writer comes first) and stores the others.
template <class S> struct BgdBits {
    S s; uint64_t acc; uint32_t nacc, word; bool first;
    BG_FN void init(uint64_t at) { acc = 0; nacc = (uint32_t)(at & 31); word = (uint32_t)(at >> 5); first = nacc != 0; }
    BG_FN void put(uint32_t v, uint32_t nb) {                      // nb <= 32
        acc |= (uint64_t)v << nacc; nacc += nb;
        if (nacc >= 32) { s.word(word++, (uint32_t)acc, first); first = false; acc >>= 32; nacc -= 32; }
    }
    BG_FN void finish() { if (acc) s.word(word, (uint32_t)acc, true); }
};

template <class B> BG_FN void bgd_put_header(B &b, const BgdPlan *p) {
    b.put(1 | p->btype << 1, 3);                                   // BFINAL, BTYPE
    if (p->btype != 2) return;
    b.put(p->hlit - 257, 5); b.put(p->hdist - 1, 5); b.put(p->hclen - 4, 4);
    for (uint32_t k = 0; k < p->hclen; ++k) b.put(p->lc[BG_CLORDER[k]], 3);
    for (uint32_t k = 0; k < p->nrle; ++k) {
        const uint32_t s = p->rle[k] & 31, x = p->rle[k] >> 5;
        b.put(p->cc[s], p->lc[s]);
        if (s >= 16) b.put(x, s == 16 ? 2 : s == 17 ? 3 : 7);
    }
}
BG_FN uint32_t bgd_lit_bits(const BgdPlan *p, uint32_t c) { return p->ll[c]; }
BG_FN uint32_t bgd_match_bits(const BgdPlan *p, uint32_t len, uint32_t dist) {
    uint32_t ls, le, ln, ds, de, dn;
    bgd_len_sym(len, ls, le, ln); bgd_dist_sym(dist, ds, de, dn);
    return p->ll[ls] + ln + p->ld[ds] + dn;
}
template <class B> BG_FN void bgd_put_lit(B &b, const BgdPlan *p, uint32_t c) { b.put(p->cl[c], p->ll[c]); }
template <class B> BG_FN void bgd_put_match(B &b, const BgdPlan *p, uint32_t len, uint32_t dist) {
    uint32_t ls, le, ln, ds, de, dn;
    bgd_len_sym(len, ls, le, ln); bgd_dist_sym(dist, ds, de, dn);
    b.put(p->cl[ls], p->ll[ls]); if (ln) b.put(le, ln);
    b.put(p->cd[ds], p->ld[ds]); if (dn) b.put(de, dn);
}

// bgzip's 18 header bytes (BSIZE = total member bytes - 1) and the trailer
BG_FN void bgd_member_header(uint8_t *m, uint32_t total) {
    const uint8_t h[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    for (int k = 0; k < 16; ++k) m[k] = h[k];
    m[16] = (uint8_t)((total - 1) & 0xff); m[17] = (uint8_t)((total - 1) >> 8);
}
BG_FN void bgd_put32(uint8_t *q, uint32_t v) { q[0] = (uint8_t)v; q[1] = (uint8_t)(v >> 8); q[2] = (uint8_t)(v >> 16); q[3] = (uint8_t)(v >> 24); }

#ifndef __CUDACC__
// ---------------------------------------------------------------- the host form: one member, one thread, the same bytes
struct BgdHostTeam { int lane = 0, nl = 1; void sync() {} };
struct BgdHostSink { uint32_t *w; void word(uint32_t i, uint32_t v, bool) { w[i] |= v; } };

// the parse of the header comment: tok[i] = length | (distance - 1) << 16 at a match start, 0 at a literal; start[i] = 1 at a token
static inline void bgd_parse_host(const uint8_t *in, uint32_t n, uint16_t *head, uint32_t *tok, uint8_t *start) {
    for (uint32_t h = 0; h < (1u << BGD_HBITS); ++h) head[h] = BGD_NONE;
    uint32_t next = 0;
    for (uint32_t i = 0; i < n; ++i) {
        uint32_t c = BGD_NONE;
        if (i + 4 <= n) { const uint32_t h = bgd_hash(in + i); c = head[h]; head[h] = (uint16_t)i; }
        tok[i] = 0; start[i] = i == next;
        if (i != next) continue;
        if (c != BGD_NONE && i - c <= 32768 && !memcmp(in + c, in + i, 4)) {
            const uint32_t maxl = n - i < 258 ? n - i : 258;
            uint32_t l = 4;
            while (l < maxl && in[c + l] == in[i + l]) ++l;
            tok[i] = l | (i - c - 1) << 16; next = i + l;
        } else next = i + 1;
    }
}

// one member of n <= BGD_BLOCK bytes into out (BGD_STORED_MAX bytes): -> member bytes
static inline uint32_t bgd_member_host(const uint8_t *in, uint32_t n, bool stored_only, uint8_t *out) {
    BgdHostTeam t;
    BgdPlan *p = new BgdPlan();
    uint16_t *head = new uint16_t[1u << BGD_HBITS];
    uint32_t *tok = new uint32_t[n + 1]; uint8_t *start = new uint8_t[n + 1];
    uint32_t *w = new uint32_t[(BGD_STORED_MAX + 3) / 4 + 1]();
    uint32_t crc = 0xffffffffu;
    for (uint32_t i = 0; i < n; ++i) crc = bg_crc_entry((crc ^ in[i]) & 0xff) ^ (crc >> 8);
    crc = ~crc;
    uint32_t dbytes;
    if (stored_only) p->btype = 0;
    else {
        bgd_parse_host(in, n, head, tok, start);
        for (uint32_t i = 0; i < n; ++i) {
            if (!start[i]) continue;
            if (!tok[i]) { p->fl[in[i]]++; continue; }
            uint32_t s, e, nb;
            bgd_len_sym(tok[i] & 0xffff, s, e, nb); p->fl[s]++;
            bgd_dist_sym((tok[i] >> 16) + 1, s, e, nb); p->fd[s]++;
        }
        p->fl[256] = 1;
        bgd_plan(t, p, n);
    }
    uint8_t *d = out + 18;
    if (p->btype == 0) {
        d[0] = 1; d[1] = (uint8_t)n; d[2] = (uint8_t)(n >> 8); d[3] = (uint8_t)~n; d[4] = (uint8_t)(~n >> 8);
        if (n) memcpy(d + 5, in, n);
        dbytes = n + 5;
    } else {
        BgdBits<BgdHostSink> b; b.s.w = w; b.init(0);
        bgd_put_header(b, p);
        for (uint32_t i = 0; i < n; ++i) {
            if (!start[i]) continue;
            if (tok[i]) bgd_put_match(b, p, tok[i] & 0xffff, (tok[i] >> 16) + 1); else bgd_put_lit(b, p, in[i]);
        }
        bgd_put_lit(b, p, 256);
        b.finish();
        dbytes = (uint32_t)((p->bits + 7) / 8);
        for (uint32_t k = 0; k < dbytes; ++k) d[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
    }
    const uint32_t total = 18 + dbytes + 8;
    bgd_member_header(out, total);
    bgd_put32(out + 18 + dbytes, crc); bgd_put32(out + 22 + dbytes, n);
    delete p; delete[] head; delete[] tok; delete[] start; delete[] w;
    return total;
}
#endif
