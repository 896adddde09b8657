// hic_writer.hpp — host-side `.hic` (version 8) container writer fed by the per-resolution COO triplets of the binning path
// (SURVEY.md §8(f)-3; stands where the driver runs `java -jar juicer_tools.jar pre -r <res,...> <sid>.final.pairs <sid>.hic
// <genome>.info`, microcket:525-529).  Host code only: the counting is done on the GPU (pairs.cu / hist.cu), this file
// lays the counts out in the container: header, one matrix per chromosome pair with every resolution's compressed blocks,
// footer with the master index and the expected-value vectors, and — when normalisation vectors are handed in with a
// resolution (norm.cu) — the normalised expected values and the vectors themselves.
//
// PARITY UNPINNED: juicer_tools is a third-party jar that is not in /root/reference and cannot run here (SURVEY §8c); the
// layout follows the published .hic v8 format description and is read back in tests/ by an independent reader written from
// the same description (tests/hic_reader.py).  Choices a reader does not depend on (block grid, list-of-rows blocks only,
// which statistics are filled) are stated where they are made.
#pragma once
#include <zlib.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace hic {

struct Rec { uint32_t x, y, c; };            // x: bin on the first chromosome (column), y: bin on the second (row)

struct Buf {                                 // little-endian byte sink
    std::vector<unsigned char> v;
    void raw(const void *p, size_t n) { const unsigned char *b = (const unsigned char *)p; v.insert(v.end(), b, b + n); }
    void i8(int x) { v.push_back((unsigned char)x); }
    void i16(int x) { int16_t t = (int16_t)x; raw(&t, 2); }
    void i32(int32_t x) { raw(&x, 4); }
    void i64(int64_t x) { raw(&x, 8); }
    void f32(float x) { raw(&x, 4); }
    void f64(double x) { raw(&x, 8); }
    void str(const std::string &s) { raw(s.c_str(), s.size() + 1); }
};

struct BlockIdx { int32_t number; int64_t off; int32_t size; };       // off: relative to the start of the zoom's block bytes

struct Zoom {                                 // one resolution of one chromosome-pair matrix
    uint32_t bin_size = 0; int res_idx = 0;
    int32_t block_bin_count = 0, block_col_count = 0;
    double sum = 0; float occupied = 0, stddev = 0, pct95 = 0;
    std::vector<BlockIdx> idx;
    std::vector<unsigned char> bytes;         // the compressed blocks, back to back
};

// block grid of a matrix: blocks of at most 1000 x 1000 bins, so that the int16 row / column offsets inside a block
// always fit (juicer's BLOCK_SIZE is 1000 as well; a reader takes both numbers from the zoom header)
static inline void block_grid(uint32_t len1, uint32_t len2, uint32_t bin_size, int32_t *bbc, int32_t *bcc) {
    const uint32_t nb = std::max(len1, len2) / bin_size + 1;
    *bcc = (int32_t)(nb / 1000 + 1);
    *bbc = (int32_t)(nb / (uint32_t)*bcc + 1);
}

// recs: all records of one matrix at one resolution.  Sorted here by (block, row, column), cut into blocks, every block
// written as "list of rows" (type 1) and deflated.
static inline void build_zoom(std::vector<Rec> &recs, uint32_t bin_size, int res_idx, int32_t bbc, int32_t bcc, bool intra, Zoom *z) {
    z->bin_size = bin_size; z->res_idx = res_idx; z->block_bin_count = bbc; z->block_col_count = bcc;
    auto blk = [&](const Rec &r) { return (uint64_t)(r.y / (uint32_t)bbc) * (uint64_t)bcc + r.x / (uint32_t)bbc; };
    std::sort(recs.begin(), recs.end(), [&](const Rec &a, const Rec &b) {
        const uint64_t ba = blk(a), bb = blk(b);
        if (ba != bb) return ba < bb;
        if (a.y != b.y) return a.y < b.y;
        return a.x < b.x; });
    double s = 0, s2 = 0;
    std::vector<uint32_t> cs; cs.reserve(recs.size());
    for (const Rec &r : recs) {
        if (!intra || r.x != r.y) s += r.c;                           // juicer leaves the diagonal out of a matrix's sum
        s2 += (double)r.c * r.c; cs.push_back(r.c);
    }
    z->sum = s; z->occupied = (float)recs.size();
    if (!cs.empty()) {
        double tot = 0; for (uint32_t c : cs) tot += c;
        const double mean = tot / cs.size();
        z->stddev = (float)std::sqrt(std::max(0.0, s2 / cs.size() - mean * mean));
        const size_t k = (size_t)(0.95 * (cs.size() - 1));
        std::nth_element(cs.begin(), cs.begin() + k, cs.end());
        z->pct95 = (float)cs[k];
    }
    Buf raw; std::vector<unsigned char> comp;
    size_t i = 0;
    while (i < recs.size()) {
        const uint64_t b = blk(recs[i]);
        size_t j = i; uint32_t xo = UINT32_MAX, yo = UINT32_MAX, cmax = 0;
        while (j < recs.size() && blk(recs[j]) == b) { xo = std::min(xo, recs[j].x); yo = std::min(yo, recs[j].y); cmax = std::max(cmax, recs[j].c); ++j; }
        const bool use_short = cmax < 32767;
        raw.v.clear();
        raw.i32((int32_t)(j - i)); raw.i32((int32_t)xo); raw.i32((int32_t)yo);
        raw.i8(use_short ? 1 : 0); raw.i8(1);                         // counts as int16 / float; type 1 = list of rows
        int rows = 0; for (size_t k = i; k < j; ++k) rows += k == i || recs[k].y != recs[k - 1].y;
        raw.i16(rows);
        for (size_t k = i; k < j;) {
            size_t e = k; while (e < j && recs[e].y == recs[k].y) ++e;
            raw.i16((int)(recs[k].y - yo)); raw.i16((int)(e - k));
            for (; k < e; ++k) { raw.i16((int)(recs[k].x - xo)); if (use_short) raw.i16((int)recs[k].c); else raw.f32((float)recs[k].c); }
        }
        uLongf clen = compressBound(raw.v.size());
        comp.resize(clen);
        compress2(comp.data(), &clen, raw.v.data(), raw.v.size(), Z_DEFAULT_COMPRESSION);
        z->idx.push_back({(int32_t)b, (int64_t)z->bytes.size(), (int32_t)clen});
        z->bytes.insert(z->bytes.end(), comp.begin(), comp.begin() + clen);
        i = j;
    }
}

// expected values of one resolution, juicer's ExpectedValueCalculation restated: counts per bin distance over all
// chromosomes divided by the number of bin pairs at that distance, with a window that widens until it holds 400 counts;
// one scale factor per chromosome so that its expected total equals its observed total
struct Expected { uint32_t bin_size; std::vector<double> values; std::vector<std::pair<int, double>> scale; };

static inline void expected_values(uint32_t bin_size, const std::vector<uint32_t> &len, const std::vector<double> &actual_in,
                                   const std::vector<double> &chr_counts, Expected *e) {
    e->bin_size = bin_size;
    uint32_t max_bins = 0; for (uint32_t l : len) max_bins = std::max(max_bins, l / bin_size + 1);
    std::vector<double> possible(max_bins, 0.0), actual(max_bins, 0.0);
    for (size_t d = 0; d < actual_in.size() && d < max_bins; ++d) actual[d] = actual_in[d];
    for (size_t c = 0; c < len.size(); ++c) {
        if (chr_counts[c] <= 0) continue;                             // a chromosome without contacts does not enter the average
        const uint32_t nb = len[c] / bin_size + 1;
        for (uint32_t d = 0; d < nb; ++d) possible[d] += nb - d;
    }
    long n = 0; for (uint32_t d = 0; d < max_bins; ++d) if (actual[d] > 0 && possible[d] > 0) n = d + 1;
    std::vector<double> avg(n, 0.0);
    if (n > 0) {
        double num = actual[0], den = possible[0]; long b1 = 0, b2 = 0;
        for (long i = 0; i < n; ++i) {
            if (num < 400) { while (num < 400 && b2 + 1 < n) { ++b2; num += actual[b2]; den += possible[b2]; } }
            else while (b2 - b1 > 0 && num - actual[b1] - actual[b2] >= 400) { num -= actual[b1] + actual[b2]; den -= possible[b1] + possible[b2]; ++b1; --b2; }
            avg[i] = den > 0 ? num / den : 0.0;
            if (b2 + 2 < n) { num += actual[b2 + 1] + actual[b2 + 2]; den += possible[b2 + 1] + possible[b2 + 2]; b2 += 2; }
            else if (b2 + 1 < n) { num += actual[b2 + 1]; den += possible[b2 + 1]; b2 += 1; }
        }
    }
    e->values = avg;
    for (size_t c = 0; c < len.size(); ++c) {
        if (chr_counts[c] <= 0) continue;
        const uint32_t nb = len[c] / bin_size + 1;
        double ex = 0; for (long d = 0; d < n && d < (long)nb; ++d) ex += avg[d] * (nb - d);
        e->scale.push_back({(int)c + 1, ex / chr_counts[c]});        // chromosome index in the file: 0 is ALL
    }
}

// one resolution's normalisation vector of one type (mk_norm_device's output): values in global bin order, and per chromosome
// whether it has a vector at all (none without intra contacts, none where KR failed)
struct NormInput { std::string type; const double *values; std::vector<bool> stored; };

class Writer {
public:
    // chromosomes in .info order; resolutions in any order (the file lists them coarse to fine, as juicer does)
    Writer(const std::string &genome_id, const std::vector<std::string> &names, const std::vector<uint32_t> &len, const std::vector<uint32_t> &res)
        : genome_(genome_id), names_(names), len_(len) {
        res_ = res; std::sort(res_.begin(), res_.end(), [](uint32_t a, uint32_t b) { return a > b; });
        res_.erase(std::unique(res_.begin(), res_.end()), res_.end());
        const size_t nc = names.size();
        zooms_.assign(nc * nc, std::vector<Zoom>());
        exp_.resize(res_.size()); done_.assign(res_.size(), false);
        uint64_t g = 0; for (uint32_t l : len) { cum_.push_back(g); g += l; }
        all_len_ = (uint32_t)(g / 1000);                              // the ALL pseudo-chromosome is measured in kb
        all_bin_ = std::max(1u, all_len_ / 500);
    }

    // one resolution's COO as pairs2bins writes it: global bin ids (bin = offset[chr] + pos / res, len / res + 1 bins per
    // chromosome, .info order), upper triangle, sorted by (bin1, bin2)
    // norms (may be NULL): the resolution's normalisation vectors; the normalised expected values are made here from the
    // same entries, with c / (n_x n_y) for the counts and only the entries whose two norms are valid (finite, > 0)
    int add(uint32_t res, const uint32_t *b1, const uint32_t *b2, const uint32_t *ct, size_t nnz, std::string *err,
            const std::vector<NormInput> *norms = nullptr) {
        int ri = -1; for (size_t k = 0; k < res_.size(); ++k) if (res_[k] == res) ri = (int)k;
        if (ri < 0) { *err = "resolution " + std::to_string(res) + " was not announced"; return 1; }
        if (done_[ri]) return 0;                                      // a resolution listed twice is stored once
        done_[ri] = true;
        const size_t nc = names_.size();
        std::vector<uint64_t> off(nc + 1, 0);
        for (size_t c = 0; c < nc; ++c) off[c + 1] = off[c] + len_[c] / res + 1;
        std::vector<std::vector<Rec>> per(nc * nc);
        std::vector<double> actual, chr_counts(nc, 0.0);
        const size_t n_types = norms ? norms->size() : 0;
        std::vector<std::vector<double>> n_actual(n_types), n_counts(n_types, std::vector<double>(nc, 0.0));
        const bool finest = res == res_.back();
        std::vector<Rec> all;                                        // whole-genome records, merged below
        size_t c1 = 0;
        for (size_t i = 0; i < nnz; ++i) {
            if (b1[i] > b2[i] || b2[i] >= off[nc] || (i && (b1[i] < b1[i - 1] || (b1[i] == b1[i - 1] && b2[i] <= b2[i - 1])))) {
                *err = "COO of resolution " + std::to_string(res) + " is not a sorted upper triangle (entry " + std::to_string(i) + ")"; return 1; }
            while (b1[i] >= off[c1 + 1]) ++c1;
            const size_t c2 = (size_t)(std::upper_bound(off.begin(), off.end(), (uint64_t)b2[i]) - off.begin()) - 1;
            const uint32_t x = (uint32_t)(b1[i] - off[c1]), y = (uint32_t)(b2[i] - off[c2]);
            per[c1 * nc + c2].push_back({x, y, ct[i]});
            if (c1 == c2) {
                const uint32_t d = y - x;
                if (d >= actual.size()) actual.resize((size_t)d + 1, 0.0);
                actual[d] += ct[i]; chr_counts[c1] += ct[i];
                for (size_t t = 0; t < n_types; ++t) {
                    const NormInput &q = (*norms)[t];
                    const double nx = q.values[b1[i]], ny = q.values[b2[i]];
                    if (!q.stored[c1] || !std::isfinite(nx) || !std::isfinite(ny) || !(nx > 0) || !(ny > 0)) continue;
                    if (d >= n_actual[t].size()) n_actual[t].resize((size_t)d + 1, 0.0);
                    const double v = ct[i] / (nx * ny);
                    n_actual[t][d] += v; n_counts[t][c1] += v;
                }
            }
            if (finest) {                                             // whole-genome view from the finest resolution's bin starts
                uint32_t gx = (uint32_t)((cum_[c1] + (uint64_t)x * res) / 1000 / all_bin_), gy = (uint32_t)((cum_[c2] + (uint64_t)y * res) / 1000 / all_bin_);
                if (gx > gy) std::swap(gx, gy);
                all.push_back({gx, gy, ct[i]});
            }
        }
        expected_values(res, len_, actual, chr_counts, &exp_[ri]);
        for (size_t t = 0; t < n_types; ++t) {
            const NormInput &q = (*norms)[t];
            norm_exp_.emplace_back(); norm_exp_.back().first = q.type;
            expected_values(res, len_, n_actual[t], n_counts[t], &norm_exp_.back().second);
            for (size_t c = 0; c < nc; ++c)
                if (q.stored[c]) norm_vec_.push_back({q.type, (int)c + 1, res, std::vector<double>(q.values + off[c], q.values + off[c + 1])});
        }
        // sort + deflate, one matrix per task
        std::vector<size_t> todo; for (size_t k = 0; k < nc * nc; ++k) if (!per[k].empty()) todo.push_back(k);
        std::sort(todo.begin(), todo.end(), [&](size_t a, size_t b) { return per[a].size() > per[b].size(); });
        std::vector<Zoom> out(todo.size());
        std::atomic<size_t> next(0);
        auto work = [&]() {
            for (size_t t; (t = next.fetch_add(1)) < todo.size();) {
                const size_t k = todo[t], a = k / nc, b = k % nc;
                int32_t bbc, bcc; block_grid(len_[a], len_[b], res, &bbc, &bcc);
                build_zoom(per[k], res, ri, bbc, bcc, a == b, &out[t]);
                std::vector<Rec>().swap(per[k]);
            }
        };
        unsigned nt = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        if (const char *e = getenv("MICROCKET_HIC_THREADS")) nt = (unsigned)std::max(1, atoi(e));
        std::vector<std::thread> th; for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
        work(); for (auto &t : th) t.join();
        for (size_t t = 0; t < todo.size(); ++t) zooms_[todo[t]].push_back(std::move(out[t]));
        if (finest) {
            std::sort(all.begin(), all.end(), [](const Rec &a, const Rec &b) { return a.y != b.y ? a.y < b.y : a.x < b.x; });
            std::vector<Rec> m;
            for (const Rec &r : all) { if (!m.empty() && m.back().x == r.x && m.back().y == r.y) m.back().c += r.c; else m.push_back(r); }
            const int32_t nb = (int32_t)(all_len_ / all_bin_ + 1);
            all_zoom_ = Zoom(); build_zoom(m, all_bin_, 0, nb, 1, true, &all_zoom_); have_all_ = true;
        }
        return 0;
    }

    int write(const std::string &path, std::string *err) {
        FILE *f = fopen(path.c_str(), "wb");
        if (!f) { *err = "cannot write " + path; return 1; }
        const size_t nc = names_.size();
        Buf h;
        h.raw("HIC", 4); h.i32(8); h.i64(0);                          // master index position, patched below
        h.str(genome_);
        h.i32(1); h.str("software"); h.str("microcket-b200 (pairs2bins / coo2hic)");
        h.i32((int32_t)nc + 1); h.str("ALL"); h.i32((int32_t)all_len_);
        for (size_t c = 0; c < nc; ++c) { h.str(names_[c]); h.i32((int32_t)len_[c]); }
        h.i32((int32_t)res_.size()); for (uint32_t r : res_) h.i32((int32_t)r);
        h.i32(0);                                                     // no fragment resolutions
        fwrite(h.v.data(), 1, h.v.size(), f);
        int64_t pos = (int64_t)h.v.size();
        struct Entry { std::string key; int64_t pos; int32_t size; };
        std::vector<Entry> master;
        auto put_matrix = [&](int i1, int i2, std::vector<Zoom> &zs) {
            std::sort(zs.begin(), zs.end(), [](const Zoom &a, const Zoom &b) { return a.res_idx < b.res_idx; });
            size_t hdr = 12; for (const Zoom &z : zs) hdr += 3 + 4 + 16 + 16 + z.idx.size() * 16;
            Buf m; m.i32(i1); m.i32(i2); m.i32((int32_t)zs.size());
            int64_t data = pos + (int64_t)hdr;
            for (const Zoom &z : zs) {
                m.str("BP"); m.i32(z.res_idx); m.f32((float)z.sum); m.f32(z.occupied); m.f32(z.stddev); m.f32(z.pct95);
                m.i32((int32_t)z.bin_size); m.i32(z.block_bin_count); m.i32(z.block_col_count); m.i32((int32_t)z.idx.size());
                for (const BlockIdx &b : z.idx) { m.i32(b.number); m.i64(data + b.off); m.i32(b.size); }
                data += (int64_t)z.bytes.size();
            }
            fwrite(m.v.data(), 1, m.v.size(), f);
            for (const Zoom &z : zs) if (!z.bytes.empty()) fwrite(z.bytes.data(), 1, z.bytes.size(), f);
            master.push_back({std::to_string(i1) + "_" + std::to_string(i2), pos, (int32_t)std::min<int64_t>(data - pos, INT32_MAX)});
            pos = data;
        };
        if (have_all_) { std::vector<Zoom> zs; zs.push_back(all_zoom_); put_matrix(0, 0, zs); }
        for (size_t a = 0; a < nc; ++a) for (size_t b = a; b < nc; ++b) if (!zooms_[a * nc + b].empty()) put_matrix((int)a + 1, (int)b + 1, zooms_[a * nc + b]);
        // footer
        Buf ft;
        ft.i32((int32_t)master.size());
        for (const Entry &e : master) { ft.str(e.key); ft.i64(e.pos); ft.i32(e.size); }
        int nexp = 0; for (const Expected &e : exp_) nexp += !e.values.empty();
        ft.i32(nexp);
        for (const Expected &e : exp_) {
            if (e.values.empty()) continue;
            ft.str("BP"); ft.i32((int32_t)e.bin_size); ft.i32((int32_t)e.values.size());
            for (double v : e.values) ft.f64(v);
            ft.i32((int32_t)e.scale.size()); for (auto &s : e.scale) { ft.i32(s.first); ft.f64(s.second); }
        }
        Buf tail; tail.i32((int32_t)ft.v.size());                     // nBytesV5: what lies between this int and the normalised section
        tail.raw(ft.v.data(), ft.v.size());
        // normalised section: expected values per (type, resolution), the vectors' index, then the vectors at their positions
        int nnexp = 0; for (auto &e : norm_exp_) nnexp += !e.second.values.empty();
        tail.i32(nnexp);
        for (auto &te : norm_exp_) {
            const Expected &e = te.second;
            if (e.values.empty()) continue;
            tail.str(te.first); tail.str("BP"); tail.i32((int32_t)e.bin_size); tail.i32((int32_t)e.values.size());
            for (double v : e.values) tail.f64(v);
            tail.i32((int32_t)e.scale.size()); for (auto &sc : e.scale) { tail.i32(sc.first); tail.f64(sc.second); }
        }
        tail.i32((int32_t)norm_vec_.size());
        int64_t vpos = pos + (int64_t)tail.v.size();
        for (const NormVec &n : norm_vec_) vpos += (int64_t)(n.type.size() + 1 + 4 + 3 + 4 + 8 + 4);
        for (const NormVec &n : norm_vec_) {
            const int32_t nbytes = (int32_t)(4 + 8 * n.values.size());
            tail.str(n.type); tail.i32(n.chr); tail.str("BP"); tail.i32((int32_t)n.bin_size); tail.i64(vpos); tail.i32(nbytes);
            vpos += nbytes;
        }
        for (const NormVec &n : norm_vec_) { tail.i32((int32_t)n.values.size()); for (double v : n.values) tail.f64(v); }
        fwrite(tail.v.data(), 1, tail.v.size(), f);
        fseek(f, 8, SEEK_SET); fwrite(&pos, 8, 1, f);
        const bool bad = ferror(f); if (fclose(f) || bad) { *err = "write error on " + path; return 1; }
        return 0;
    }

private:
    std::string genome_; std::vector<std::string> names_; std::vector<uint32_t> len_, res_;
    std::vector<uint64_t> cum_; uint32_t all_len_ = 0, all_bin_ = 1;
    std::vector<std::vector<Zoom>> zooms_;                           // [c1 * n + c2] -> the resolutions added so far
    std::vector<Expected> exp_; std::vector<bool> done_; Zoom all_zoom_; bool have_all_ = false;
    struct NormVec { std::string type; int chr; uint32_t bin_size; std::vector<double> values; };
    std::vector<std::pair<std::string, Expected>> norm_exp_;        // normalised expected values, in the order added
    std::vector<NormVec> norm_vec_;                                   // chromosome index in the file: 1..n (0 is ALL: no vectors)
};

}  // namespace hic
