// cli_sam2bam.cpp — `sam2bam -o OUT.bam [IN.sam ...]`: SAM text to a coordinate-sorted BAM and its .bai, on the GPU (stands where
// the driver runs `samtools view | samtools sort | samtools index` on `$header $sid.flash.sam $sid.unc.sam`, microcket:537-539).
// The inputs are one SAM stream.  A reader thread fills two pinned slots of whole lines (MICROCKET_CHUNK_MB, default 256); the
// GPU encodes each slot's lines into BAM records of the current run (mk_bam_encode_*); a run that reaches the sort budget
// (MICROCKET_SORT_MB) is sorted on the GPU and spilled to OUT.bam.tmp.<k> (record bytes) and OUT.bam.tmp.<k>.len (u32 lengths).
// Without a spill the run is sorted once in core.  Otherwise merge rounds load a window of whole records of every run, take
// from every run the records whose (key, run) is at most the smallest (key of the last loaded record, run) over the runs not
// yet read to the end, and sort their concatenation in run order stably on the GPU: that is the in-core order.
// Sorted records are gathered in windows, compressed by mk_bgzf_deflate_device at multiples of 65 280 bytes of the record
// stream (the partial last member is carried into the next window), and written by a writer thread; the index is built on the
// device as the records go out (mk_bam_index_add_device) and laid out from the member table at the end.  So OUT.bam and its
// .bai are the same bytes whatever the budget and chunk size.
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "../../include/microcket_b200.h"
#include "bam_encode.h"
using namespace std;

static const unsigned char BGZF_EOF[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
static const size_t BLOCK = 65280;

static int usage(const char *prg, int rc) {
    fprintf(stderr,
            "\nUsage: %s -o OUT.bam [IN.sam ...]\n"
            "  Reads the SAM inputs one after another as one stream (no IN, or IN '-': standard input) and writes the\n"
            "  coordinate-sorted BAM OUT.bam and its index OUT.bam.bai, encoding, sorting, compressing and indexing on the GPU.\n"
            "  The header is the '@' lines before the first record: @HD gets SO:coordinate (an @HD line is added first when\n"
            "  there is none), the references are the @SQ SN/LN pairs in order.  Records are ordered by (reference, position,\n"
            "  reverse strand) with unplaced records last; ties keep input order.\n"
            "Environment:\n"
            "  MICROCKET_DEVICE    CUDA device (default 0)\n"
            "  MICROCKET_CHUNK_MB  input chunk (default 256); a line must fit in one chunk\n"
            "  MICROCKET_SORT_MB   device bytes of one in-memory run (at least 4 chunks).  Default: (free device memory at\n"
            "                      start-up - 8 chunks - 512 MB) / 2.2.  Larger inputs are sorted in runs spilled to\n"
            "                      OUT.bam.tmp.<k> and merged; the output bytes do not depend on either size.\n"
            "Exit codes: 0 success; 2 usage; 10 an input that cannot be read, an output or temp file that cannot be written,\n"
            "  a malformed line (named by its line number in the stream) or a reference not in @SQ; 20 a CUDA or library\n"
            "  error.  A failed run leaves no OUT.bam, OUT.bam.bai or temp file behind.\n\n",
            prg);
    return rc;
}

struct Fail { int rc; };
static vector<string> g_cleanup;                                          // removed when the run fails
[[noreturn]] static void fail(int rc, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
static void fail(int rc, const char *fmt, ...) {
    va_list ap; va_start(ap, fmt);
    fprintf(stderr, "Error: "); vfprintf(stderr, fmt, ap); fprintf(stderr, "\n");
    va_end(ap);
    throw Fail{rc};
}
static void lib(int r) { if (r != MK_OK) fail(20, "%s", mk_last_error()); }

template <class T> struct Chan {                                        // blocking queue
    deque<T> q; mutex m; condition_variable cv;
    void put(T v) { { lock_guard<mutex> l(m); q.push_back(v); } cv.notify_one(); }
    T get() { unique_lock<mutex> l(m); cv.wait(l, [&] { return !q.empty(); }); T v = q.front(); q.pop_front(); return v; }
};
struct Slot { char *p = NULL; size_t n = 0; bool last = false; };

// the inputs one after another
struct Input {
    vector<FILE *> f; vector<string> name; size_t k = 0; bool err = false;
    size_t read(char *p, size_t n) {
        size_t got = 0;
        while (got < n && k < f.size()) {
            const size_t g = fread(p + got, 1, n - got, f[k]);
            got += g;
            if (g == 0 || got < n) {
                if (ferror(f[k])) { err = true; return got; }
                if (feof(f[k])) ++k;
            }
        }
        return got;
    }
};

struct Key { uint32_t hi, lo; int run; };
static bool key_le(const Key &a, const Key &b) {
    if (a.hi != b.hi) return a.hi < b.hi;
    if (a.lo != b.lo) return a.lo < b.lo;
    return a.run <= b.run;
}

struct Sam2Bam {
    int dev = 0;
    size_t chunk = 0, budget = 0, max_records = 0, out_cap = 0, z_cap = 0;
    string out_path;
    FILE *fo = NULL;
    mk_bam *bam = NULL; mk_bgzf_enc *enc = NULL;
    void *d_text = NULL, *d_run = NULL, *d_runoff = NULL, *d_out = NULL, *d_z = NULL;
    int32_t n_refs = 0;
    // the run on the device
    size_t n_run = 0, run_bytes = 0;
    // output
    size_t carry = 0;                                                   // record-stream bytes at the front of d_out not yet compressed
    uint64_t u = 0, file_pos = 0, records = 0;
    vector<uint64_t> coff;                                              // file offset of every record-stream member
    Slot oslot[2]; Chan<Slot *> o_free, o_full; thread writer; bool write_err = false;
    vector<unsigned char> h_tmp;
    // spill
    vector<string> runs;
    uint64_t rounds = 0;

    void start_writer() {
        for (int k = 0; k < 2; ++k) { lib(mk_host_alloc(z_cap + 28, (void **)&oslot[k].p)); o_free.put(&oslot[k]); }
        writer = thread([this] {
            while (true) {
                Slot *s = o_full.get();
                if (s->n && !write_err && fwrite(s->p, 1, s->n, fo) != s->n) write_err = true;
                const bool last = s->last;
                o_free.put(s);
                if (last) break;
            }
        });
    }
    void stop_writer() {
        if (!writer.joinable()) return;
        Slot *s = o_free.get(); s->n = 0; s->last = true; o_full.put(s);
        writer.join();
        for (int k = 0; k < 2; ++k) mk_host_free(oslot[k].p);
    }
    // n bytes at d_in compressed into members and handed to the writer; rec: they are record-stream bytes
    void compress(const void *d_in, size_t n, bool rec) {
        if (!n) return;
        size_t len = 0, nm = 0;
        vector<mk_bgzf_member> mem((n + BLOCK - 1) / BLOCK);
        lib(mk_bgzf_deflate_device(enc, d_in, n, -1, d_z, z_cap, &len, mem.data(), mem.size(), &nm, NULL));
        Slot *s = o_free.get();
        if (mk_copy_to_host(s->p, d_z, len) != MK_OK) { o_free.put(s); lib(MK_ERR_CUDA); }
        for (size_t k = 0; k < nm && rec; ++k) coff.push_back(file_pos + mem[k].in_off);
        file_pos += len;
        s->n = len; s->last = false;
        o_full.put(s);
    }

    void create(const vector<string> &names, const vector<uint32_t> &lens) {
        vector<const char *> np;
        for (auto &s : names) np.push_back(s.c_str());
        n_refs = (int32_t)names.size();
        lib(mk_bam_create(dev, np.data(), lens.data(), n_refs, chunk + 1, max_records, &bam));
        lib(mk_dev_alloc(dev, chunk + 64, &d_text));
        lib(mk_dev_alloc(dev, budget, &d_run));
        lib(mk_dev_alloc(dev, (max_records + 1) * 8, &d_runoff));
        out_cap = 2 * chunk + 2 * BLOCK + 64;
        lib(mk_dev_alloc(dev, out_cap, &d_out));
        lib(mk_bgzf_enc_create(dev, out_cap, &enc));
        z_cap = mk_bgzf_deflate_bound(out_cap);
        lib(mk_dev_alloc(dev, z_cap, &d_z));
        const uint64_t zero = 0;
        lib(mk_copy_to_device(d_runoff, &zero, 8));
    }

    // the BAM header: magic, text, references; into members of its own
    void write_header(const string &text, const vector<string> &names, const vector<uint32_t> &lens) {
        vector<unsigned char> h;
        auto p32 = [&](uint32_t v) { for (int b = 0; b < 4; ++b) h.push_back((unsigned char)(v >> 8 * b)); };
        h.insert(h.end(), {'B', 'A', 'M', 1});
        p32((uint32_t)text.size()); h.insert(h.end(), text.begin(), text.end());
        p32((uint32_t)names.size());
        for (size_t k = 0; k < names.size(); ++k) { p32((uint32_t)names[k].size() + 1); h.insert(h.end(), names[k].begin(), names[k].end()); h.push_back(0); p32(lens[k]); }
        for (size_t o = 0; o < h.size(); o += out_cap / BLOCK * BLOCK) {
            const size_t n = min(h.size() - o, out_cap / BLOCK * BLOCK);
            lib(mk_copy_to_device(d_out, h.data() + o, n));
            compress(d_out, n, false);
        }
    }

    // the sorted order of the n records at d_run, out in windows of about one chunk: to the record stream, or to a spill file
    void emit_sorted(size_t n, FILE *spill, FILE *spill_len) {
        size_t total = 0;
        lib(mk_bam_sort_device(bam, (const uint8_t *)d_run, (const uint64_t *)d_runoff, n, &total, NULL));
        vector<uint64_t> off;
        vector<uint32_t> lens;
        for (size_t i0 = 0; i0 < n;) {
            size_t i1 = 0, bytes = 0;
            const uint64_t *d_off = NULL;
            unsigned char *dst = (unsigned char *)d_out + (spill ? 0 : carry);
            lib(mk_bam_gather_device(bam, i0, chunk, dst, out_cap - (spill ? 0 : carry), &i1, &bytes, &d_off, NULL));
            if (spill) {
                h_tmp.resize(bytes);
                off.resize(i1 - i0 + 1); lens.resize(i1 - i0);
                lib(mk_copy_to_host(h_tmp.data(), d_out, bytes));
                lib(mk_copy_to_host(off.data(), d_off, off.size() * 8));
                for (size_t k = 0; k < lens.size(); ++k) lens[k] = (uint32_t)(off[k + 1] - off[k]);
                if (fwrite(h_tmp.data(), 1, bytes, spill) != bytes || fwrite(lens.data(), 4, lens.size(), spill_len) != lens.size())
                    fail(10, "writing the temp file %s failed", runs.back().c_str());
            } else {
                lib(mk_bam_index_add_device(bam, dst, d_off, i1 - i0, u, NULL));
                u += bytes; records += i1 - i0; carry += bytes;
                const size_t whole = carry / BLOCK * BLOCK;
                compress(d_out, whole, true);
                if (whole && carry > whole) lib(mk_copy_device(d_out, (unsigned char *)d_out + whole, carry - whole));   // disjoint: whole >= 65 280 > the rest
                carry -= whole;
            }
            i0 = i1;
        }
    }

    void spill_run() {
        const string path = out_path + ".tmp." + to_string(runs.size());
        runs.push_back(path);
        g_cleanup.push_back(path); g_cleanup.push_back(path + ".len");
        FILE *f = fopen(path.c_str(), "wb"), *fl = fopen((path + ".len").c_str(), "wb");
        if (!f || !fl) { if (f) fclose(f); if (fl) fclose(fl); fail(10, "cannot write the temp file %s", path.c_str()); }
        emit_sorted(n_run, f, fl);
        const bool bad = fclose(f) != 0, bad2 = fclose(fl) != 0;
        if (bad || bad2) fail(10, "writing the temp file %s failed", path.c_str());
        n_run = run_bytes = 0;
    }

    // merge rounds over the spilled runs
    struct Run {
        FILE *f = NULL, *fl = NULL; bool disk_done = false;
        uint32_t next = 0; bool has_next = false;                                 // the length of the next record on disk
        vector<unsigned char> bytes; vector<uint32_t> lens; vector<size_t> at;   // loaded records not yet taken (at: start offsets)
    };
    void merge() {
        const size_t R = runs.size(), win = max<size_t>(budget / R, 1), wrec = max<size_t>(max_records / R, 1);
        vector<Run> rs(R);
        for (size_t r = 0; r < R; ++r) {
            rs[r].f = fopen(runs[r].c_str(), "rb"); rs[r].fl = fopen((runs[r] + ".len").c_str(), "rb");
            if (!rs[r].f || !rs[r].fl) fail(10, "cannot read the temp file %s", runs[r].c_str());
        }
        auto key_of = [&](const Run &x, size_t i, int r) { Key k; be_key(x.bytes.data() + x.at[i], n_refs, k.hi, k.lo); k.run = r; return k; };
        vector<uint64_t> off;
        while (true) {
            bool any = false;
            for (size_t r = 0; r < R; ++r) {                               // top every run up to its window
                Run &x = rs[r];
                while (!x.disk_done) {
                    if (!x.has_next && fread(&x.next, 4, 1, x.fl) != 1) { x.disk_done = true; break; }
                    x.has_next = true;
                    const uint32_t len = x.next;
                    if (!x.lens.empty() && (x.bytes.size() + len > win || x.lens.size() >= wrec)) break;
                    x.has_next = false;
                    const size_t o = x.bytes.size();
                    x.bytes.resize(o + len);
                    if (fread(x.bytes.data() + o, 1, len, x.f) != len) fail(10, "the temp file %s is short", runs[r].c_str());
                    x.lens.push_back(len); x.at.push_back(o);
                }
                any |= !x.lens.empty();
            }
            if (!any) break;
            bool bounded = false; Key bound{0, 0, 0};
            for (size_t r = 0; r < R; ++r) {
                const Run &x = rs[r];
                if (x.disk_done || x.lens.empty()) continue;
                const Key l = key_of(x, x.lens.size() - 1, (int)r);
                if (!bounded || !key_le(bound, l)) { bound = l; bounded = true; }
            }
            size_t n = 0, bytes = 0;
            off.assign(1, 0);
            for (size_t r = 0; r < R; ++r) {
                Run &x = rs[r];
                size_t lo = 0, hi = x.lens.size();                         // the records with (key, r) <= bound: a prefix
                if (bounded) while (lo < hi) { const size_t m = (lo + hi) / 2; if (key_le(key_of(x, m, (int)r), bound)) lo = m + 1; else hi = m; }
                else lo = x.lens.size();
                const size_t take = lo, tb = take ? x.at[take - 1] + x.lens[take - 1] : 0;
                if (bytes + tb > budget) fail(20, "a merge window of %zu bytes exceeds MICROCKET_SORT_MB", bytes + tb);
                if (take) lib(mk_copy_to_device((unsigned char *)d_run + bytes, x.bytes.data(), tb));
                for (size_t i = 0; i < take; ++i) off.push_back(off.back() + x.lens[i]);
                n += take; bytes += tb;
                x.bytes.erase(x.bytes.begin(), x.bytes.begin() + tb);
                x.lens.erase(x.lens.begin(), x.lens.begin() + take);
                x.at.erase(x.at.begin(), x.at.begin() + take);
                for (auto &a : x.at) a -= tb;
            }
            lib(mk_copy_to_device(d_runoff, off.data(), off.size() * 8));
            emit_sorted(n, NULL, NULL);
            ++rounds;
        }
        for (auto &x : rs) { fclose(x.f); fclose(x.fl); }
        for (auto &p : runs) { unlink(p.c_str()); unlink((p + ".len").c_str()); }
    }
};

// the header lines -> the BAM header text and the reference dictionary
static string make_header(const string &hdr, vector<string> &names, vector<uint32_t> &lens) {
    vector<string> lines;
    for (size_t p = 0; p < hdr.size();) { const size_t e = hdr.find('\n', p); lines.push_back(hdr.substr(p, e - p)); p = e + 1; }
    if (!lines.empty() && lines[0].compare(0, 3, "@HD") == 0 && (lines[0].size() == 3 || lines[0][3] == '\t')) {
        string &h = lines[0];
        const size_t so = h.find("\tSO:");
        if (so == string::npos) h += "\tSO:coordinate";
        else { const size_t e = h.find('\t', so + 4); h.replace(so + 4, (e == string::npos ? h.size() : e) - so - 4, "coordinate"); }
    } else lines.insert(lines.begin(), "@HD\tVN:1.6\tSO:coordinate");
    string text;
    for (size_t k = 0; k < lines.size(); ++k) {
        const string &l = lines[k];
        text += l; text += '\n';
        if (l.compare(0, 4, "@SQ\t") != 0) continue;
        string sn; long long ln = -1; bool has_sn = false;
        for (size_t p = 4; p <= l.size();) {
            size_t e = l.find('\t', p); if (e == string::npos) e = l.size();
            const string f = l.substr(p, e - p);
            if (f.compare(0, 3, "SN:") == 0) { sn = f.substr(3); has_sn = true; }
            else if (f.compare(0, 3, "LN:") == 0) {
                char *end = NULL; ln = strtoll(f.c_str() + 3, &end, 10);
                if (f.size() == 3 || *end || ln < 1 || ln > 2147483647ll) fail(10, "@SQ line %zu: bad LN", k + 1);
            }
            p = e + 1;
        }
        if (!has_sn || sn.empty()) fail(10, "@SQ line without SN: %s", l.c_str());
        if (ln < 0) fail(10, "@SQ %s has no LN", sn.c_str());
        if (find(names.begin(), names.end(), sn) != names.end()) fail(10, "@SQ %s appears twice", sn.c_str());
        names.push_back(sn); lens.push_back((uint32_t)ln);
    }
    return text;
}

static int run(Sam2Bam &S, Input &in) {
    // reader: slots of whole lines, the partial last line carried into the next slot
    Slot slot[2];
    Chan<Slot *> in_free, in_full;
    for (int k = 0; k < 2; ++k) { lib(mk_host_alloc(S.chunk + 1, (void **)&slot[k].p)); in_free.put(&slot[k]); }
    bool too_long = false;
    atomic<bool> stop{false};
    thread reader([&] {
        vector<char> carry;
        while (true) {
            Slot *s = in_free.get();
            if (stop) { s->n = 0; s->last = true; in_full.put(s); break; }
            memcpy(s->p, carry.data(), carry.size());
            size_t n = carry.size();
            n += in.read(s->p + n, S.chunk - n);
            s->last = n < S.chunk || in.err;
            size_t keep = n;
            if (!s->last) {
                while (keep && s->p[keep - 1] != '\n') --keep;
                if (!keep) { too_long = true; s->last = true; s->n = 0; in_full.put(s); break; }
            } else if (n && s->p[n - 1] != '\n') s->p[keep++] = '\n';
            carry.assign(s->p + keep, s->p + max(n, keep));
            s->n = keep;
            in_full.put(s);
            if (s->last) break;
        }
    });
    string hdr;
    bool in_header = true;
    uint64_t lines = 0;                                                 // lines of the stream before the current slot's records
    vector<string> names; vector<uint32_t> lens;
    int rc = 0;
    Slot *cur = NULL;
    bool reader_done = false;
    try {
        while (true) {
            Slot *s = cur = in_full.get();
            reader_done = s->last;
            if (too_long) fail(10, "line %llu is longer than MICROCKET_CHUNK_MB", (unsigned long long)lines + 1);
            if (in.err) fail(10, "reading %s failed", in.name[min(in.k, in.name.size() - 1)].c_str());
            size_t at = 0;
            while (in_header && at < s->n && s->p[at] == '@') {
                const char *e = (const char *)memchr(s->p + at, '\n', s->n - at);
                hdr.append(s->p + at, e + 1 - (s->p + at));
                at = e + 1 - s->p; ++lines;
            }
            if (in_header && (at < s->n || s->last)) {
                in_header = false;
                const string text = make_header(hdr, names, lens);
                S.create(names, lens);
                S.start_writer();
                S.write_header(text, names, lens);
            }
            const size_t n = s->n - at;
            if (n) {
                lib(mk_copy_to_device(S.d_text, s->p + at, n));
                size_t nl = 0, rb = 0; uint64_t bad = 0; int code = 0;
                const int r = mk_bam_encode_size_device(S.bam, (const char *)S.d_text, n, &nl, &rb, &bad, &code, NULL);
                if (r == MK_ERR_INPUT) fail(10, "line %llu: %s", (unsigned long long)(lines + bad + 1), be_errstr[code]);
                lib(r);
                if (S.n_run + nl > S.max_records || S.run_bytes + rb > S.budget) S.spill_run();
                if (nl > S.max_records || rb > S.budget) fail(20, "one chunk's records exceed MICROCKET_SORT_MB");
                lib(mk_bam_encode_write_device(S.bam, (uint8_t *)S.d_run, S.run_bytes, S.budget, (uint64_t *)S.d_runoff + S.n_run, NULL, NULL));
                S.n_run += nl; S.run_bytes += rb; lines += nl;
            }
            const bool last = s->last;
            cur = NULL;
            in_free.put(s);
            if (last) break;
        }
        reader.join();
        if (S.runs.empty()) { if (S.n_run) S.emit_sorted(S.n_run, NULL, NULL); }
        else { if (S.n_run) S.spill_run(); S.merge(); }
        S.compress(S.d_out, S.carry, true);
        S.coff.push_back(S.file_pos);
        const uint8_t *bai = NULL; size_t blen = 0;
        lib(mk_bam_bai(S.bam, S.coff.data(), S.coff.size(), &bai, &blen));
        Slot *e = S.o_free.get();
        memcpy(e->p, BGZF_EOF, 28); e->n = 28; e->last = false;
        S.o_full.put(e);
        S.stop_writer();
        if (S.write_err) fail(10, "writing %s failed", S.out_path.c_str());
        const string bp = S.out_path + ".bai";
        FILE *fb = fopen(bp.c_str(), "wb");
        if (!fb) fail(10, "cannot write %s", bp.c_str());
        const bool bad = fwrite(bai, 1, blen, fb) != blen;
        if (fclose(fb) != 0 || bad) fail(10, "writing %s failed", bp.c_str());
        fprintf(stderr, "INFO: %llu records, %zu runs spilled, %llu merge rounds\n", (unsigned long long)S.records, S.runs.size(),
                (unsigned long long)S.rounds);
    } catch (Fail &f) {
        rc = f.rc;
    }
    if (reader.joinable()) {                                            // stop the reader: it ends with a last slot
        stop = true;
        if (cur) in_free.put(cur);
        while (!reader_done) { Slot *s = in_full.get(); reader_done = s->last; in_free.put(s); }
        reader.join();
    }
    S.stop_writer();
    for (int k = 0; k < 2; ++k) mk_host_free(slot[k].p);
    return rc;
}

int main(int argc, char *argv[]) {
    string out;
    vector<string> files;
    for (int a = 1; a < argc; ++a) {
        const char *s = argv[a];
        if (!strcmp(s, "-h")) return usage(argv[0], 0);
        if (!strcmp(s, "-o")) { if (a + 1 >= argc || !out.empty()) return usage(argv[0], 2); out = argv[++a]; continue; }
        if (s[0] == '-' && s[1]) return usage(argv[0], 2);
        files.push_back(s);
    }
    if (out.empty()) return usage(argv[0], 2);
    if (files.empty()) files.push_back("-");
    Input in;
    for (auto &f : files) {
        FILE *x = f == "-" ? stdin : fopen(f.c_str(), "rb");
        if (!x) { fprintf(stderr, "Error: cannot read %s\n", f.c_str()); for (auto *y : in.f) if (y != stdin) fclose(y); return 10; }
        in.f.push_back(x); in.name.push_back(f == "-" ? "stdin" : f);
    }
    Sam2Bam S;
    S.out_path = out;
    S.dev = getenv("MICROCKET_DEVICE") ? atoi(getenv("MICROCKET_DEVICE")) : 0;
    int rc = 0;
    try {
        if (mk_device_count() < 1) fail(20, "no CUDA device: microcket_b200 has no CPU fallback");
        S.chunk = (size_t)max(1L, getenv("MICROCKET_CHUNK_MB") ? atol(getenv("MICROCKET_CHUNK_MB")) : 256L) << 20;
        size_t b = 0;
        if (getenv("MICROCKET_SORT_MB")) b = (size_t)max(0L, atol(getenv("MICROCKET_SORT_MB"))) << 20;
        else lib(mk_bam_sort_budget(S.dev, S.chunk, &b));
        S.budget = max(b, 4 * S.chunk);
        S.max_records = min<size_t>(S.budget / 64 + S.chunk / BE_MIN_LINE + 2, (1u << 30) - 1);
        g_cleanup = {out, out + ".bai"};
        S.fo = fopen(out.c_str(), "wb");
        if (!S.fo) fail(10, "cannot write %s", out.c_str());
        rc = run(S, in);
    } catch (Fail &f) {
        rc = f.rc;
    }
    if (S.fo && fclose(S.fo) != 0 && !rc) { fprintf(stderr, "Error: writing %s failed\n", out.c_str()); rc = 10; }
    for (auto *x : in.f) if (x != stdin) fclose(x);
    mk_bam_destroy(S.bam); mk_bgzf_enc_destroy(S.enc);
    for (void *p : {S.d_text, S.d_run, S.d_runoff, S.d_out, S.d_z}) if (p) mk_dev_free(p);
    if (rc) for (auto &p : g_cleanup) unlink(p.c_str());
    return rc;
}
