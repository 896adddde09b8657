// cli_bgzip.cpp — drop-in `bgzip` for whole files, compressing on the GPU (stands where the driver calls bin/bgzip,
// microcket:548-551).  BGZF members are written in HBM by mk_bgzf_deflate_device (bgzf_deflate.cu) and read back by
// mk_bgzf_scan + mk_bgzf_inflate_device (bgzf.cu, -d).
// The input streams through two pinned slots of MICROCKET_CHUNK_MB (default 256, rounded down to a multiple of 65 280
// bytes): a reader thread fills one while the GPU compresses the other, and a writer thread writes the previous output.
// Members are cut at multiples of 65 280 input bytes whatever the chunk size, so a file, stdin and every chunk size give the
// same bytes.  The compressed bytes are this project's own, not htslib's; gzip, zlib and htslib read them back.
#include <sys/stat.h>
#include <unistd.h>
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
using namespace std;

static const unsigned char BGZF_EOF[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
static const size_t BLOCK = 65280;

static int usage(const char *prg, int rc) {
    fprintf(stderr,
            "\nUsage: %s [-c] [-d] [-f] [-k] [-l LEVEL] [-@ THREADS] [FILE]\n"
            "  Compresses FILE to FILE.gz in bgzip's BGZF format on the GPU and removes FILE; with no FILE, or FILE '-',\n"
            "  reads standard input and writes standard output.\n"
            "  -c        write to standard output and keep FILE\n"
            "  -d        decompress FILE.gz to FILE (any BGZF input; gzip that is not BGZF is refused)\n"
            "  -f        overwrite an existing output file\n"
            "  -k        keep FILE\n"
            "  -l LEVEL  -1..9.  0 writes stored (uncompressed) members; -1 (the default) and 1-9 all write the same bytes:\n"
            "            one greedy parse with one match candidate per position and per-member Huffman codes\n"
            "  -@ N      accepted and ignored (the GPU does the work)\n"
            "  -h        this text\n"
            "  Other bgzip options (-i, -b, -s, -r, ...) are refused.  The output is read back by gzip, zlib and htslib; its\n"
            "  bytes are not those of htslib's bgzip.\n"
            "Exit codes: 0 success; 2 usage; 10 a file that cannot be read or written, an output that exists without -f, or\n"
            "  input that is not BGZF or is damaged (-d); 20 a CUDA or library error.\n\n",
            prg);
    return rc;
}

template <class T> struct Chan {                                        // blocking queue
    deque<T> q; mutex m; condition_variable cv;
    void put(T v) { { lock_guard<mutex> l(m); q.push_back(v); } cv.notify_one(); }
    T get() { unique_lock<mutex> l(m); cv.wait(l, [&] { return !q.empty(); }); T v = q.front(); q.pop_front(); return v; }
};
struct Slot { unsigned char *p = NULL; size_t n = 0; bool last = false; };

static int lib_fail() { fprintf(stderr, "Error: %s\n", mk_last_error()); return 20; }

// input -> BGZF members + the EOF member
static int compress(FILE *fi, FILE *fo, int level, size_t chunk, int dev, bool &write_err) {
    const size_t cap = mk_bgzf_deflate_bound(chunk);
    mk_bgzf_enc *enc = NULL;
    void *d_in = NULL, *d_out = NULL;
    if (mk_bgzf_enc_create(dev, chunk, &enc) != MK_OK || mk_dev_alloc(dev, chunk, &d_in) != MK_OK || mk_dev_alloc(dev, cap, &d_out) != MK_OK) return lib_fail();
    Slot in[2], out[2];
    for (int k = 0; k < 2; ++k)
        if (mk_host_alloc(chunk, (void **)&in[k].p) != MK_OK || mk_host_alloc(cap, (void **)&out[k].p) != MK_OK) return lib_fail();
    Chan<Slot *> in_free, in_full, out_free, out_full;
    for (int k = 0; k < 2; ++k) { in_free.put(&in[k]); out_free.put(&out[k]); }
    bool read_err = false;
    thread reader([&] {
        while (true) {
            Slot *s = in_free.get();
            s->n = fread(s->p, 1, chunk, fi);                               // short only at the end of the input
            s->last = s->n < chunk;
            if (s->last && ferror(fi)) read_err = true;
            in_full.put(s);
            if (s->last) break;
        }
    });
    thread writer([&] {
        while (true) {
            Slot *s = out_full.get();
            if (s->n && fwrite(s->p, 1, s->n, fo) != s->n) write_err = true;
            const bool last = s->last;
            out_free.put(s);
            if (last) break;
        }
    });
    int rc = 0;
    while (true) {
        Slot *s = in_full.get();
        const bool last = s->last;
        size_t len = 0, nm = 0;
        if (!rc && s->n) {
            if (mk_copy_to_device(d_in, s->p, s->n) != MK_OK) rc = lib_fail();
        }
        const size_t n = s->n;
        in_free.put(s);                                                 // the reader fills it while the GPU works
        Slot *o = out_free.get();
        if (!rc && n && mk_bgzf_deflate_device(enc, d_in, n, level, d_out, cap, &len, NULL, 0, &nm, NULL) != MK_OK) rc = lib_fail();
        if (!rc && len && mk_copy_to_host(o->p, d_out, len) != MK_OK) rc = lib_fail();
        if (rc) len = 0;
        if (last && !rc) { memcpy(o->p + len, BGZF_EOF, 28); len += 28; }
        o->n = len; o->last = last;
        out_full.put(o);
        if (last) break;
    }
    reader.join(); writer.join();
    for (int k = 0; k < 2; ++k) { mk_host_free(in[k].p); mk_host_free(out[k].p); }
    mk_dev_free(d_in); mk_dev_free(d_out); mk_bgzf_enc_destroy(enc);
    if (read_err) { fprintf(stderr, "Error: reading the input failed\n"); return 10; }
    return rc;
}

// BGZF -> its text: whole members go to the device and are inflated there, as pairs2bins reads .pairs.gz
static int decompress(FILE *fi, FILE *fo, const char *name, size_t chunk, int dev, bool &write_err) {
    const size_t CIN = chunk > (1u << 20) ? chunk : (1u << 20), OUT = CIN + 65536, MAXM = 65536;
    unsigned char *h_in = NULL, *h_out = NULL; void *d_in = NULL, *d_out = NULL; mk_bgzf *bz = NULL;
    if (mk_host_alloc(CIN, (void **)&h_in) != MK_OK || mk_host_alloc(OUT, (void **)&h_out) != MK_OK || mk_dev_alloc(dev, CIN, &d_in) != MK_OK ||
        mk_dev_alloc(dev, OUT, &d_out) != MK_OK || mk_bgzf_create(dev, MAXM, &bz) != MK_OK) return lib_fail();
    vector<mk_bgzf_member> mem(MAXM);
    size_t have = 0; uint64_t at = 0; bool in_eof = false; int rc = 0;
    while (!rc) {
        if (!in_eof) { const size_t got = fread(h_in + have, 1, CIN - have, fi); in_eof = got < CIN - have; have += got; }
        if (in_eof && ferror(fi)) { fprintf(stderr, "Error: reading %s failed\n", name); rc = 10; break; }
        if (have == 0) break;
        size_t nm = 0, nb = 0;
        if (mk_bgzf_scan(h_in, have, mem.data(), MAXM, &nm, &nb, NULL) != MK_OK) {
            const char *why = mk_last_error();
            fprintf(stderr, "Error: %s: compressed bytes from %llu on: %s%s\n", name, (unsigned long long)at, why,
                    strstr(why, "not BGZF") ? "; a single gzip stream cannot be inflated in parallel: use `gzip -dc`" : "");
            rc = 10; break;
        }
        if (nm == 0) {
            if (in_eof) { fprintf(stderr, "Error: %s: a truncated BGZF member at byte %llu\n", name, (unsigned long long)at); rc = 10; break; }
            continue;
        }
        size_t k = 0, out = 0;
        while (k < nm && (k == 0 || out + mem[k].isize <= OUT)) out += mem[k++].isize;
        const size_t cb = mem[k - 1].in_off + mem[k - 1].in_len;
        if (mk_copy_to_device(d_in, h_in, cb) != MK_OK) { rc = lib_fail(); break; }
        const int r = mk_bgzf_inflate_device(bz, d_in, mem.data(), k, d_out, OUT, NULL);
        if (r == MK_ERR_INPUT) { fprintf(stderr, "Error: %s: compressed bytes from %llu on: %s\n", name, (unsigned long long)at, mk_last_error()); rc = 10; break; }
        if (r != MK_OK || (out && mk_copy_to_host(h_out, d_out, out) != MK_OK)) { rc = lib_fail(); break; }
        if (out && fwrite(h_out, 1, out, fo) != out) { write_err = true; break; }
        at += cb; have -= cb;
        if (have) memmove(h_in, h_in + cb, have);
    }
    mk_bgzf_destroy(bz); mk_dev_free(d_in); mk_dev_free(d_out); mk_host_free(h_in); mk_host_free(h_out);
    return rc;
}

int main(int argc, char *argv[]) {
    bool to_stdout = false, dec = false, force = false, keep = false;
    int level = -1;
    vector<const char *> files;
    for (int a = 1; a < argc; ++a) {
        const char *s = argv[a];
        if (s[0] != '-' || !s[1]) { files.push_back(s); continue; }
        if (s[1] == '-') return usage(argv[0], 2);                      // no long options
        for (int j = 1; s[j]; ++j) {
            const char c = s[j];
            if (c == 'c') to_stdout = true;
            else if (c == 'd') dec = true;
            else if (c == 'f') force = true;
            else if (c == 'k') keep = true;
            else if (c == 'h') return usage(argv[0], 0);
            else if (c == 'l' || c == '@') {                            // -l6, -l 6, -@8, -@ 8
                const char *v = s[j + 1] ? s + j + 1 : a + 1 < argc ? argv[++a] : NULL;
                char *end = NULL;
                const long x = v ? strtol(v, &end, 10) : 0;
                if (!v || !*v || *end) return usage(argv[0], 2);
                if (c == 'l') { if (x < -1 || x > 9) return usage(argv[0], 2); level = (int)x; }
                break;
            } else return usage(argv[0], 2);
        }
    }
    if (files.size() > 1) return usage(argv[0], 2);
    const char *file = files.empty() || !strcmp(files[0], "-") ? NULL : files[0];
    string out_path;
    if (file && !to_stdout) {
        if (dec) {
            const size_t l = strlen(file);
            if (l < 4 || strcmp(file + l - 3, ".gz")) { fprintf(stderr, "Error: %s: unknown suffix (expected .gz)\n", file); return 10; }
            out_path.assign(file, l - 3);
        } else out_path = string(file) + ".gz";
        struct stat st;
        if (!force && stat(out_path.c_str(), &st) == 0) { fprintf(stderr, "Error: %s already exists; use -f to overwrite it\n", out_path.c_str()); return 10; }
    }
    FILE *fi = file ? fopen(file, "rb") : stdin;
    if (!fi) { fprintf(stderr, "Error: cannot read %s\n", file); return 10; }
    const int dev = getenv("MICROCKET_DEVICE") ? atoi(getenv("MICROCKET_DEVICE")) : 0;
    if (mk_device_count() < 1) { fprintf(stderr, "Error: no CUDA device: microcket_b200 has no CPU fallback\n"); return 20; }
    size_t chunk = (size_t)(getenv("MICROCKET_CHUNK_MB") ? atol(getenv("MICROCKET_CHUNK_MB")) : 256) << 20;
    chunk = chunk / BLOCK * BLOCK;
    if (chunk == 0) chunk = BLOCK;
    FILE *fo = out_path.empty() ? stdout : fopen(out_path.c_str(), "wb");
    if (!fo) { fprintf(stderr, "Error: cannot write %s\n", out_path.c_str()); return 10; }
    bool write_err = false;
    int rc = dec ? decompress(fi, fo, file ? file : "stdin", chunk, dev, write_err) : compress(fi, fo, level, chunk, dev, write_err);
    if (fflush(fo) != 0) write_err = true;
    if (fo != stdout && fclose(fo) != 0) write_err = true;
    if (!rc && write_err) { fprintf(stderr, "Error: writing %s failed\n", out_path.empty() ? "stdout" : out_path.c_str()); rc = 10; }
    if (fi != stdin) fclose(fi);
    if (rc) { if (!out_path.empty()) unlink(out_path.c_str()); return rc; }
    if (file && !to_stdout && !keep && unlink(file) != 0) { fprintf(stderr, "Error: cannot remove %s\n", file); return 10; }
    return 0;
}
