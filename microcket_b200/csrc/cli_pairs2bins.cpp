// cli_pairs2bins.cpp — contact binning of a .pairs file on the GPU (new tool; stands where the driver calls
// `java -jar juicer_tools.jar pre -r <res,...> <sid>.final.pairs <sid>.hic <genome>.info`, microcket:525-529).
//   pairs2bins [-d] [-b] [-H <out.hic>] [-g <genomeId>] -r <res[,res...]> <in.pairs|-> <out.prefix> <genome.info>
// Writes <out.prefix>.<res>.coo with `bin1<TAB>bin2<TAB>count` (upper triangle, sorted), bins numbered in .info order with
// bin = offset[chr] + pos / res.  -d removes coordinate duplicates first (first occurrence wins).
// -b also writes <out.prefix>.<res>.bins.bed (`chrom<TAB>start<TAB>end`, one line per bin id): the pair of files is what
// `cooler load -f coo <bins.bed> <coo> out.cool` takes, i.e. the hand-over point to the .cool branch of the driver
// (microcket:531-551) without `cooler cload pairs` re-reading and re-binning the pairs.
// The file is streamed in 256 MiB chunks from pinned memory and PARSED ON THE GPU (mk_pairs_parse_text_device); resolutions
// whose upper triangle fits MICROCKET_DENSE_MB (default 4096) all come from one pass of the dense histogram (mk_hist_*), the
// finer ones from the sort path.
// -H <out.hic> also packs every resolution's counts into one `.hic` (version 8) container, i.e. the file the driver's
// `juicer_tools pre` call produces (host code over the arrays copied back for the .coo files: hic_writer.hpp; -g names the
// genome in its header, default: the .info file's stem).
// -n <types> (with -H; any of VC,VC_SQRT,KR, comma separated) also balances every resolution's matrices on the GPU (norm.cu,
// mk_norm_device on the COO while it is still in device memory) and stores the normalisation vectors and the normalised
// expected values in the container, what `juicer_tools pre` computes by default (and `addNorm` adds to a file without them).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>
#include "../../include/microcket_b200.h"
#include "hic_writer.hpp"
using namespace std;

#define CHECK(call) do { if ((call) != MK_OK) { cerr << "Error: " << mk_last_error() << "\n"; return 20; } } while (0)

static hic::Writer *g_hic = NULL;                                         // -H: every resolution's arrays also go into the container
static int g_norm_types = 0, g_dev = 0;                                   // -n: MK_NORM_* bits
static vector<uint32_t> g_len; static vector<string> g_names;

// -n: the resolution's normalisation vectors from its device COO, copied to the host for the writer
static int balance(uint32_t res, const void *d_b1, const void *d_b2, const void *d_ct, size_t nnz, vector<vector<double>> &vals, vector<hic::NormInput> &norms) {
    static const char *names[3] = {"VC", "VC_SQRT", "KR"};
    uint64_t nb = 0; CHECK(mk_hist_cells(g_len.data(), (int)g_len.size(), res, &nb, NULL));
    mk_norm *nm = NULL;
    CHECK(mk_norm_create(g_dev, g_len.data(), (int)g_len.size(), res, nnz, &nm));
    void *d_out[3] = {NULL, NULL, NULL};
    for (int t = 0; t < 3; ++t) if (g_norm_types & (1 << t)) CHECK(mk_dev_alloc(g_dev, nb * 8 + 8, &d_out[t]));
    vector<uint8_t> status(g_len.size(), 0); mk_norm_stats st;
    CHECK(mk_norm_device(nm, (const uint32_t *)d_b1, (const uint32_t *)d_b2, (const uint32_t *)d_ct, nnz, g_norm_types,
                         (double *)d_out[0], (double *)d_out[1], (double *)d_out[2], status.data(), &st, NULL));
    mk_norm_destroy(nm);
    vals.assign(3, vector<double>());
    for (int t = 0; t < 3; ++t) {
        if (!d_out[t]) continue;
        vals[t].resize(nb);
        CHECK(mk_copy_to_host(vals[t].data(), d_out[t], nb * 8));
        mk_dev_free(d_out[t]);
        hic::NormInput q; q.type = names[t]; q.values = vals[t].data();
        for (size_t c = 0; c < g_len.size(); ++c) q.stored.push_back(status[c] == 0 || (status[c] == 2 && t < 2));
        norms.push_back(q);
    }
    if (g_norm_types & MK_NORM_KR) {
        string failed;
        for (size_t c = 0; c < g_len.size(); ++c) if (status[c] == 2) failed += (failed.empty() ? "" : ", ") + g_names[c];
        cerr << "INFO: KR at " << res << " bp: " << st.kr_matvecs << " steps, " << st.kr_failed << " chromosome(s) failed"
             << (failed.empty() ? "" : ": " + failed) << ".\n";
    }
    return 0;
}

static int write_coo(const string &prefix, uint32_t res, const void *d_b1, const void *d_b2, const void *d_ct, size_t nnz) {
    const string path = prefix + "." + to_string(res) + ".coo";
    vector<vector<double>> vals; vector<hic::NormInput> norms;           // before the copy: the device arrays are reused afterwards
    if (g_norm_types) if (int rc = balance(res, d_b1, d_b2, d_ct, nnz, vals, norms)) return rc;
    vector<uint32_t> b1(nnz + 1), b2(nnz + 1), ct(nnz + 1);
    if (nnz) { CHECK(mk_copy_to_host(b1.data(), d_b1, nnz * 4)); CHECK(mk_copy_to_host(b2.data(), d_b2, nnz * 4)); CHECK(mk_copy_to_host(ct.data(), d_ct, nnz * 4)); }
    if (g_hic) { string err; if (g_hic->add(res, b1.data(), b2.data(), ct.data(), nnz, &err, g_norm_types ? &norms : NULL)) { cerr << "Error: " << err << "\n"; return 10; } }
    FILE *fo = fopen(path.c_str(), "w");
    if (!fo) { cerr << "Error: cannot write " << path << "\n"; return 10; }
    static char big[1 << 22];
    setvbuf(fo, big, _IOFBF, sizeof big);
    for (size_t i = 0; i < nnz; ++i) fprintf(fo, "%u\t%u\t%u\n", b1[i], b2[i], ct[i]);
    fclose(fo);
    return 0;
}

int main(int argc, char *argv[]) {
    bool dedup = false, bins_bed = false; string reslist, hic_path, genome, normlist;
    int a = 1;
    while (a < argc && argv[a][0] == '-' && argv[a][1]) {
        if (!strcmp(argv[a], "-d")) { dedup = true; ++a; }
        else if (!strcmp(argv[a], "-b")) { bins_bed = true; ++a; }
        else if (!strcmp(argv[a], "-r") && a + 1 < argc) { reslist = argv[a + 1]; a += 2; }
        else if (!strcmp(argv[a], "-H") && a + 1 < argc) { hic_path = argv[a + 1]; a += 2; }
        else if (!strcmp(argv[a], "-g") && a + 1 < argc) { genome = argv[a + 1]; a += 2; }
        else if (!strcmp(argv[a], "-n") && a + 1 < argc) { normlist = argv[a + 1]; a += 2; }
        else break;
    }
    if (!normlist.empty()) {
        stringstream ss(normlist); string t;
        while (getline(ss, t, ',')) {
            if (t == "VC") g_norm_types |= MK_NORM_VC;
            else if (t == "VC_SQRT") g_norm_types |= MK_NORM_VC_SQRT;
            else if (t == "KR") g_norm_types |= MK_NORM_KR;
            else { cerr << "Error: unknown normalisation '" << t << "' (VC, VC_SQRT, KR)\n"; return 2; }
        }
    }
    if (argc - a < 3 || reslist.empty() || (!normlist.empty() && hic_path.empty())) {
        cerr << "\nUsage: " << argv[0] << " [-d] [-b] [-H <out.hic> [-n VC,VC_SQRT,KR]] [-g <genomeId>] -r <res[,res...]> <in.pairs|-> <out.prefix> <genome.info>\n\n";
        return 2;
    }
    vector<uint32_t> res;
    { stringstream ss(reslist); string t; while (getline(ss, t, ',')) if (!t.empty()) res.push_back((uint32_t)strtoul(t.c_str(), NULL, 10)); }
    for (uint32_t r : res) if (r == 0) { cerr << "Error: resolution 0\n"; return 2; }
    vector<string> names; vector<uint32_t> chr_len;
    { ifstream fi(argv[a + 2]); if (fi.fail()) { cerr << "Error: cannot read " << argv[a + 2] << "\n"; return 10; }
      string n; uint32_t l; while (fi >> n >> l) { names.push_back(n); chr_len.push_back(l); } }
    if (names.empty()) { cerr << "Error: no chromosomes in " << argv[a + 2] << "\n"; return 10; }
    vector<const char *> cnames; for (auto &s : names) cnames.push_back(s.c_str());
    if (!hic_path.empty()) {
        if (genome.empty()) {                                            // hg38.info -> hg38, as the driver names its genomes
            genome = argv[a + 2];
            const size_t sl = genome.find_last_of('/'); if (sl != string::npos) genome = genome.substr(sl + 1);
            const size_t dt = genome.find_last_of('.'); if (dt != string::npos && dt > 0) genome = genome.substr(0, dt);
        }
        g_hic = new hic::Writer(genome, names, chr_len, res);
    }
    if (bins_bed) for (uint32_t r : res) {                                // bin id = line number: chromosomes in .info order, pos / res
        const string path = string(argv[a + 1]) + "." + to_string(r) + ".bins.bed";
        FILE *fb = fopen(path.c_str(), "w");
        if (!fb) { cerr << "Error: cannot write " << path << "\n"; return 10; }
        for (size_t c = 0; c < names.size(); ++c)
            for (uint64_t s0 = 0; s0 <= chr_len[c]; s0 += r) {           // pos / res of a 1-based pos <= len: bins 0 .. len / res
                const uint64_t e0 = s0 + r < (uint64_t)chr_len[c] + 1 ? s0 + r : (uint64_t)chr_len[c] + 1;
                fprintf(fb, "%s\t%llu\t%llu\n", names[c].c_str(), (unsigned long long)s0, (unsigned long long)e0);
            }
        fclose(fb);
    }
    FILE *fp = strcmp(argv[a], "-") ? fopen(argv[a], "rb") : stdin;
    if (!fp) { cerr << "Error: cannot read " << argv[a] << "\n"; return 10; }
    const int dev = getenv("MICROCKET_DEVICE") ? atoi(getenv("MICROCKET_DEVICE")) : 0;
    g_dev = dev; g_len = chr_len; g_names = names;
    if (mk_device_count() < 1) { cerr << "Error: no CUDA device: microcket_b200 has no CPU fallback\n"; return 20; }

    // ---- stream the text to the GPU and parse it there
    const size_t CHUNK = (size_t)(getenv("MICROCKET_CHUNK_MB") ? atol(getenv("MICROCKET_CHUNK_MB")) : 256) << 20;
    size_t cap = 1u << 22;                                               // pairs capacity, grown as the file goes by
    void *d_pairs = NULL, *d_text = NULL; char *h_text = NULL;
    CHECK(mk_dev_alloc(dev, cap * sizeof(mk_pair), &d_pairs));
    CHECK(mk_dev_alloc(dev, CHUNK + 64, &d_text));
    CHECK(mk_host_alloc(CHUNK + 64, (void **)&h_text));
    mk_pairs_ws *pws = NULL;                                             // parser workspace (sized per chunk: a line is >= 14 bytes)
    const size_t chunk_lines = CHUNK / 14 + 16;
    CHECK(mk_pairs_ws_create(dev, chunk_lines, &pws));
    size_t n = 0, have = 0, skipped = 0;
    while (true) {
        const size_t got = fread(h_text + have, 1, CHUNK - have, fp);
        const bool eof = got == 0;
        size_t tot = have + got;
        if (tot == 0) break;
        size_t cut = tot;
        if (!eof) { while (cut > 0 && h_text[cut - 1] != '\n') --cut; if (cut == 0) { if (tot == CHUNK) { cerr << "Error: a line longer than " << CHUNK << " bytes\n"; return 10; } have = tot; continue; } }
        else if (h_text[tot - 1] != '\n') { h_text[tot++] = '\n'; cut = tot; }   // last line without a newline
        size_t lines_max = 0; for (size_t i = 0; i < cut; ++i) lines_max += h_text[i] == '\n';
        if (n + lines_max > cap) {                                       // grow the pair array (device-to-device copy of what is there)
            size_t ncap = cap; while (ncap < n + lines_max) ncap *= 2;
            void *bigger = NULL;
            CHECK(mk_dev_alloc(dev, ncap * sizeof(mk_pair), &bigger));
            if (n) CHECK(mk_copy_device(bigger, d_pairs, n * sizeof(mk_pair)));
            mk_dev_free(d_pairs); d_pairs = bigger; cap = ncap;
        }
        CHECK(mk_copy_to_device(d_text, h_text, cut));
        size_t nl = 0, ns = 0;
        CHECK(mk_pairs_parse_text_device(pws, (const char *)d_text, cut, cnames.data(), (int)cnames.size(), (mk_pair *)d_pairs + n, cap - n, &nl, &ns, NULL));
        n += nl; skipped += ns;
        have = tot - cut;
        if (have) memmove(h_text, h_text + cut, have);
        if (eof) break;
    }
    if (fp != stdin) fclose(fp);
    mk_pairs_ws_destroy(pws); mk_dev_free(d_text); mk_host_free(h_text);

    // ---- bins
    mk_pairs_ws *ws = NULL;
    CHECK(mk_pairs_ws_create(dev, n + 1, &ws));
    void *d_b1 = NULL, *d_b2 = NULL, *d_ct = NULL;
    CHECK(mk_dev_alloc(dev, (n + 1) * 4, &d_b1)); CHECK(mk_dev_alloc(dev, (n + 1) * 4, &d_b2)); CHECK(mk_dev_alloc(dev, (n + 1) * 4, &d_ct));
    const double dense_budget = (double)(getenv("MICROCKET_DENSE_MB") ? atol(getenv("MICROCKET_DENSE_MB")) : 4096) * 1048576.0;
    vector<int> dense, sparse; double used = 0;
    {   // coarsest first into the dense set while the triangles fit the budget
        vector<int> order(res.size()); for (size_t k = 0; k < res.size(); ++k) order[k] = (int)k;
        for (size_t i = 0; i < order.size(); ++i) for (size_t j = i + 1; j < order.size(); ++j) if (res[order[j]] > res[order[i]]) swap(order[i], order[j]);
        for (int k : order) {
            uint64_t nb = 0, nc = 0; CHECK(mk_hist_cells(chr_len.data(), (int)chr_len.size(), res[k], &nb, &nc));
            if (used + nc * 4.0 <= dense_budget && dense.size() < 12) { dense.push_back(k); used += nc * 4.0; } else sparse.push_back(k);
        }
    }
    size_t m = n;                                                        // pairs after duplicate removal
    bool deduped = !dedup;
    if (dedup) {                                                         // one sort: duplicates out, and the finest sparse resolution's COO for free
        int k = sparse.empty() ? -1 : sparse.back();
        for (int q : sparse) if (res[q] < res[k]) k = q;
        const uint32_t r0 = k >= 0 ? res[k] : 5000u;
        size_t kept = 0, nnz = 0;
        CHECK(mk_pairs_dedup_bin_device(ws, (mk_pair *)d_pairs, n, chr_len.data(), (int)chr_len.size(), NULL, 0, r0, 0,
                                        (uint32_t *)d_b1, (uint32_t *)d_b2, (uint32_t *)d_ct, n + 1, &kept, &nnz, NULL));
        m = kept; deduped = true;
        if (k >= 0) {
            if (int rc = write_coo(argv[a + 1], res[k], d_b1, d_b2, d_ct, nnz)) return rc;
            vector<int> rest; for (int q : sparse) if (q != k) rest.push_back(q);
            sparse = rest;
        }
    }
    (void)deduped;
    for (int k : sparse) {
        size_t nnz = 0;
        CHECK(mk_pairs_bin_device(ws, (const mk_pair *)d_pairs, m, chr_len.data(), (int)chr_len.size(), NULL, 0, res[k],
                                  (uint32_t *)d_b1, (uint32_t *)d_b2, (uint32_t *)d_ct, n + 1, &nnz, NULL));
        if (int rc = write_coo(argv[a + 1], res[k], d_b1, d_b2, d_ct, nnz)) return rc;
    }
    if (!dense.empty()) {
        vector<uint32_t> dres; for (int k : dense) dres.push_back(res[k]);
        mk_hist *h = NULL;
        CHECK(mk_hist_create(dev, chr_len.data(), (int)chr_len.size(), dres.data(), (int)dres.size(), NULL, &h));
        CHECK(mk_hist_add_device(h, (const mk_pair *)d_pairs, m, NULL, 0, NULL));
        for (size_t i = 0; i < dense.size(); ++i) {
            size_t nnz = 0; uint64_t total = 0;
            CHECK(mk_hist_coo_device(h, (int)i, (uint32_t *)d_b1, (uint32_t *)d_b2, (uint32_t *)d_ct, n + 1, &nnz, &total, NULL));
            if (int rc = write_coo(argv[a + 1], dres[i], d_b1, d_b2, d_ct, nnz)) return rc;
        }
        mk_hist_destroy(h);
    }
    cerr << "INFO: " << n << " lines, " << skipped << " of them headers / unknown chromosomes; " << m << " pairs binned"
         << (dedup ? " after duplicate removal" : "") << " at " << res.size() << " resolutions (" << dense.size() << " dense).\n";
    mk_pairs_ws_destroy(ws); mk_dev_free(d_pairs); mk_dev_free(d_b1); mk_dev_free(d_b2); mk_dev_free(d_ct);
    if (g_hic) { string err; if (g_hic->write(hic_path, &err)) { cerr << "Error: " << err << "\n"; return 10; } }
    return 0;
}
