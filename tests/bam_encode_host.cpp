// bam_encode_host.cpp — the host form of the SAM -> BAM record encoder (microcket_b200/csrc/bam_encode.h, the code every GPU
// thread of bam_out.cu runs on one line) for tests/test_bam_encode.py, which builds it with AddressSanitizer and UBSan:
//   g++ -std=c++17 -g -O1 -fsanitize=address,undefined -I microcket_b200/csrc tests/bam_encode_host.cpp -o <tmp>/bam_encode_host
//   bam_encode_host <refs> <in.sam> <out.bin>
// <refs>: one "name<TAB>length" line per reference.  Every line of <in.sam> is encoded (exact floats, strtof); the records go
// to <out.bin> back to back.  The first refused line prints "line <1-based> code <c>: <reason>" on stderr and exits 10.
// Each line gets a heap block of exactly its size (no newline), so that a read past it is an ASan report.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "bam_encode.h"

static bool slurp(const char *path, std::string &out) {
    FILE *f = fopen(path, "rb");
    if (!f) return false;
    char buf[1 << 16]; size_t g;
    while ((g = fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, g);
    fclose(f);
    return true;
}

int main(int argc, char **argv) {
    if (argc != 4) { fprintf(stderr, "usage: bam_encode_host <refs> <in.sam> <out.bin>\n"); return 2; }
    std::string refs, sam;
    if (!slurp(argv[1], refs) || !slurp(argv[2], sam)) return 1;
    std::string names; std::vector<uint32_t> off(1, 0);
    for (size_t p = 0; p < refs.size();) {
        size_t e = refs.find('\n', p); if (e == std::string::npos) e = refs.size();
        const size_t t = refs.find('\t', p);
        names.append(refs, p, t - p); off.push_back((uint32_t)names.size());
        p = e + 1;
    }
    const int n_ref = (int)off.size() - 1;
    uint32_t bits = 4;
    while ((1u << bits) < 2u * (uint32_t)n_ref + 2) ++bits;
    std::vector<int32_t> slot(1u << bits, 0);
    for (int k = 0; k < n_ref; ++k) {
        uint32_t h = be_hash(names.data() + off[k], off[k + 1] - off[k]) & ((1u << bits) - 1);
        while (slot[h]) h = (h + 1) & ((1u << bits) - 1);
        slot[h] = k + 1;
    }
    const BeDict d{names.data(), off.data(), slot.data(), (1u << bits) - 1, n_ref};
    FILE *fo = fopen(argv[3], "wb");
    if (!fo) return 1;
    uint64_t line = 0;
    for (size_t p = 0; p < sam.size();) {
        size_t e = sam.find('\n', p); if (e == std::string::npos) e = sam.size();
        ++line;
        const uint32_t n = (uint32_t)(e - p);
        char *ln = (char *)malloc(n ? n : 1);
        memcpy(ln, sam.data() + p, n);
        BeOut<false> c{nullptr, 0};
        bool patch = false;
        int r = be_line<false>(ln, n, d, true, c, &patch);
        if (r == BE_OK) {
            uint8_t *rec = (uint8_t *)malloc(c.at);
            BeOut<true> o{rec, 0};
            r = be_line<true>(ln, n, d, true, o, &patch);
            if (r == BE_OK && o.at != c.at) { fprintf(stderr, "line %llu: size pass %u, write pass %u\n", (unsigned long long)line, c.at, o.at); return 1; }
            if (r == BE_OK) fwrite(rec, 1, o.at, fo);
            free(rec);
        }
        free(ln);
        if (r != BE_OK) { fprintf(stderr, "line %llu code %d: %s\n", (unsigned long long)line, r, be_errstr[r]); fclose(fo); return 10; }
        p = e + 1;
    }
    fclose(fo);
    return 0;
}
