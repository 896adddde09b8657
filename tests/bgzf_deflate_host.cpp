// bgzf_deflate_host.cpp — the host form of the BGZF member encoder (microcket_b200/csrc/bgzf_deflate.h, the per-member
// decisions the GPU kernel makes) for tests/test_bgzf_deflate.py, which builds it with AddressSanitizer and UBSan:
//   g++ -std=c++17 -g -O1 -fsanitize=address,undefined -I microcket_b200/csrc tests/bgzf_deflate_host.cpp -o <tmp>/bgzf_deflate_host
//   bgzf_deflate_host c <level> <in> <out>   BGZF members of <in> (65 280-byte cuts, no EOF member) to <out>
//   bgzf_deflate_host h                      per stdin line "<maxlen> <count>...": prints the code lengths
// Every member's input and output get heap blocks of exactly their size, so that an access outside them is an ASan report.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sstream>
#include <string>
#include <vector>
#include "bgzf_deflate.h"

static int compress(int level, const char *in, const char *out) {
    std::vector<uint8_t> f;
    if (FILE *fi = fopen(in, "rb")) {
        uint8_t buf[1 << 16]; size_t g;
        while ((g = fread(buf, 1, sizeof buf, fi)) > 0) f.insert(f.end(), buf, buf + g);
        fclose(fi);
    } else return 1;
    FILE *fo = fopen(out, "wb");
    if (!fo) return 1;
    for (size_t off = 0; off < f.size(); off += BGD_BLOCK) {
        const uint32_t n = (uint32_t)(f.size() - off < BGD_BLOCK ? f.size() - off : BGD_BLOCK);
        uint8_t *m = (uint8_t *)malloc(n ? n : 1), *o = (uint8_t *)malloc(n + 31);
        memcpy(m, f.data() + off, n);
        const uint32_t len = bgd_member_host(m, n, level == 0, o);
        if (len > n + 31) { fprintf(stderr, "member of %u bytes for %u input bytes\n", len, n); return 1; }
        fwrite(o, 1, len, fo);
        free(m); free(o);
    }
    fclose(fo);
    return 0;
}

static int lengths() {
    std::string line;
    char buf[1 << 16];
    while (fgets(buf, sizeof buf, stdin)) {
        std::istringstream ss(buf);
        int maxlen; ss >> maxlen;
        std::vector<uint32_t> f; uint32_t v;
        while (ss >> v) f.push_back(v);
        BgdPlan *p = new BgdPlan();
        uint8_t *len = new uint8_t[f.size()];
        uint32_t *fa = new uint32_t[f.size()];
        for (size_t k = 0; k < f.size(); ++k) fa[k] = f[k];
        BgdHostTeam t;
        bgd_lengths(t, p, fa, (int)f.size(), maxlen, len);
        for (size_t k = 0; k < f.size(); ++k) printf(k ? " %d" : "%d", len[k]);
        printf("\n");
        delete p; delete[] len; delete[] fa;
    }
    return 0;
}

int main(int argc, char **argv) {
    if (argc == 5 && !strcmp(argv[1], "c")) return compress(atoi(argv[2]), argv[3], argv[4]);
    if (argc == 2 && !strcmp(argv[1], "h")) return lengths();
    fprintf(stderr, "usage: bgzf_deflate_host c <level> <in> <out> | h\n");
    return 2;
}
