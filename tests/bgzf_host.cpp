// bgzf_host.cpp — the host form of the BGZF member decoder (microcket_b200/csrc/bgzf_member.h, the control logic the GPU
// kernel runs) for tests/test_bgzf.py, which builds it with AddressSanitizer into a temporary directory:
//   g++ -std=c++17 -g -O1 -fsanitize=address,undefined -I microcket_b200/csrc tests/bgzf_host.cpp -o <tmp>/bgzf_host
//   bgzf_host <file>...   for each file: walk its members, inflate each one, write the output to <file>.out and print
//                         "ok <bytes>" or "error: ..." (one line per file); a truncated last member is an error.
// Every member's compressed bytes and its output get heap blocks of exactly their size, so that a read or write outside
// them is an ASan report, not a silent pass.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "bgzf_member.h"

struct HostW {                                                         // the output side, one byte at a time
    int lane = 0, nl = 1;
    uint8_t *out = nullptr; uint32_t cap = 0, pos = 0;
    void sync() {}
    void flush() {}
    int lit(uint32_t c) { if (pos >= cap) return BG_OVERFLOW; out[pos++] = (uint8_t)c; return 0; }
    int match(uint32_t len, uint32_t dist) {
        if (dist > pos) return BG_TOO_FAR;
        if (pos + len > cap) return BG_OVERFLOW;
        for (uint32_t i = 0; i < len; ++i) out[pos + i] = out[pos + i - dist];
        pos += len;
        return 0;
    }
    int stored(const uint8_t *in, uint32_t len) {
        if (pos + len > cap) return BG_OVERFLOW;
        if (len) memcpy(out + pos, in, len);
        pos += len;
        return 0;
    }
    uint32_t crc() {
        uint32_t c = 0xffffffffu;
        for (uint32_t i = 0; i < pos; ++i) c = bg_crc_entry((c ^ out[i]) & 0xff) ^ (c >> 8);
        return ~c;
    }
};

static std::string run(const std::vector<uint8_t> &f, std::vector<uint8_t> &text) {
    BgTables *t = (BgTables *)malloc(sizeof(BgTables));
    std::string res;
    size_t off = 0, k = 0;
    while (off < f.size() && res.empty()) {
        uint32_t len = 0, isize = 0; const char *why = "";
        const int h = bg_header(f.data() + off, f.size() - off, &len, &isize, &why);
        if (h) { res = "error: member " + std::to_string(k) + " at byte " + std::to_string(off) + ": " + (h < 0 ? why : "truncated"); break; }
        uint8_t *m = (uint8_t *)malloc(len), *o = (uint8_t *)malloc(isize ? isize : 1);
        memcpy(m, f.data() + off, len);
        HostW w; w.out = o; w.cap = isize;
        const int r = bg_member(w, t, m, len, isize);
        if (r) res = "error: member " + std::to_string(k) + " at byte " + std::to_string(off) + ": " + bg_reason(r);
        else text.insert(text.end(), o, o + isize);
        free(m); free(o);
        off += len; ++k;
    }
    free(t);
    return res.empty() ? "ok " + std::to_string(text.size()) : res;
}

int main(int argc, char **argv) {
    for (int a = 1; a < argc; ++a) {
        std::vector<uint8_t> f, text;
        if (FILE *fi = fopen(argv[a], "rb")) {
            uint8_t buf[1 << 16]; size_t g;
            while ((g = fread(buf, 1, sizeof buf, fi)) > 0) f.insert(f.end(), buf, buf + g);
            fclose(fi);
        } else { printf("error: cannot read %s\n", argv[a]); continue; }
        const std::string r = run(f, text);
        if (r[0] == 'o') {
            FILE *fo = fopen((std::string(argv[a]) + ".out").c_str(), "wb");
            if (!text.empty()) fwrite(text.data(), 1, text.size(), fo);
            fclose(fo);
        }
        printf("%s\n", r.c_str());
    }
    return 0;
}
