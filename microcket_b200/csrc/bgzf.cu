// bgzf.cu — BGZF members inflated in HBM (mk_bgzf_*): the input side of `pairs2bins x.pairs.gz`, and the first half of a
// device-side BAM decode.  A BGZF file is a chain of independent raw-deflate members of at most 64 KiB of output each, whose
// boundaries the host finds from their 18-byte headers (mk_bgzf_scan); every member is one job.
//   k_bgzf_inflate: one warp per member, a grid-stride loop over the call's members.  The warp decodes the symbols
//   warp-uniformly (every lane holds the same bit buffer; bgzf_member.h), builds the member's Huffman tables in its own
//   shared memory, and shares the copies: a literal run is gathered one byte per lane and stored 32 at a time, a match
//   or stored block is copied by all lanes.  Then every lane takes the CRC-32 and the '\n' count of one 32nd of the
//   output, and the partial CRCs are combined with the x^(8n) mod P shift.  A failing member sets the call's error word
//   to min(member index, reason): the first failing member in file order.  No floating point, no atomics on the output.
#include <algorithm>
#include <vector>
#include "mk_common.cuh"
#include "bgzf_member.h"

#define BG_WPB 4                                                  // warps (members in flight) per CTA

struct BgWarp {                                                    // the output side of bg_member for one warp
    int lane, nl;
    uint8_t *out; uint32_t cap, pos, npend, mine;                  // npend literals gathered, lane k holds the k-th
    const uint32_t *crc_tab, *x2n;
    uint32_t newlines; int32_t last_nl;                            // of the member's output, after crc()
    __device__ void sync() { __syncwarp(); }
    __device__ void flush() {
        if (lane < (int)npend) out[pos + lane] = (uint8_t)mine;
        pos += npend; npend = 0;
    }
    __device__ int lit(uint32_t c) {
        if (pos + npend >= cap) return BG_OVERFLOW;
        if (lane == (int)npend) mine = c;
        if (++npend == 32) flush();
        return 0;
    }
    __device__ int match(uint32_t len, uint32_t dist) {
        if (dist > pos + npend) return BG_TOO_FAR;
        if (pos + npend + len > cap) return BG_OVERFLOW;
        flush();
        __syncwarp();                                              // the bytes other lanes stored are visible
        // byte k comes from k - per for any multiple per of dist that reaches back to written bytes: per grows with them,
        // so a distance below the length takes log2(len / dist) rounds and no division
        for (uint32_t done = 0, per = dist; done < len; per = done + dist) {
            const uint32_t c = min(per, len - done);
            uint8_t *o = out + pos + done;
            for (uint32_t i = lane; i < c; i += 32) o[i] = o[(int)i - (int)per];
            done += c;
            if (done < len) __syncwarp();
        }
        pos += len;
        return 0;
    }
    __device__ int stored(const uint8_t *in, uint32_t len) {
        if (pos + npend + len > cap) return BG_OVERFLOW;
        flush();
        for (uint32_t i = lane; i < len; i += 32) out[pos + i] = in[i];
        pos += len;
        return 0;
    }
    __device__ uint32_t crc() {
        __syncwarp();
        const uint32_t per = (pos + 31) / 32, a = min(pos, per * lane), e = min(pos, a + per);
        uint32_t c = 0xffffffffu, nlc = 0; int32_t last = -1;
        for (uint32_t i = a; i < e; ++i) {
            const uint32_t b = out[i];
            c = crc_tab[(c ^ b) & 0xff] ^ (c >> 8);
            if (b == '\n') { ++nlc; last = (int32_t)i; }
        }
        c = bg_multmodp(bg_x8nmodp(pos - e, x2n), ~c);            // shifted past the bytes of the later lanes
        for (int s = 16; s; s >>= 1) {
            c ^= __shfl_xor_sync(0xffffffffu, c, s);
            nlc += __shfl_xor_sync(0xffffffffu, nlc, s);
            last = max(last, __shfl_xor_sync(0xffffffffu, last, s));
        }
        newlines = nlc; last_nl = last;
        return c;
    }
};

// err[0]: min(member << 8 | reason) over the failing members (~0: none); err[1]: '\n' bytes; err[2]: 1 + offset of the last '\n'
__global__ void __launch_bounds__(BG_WPB * 32, 8) k_bgzf_inflate(const uint8_t *__restrict__ in, const mk_bgzf_member *__restrict__ mem,
                                                               uint32_t n, uint8_t *out, unsigned long long *err) {
    __shared__ BgTables tabs[BG_WPB];
    __shared__ uint32_t crc_tab[256], x2n[32];
    for (int i = threadIdx.x; i < 256; i += BG_WPB * 32) crc_tab[i] = bg_crc_entry(i);
    if (threadIdx.x == 0) { uint32_t p = 1u << 30; for (int k = 0; k < 32; ++k) { x2n[k] = p; p = bg_multmodp(p, p); } }
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint32_t i = blockIdx.x * BG_WPB + wid; i < n; i += gridDim.x * BG_WPB) {
        const mk_bgzf_member mb = mem[i];
        BgWarp w;
        w.lane = lane; w.nl = 32; w.out = out + mb.out_off; w.cap = mb.isize; w.pos = 0; w.npend = 0; w.mine = 0;
        w.crc_tab = crc_tab; w.x2n = x2n; w.newlines = 0; w.last_nl = -1;
        const int r = bg_member(w, &tabs[wid], in + mb.in_off, mb.in_len, mb.isize);
        if (lane == 0) {
            if (r) atomicMin(&err[0], (unsigned long long)i << 8 | (unsigned)r);
            else {
                if (w.newlines) atomicAdd(&err[1], (unsigned long long)w.newlines);
                if (w.last_nl >= 0) atomicMax(&err[2], mb.out_off + (unsigned long long)w.last_nl + 1);
            }
        }
        __syncwarp();                                              // the tables are rebuilt by the next member
    }
}

struct mk_bgzf {
    int device = 0, grid_max = 148;
    size_t max_members = 0;
    DevBuf d_mem, d_err;
    PinBuf h_mem, h_err;
    uint64_t newlines = 0; int64_t last_nl = -1, launches = 0;
};

extern "C" int mk_bgzf_scan(const void *buf, size_t n, mk_bgzf_member *members, size_t cap, size_t *n_members, size_t *n_bytes, uint64_t *n_out) {
    if ((n && !buf) || (cap && !members) || !n_members) { mk_set_error("mk_bgzf_scan: bad argument"); return MK_ERR_ARG; }
    const uint8_t *p = (const uint8_t *)buf;
    size_t off = 0, k = 0; uint64_t out = 0;
    while (k < cap && off < n) {
        uint32_t len = 0, isize = 0; const char *why = "";
        const int r = bg_header(p + off, n - off, &len, &isize, &why);
        if (r < 0) { mk_set_error("mk_bgzf_scan: the member at byte %zu: %s", off, why); return MK_ERR_INPUT; }
        if (r > 0) break;
        members[k].in_off = off; members[k].in_len = len; members[k].out_off = out; members[k].isize = isize;
        off += len; out += isize; ++k;
    }
    *n_members = k;
    if (n_bytes) *n_bytes = off;
    if (n_out) *n_out = out;
    return MK_OK;
}

extern "C" int mk_bgzf_create(int device, size_t max_members, mk_bgzf **out) {
    if (!out || max_members == 0 || max_members >= (1ull << 32)) { mk_set_error("mk_bgzf_create: bad argument"); return MK_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(device));
    int per_sm = 0;
    MK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bgzf_inflate, BG_WPB * 32, 0));
    mk_bgzf *h = new mk_bgzf();
    h->device = device; h->max_members = max_members; h->grid_max = std::max(1, per_sm) * mk_sm_count(device);
    int rc = h->d_mem.alloc(max_members * sizeof(mk_bgzf_member));
    if (rc == MK_OK) rc = h->d_err.alloc(3 * 8);
    if (rc == MK_OK) rc = h->h_mem.alloc(max_members * sizeof(mk_bgzf_member));
    if (rc == MK_OK) rc = h->h_err.alloc(3 * 8);
    if (rc != MK_OK) { delete h; return rc; }
    *out = h;
    return MK_OK;
}

extern "C" void mk_bgzf_destroy(mk_bgzf *h) { if (h) { cudaSetDevice(h->device); delete h; } }

extern "C" int mk_bgzf_inflate_device(mk_bgzf *h, const void *d_in, const mk_bgzf_member *members, size_t n, void *d_out, size_t out_cap, void *stream) {
    if (!h || (n && (!d_in || !members || !d_out))) { mk_set_error("mk_bgzf_inflate_device: bad argument"); return MK_ERR_ARG; }
    if (n > h->max_members) { mk_set_error("mk_bgzf_inflate_device: %zu members, the object holds %zu", n, h->max_members); return MK_ERR_CAPACITY; }
    uint64_t total = 0;
    for (size_t i = 0; i < n; ++i) {
        const mk_bgzf_member &m = members[i];
        if (m.isize > BG_MAX_ISIZE || m.in_len < 20 || m.in_len > 65536 || m.out_off + m.isize > out_cap) {
            mk_set_error("mk_bgzf_inflate_device: member %zu: ISIZE %u, %u compressed bytes, output [%llu, +%u) of %zu", i, m.isize, m.in_len,
                         (unsigned long long)m.out_off, m.isize, out_cap);
            return MK_ERR_ARG;
        }
        total += m.isize;
    }
    if (total > out_cap) { mk_set_error("mk_bgzf_inflate_device: the members inflate to %llu bytes, out_cap %zu", (unsigned long long)total, out_cap); return MK_ERR_ARG; }
    h->newlines = 0; h->last_nl = -1;
    if (n == 0) return MK_OK;
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *he = h->h_err.as<unsigned long long>();
    MK_CUDA(cudaStreamSynchronize(s));                            // the staging buffers may still feed the previous call's copies
    memcpy(h->h_mem.p, members, n * sizeof(mk_bgzf_member));
    he[0] = ~0ull; he[1] = 0; he[2] = 0;
    MK_CUDA(cudaMemcpyAsync(h->d_mem.p, h->h_mem.p, n * sizeof(mk_bgzf_member), cudaMemcpyHostToDevice, s));
    MK_CUDA(cudaMemcpyAsync(h->d_err.p, h->h_err.p, 24, cudaMemcpyHostToDevice, s));
    const int grid = (int)std::min<size_t>((n + BG_WPB - 1) / BG_WPB, (size_t)h->grid_max);
    k_bgzf_inflate<<<grid, BG_WPB * 32, 0, s>>>((const uint8_t *)d_in, h->d_mem.as<mk_bgzf_member>(), (uint32_t)n, (uint8_t *)d_out,
                                                h->d_err.as<unsigned long long>());
    ++h->launches;
    MK_CUDA(cudaGetLastError());
    MK_CUDA(cudaMemcpyAsync(h->h_err.p, h->d_err.p, 24, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (he[0] != ~0ull) {
        const size_t i = (size_t)(he[0] >> 8);
        mk_set_error("BGZF member %zu (compressed bytes at %llu): %s", i, (unsigned long long)members[i].in_off, bg_reason((int)(he[0] & 0xff)));
        return MK_ERR_INPUT;
    }
    h->newlines = he[1]; h->last_nl = (int64_t)he[2] - 1;
    return MK_OK;
}

extern "C" int mk_bgzf_text_stats(mk_bgzf *h, uint64_t *newlines, int64_t *last_newline) {
    if (!h || !newlines || !last_newline) { mk_set_error("mk_bgzf_text_stats: bad argument"); return MK_ERR_ARG; }
    *newlines = h->newlines; *last_newline = h->last_nl;
    return MK_OK;
}

extern "C" uint64_t mk_bgzf_launch_count(mk_bgzf *h) { return h ? (uint64_t)h->launches : 0; }
