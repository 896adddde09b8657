// bgzf_deflate.cu — BGZF members written in HBM (mk_bgzf_deflate_device): the output side of `bgzip`, the counterpart of
// bgzf.cu.  Member k holds input bytes [k * 65 280, (k + 1) * 65 280), the cut bgzip makes; members are independent jobs.
//   k_bgzf_deflate: one CTA per member, a grid-stride loop over the call's members.  The member's input is staged in shared
//   memory.  Every thread takes the CRC-32 of 256 bytes; the partial CRCs are combined with the x^(8n) mod P shift.  Warp 0
//   sweeps the member 32 positions at a time: the head-table candidate of each position (__match_any_sync finds the latest
//   earlier lane with the same hash, so the table is updated as if one position at a time), and the greedy walk over the
//   tokens that start in those 32 positions (match lengths compared by the whole warp).  Token starts and match starts
//   go to two bit masks, match lengths and distances to a per-CTA scratch.  Then the CTA counts symbols, one thread builds
//   the codes (bgzf_deflate.h), every thread sizes the tokens of its 256 positions, a CTA scan gives each one its bit
//   offset, and every thread writes its bits: words it shares with a neighbour are ORed in, so the words do not depend
//   on which thread comes first.  The member goes to a staging slot of 65 316 bytes.
//   k_bgzf_offsets: one CTA, the exclusive sum of the member sizes.   k_bgzf_pack: the members back to back.
// No floating point; the only atomics are integer counts and ORs into zeroed words, whose results do not depend on order.
#include <algorithm>
#include <vector>
#include "mk_common.cuh"
#include "bgzf_deflate.h"

#define BGD_NT 256                                            // threads per CTA: thread t owns positions [256 t, 256 t + 256)
#define BGD_SLOT 65316u                                       // staging bytes per member (>= 2 + BGD_STORED_MAX, a multiple of 4)
#define BGD_WORDS (BGD_BLOCK / 32)                            // mask words per member
#define BGD_SCRATCH (2 * BGD_WORDS + BGD_BLOCK / 4)           // per-CTA scratch words: two masks, matches indexed by position / 4

struct BgdCta { int lane, nl; __device__ void sync() { __syncthreads(); } };
struct BgdDevSink {
    uint32_t *w;
    __device__ void word(uint32_t i, uint32_t v, bool shared) { if (shared) atomicOr(&w[i], v); else w[i] = v; }
};

struct BgdShared {
    uint8_t in[BGD_BLOCK];
    union {                                                    // one phase at a time
        uint16_t head[1u << BGD_HBITS];
        uint32_t crc_tab[256];
        BgdPlan plan;
    } u;
    uint32_t x2n[32], part[BGD_NT / 32], scan[BGD_NT / 32];
    uint32_t crc;
};

// the candidate sweep and the greedy walk of one member (warp 0)
__device__ void bgd_sweep(BgdShared &S, uint32_t n, uint32_t *mstart, uint32_t *mmatch, uint32_t *tok, int lane) {
    uint32_t p = 0;                                            // the next token start (warp-uniform)
    for (uint32_t g = 0; g < n; g += 32) {
        const uint32_t i = g + lane;
        const bool v = i + 4 <= n;
        const uint32_t h = v ? bgd_hash(S.in + i) : (1u << BGD_HBITS) + lane;
        const uint32_t peers = __match_any_sync(0xffffffffu, h), below = peers & ((1u << lane) - 1);
        uint32_t c = below ? g + 31 - __clz(below) : v ? S.u.head[h] : BGD_NONE;
        const bool ok = v && c != BGD_NONE && i - c <= 32768 && S.in[c] == S.in[i] && S.in[c + 1] == S.in[i + 1] &&
                        S.in[c + 2] == S.in[i + 2] && S.in[c + 3] == S.in[i + 3];
        __syncwarp();
        if (v && (peers >> lane) == 1) S.u.head[h] = (uint16_t)i;   // the latest lane of each hash
        const uint32_t vm = __ballot_sync(0xffffffffu, ok);
        const uint32_t in_n = n - g >= 32 ? 0xffffffffu : (1u << (n - g)) - 1;
        uint32_t st = 0, ms = 0;
        while (p < g + 32 && p < n) {
            const uint32_t k = p - g, rest = vm >> k;
            if (!rest) { st |= (0xffffffffu << k) & in_n; p = g + 32; break; }
            const uint32_t j = k + __ffs(rest) - 1;
            st |= (j == 31 ? 0xffffffffu : (2u << j) - 1) & (0xffffffffu << k);   // literals k..j-1, the match at j
            ms |= 1u << j;
            const uint32_t q = g + j, cq = __shfl_sync(0xffffffffu, c, j), maxl = min(258u, n - q);
            uint32_t len = maxl;
            for (uint32_t o = 4; o < maxl; o += 32) {              // the first 4 bytes are equal
                const uint32_t x = o + lane;
                const uint32_t miss = __ballot_sync(0xffffffffu, x < maxl && S.in[cq + x] != S.in[q + x]);
                if (miss) { len = o + __ffs(miss) - 1; break; }
            }
            if (lane == 0) tok[q >> 2] = len | (q - cq - 1) << 16;
            p = q + len;
        }
        if (lane == 0) { mstart[g >> 5] = st; mmatch[g >> 5] = ms; }
    }
}

__global__ void __launch_bounds__(BGD_NT, 2) k_bgzf_deflate(const uint8_t *__restrict__ in, uint64_t n_in, uint32_t n_mem, int stored_only,
                                                           uint8_t *stage, uint32_t *sizes, uint32_t *scratch) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    BgdShared &S = *(BgdShared *)smem_raw;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    uint32_t *mstart = scratch + (size_t)blockIdx.x * BGD_SCRATCH, *mmatch = mstart + BGD_WORDS, *tok = mmatch + BGD_WORDS;
    if (tid == 0) { uint32_t p = 1u << 30; for (int k = 0; k < 32; ++k) { S.x2n[k] = p; p = bg_multmodp(p, p); } }
    BgdCta team{tid, BGD_NT};
    for (uint32_t k = blockIdx.x; k < n_mem; k += gridDim.x) {
        const uint64_t off = (uint64_t)k * BGD_BLOCK;
        const uint32_t n = (uint32_t)(n_in - off < BGD_BLOCK ? n_in - off : BGD_BLOCK);
        const uint8_t *src = in + off;
        uint8_t *slot = stage + (size_t)k * BGD_SLOT;
        uint32_t *dw = (uint32_t *)(slot + 20);                // the deflate data, word-aligned; the header goes in [2, 20)
        if (((uintptr_t)src & 15) == 0) {
            for (uint32_t i = tid; i < n / 16; i += BGD_NT) ((uint4 *)S.in)[i] = __ldg((const uint4 *)src + i);
            for (uint32_t i = n / 16 * 16 + tid; i < n; i += BGD_NT) S.in[i] = src[i];
        } else for (uint32_t i = tid; i < n; i += BGD_NT) S.in[i] = src[i];
        S.u.crc_tab[tid] = bg_crc_entry(tid);
        __syncthreads();
        {                                                      // CRC-32 of the member's input
            const uint32_t a = min(n, (uint32_t)tid * 256), e = min(n, a + 256);
            uint32_t c = 0xffffffffu;
            for (uint32_t i = a; i < e; ++i) c = S.u.crc_tab[(c ^ S.in[i]) & 0xff] ^ (c >> 8);
            c = bg_multmodp(bg_x8nmodp(n - e, S.x2n), ~c);     // shifted past the bytes of the later threads
            for (int s = 16; s; s >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, s);
            if (lane == 0) S.part[wid] = c;
        }
        __syncthreads();
        if (tid == 0) { uint32_t c = 0; for (int w = 0; w < BGD_NT / 32; ++w) c ^= S.part[w]; S.crc = c; }
        uint32_t dbytes;
        if (stored_only) dbytes = n + 5;
        else {
            for (uint32_t i = tid; i < (1u << BGD_HBITS) / 2; i += BGD_NT) ((uint32_t *)S.u.head)[i] = 0xffffffffu;
            __syncthreads();
            if (wid == 0) bgd_sweep(S, n, mstart, mmatch, tok, lane);
            __syncthreads();
            BgdPlan *P = &S.u.plan;
            for (int s = tid; s < BGD_NL; s += BGD_NT) P->fl[s] = s == 256;
            if (tid < BGD_ND) P->fd[tid] = 0;
            __syncthreads();
            const uint32_t w0 = tid * 8, w1 = min(w0 + 8, (n + 31) / 32);
            for (uint32_t w = w0; w < w1; ++w) {               // symbol counts of the thread's tokens
                uint32_t st = mstart[w];
                const uint32_t ms = mmatch[w];
                while (st) {
                    const uint32_t b = __ffs(st) - 1, q = w * 32 + b;
                    st &= st - 1;
                    if (ms >> b & 1) {
                        const uint32_t t = tok[q >> 2], len = t & 0xffff, dist = (t >> 16) + 1;
                        uint32_t s, e, nb;
                        bgd_len_sym(len, s, e, nb); atomicAdd(&P->fl[s], 1u);
                        bgd_dist_sym(dist, s, e, nb); atomicAdd(&P->fd[s], 1u);
                    } else atomicAdd(&P->fl[S.in[q]], 1u);
                }
            }
            __syncthreads();
            bgd_plan(team, P, n);
            if (P->btype == 0) dbytes = n + 5;
            else {
                uint32_t bits = 0;                             // the thread's token bits, then its offset from a CTA scan
                for (uint32_t w = w0; w < w1; ++w) {
                    uint32_t st = mstart[w];
                    const uint32_t ms = mmatch[w];
                    while (st) {
                        const uint32_t b = __ffs(st) - 1, q = w * 32 + b;
                        st &= st - 1;
                        if (ms >> b & 1) { const uint32_t t = tok[q >> 2]; bits += bgd_match_bits(P, t & 0xffff, (t >> 16) + 1); }
                        else bits += bgd_lit_bits(P, S.in[q]);
                    }
                }
                uint32_t x = bits;
                for (int s = 1; s < 32; s <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, s); if (lane >= s) x += y; }
                if (lane == 31) S.scan[wid] = x;
                __syncthreads();
                uint32_t before = x - bits;
                for (int w = 0; w < wid; ++w) before += S.scan[w];
                dbytes = (uint32_t)((P->bits + 7) / 8);
                for (uint32_t i = tid; i < (dbytes + 3) / 4; i += BGD_NT) dw[i] = 0;
                __syncthreads();
                BgdBits<BgdDevSink> out; out.s.w = dw;
                out.init(P->hdr_bits + before);
                for (uint32_t w = w0; w < w1; ++w) {
                    uint32_t st = mstart[w];
                    const uint32_t ms = mmatch[w];
                    while (st) {
                        const uint32_t b = __ffs(st) - 1, q = w * 32 + b;
                        st &= st - 1;
                        if (ms >> b & 1) { const uint32_t t = tok[q >> 2]; bgd_put_match(out, P, t & 0xffff, (t >> 16) + 1); }
                        else bgd_put_lit(out, P, S.in[q]);
                    }
                }
                out.finish();
                if (tid == 0) {
                    BgdBits<BgdDevSink> h; h.s.w = dw;
                    h.init(0); bgd_put_header(h, P); h.finish();
                    h.init(P->bits - P->ll[256]); bgd_put_lit(h, P, 256); h.finish();
                }
            }
        }
        const bool stored = stored_only || S.u.plan.btype == 0;
        if (stored) {
            uint8_t *d = slot + 20;
            for (uint32_t i = tid; i < n; i += BGD_NT) d[5 + i] = S.in[i];
            if (tid == 0) { d[0] = 1; d[1] = (uint8_t)n; d[2] = (uint8_t)(n >> 8); d[3] = (uint8_t)~n; d[4] = (uint8_t)(~n >> 8); }
        }
        __syncthreads();                                       // the deflate bytes are complete: the trailer may follow them
        if (tid == 0) {
            const uint32_t total = 18 + dbytes + 8;
            bgd_member_header(slot + 2, total);
            bgd_put32(slot + 20 + dbytes, S.crc); bgd_put32(slot + 24 + dbytes, n);
            sizes[k] = total;
        }
        __syncthreads();                                       // shared memory is reused by the next member
    }
}

// off[k] = sum of sizes[0..k), off[n] = the total (one CTA; the thread sums are added in thread order)
__global__ void __launch_bounds__(1024) k_bgzf_offsets(const uint32_t *sizes, uint32_t n, uint64_t *off) {
    __shared__ uint64_t part[1024];
    const uint32_t per = (n + 1023) / 1024, a = min(n, threadIdx.x * per), e = min(n, a + per);
    uint64_t s = 0;
    for (uint32_t i = a; i < e; ++i) s += sizes[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) { uint64_t acc = 0; for (int t = 0; t < 1024; ++t) { const uint64_t v = part[t]; part[t] = acc; acc += v; } off[n] = acc; }
    __syncthreads();
    s = part[threadIdx.x];
    for (uint32_t i = a; i < e; ++i) { off[i] = s; s += sizes[i]; }
}

__global__ void __launch_bounds__(BGD_NT) k_bgzf_pack(const uint8_t *stage, const uint32_t *sizes, const uint64_t *off, uint32_t n, uint8_t *out) {
    for (uint32_t k = blockIdx.x; k < n; k += gridDim.x) {
        const uint8_t *s = stage + (size_t)k * BGD_SLOT + 2;
        uint8_t *d = out + off[k];
        const uint32_t len = sizes[k];
        for (uint32_t i = threadIdx.x; i < len; i += BGD_NT) d[i] = s[i];
    }
}

struct mk_bgzf_enc {
    int device = 0, grid_max = 148;
    size_t max_bytes = 0, max_members = 0;
    DevBuf d_stage, d_sizes, d_off, d_scratch;
    PinBuf h_sizes;
    int64_t launches = 0;
};

extern "C" size_t mk_bgzf_deflate_bound(size_t n) { return n + (n + BGD_BLOCK - 1) / BGD_BLOCK * 31; }

extern "C" int mk_bgzf_enc_create(int device, size_t max_bytes, mk_bgzf_enc **out) {
    if (!out || max_bytes == 0 || max_bytes / BGD_BLOCK >= (1ull << 31)) { mk_set_error("mk_bgzf_enc_create: bad argument"); return MK_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(device));
    MK_CUDA(cudaFuncSetAttribute(k_bgzf_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BgdShared)));
    int per_sm = 0;
    MK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bgzf_deflate, BGD_NT, sizeof(BgdShared)));
    mk_bgzf_enc *h = new mk_bgzf_enc();
    h->device = device; h->max_bytes = max_bytes; h->max_members = (max_bytes + BGD_BLOCK - 1) / BGD_BLOCK;
    h->grid_max = (int)std::min<size_t>((size_t)std::max(1, per_sm) * mk_sm_count(device), h->max_members);
    int rc = h->d_stage.alloc(h->max_members * BGD_SLOT);
    if (rc == MK_OK) rc = h->d_sizes.alloc(h->max_members * 4);
    if (rc == MK_OK) rc = h->d_off.alloc((h->max_members + 1) * 8);
    if (rc == MK_OK) rc = h->d_scratch.alloc((size_t)h->grid_max * BGD_SCRATCH * 4);
    if (rc == MK_OK) rc = h->h_sizes.alloc(h->max_members * 4);
    if (rc != MK_OK) { delete h; return rc; }
    *out = h;
    return MK_OK;
}

extern "C" void mk_bgzf_enc_destroy(mk_bgzf_enc *h) { if (h) { cudaSetDevice(h->device); delete h; } }

extern "C" int mk_bgzf_deflate_device(mk_bgzf_enc *h, const void *d_in, size_t n, int level, void *d_out, size_t out_cap, size_t *out_len,
                                      mk_bgzf_member *members, size_t members_cap, size_t *n_members, void *stream) {
    if (!h || (n && (!d_in || !d_out)) || !out_len || !n_members || level < -1 || level > 9) {
        mk_set_error("mk_bgzf_deflate_device: bad argument (level %d)", level); return MK_ERR_ARG;
    }
    const size_t nm = (n + BGD_BLOCK - 1) / BGD_BLOCK;
    if (n > h->max_bytes) { mk_set_error("mk_bgzf_deflate_device: %zu input bytes, the object holds %zu", n, h->max_bytes); return MK_ERR_CAPACITY; }
    if (out_cap < mk_bgzf_deflate_bound(n)) { mk_set_error("mk_bgzf_deflate_device: out_cap %zu below the bound %zu", out_cap, mk_bgzf_deflate_bound(n)); return MK_ERR_ARG; }
    if (members && members_cap < nm) { mk_set_error("mk_bgzf_deflate_device: %zu members, the table holds %zu", nm, members_cap); return MK_ERR_ARG; }
    *out_len = 0; *n_members = 0;
    if (n == 0) return MK_OK;
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = (int)std::min<size_t>(nm, (size_t)h->grid_max);
    k_bgzf_deflate<<<grid, BGD_NT, sizeof(BgdShared), s>>>((const uint8_t *)d_in, n, (uint32_t)nm, level == 0, h->d_stage.as<uint8_t>(),
                                                           h->d_sizes.as<uint32_t>(), h->d_scratch.as<uint32_t>());
    MK_CUDA(cudaGetLastError());
    k_bgzf_offsets<<<1, 1024, 0, s>>>(h->d_sizes.as<uint32_t>(), (uint32_t)nm, h->d_off.as<uint64_t>());
    MK_CUDA(cudaGetLastError());
    k_bgzf_pack<<<(int)std::min<size_t>(nm, 4 * (size_t)h->grid_max), BGD_NT, 0, s>>>(h->d_stage.as<uint8_t>(), h->d_sizes.as<uint32_t>(),
                                                                                        h->d_off.as<uint64_t>(), (uint32_t)nm, (uint8_t *)d_out);
    MK_CUDA(cudaGetLastError());
    h->launches += 3;
    MK_CUDA(cudaMemcpyAsync(h->h_sizes.p, h->d_sizes.p, nm * 4, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    const uint32_t *sz = h->h_sizes.as<uint32_t>();
    uint64_t o = 0;
    for (size_t k = 0; k < nm; ++k) {
        if (members) {
            members[k].in_off = o; members[k].in_len = sz[k];
            members[k].out_off = (uint64_t)k * BGD_BLOCK; members[k].isize = (uint32_t)std::min<uint64_t>(BGD_BLOCK, n - (uint64_t)k * BGD_BLOCK);
        }
        o += sz[k];
    }
    *out_len = o; *n_members = nm;
    return MK_OK;
}

extern "C" uint64_t mk_bgzf_enc_launch_count(mk_bgzf_enc *h) { return h ? (uint64_t)h->launches : 0; }
