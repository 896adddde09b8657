// bam_out.cu — coordinate-sorted BAM records and their .bai index in HBM (mk_bam_*): the device side of `sam2bam`.
//   encode   k_bam_nl_count / k_bam_nl_write: the line index of a text chunk (newlines per 4 KiB tile, a scan, the starts).
//            k_bam_size: one thread per line runs bam_encode.h's encoder in counting mode; the record sizes, and the first
//            bad line (a 64-bit atomicMin on line << 8 | code, so the lowest line wins whatever the thread order).
//            A scan gives the record offsets; k_bam_write runs the same encoder in writing mode.  Lines with a float off
//            the exact fast path are listed and re-encoded on the host with strtof inside the same call.
//   sort     k_bam_keys: 16-byte records (input index | (pos + 1) << 1 | rev | tid'), radix_sort.cuh on the key bytes that
//            can vary (stable: ties keep input order); a scan of the sizes in sorted order gives the output offsets.
//   gather   k_bam_gather: one warp per record copies it to its sorted place, for a slice [i0, i1) of the sorted order.
//   index    k_bam_index: per record its bin (the record's field), end, per-reference counts and pseudo-bin offsets
//            (atomics), the linear index (a 64-bit atomicMin of the record's stream offset per 16 kb window it overlaps),
//            and a flag where a run of equal (tid, bin) starts; a scan and k_bam_chunks compact the run starts.  A reference
//            starts with the windows its length needs; records that end past it grow its table (k_bam_wneed, k_bam_regrow).  Offsets
//            are kept as offsets of the uncompressed record stream, which orders them as their virtual offsets do; at the
//            end the chunks are grouped per (tid, bin) by a stable radix sort and every offset becomes a virtual offset
//            from the deflate's member table (k_bam_voff).  The host only lays out the .bai bytes.
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>
#include "mk_common.cuh"
#include "radix_sort.cuh"
#include "bam_encode.h"

#define BO_T 256
#define BO_ITEMS 16
#define BO_TILE (BO_T * BO_ITEMS)                 // items per scan tile / bytes per line-index tile
#define BO_BLOCK 65280ull                         // BGZF member payload: virtual offsets are made of these cuts
#define BO_WIN_MAX (1u << 15)                     // linear-index windows per reference (BAI covers positions below 2^29)
#define BO_NONE 0xffffffffffffffffull

// ---------------------------------------------------------------- a device-wide exclusive scan (u64) of any item function
__device__ __forceinline__ u64 bo_warp_incl(u64 v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const u64 t = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += t; }
    return v;
}
// exclusive scan over the CTA of one u64 per thread; *total = the CTA's sum
__device__ __forceinline__ u64 bo_block_excl(u64 v, u64 *sh, u64 *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const u64 inc = bo_warp_incl(v, lane);
    if (lane == 31) sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const u64 w = lane < BO_T / 32 ? sh[lane] : 0, wi = bo_warp_incl(w, lane);
        if (lane < BO_T / 32) sh[lane] = wi - w;
        if (lane == BO_T / 32 - 1) sh[BO_T / 32] = wi;
    }
    __syncthreads();
    const u64 r = inc - v + sh[wid];
    *total = sh[BO_T / 32];
    __syncthreads();
    return r;
}

template <class F> __global__ void __launch_bounds__(BO_T) k_bo_scan_part(F f, u64 n, u64 *part) {
    __shared__ u64 sh[BO_T / 32 + 1];
    const u64 a = (u64)blockIdx.x * BO_TILE + (u64)threadIdx.x * BO_ITEMS;
    u64 s = 0;
    for (int k = 0; k < BO_ITEMS; ++k) if (a + k < n) s += f(a + k);
    u64 tot;
    bo_block_excl(s, sh, &tot);
    if (threadIdx.x == 0) part[blockIdx.x] = tot;
}
// one CTA: part[0..nb) -> exclusive offsets, part[nb] = the total
__global__ void __launch_bounds__(BO_T) k_bo_scan_top(u64 *part, u64 nb) {
    __shared__ u64 sh[BO_T / 32 + 1];
    u64 carry = 0;
    for (u64 b = 0; b < nb; b += BO_T) {
        const u64 i = b + threadIdx.x;
        const u64 v = i < nb ? part[i] : 0;
        u64 tot;
        const u64 ex = bo_block_excl(v, sh, &tot);
        if (i < nb) part[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) part[nb] = carry;
}
// out[i] = base + sum of f(0..i), for i in [0, n]
template <class F> __global__ void __launch_bounds__(BO_T) k_bo_scan_down(F f, u64 n, const u64 *part, u64 *out, u64 base) {
    __shared__ u64 sh[BO_T / 32 + 1];
    const u64 a = (u64)blockIdx.x * BO_TILE + (u64)threadIdx.x * BO_ITEMS;
    u64 v[BO_ITEMS], s = 0;
    for (int k = 0; k < BO_ITEMS; ++k) { v[k] = a + k < n ? f(a + k) : 0; s += v[k]; }
    u64 tot;
    u64 run = base + part[blockIdx.x] + bo_block_excl(s, sh, &tot);
    for (int k = 0; k < BO_ITEMS; ++k) {
        if (a + k < n) out[a + k] = run;
        run += v[k];
        if (a + k + 1 == n) out[n] = run;
    }
    if (n == 0 && blockIdx.x == 0 && threadIdx.x == 0) out[0] = base;
}

struct BoScanWs {
    DevBuf part;
    int alloc(u64 max_n) { return part.alloc((max_n / BO_TILE + 2) * 8); }
};
template <class F> static int bo_scan(F f, u64 n, u64 *out, u64 base, BoScanWs &ws, cudaStream_t s, u64 *launches) {
    const u64 nb = std::max<u64>(1, (n + BO_TILE - 1) / BO_TILE);
    if ((nb + 1) * 8 > ws.part.n) { mk_set_error("bam scan: %llu items over the workspace", (unsigned long long)n); return MK_ERR_CAPACITY; }
    u64 *part = ws.part.as<u64>();
    k_bo_scan_part<<<(unsigned)nb, BO_T, 0, s>>>(f, n, part);
    k_bo_scan_top<<<1, BO_T, 0, s>>>(part, nb);
    k_bo_scan_down<<<(unsigned)nb, BO_T, 0, s>>>(f, n, part, out, base);
    MK_CUDA(cudaGetLastError());
    *launches += 3;
    return MK_OK;
}
struct BoGetU32 { const u32 *p; __device__ u64 operator()(u64 i) const { return p[i]; } };

// ---------------------------------------------------------------- encode
__global__ void __launch_bounds__(BO_T) k_bam_nl_count(const char *t, u64 n, u32 *cnt) {
    __shared__ u32 sh[BO_T / 32 + 1];
    const u64 a = (u64)blockIdx.x * BO_TILE + (u64)threadIdx.x * BO_ITEMS;
    u32 c = 0;
    for (int k = 0; k < BO_ITEMS; ++k) c += a + k < n && t[a + k] == '\n';
    u32 tot;
    block_excl_scan<BO_T>(c, sh, &tot);
    if (threadIdx.x == 0) cnt[blockIdx.x] = tot;
}
// ls[k + 1] = the byte after newline k, for k + 1 <= cap; ls[0] = 0
__global__ void __launch_bounds__(BO_T) k_bam_nl_write(const char *t, u64 n, const u64 *tile_base, u32 *ls, u64 cap) {
    __shared__ u32 sh[BO_T / 32 + 1];
    const u64 a = (u64)blockIdx.x * BO_TILE + (u64)threadIdx.x * BO_ITEMS;
    u32 c = 0;
    for (int k = 0; k < BO_ITEMS; ++k) c += a + k < n && t[a + k] == '\n';
    u32 tot;
    u64 idx = tile_base[blockIdx.x] + block_excl_scan<BO_T>(c, sh, &tot);
    for (int k = 0; k < BO_ITEMS; ++k)
        if (a + k < n && t[a + k] == '\n') { if (++idx <= cap) ls[idx] = (u32)(a + k + 1); }
    if (blockIdx.x == 0 && threadIdx.x == 0) ls[0] = 0;
}

__global__ void __launch_bounds__(BO_T) k_bam_size(const char *t, const u32 *ls, u64 n_lines, BeDict d, u32 *size, unsigned long long *err) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n_lines; i += (u64)gridDim.x * BO_T) {
        BeOut<false> o{nullptr, 0};
        bool patch = false;
        const int r = be_line<false>(t + ls[i], ls[i + 1] - ls[i] - 1, d, false, o, &patch);
        size[i] = o.at;
        if (r) atomicMin(err, (unsigned long long)i << 8 | (unsigned)r);
    }
}

__global__ void __launch_bounds__(BO_T) k_bam_write(const char *t, const u32 *ls, u64 n_lines, BeDict d, const u64 *off, u64 off_base,
                                                    u8 *out, u32 *patch_list, u32 *n_patch) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n_lines; i += (u64)gridDim.x * BO_T) {
        BeOut<true> o{out + (off[i] - off_base), 0};
        bool patch = false;
        be_line<true>(t + ls[i], ls[i + 1] - ls[i] - 1, d, false, o, &patch);
        if (patch) patch_list[atomicAdd(n_patch, 1u)] = (u32)i;
    }
}

// ---------------------------------------------------------------- sort + gather
__global__ void __launch_bounds__(BO_T) k_bam_keys(const u8 *rec, const u64 *off, u64 n, int32_t n_refs, uint4 *k0) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n; i += (u64)gridDim.x * BO_T) {
        u32 hi, lo;
        be_key(rec + off[i] - off[0], n_refs, hi, lo);
        k0[i] = make_uint4((u32)i, lo, hi, 0);
    }
}
struct BoSortedSize {
    const uint4 *b0, *b1; const RadixPlan *plan; const u64 *off;
    __device__ u64 operator()(u64 i) const { const u32 x = (plan->final_buf ? b1 : b0)[i].x; return off[x + 1] - off[x]; }
};
// the last i1 in (i0, n] with dst[i1] - dst[i0] <= max_bytes (at least i0 + 1)
__global__ void k_bam_slice_end(const u64 *dst, u64 i0, u64 n, u64 max_bytes, u64 *res) {
    u64 lo = i0 + 1, hi = n;
    while (lo < hi) { const u64 m = (lo + hi + 1) / 2; if (dst[m] - dst[i0] <= max_bytes) lo = m; else hi = m - 1; }
    res[0] = lo; res[1] = dst[lo] - dst[i0];
}
__global__ void __launch_bounds__(BO_T) k_bam_gather(const u8 *rec, const u64 *off, const uint4 *b0, const uint4 *b1, const RadixPlan *plan,
                                                     const u64 *dst, u64 i0, u64 i1, u8 *out) {
    const uint4 *order = plan->final_buf ? b1 : b0;
    const int lane = threadIdx.x & 31;
    const u64 base = dst[i0], o0 = off[0];
    for (u64 i = i0 + ((u64)blockIdx.x * BO_T + threadIdx.x) / 32; i < i1; i += (u64)gridDim.x * BO_T / 32) {
        const u32 x = order[i].x;
        const u8 *s = rec + off[x] - o0;
        u8 *d = out + dst[i] - base;
        const u64 len = off[x + 1] - off[x];
        for (u64 k = lane; k < len; k += 32) d[k] = s[k];
    }
}

// ---------------------------------------------------------------- index
struct BoRef { unsigned long long first, last, n_mapped, n_unmapped, max_end; };
__global__ void __launch_bounds__(BO_T) k_bam_index(const u8 *rec, const u64 *off, u64 n, u64 u_base, const u32 *win_base, const u32 *win_n,
                                                    unsigned long long *lin, BoRef *ref, unsigned long long *no_coor, u32 *flag) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n; i += (u64)gridDim.x * BO_T) {
        const u8 *r = rec + off[i] - off[0];
        const int32_t tid = (int32_t)be_rd32(r + 4);
        const u32 bin = (u32)r[14] | (u32)r[15] << 8;
        bool start = i == 0;
        if (!start) {
            const u8 *q = rec + off[i - 1] - off[0];
            start = (int32_t)be_rd32(q + 4) != tid || ((u32)q[14] | (u32)q[15] << 8) != bin;
        }
        flag[i] = start;
        if (tid < 0) { atomicAdd(no_coor, 1ull); continue; }
        const u64 u = u_base + off[i] - off[0], ue = u + (off[i + 1] - off[i]);
        const int64_t beg = (int32_t)be_rd32(r + 8), end = be_end(r);
        BoRef &R = ref[tid];
        atomicMin(&R.first, (unsigned long long)u);
        atomicMax(&R.last, (unsigned long long)ue);
        atomicAdd((r[18] & 4) ? &R.n_unmapped : &R.n_mapped, 1ull);
        atomicMax(&R.max_end, (unsigned long long)std::max<int64_t>(end, 1));
        const u32 wn = win_n[tid];
        const u64 w0 = std::min<u64>(beg < 0 ? 0 : (u64)beg >> 14, wn - 1), w1 = std::min<u64>((u64)std::max<int64_t>(end - 1, 0) >> 14, wn - 1);
        for (u64 w = w0; w <= w1; ++w) atomicMin(&lin[win_base[tid] + w], (unsigned long long)u);
    }
}
// the linear-index windows each reference needs for these records (a record may end past its reference's length)
__global__ void __launch_bounds__(BO_T) k_bam_wneed(const u8 *rec, const u64 *off, u64 n, u32 *need) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n; i += (u64)gridDim.x * BO_T) {
        const u8 *r = rec + off[i] - off[0];
        const int32_t tid = (int32_t)be_rd32(r + 4);
        if (tid >= 0) atomicMax(&need[tid], (u32)std::min<u64>((u64)std::max<int64_t>(be_end(r) - 1, 0) >> 14, BO_WIN_MAX - 1) + 1);
    }
}
// the window table re-laid out for larger per-reference counts: window i of the old table (reference t: the last t with
// old_base[t] <= i) moves to new_base[t] + i - old_base[t]
__global__ void __launch_bounds__(BO_T) k_bam_regrow(const unsigned long long *old, u64 n_old, const u32 *old_base, int n_refs, const u32 *new_base,
                                                     unsigned long long *nw) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n_old; i += (u64)gridDim.x * BO_T) {
        int lo = 0, hi = n_refs - 1;
        while (lo < hi) { const int m = (lo + hi + 1) / 2; if (old_base[m] <= i) lo = m; else hi = m - 1; }
        nw[new_base[lo] + (i - old_base[lo])] = old[i];
    }
}
__global__ void __launch_bounds__(BO_T) k_bam_chunks(const u8 *rec, const u64 *off, u64 n, u64 u_base, const u32 *flag, const u64 *idx, uint4 *chunks) {
    for (u64 i = (u64)blockIdx.x * BO_T + threadIdx.x; i < n; i += (u64)gridDim.x * BO_T) {
        if (!flag[i]) continue;
        const u8 *r = rec + off[i] - off[0];
        const u64 u = u_base + off[i] - off[0];
        chunks[idx[i]] = make_uint4(be_rd32(r + 4), (u32)r[14] | (u32)r[15] << 8, (u32)u, (u32)(u >> 32));
    }
}
__device__ __forceinline__ u64 bo_voff(const u64 *coff, u64 u) { return coff[u / BO_BLOCK] << 16 | u % BO_BLOCK; }
// every stream offset of the index -> its virtual offset; the chunks in (tid, bin) order
__global__ void __launch_bounds__(BO_T) k_bam_voff(const uint4 *k0, const uint4 *k1, const RadixPlan *plan, const u64 *cbeg, const u64 *cend, u64 nc,
                                                   u64 *cout, unsigned long long *lin, u64 nlin, BoRef *ref, int n_refs, const u64 *coff) {
    const uint4 *order = plan->final_buf ? k1 : k0;
    const u64 g = (u64)blockIdx.x * BO_T + threadIdx.x, stride = (u64)gridDim.x * BO_T;
    for (u64 i = g; i < nc; i += stride) {
        const u32 x = order[i].x;
        cout[4 * i] = order[i].z; cout[4 * i + 1] = order[i].y;
        cout[4 * i + 2] = bo_voff(coff, cbeg[x]); cout[4 * i + 3] = bo_voff(coff, cend[x]);
    }
    for (u64 i = g; i < nlin; i += stride) if (lin[i] != BO_NONE) lin[i] = bo_voff(coff, lin[i]);
    for (u64 i = g; i < (u64)n_refs; i += stride)
        if (ref[i].first != BO_NONE) { ref[i].first = bo_voff(coff, ref[i].first); ref[i].last = bo_voff(coff, ref[i].last); }
}

// ---------------------------------------------------------------- the object
struct mk_bam {
    int device = 0, sms = 148;
    int32_t n_refs = 0;
    std::vector<uint32_t> ref_len;
    size_t max_text = 0, max_records = 0, cap_lines = 0;
    DevBuf d_names, d_noff, d_slot;
    std::string h_names; std::vector<uint32_t> h_noff; std::vector<int32_t> h_slot;   // the host copy, for the float patches
    BeDict dict{};
    // encode
    DevBuf d_ls, d_tcnt, d_tbase, d_size, d_roff, d_patch, d_misc;   // misc: err word, patch count, slice result
    u64 n_lines = 0, rec_bytes = 0;
    const char *enc_text = nullptr; size_t enc_n = 0;
    // sort
    DevBuf d_k[2], d_dst;
    RadixWs rws;
    u64 sorted_n = 0;
    const u8 *sorted_rec = nullptr; const u64 *sorted_off = nullptr;
    BoScanWs scan;
    // index
    std::vector<uint32_t> win_base, win_n;
    DevBuf d_wbase, d_wn, d_wneed, d_lin, d_refstat, d_flag, d_fidx, d_chunks;
    u64 n_win = 0;
    struct Chunk { int32_t tid; uint32_t bin; uint64_t beg, end; };
    std::vector<Chunk> chunks;
    u64 u_end = 0;
    std::vector<u8> bai;
    u64 launches = 0;
};

static int bo_index_reset(mk_bam *h, cudaStream_t s) {
    MK_CUDA(cudaMemsetAsync(h->d_lin.p, 0xff, h->n_win * 8, s));
    std::vector<BoRef> r(std::max(h->n_refs, 1));
    for (auto &x : r) { x.first = BO_NONE; x.last = 0; x.n_mapped = x.n_unmapped = x.max_end = 0; }
    MK_CUDA(cudaMemcpyAsync(h->d_refstat.p, r.data(), r.size() * sizeof(BoRef), cudaMemcpyHostToDevice, s));
    MK_CUDA(cudaMemsetAsync(h->d_misc.as<u64>() + 4, 0, 8, s));                 // n_no_coor
    MK_CUDA(cudaStreamSynchronize(s));
    h->chunks.clear(); h->u_end = 0;
    return MK_OK;
}

// more linear-index windows for the references whose records need them (a new table, the old windows moved over)
static int bo_grow(mk_bam *h, cudaStream_t s) {
    std::vector<u32> need(h->n_refs);
    MK_CUDA(cudaMemcpyAsync(need.data(), h->d_wneed.p, h->n_refs * 4, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    bool grow = false;
    for (int t = 0; t < h->n_refs; ++t) grow |= need[t] > h->win_n[t];
    if (!grow) return MK_OK;
    std::vector<u32> nb(h->n_refs), nn(h->n_refs);
    u64 tot = 0;
    for (int t = 0; t < h->n_refs; ++t) { nb[t] = (u32)tot; nn[t] = std::max(need[t], h->win_n[t]); tot += nn[t]; }
    DevBuf lin, nbase;
    MK_TRY(lin.alloc(tot * 8)); MK_TRY(nbase.alloc(h->n_refs * 4));
    MK_CUDA(cudaMemsetAsync(lin.p, 0xff, tot * 8, s));
    MK_CUDA(cudaMemcpyAsync(nbase.p, nb.data(), h->n_refs * 4, cudaMemcpyHostToDevice, s));
    const int grid = (int)std::max<u64>(1, std::min<u64>((h->n_win + BO_T - 1) / BO_T, (u64)h->sms * 8));
    k_bam_regrow<<<grid, BO_T, 0, s>>>((const unsigned long long *)h->d_lin.p, h->n_win, h->d_wbase.as<u32>(), h->n_refs, nbase.as<u32>(),
                                       (unsigned long long *)lin.p);
    MK_CUDA(cudaGetLastError());
    h->launches += 1;
    MK_CUDA(cudaMemcpyAsync(h->d_wbase.p, nb.data(), h->n_refs * 4, cudaMemcpyHostToDevice, s));
    MK_CUDA(cudaMemcpyAsync(h->d_wn.p, nn.data(), h->n_refs * 4, cudaMemcpyHostToDevice, s));
    MK_CUDA(cudaStreamSynchronize(s));
    std::swap(h->d_lin.p, lin.p); std::swap(h->d_lin.n, lin.n);
    h->win_base = nb; h->win_n = nn; h->n_win = tot;
    return MK_OK;
}

extern "C" int mk_bam_create(int device, const char *const *ref_names, const uint32_t *ref_len, int n_refs, size_t max_text, size_t max_records, mk_bam **out) {
    if (!out || n_refs < 0 || (n_refs && (!ref_names || !ref_len)) || max_text == 0 || max_text >= (1ull << 32) - 1 || max_records == 0 || max_records >= (1ull << 30)) {
        mk_set_error("mk_bam_create: bad argument (max_text below 4 GiB, max_records below 2^30)"); return MK_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(device));
    mk_bam *h = new mk_bam();
    h->device = device; h->sms = mk_sm_count(device); h->n_refs = n_refs; h->max_text = max_text; h->max_records = max_records;
    h->ref_len.assign(ref_len, ref_len + n_refs);
    // the dictionary: names back to back, open addressing on FNV-1a
    std::string names; std::vector<uint32_t> noff(1, 0);
    for (int k = 0; k < n_refs; ++k) { names += ref_names[k]; noff.push_back((uint32_t)names.size()); }
    uint32_t bits = 4;
    while ((1u << bits) < 2u * (uint32_t)n_refs + 2) ++bits;
    std::vector<int32_t> slot(1u << bits, 0);
    BeDict hd{names.data(), noff.data(), slot.data(), (1u << bits) - 1, n_refs};
    for (int k = 0; k < n_refs; ++k) {
        const uint32_t len = noff[k + 1] - noff[k];
        if (len == 0 || be_lookup(hd, names.data() + noff[k], len) >= 0) { delete h; mk_set_error("mk_bam_create: reference %d is empty or a duplicate", k); return MK_ERR_ARG; }
        uint32_t p = be_hash(names.data() + noff[k], len) & hd.mask;
        while (slot[p]) p = (p + 1) & hd.mask;
        slot[p] = k + 1;
    }
    h->cap_lines = max_text / BE_MIN_LINE + 2;                   // lines before the first short one; see mk_bam_encode_size_device
    const u64 tiles = max_text / BO_TILE + 2;
    for (int k = 0; k < n_refs; ++k) {
        h->win_base.push_back((uint32_t)h->n_win);
        const uint32_t w = (uint32_t)std::min<u64>(((u64)std::max<uint32_t>(ref_len[k], 1) - 1) / 16384 + 1, BO_WIN_MAX);
        h->win_n.push_back(w); h->n_win += w;
    }
    int rc = MK_OK;
    auto A = [&](DevBuf &b, size_t bytes) { if (rc == MK_OK) rc = b.alloc(bytes); };
    A(h->d_names, names.size() + 1); A(h->d_noff, noff.size() * 4); A(h->d_slot, slot.size() * 4);
    A(h->d_ls, (h->cap_lines + 1) * 4); A(h->d_tcnt, tiles * 4); A(h->d_tbase, (tiles + 1) * 8); A(h->d_size, h->cap_lines * 4);
    A(h->d_roff, (h->cap_lines + 1) * 8); A(h->d_patch, h->cap_lines * 4); A(h->d_misc, 64);
    A(h->d_k[0], max_records * 16); A(h->d_k[1], max_records * 16); A(h->d_dst, (max_records + 1) * 8);
    A(h->d_wbase, (n_refs + 1) * 4); A(h->d_wn, (n_refs + 1) * 4); A(h->d_wneed, (n_refs + 1) * 4); A(h->d_lin, h->n_win * 8); A(h->d_refstat, (n_refs + 1) * sizeof(BoRef));
    A(h->d_flag, max_records * 4); A(h->d_fidx, (max_records + 1) * 8); A(h->d_chunks, max_records * 16);
    if (rc == MK_OK) rc = h->rws.alloc(max_records);
    if (rc == MK_OK) rc = h->scan.alloc(std::max<u64>(max_records, h->cap_lines) + tiles);
    if (rc != MK_OK) { delete h; return rc; }
    if (!names.empty()) MK_CUDA(cudaMemcpy(h->d_names.p, names.data(), names.size(), cudaMemcpyHostToDevice));
    MK_CUDA(cudaMemcpy(h->d_noff.p, noff.data(), noff.size() * 4, cudaMemcpyHostToDevice));
    MK_CUDA(cudaMemcpy(h->d_slot.p, slot.data(), slot.size() * 4, cudaMemcpyHostToDevice));
    if (n_refs) {
        MK_CUDA(cudaMemcpy(h->d_wbase.p, h->win_base.data(), n_refs * 4, cudaMemcpyHostToDevice));
        MK_CUDA(cudaMemcpy(h->d_wn.p, h->win_n.data(), n_refs * 4, cudaMemcpyHostToDevice));
    }
    h->h_names = names; h->h_noff = noff; h->h_slot = slot;
    if (n_refs) MK_CUDA(cudaMemset(h->d_wneed.p, 0, n_refs * 4));
    h->dict = BeDict{h->d_names.as<char>(), h->d_noff.as<uint32_t>(), h->d_slot.as<int32_t>(), (1u << bits) - 1, n_refs};
    rc = bo_index_reset(h, 0);
    if (rc != MK_OK) { delete h; return rc; }
    *out = h;
    return MK_OK;
}

extern "C" void mk_bam_destroy(mk_bam *h) { if (h) { cudaSetDevice(h->device); delete h; } }

extern "C" int mk_bam_encode_size_device(mk_bam *h, const char *d_text, size_t n, size_t *n_lines, size_t *rec_bytes, uint64_t *bad_line, int *bad_code,
                                         void *stream) {
    if (!h || (n && !d_text) || !n_lines || !rec_bytes || !bad_line || !bad_code) { mk_set_error("mk_bam_encode_size_device: bad argument"); return MK_ERR_ARG; }
    if (n > h->max_text) { mk_set_error("mk_bam_encode_size_device: %zu bytes, the object holds %zu", n, h->max_text); return MK_ERR_CAPACITY; }
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    *n_lines = *rec_bytes = 0; *bad_line = 0; *bad_code = 0;
    h->n_lines = h->rec_bytes = 0; h->enc_text = d_text; h->enc_n = n;
    if (n == 0) return MK_OK;
    char last;
    MK_CUDA(cudaMemcpyAsync(&last, d_text + n - 1, 1, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (last != '\n') { mk_set_error("mk_bam_encode_size_device: the text does not end with a newline"); return MK_ERR_ARG; }
    const u64 tiles = (n + BO_TILE - 1) / BO_TILE;
    k_bam_nl_count<<<(unsigned)tiles, BO_T, 0, s>>>(d_text, n, h->d_tcnt.as<u32>());
    h->launches += 1;
    MK_TRY(bo_scan(BoGetU32{h->d_tcnt.as<u32>()}, tiles, h->d_tbase.as<u64>(), 0, h->scan, s, &h->launches));
    k_bam_nl_write<<<(unsigned)tiles, BO_T, 0, s>>>(d_text, n, h->d_tbase.as<u64>(), h->d_ls.as<u32>(), h->cap_lines);
    u64 *misc = h->d_misc.as<u64>();
    MK_CUDA(cudaMemsetAsync(misc, 0xff, 8, s));
    u64 total = 0;
    MK_CUDA(cudaMemcpyAsync(&total, h->d_tbase.as<u64>() + tiles, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    // lines before the first line shorter than BE_MIN_LINE are at least BE_MIN_LINE + 1 bytes each, so that line lies below
    // cap_lines: the first bad line is always among the lines encoded here
    const u64 nl = std::min<u64>(total, h->cap_lines);
    const int grid = (int)std::min<u64>((nl + BO_T - 1) / BO_T, (u64)h->sms * 8);
    k_bam_size<<<std::max(grid, 1), BO_T, 0, s>>>(d_text, h->d_ls.as<u32>(), nl, h->dict, h->d_size.as<u32>(), (unsigned long long *)misc);
    h->launches += 2;
    MK_CUDA(cudaGetLastError());
    u64 err = 0;
    MK_CUDA(cudaMemcpyAsync(&err, misc, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (err != BO_NONE) {
        *bad_line = err >> 8; *bad_code = (int)(err & 255);
        mk_set_error("line %llu of the chunk: %s", (unsigned long long)(err >> 8) + 1, be_errstr[err & 255]);
        return MK_ERR_INPUT;
    }
    if (total > h->cap_lines) { mk_set_error("mk_bam_encode_size_device: more lines than the object holds"); return MK_ERR_CAPACITY; }
    MK_TRY(bo_scan(BoGetU32{h->d_size.as<u32>()}, nl, h->d_roff.as<u64>(), 0, h->scan, s, &h->launches));
    u64 bytes = 0;
    MK_CUDA(cudaMemcpyAsync(&bytes, h->d_roff.as<u64>() + nl, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    h->n_lines = nl; h->rec_bytes = bytes;
    *n_lines = nl; *rec_bytes = bytes;
    return MK_OK;
}

// the host form of the encoder on the lines the device marked (a float off the exact fast path): same length, strtof values
static int bo_patch(mk_bam *h, u8 *d_out, u32 np, cudaStream_t s) {
    std::vector<u32> list(np), ls(h->n_lines + 1);
    std::vector<u64> off(h->n_lines + 1);
    std::vector<char> text(h->enc_n);
    MK_CUDA(cudaMemcpyAsync(list.data(), h->d_patch.p, np * 4, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(ls.data(), h->d_ls.p, ls.size() * 4, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(off.data(), h->d_roff.p, off.size() * 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(text.data(), h->enc_text, h->enc_n, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    const BeDict d{h->h_names.data(), h->h_noff.data(), h->h_slot.data(), h->dict.mask, h->n_refs};
    std::vector<u8> rec;
    for (u32 i : list) {
        rec.assign(off[i + 1] - off[i], 0);
        BeOut<true> o{rec.data(), 0};
        bool patch = false;
        const int r = be_line<true>(text.data() + ls[i], ls[i + 1] - ls[i] - 1, d, true, o, &patch);
        if (r != BE_OK || o.at != rec.size()) { mk_set_error("bam float patch: line %u re-encoded with code %d", i + 1, r); return MK_ERR_STATE; }
        MK_CUDA(cudaMemcpy(d_out + off[i], rec.data(), rec.size(), cudaMemcpyHostToDevice));
    }
    return MK_OK;
}

extern "C" int mk_bam_encode_write_device(mk_bam *h, uint8_t *d_out, uint64_t base, size_t out_cap, uint64_t *d_off, size_t *n_patched, void *stream) {
    if (!h || !d_out || !d_off) { mk_set_error("mk_bam_encode_write_device: bad argument"); return MK_ERR_ARG; }
    if (base + h->rec_bytes > out_cap) { mk_set_error("mk_bam_encode_write_device: %llu record bytes past the output's %zu", (unsigned long long)(base + h->rec_bytes), out_cap); return MK_ERR_CAPACITY; }
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (n_patched) *n_patched = 0;
    if (h->n_lines == 0) { MK_CUDA(cudaMemcpyAsync(d_off, &base, 8, cudaMemcpyHostToDevice, s)); MK_CUDA(cudaStreamSynchronize(s)); return MK_OK; }
    u32 *np = (u32 *)(h->d_misc.as<u64>() + 1);
    MK_CUDA(cudaMemsetAsync(np, 0, 4, s));
    const int grid = (int)std::min<u64>((h->n_lines + BO_T - 1) / BO_T, (u64)h->sms * 8);
    k_bam_write<<<grid, BO_T, 0, s>>>(h->enc_text, h->d_ls.as<u32>(), h->n_lines, h->dict, h->d_roff.as<u64>(), 0, d_out + base, h->d_patch.as<u32>(), np);
    MK_TRY(bo_scan(BoGetU32{h->d_size.as<u32>()}, h->n_lines, d_off, base, h->scan, s, &h->launches));
    h->launches += 1;
    MK_CUDA(cudaGetLastError());
    u32 hp = 0;
    MK_CUDA(cudaMemcpyAsync(&hp, np, 4, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (hp) MK_TRY(bo_patch(h, d_out + base, hp, s));
    if (n_patched) *n_patched = hp;
    return MK_OK;
}

extern "C" int mk_bam_sort_device(mk_bam *h, const uint8_t *d_rec, const uint64_t *d_off, size_t n, size_t *total_bytes, void *stream) {
    if (!h || (n && (!d_rec || !d_off)) || !total_bytes) { mk_set_error("mk_bam_sort_device: bad argument"); return MK_ERR_ARG; }
    if (n > h->max_records) { mk_set_error("mk_bam_sort_device: %zu records, the object holds %zu", n, h->max_records); return MK_ERR_CAPACITY; }
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    h->sorted_n = n; h->sorted_rec = d_rec; h->sorted_off = d_off;
    *total_bytes = 0;
    uint4 *k0 = h->d_k[0].as<uint4>(), *k1 = h->d_k[1].as<uint4>();
    const int grid = (int)std::max<u64>(1, std::min<u64>((n + BO_T - 1) / BO_T, (u64)h->sms * 8));
    k_bam_keys<<<grid, BO_T, 0, s>>>(d_rec, d_off, n, h->n_refs, k0);
    h->launches += 1;
    RadixSchedule sch; sch.n_pass = 0;
    for (int b = 4; b < 8; ++b) sch.byte_of[sch.n_pass++] = b;                  // (pos + 1) << 1 | rev
    for (u32 v = (u32)h->n_refs, b = 8; b < 12; ++b, v >>= 8) { sch.byte_of[sch.n_pass++] = (int)b; if (v < 256) break; }   // tid'
    Rec16::Bufs bufs; bufs.k[0] = k0; bufs.k[1] = k1; bufs.v[0] = bufs.v[1] = nullptr;
    MK_TRY(radix_sort<Rec16>(bufs, n, sch, h->rws, 0, h->sms, s, &h->launches));
    MK_TRY(bo_scan(BoSortedSize{k0, k1, h->rws.plan.as<RadixPlan>(), d_off}, n, h->d_dst.as<u64>(), 0, h->scan, s, &h->launches));
    u64 tot = 0;
    MK_CUDA(cudaMemcpyAsync(&tot, h->d_dst.as<u64>() + n, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    *total_bytes = tot;
    return MK_OK;
}

extern "C" int mk_bam_gather_device(mk_bam *h, size_t i0, size_t max_bytes, uint8_t *d_out, size_t out_cap, size_t *i1, size_t *bytes,
                                    const uint64_t **d_out_off, void *stream) {
    if (!h || !d_out || !i1 || !bytes || i0 >= h->sorted_n) { mk_set_error("mk_bam_gather_device: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    u64 *res = h->d_misc.as<u64>() + 2, hr[2];
    k_bam_slice_end<<<1, 1, 0, s>>>(h->d_dst.as<u64>(), i0, h->sorted_n, max_bytes, res);
    MK_CUDA(cudaMemcpyAsync(hr, res, 16, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (hr[1] > out_cap) { mk_set_error("mk_bam_gather_device: a record of %llu bytes past the output's %zu", (unsigned long long)hr[1], out_cap); return MK_ERR_CAPACITY; }
    const u64 m = hr[0] - i0;
    const int grid = (int)std::min<u64>((m * 32 + BO_T - 1) / BO_T, (u64)h->sms * 16);
    k_bam_gather<<<grid, BO_T, 0, s>>>(h->sorted_rec, h->sorted_off, h->d_k[0].as<uint4>(), h->d_k[1].as<uint4>(), h->rws.plan.as<RadixPlan>(),
                                      h->d_dst.as<u64>(), i0, hr[0], d_out);
    MK_CUDA(cudaGetLastError());
    h->launches += 2;
    *i1 = hr[0]; *bytes = hr[1];
    if (d_out_off) *d_out_off = h->d_dst.as<u64>() + i0;
    return MK_OK;
}

extern "C" int mk_bam_index_reset(mk_bam *h) {
    if (!h) { mk_set_error("mk_bam_index_reset: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(h->device));
    return bo_index_reset(h, 0);
}

extern "C" int mk_bam_index_add_device(mk_bam *h, const uint8_t *d_rec, const uint64_t *d_off, size_t n, uint64_t u_base, void *stream) {
    if (!h || (n && (!d_rec || !d_off))) { mk_set_error("mk_bam_index_add_device: bad argument"); return MK_ERR_ARG; }
    if (n > h->max_records) { mk_set_error("mk_bam_index_add_device: %zu records, the object holds %zu", n, h->max_records); return MK_ERR_CAPACITY; }
    if (u_base != h->u_end) { mk_set_error("mk_bam_index_add_device: records at stream offset %llu, the index ends at %llu", (unsigned long long)u_base, (unsigned long long)h->u_end); return MK_ERR_ARG; }
    if (n == 0) return MK_OK;
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int grid = (int)std::min<u64>((n + BO_T - 1) / BO_T, (u64)h->sms * 8);
    if (h->n_refs) {
        k_bam_wneed<<<grid, BO_T, 0, s>>>(d_rec, d_off, n, h->d_wneed.as<u32>());
        h->launches += 1;
        MK_TRY(bo_grow(h, s));
    }
    k_bam_index<<<grid, BO_T, 0, s>>>(d_rec, d_off, n, u_base, h->d_wbase.as<u32>(), h->d_wn.as<u32>(), (unsigned long long *)h->d_lin.p,
                                      h->d_refstat.as<BoRef>(), (unsigned long long *)(h->d_misc.as<u64>() + 4), h->d_flag.as<u32>());
    MK_TRY(bo_scan(BoGetU32{h->d_flag.as<u32>()}, n, h->d_fidx.as<u64>(), 0, h->scan, s, &h->launches));
    k_bam_chunks<<<grid, BO_T, 0, s>>>(d_rec, d_off, n, u_base, h->d_flag.as<u32>(), h->d_fidx.as<u64>(), h->d_chunks.as<uint4>());
    MK_CUDA(cudaGetLastError());
    h->launches += 2;
    u64 nc = 0, o[2];
    MK_CUDA(cudaMemcpyAsync(&nc, h->d_fidx.as<u64>() + n, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(o, d_off, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(o + 1, d_off + n, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    std::vector<uint4> c(nc);
    MK_CUDA(cudaMemcpyAsync(c.data(), h->d_chunks.p, nc * 16, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    const u64 end = u_base + (o[1] - o[0]);
    // a run that goes on across the cut between two calls is one chunk; ends are the next run's start, the last one the call's end
    size_t from = h->chunks.size(), k = 0;
    if (nc && from && h->chunks.back().tid == (int32_t)c[0].x && h->chunks.back().bin == c[0].y) { from -= 1; k = 1; }
    for (; k < nc; ++k) h->chunks.push_back({(int32_t)c[k].x, c[k].y, (u64)c[k].z | (u64)c[k].w << 32, 0});
    for (size_t j = from; j < h->chunks.size(); ++j) h->chunks[j].end = j + 1 < h->chunks.size() ? h->chunks[j + 1].beg : end;
    h->u_end = end;
    return MK_OK;
}

// the .bai (SAMv1 §5.2) of every record added since the reset.  coff[k] = the file offset of record-stream member k, for
// k = 0 .. n_members (coff[n_members]: where the member after the last one starts, the EOF member).  *bai: the bytes, owned by
// the object until its next call.  The index starts over afterwards.
extern "C" int mk_bam_bai(mk_bam *h, const uint64_t *coff, size_t n_coff, const uint8_t **bai, size_t *len) {
    if (!h || !coff || !bai || !len || n_coff < (h->u_end + BO_BLOCK - 1) / BO_BLOCK + 1) { mk_set_error("mk_bam_bai: bad argument (member table)"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = 0;
    // chunks without a reference (tid -1) are not indexed
    std::vector<mk_bam::Chunk> ch;
    for (auto &c : h->chunks) if (c.tid >= 0) ch.push_back(c);
    const u64 nc = ch.size();
    DevBuf k[2], cb, ce, co, dc;
    RadixWs rws;
    MK_TRY(k[0].alloc(nc * 16)); MK_TRY(k[1].alloc(nc * 16)); MK_TRY(cb.alloc(nc * 8)); MK_TRY(ce.alloc(nc * 8)); MK_TRY(co.alloc(nc * 32));
    MK_TRY(dc.alloc(n_coff * 8)); MK_TRY(rws.alloc(std::max<u64>(nc, 1)));
    {
        std::vector<uint4> kh(nc); std::vector<u64> bh(nc), eh(nc);
        for (u64 i = 0; i < nc; ++i) { kh[i] = make_uint4((u32)i, ch[i].bin, (u32)ch[i].tid, 0); bh[i] = ch[i].beg; eh[i] = ch[i].end; }
        MK_CUDA(cudaMemcpyAsync(k[0].p, kh.data(), nc * 16, cudaMemcpyHostToDevice, s));
        MK_CUDA(cudaMemcpyAsync(cb.p, bh.data(), nc * 8, cudaMemcpyHostToDevice, s));
        MK_CUDA(cudaMemcpyAsync(ce.p, eh.data(), nc * 8, cudaMemcpyHostToDevice, s));
        MK_CUDA(cudaMemcpyAsync(dc.p, coff, n_coff * 8, cudaMemcpyHostToDevice, s));
        RadixSchedule sch; sch.n_pass = 0;
        sch.byte_of[sch.n_pass++] = 4; sch.byte_of[sch.n_pass++] = 5;                // bin
        for (u32 v = (u32)h->n_refs, b = 8; b < 12; ++b, v >>= 8) { sch.byte_of[sch.n_pass++] = (int)b; if (v < 256) break; }
        Rec16::Bufs bufs; bufs.k[0] = k[0].as<uint4>(); bufs.k[1] = k[1].as<uint4>(); bufs.v[0] = bufs.v[1] = nullptr;
        MK_TRY(radix_sort<Rec16>(bufs, nc, sch, rws, 0, h->sms, s, &h->launches));
        const u64 work = std::max<u64>(std::max<u64>(nc, h->n_win), (u64)h->n_refs);
        const int grid = (int)std::max<u64>(1, std::min<u64>((work + BO_T - 1) / BO_T, (u64)h->sms * 8));
        k_bam_voff<<<grid, BO_T, 0, s>>>(k[0].as<uint4>(), k[1].as<uint4>(), rws.plan.as<RadixPlan>(), cb.as<u64>(), ce.as<u64>(), nc, co.as<u64>(),
                                         (unsigned long long *)h->d_lin.p, h->n_win, h->d_refstat.as<BoRef>(), h->n_refs, dc.as<u64>());
        MK_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    std::vector<u64> cs(nc * 4), lin(h->n_win);
    std::vector<BoRef> ref(std::max(h->n_refs, 1));
    u64 no_coor = 0;
    MK_CUDA(cudaMemcpyAsync(cs.data(), co.p, nc * 32, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(lin.data(), h->d_lin.p, h->n_win * 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(ref.data(), h->d_refstat.p, h->n_refs * sizeof(BoRef), cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaMemcpyAsync(&no_coor, h->d_misc.as<u64>() + 4, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    MK_TRY(bo_index_reset(h, s));                                // the device state holds virtual offsets now
    std::vector<u8> &o = h->bai;
    o.clear();
    auto p32 = [&](uint32_t v) { for (int b = 0; b < 4; ++b) o.push_back((u8)(v >> 8 * b)); };
    auto p64 = [&](uint64_t v) { for (int b = 0; b < 8; ++b) o.push_back((u8)(v >> 8 * b)); };
    o.insert(o.end(), {'B', 'A', 'I', 1});
    p32((uint32_t)h->n_refs);
    u64 c = 0;
    for (int t = 0; t < h->n_refs; ++t) {
        const u64 c0 = c;
        while (c < nc && cs[4 * c] == (u64)t) ++c;
        const BoRef &R = ref[t];
        if (R.n_mapped + R.n_unmapped == 0) { p32(0); p32(0); continue; }
        uint32_t nbin = 1;
        for (u64 j = c0; j < c; ++j) if (j == c0 || cs[4 * j + 1] != cs[4 * j - 3]) ++nbin;
        p32(nbin);
        for (u64 j = c0; j < c;) {
            u64 e = j;
            while (e < c && cs[4 * e + 1] == cs[4 * j + 1]) ++e;
            p32((uint32_t)cs[4 * j + 1]); p32((uint32_t)(e - j));
            for (; j < e; ++j) { p64(cs[4 * j + 2]); p64(cs[4 * j + 3]); }
        }
        p32(37450); p32(2); p64(R.first); p64(R.last); p64(R.n_mapped); p64(R.n_unmapped);
        const uint32_t nint = (uint32_t)std::min<u64>((R.max_end - 1) / 16384 + 1, h->win_n[t]);
        p32(nint);
        u64 prev = 0;
        for (uint32_t w = 0; w < nint; ++w) { const u64 v = lin[h->win_base[t] + w]; if (v != BO_NONE) prev = v; p64(prev); }
    }
    p64(no_coor);
    *bai = o.data(); *len = o.size();
    return MK_OK;
}

extern "C" uint64_t mk_bam_launch_count(mk_bam *h) { return h ? h->launches : 0; }

// What one sorted run may hold when the caller reads text in chunks of `chunk` bytes: the device memory free now, less 8
// chunks (text, line index, output window, deflate staging and output) and 512 MiB, over 2.2 (the run's bytes, and the
// per-record sort, gather and index workspace of mk_bam_create with max_records = bytes / 64).
extern "C" int mk_bam_sort_budget(int device, size_t chunk, size_t *bytes) {
    if (!bytes) { mk_set_error("mk_bam_sort_budget: bad argument"); return MK_ERR_ARG; }
    MK_CUDA(cudaSetDevice(device));
    size_t fr = 0, tot = 0;
    MK_CUDA(cudaMemGetInfo(&fr, &tot));
    const double left = (double)fr - 8.0 * (double)chunk - 512.0 * (1 << 20);
    *bytes = left > 0 ? (size_t)(left / 2.2) : 0;
    return MK_OK;
}
