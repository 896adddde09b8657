// radix_sort.cuh — hand-written single-sweep LSD radix sort for sm_100a (8-bit digits).
//
//   k_radix_hist   one read of the input: all digit histograms at once (shared-memory privatised,
//                  warp-aggregated with match.any so constant digits do not serialise)
//   k_radix_plan   exclusive scan of every histogram, detection of trivial passes (one bin holds
//                  everything: the pass is skipped), ping-pong buffer assignment — all on the device
//   k_radix_pass   one kernel per digit: tile histogram -> 256 parallel decoupled look-back chains
//                  -> stable in-tile ranking (match.any) -> shared-memory reorder -> coalesced scatter
//
// The element type is a policy: KV64 = (u64 key, u32 value) in separate arrays (krmdup keys with their
// pair index), Rec16 = 16-byte records sorted on an arbitrary byte schedule (mk_pair records sorted on
// lane,chr1,pos1,chr2,pos2,strands without building a separate key).
// Replaces the reference's unordered_set probe (src/preprocess/krmdup.cpp:201-203): a stable sort keeps
// equal keys in input order, so the first element of each run is the occurrence krmdup would keep.
#pragma once
#include "mk_common.cuh"

#define RS_THREADS 256
#ifndef RS_BALLOT_MATCH
#define RS_BALLOT_MATCH 1
#endif
#define RS_MAX_PASSES 16

struct RadixPlan {                 // device resident
    u32 hist[RS_MAX_PASSES][256];  // counts, then exclusive offsets
    u32 skip[RS_MAX_PASSES];
    u32 src[RS_MAX_PASSES];        // which buffer (0/1) the pass reads
    u32 first[RS_MAX_PASSES];      // first executed pass (values are still the implicit iota)
    u32 ticket[RS_MAX_PASSES];
    u32 final_buf, n_exec;
};

struct RadixSchedule { int n_pass; int byte_of[RS_MAX_PASSES]; };   // LSD order: byte index inside the key/record

// ---------------------------------------------------------------- element policies
struct KV64 {
    typedef u64 Key;
    static constexpr int ITEMS = 16;
    static constexpr int MIN_BLOCKS = 1;
    static constexpr bool HAS_VAL = true;
    struct Bufs { u64 *k[2]; u32 *v[2]; };
    __device__ static __forceinline__ u32 digit(const u64 &k, int byte) { return (u32)(k >> (8 * byte)) & 255u; }
    __device__ static __forceinline__ u64 load_key(const Bufs &b, int which, u64 i) { return b.k[which][i]; }
    __device__ static __forceinline__ void store_key(const Bufs &b, int which, u64 i, const u64 &k) { b.k[which][i] = k; }
};
struct Rec16 {
    typedef uint4 Key;
#ifndef RS_REC16_ITEMS
#define RS_REC16_ITEMS 8
#endif
#ifndef RS_REC16_MINB
#define RS_REC16_MINB 4
#endif
    static constexpr int ITEMS = RS_REC16_ITEMS;
    static constexpr int MIN_BLOCKS = RS_REC16_MINB;   // 64 registers: four resident tiles per SM hide the look-back and scatter latency
    static constexpr bool HAS_VAL = false;
    struct Bufs { uint4 *k[2]; u32 *v[2]; };
    __device__ static __forceinline__ u32 digit(const uint4 &k, int byte) {
        const u32 lo = (byte & 8) ? k.z : k.x, hi = (byte & 8) ? k.w : k.y;      // two selects + one byte permute
        return __byte_perm(lo, hi, (u32)(byte & 7)) & 255u;
    }
    __device__ static __forceinline__ uint4 load_key(const Bufs &b, int which, u64 i) { return b.k[which][i]; }
    __device__ static __forceinline__ void store_key(const Bufs &b, int which, u64 i, const uint4 &k) { b.k[which][i] = k; }
};

// ---------------------------------------------------------------- histogram of every digit in one read
// one element's digits into the CTA's shared-memory histograms (n_pass * 256 counters); called by whole warps
// (`valid` false for lanes past the end).  Fully unrolled over the schedule: byte_of[p] is then a constant-bank operand (no
// dynamic indexing of the parameter array) and a pass costs ~12 instructions instead of ~75.
template <class P>
__device__ __forceinline__ void radix_hist_add(u32 *s_hist, const RadixSchedule &sch, const typename P::Key &k, bool valid, int lane) {
    const u32 vmask = __ballot_sync(0xffffffffu, valid);
#pragma unroll
    for (int p = 0; p < RS_MAX_PASSES; ++p) {
        if (p >= sch.n_pass) break;
        const u32 d = valid ? P::digit(k, sch.byte_of[p]) : 0u;
        // constant digits (high bytes, unused fields) would serialise 32 ways on one counter: one add per warp instead
        if (vmask == 0xffffffffu) {
            const u32 d0 = __shfl_sync(0xffffffffu, d, 0);
            if (__all_sync(0xffffffffu, d == d0)) { if (lane == 0) atomicAdd(&s_hist[p * 256 + d], 32u); }
            else atomicAdd(&s_hist[p * 256 + d], 1u);
        } else if (valid) atomicAdd(&s_hist[p * 256 + d], 1u);
    }
}
__device__ __forceinline__ void radix_hist_flush(const u32 *s_hist, int n_pass, RadixPlan *plan) {      // after a __syncthreads()
    for (int i = threadIdx.x; i < n_pass * 256; i += blockDim.x) {
        u32 v = s_hist[i];
        if (v) atomicAdd(&plan->hist[i >> 8][i & 255], v);
    }
}

template <class P>
static __global__ void __launch_bounds__(RS_THREADS) k_radix_hist(typename P::Bufs bufs, u64 n, RadixSchedule sch, RadixPlan *plan) {
    extern __shared__ u32 s_hist[];                  // n_pass * 256
    for (int i = threadIdx.x; i < sch.n_pass * 256; i += RS_THREADS) s_hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const u64 stride = (u64)gridDim.x * RS_THREADS;
    const u64 n_round = (n + 31) & ~(u64)31;         // keep warps converged
    for (u64 i = (u64)blockIdx.x * RS_THREADS + threadIdx.x; i < n_round; i += stride) {
        const bool valid = i < n;
        typename P::Key k;
        if (valid) k = P::load_key(bufs, 0, i);
        radix_hist_add<P>(s_hist, sch, k, valid, lane);
    }
    __syncthreads();
    radix_hist_flush(s_hist, sch.n_pass, plan);
}

// one CTA: scan histograms, decide which passes run and which buffer each reads
static __global__ void __launch_bounds__(256) k_radix_plan(RadixPlan *plan, u64 n, int n_pass) {
    __shared__ u32 s_scan[256 / 32 + 1];
    __shared__ u32 s_skip[RS_MAX_PASSES];
    for (int p = 0; p < n_pass; ++p) {
        u32 c = plan->hist[p][threadIdx.x];
        if (threadIdx.x == 0) s_skip[p] = 0;
        __syncthreads();
        if ((u64)c == n) s_skip[p] = 1;              // every key has the same digit here: nothing to do
        u32 tot;
        u32 ex = block_excl_scan<256>(c, s_scan, &tot);
        plan->hist[p][threadIdx.x] = ex;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        u32 cur = 0, n_exec = 0;
        for (int p = 0; p < n_pass; ++p) {
            plan->skip[p] = s_skip[p] || n == 0;
            plan->src[p] = cur;
            plan->first[p] = (!plan->skip[p] && n_exec == 0) ? 1u : 0u;
            plan->ticket[p] = 0;
            if (!plan->skip[p]) { cur ^= 1u; ++n_exec; }
        }
        plan->final_buf = cur; plan->n_exec = n_exec;
    }
}

// ---------------------------------------------------------------- one digit pass
#define RS_ST_AGG (1u << 30)
#define RS_ST_INC (2u << 30)
#define RS_VAL(x) ((x) & 0x3FFFFFFFu)
#define RS_LB 8                                  // look-back descriptor loads in flight per digit thread

template <class P>
static __global__ void __launch_bounds__(RS_THREADS, P::MIN_BLOCKS) k_radix_pass(typename P::Bufs bufs, u64 n, int pass, int byte, RadixPlan *plan,
                                                          u32 *desc /* n_tiles * 256 */, int iota_vals) {
    constexpr int ITEMS = P::ITEMS;
    constexpr int TILE = RS_THREADS * ITEMS;
    typedef typename P::Key Key;
    extern __shared__ __align__(16) unsigned char s_raw[];
    Key *s_keys = (Key *)s_raw;                                        // TILE keys
    u32 *s_vals = (u32 *)(s_raw + sizeof(Key) * TILE);                 // TILE values (when HAS_VAL)
    u32 *s_wcnt = (u32 *)(s_raw + sizeof(Key) * TILE + (P::HAS_VAL ? 4 * TILE : 0));   // [8 warps][256]
    u32 *s_dig_excl = s_wcnt + (RS_THREADS / 32) * 256;                // [256] start of each digit inside the tile
    u32 *s_gbase = s_dig_excl + 256;                                   // [256] global position of the digit's first key of this tile
    u32 *s_scan = s_gbase + 256;                                       // block scan scratch (9) + ticket (1)
    if (plan->skip[pass]) return;
    const int which = (int)plan->src[pass];
    const bool use_iota = P::HAS_VAL && iota_vals && plan->first[pass];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) s_scan[16] = atomicAdd(&plan->ticket[pass], 1u);
    for (int i = tid; i < (RS_THREADS / 32) * 256 + 256; i += RS_THREADS) s_wcnt[i] = 0;       // warp counters and s_dig_excl (tile histogram below)
    __syncthreads();
    const u32 tile = s_scan[16];
    const u64 tile_base = (u64)tile * TILE;
    // ---- load (warp-striped: warp w owns keys [w*32*ITEMS, (w+1)*32*ITEMS), item j lane l -> + j*32 + l)
    Key key[ITEMS]; u32 val[ITEMS]; u32 rank[ITEMS]; u32 dig[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const u64 i = tile_base + (u64)wid * 32 * ITEMS + j * 32 + lane;
        if (i < n) {
            key[j] = P::load_key(bufs, which, i);
            if (P::HAS_VAL) val[j] = use_iota ? (u32)i : bufs.v[which][i];
            dig[j] = P::digit(key[j], byte);
        } else dig[j] = 255u;                                            // padding sorts last inside the last tile
    }
    // ---- the tile's digit counts first (plain shared-memory atomics), so that its aggregate is published BEFORE the slow
    // stable ranking: the successors' look-back then finds it ready instead of spinning (ncu: 29 % of the stall samples)
    u32 *my = desc + (u64)tile * 256 + tid;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) atomicAdd(&s_dig_excl[dig[j]], 1u);
    __syncthreads();
    {
        const u32 c0 = s_dig_excl[tid];
        atomicExch(my, (tile == 0 ? RS_ST_INC : RS_ST_AGG) | c0);
    }
    // ---- stable rank inside the warp, digit by digit
    u32 *wc = s_wcnt + wid * 256;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const u32 d = dig[j];
#if RS_BALLOT_MATCH
        u32 peers = 0xffffffffu;                                         // lanes with the same 8-bit digit, from eight ballots (A/B against match.any)
#pragma unroll
        for (int bit = 0; bit < 8; ++bit) { const bool on = (d >> bit) & 1u; const u32 bl = __ballot_sync(0xffffffffu, on); peers &= on ? bl : ~bl; }
#else
        const u32 peers = __match_any_sync(0xffffffffu, d);
#endif
        const int leader = __ffs(peers) - 1;
        u32 old = 0;
        if (lane == leader) { old = wc[d]; wc[d] = old + (u32)__popc(peers); }
        old = __shfl_sync(0xffffffffu, old, leader);
        rank[j] = old + (u32)__popc(peers & ((1u << lane) - 1u));
        __syncwarp();
    }
    __syncthreads();
    // ---- per digit (thread d): offsets of each warp, tile count, look-back over previous tiles
    {
        const int d = tid;
        u32 run = 0;
#pragma unroll
        for (int w = 0; w < RS_THREADS / 32; ++w) { u32 c = s_wcnt[w * 256 + d]; s_wcnt[w * 256 + d] = run; run += c; }
        const u32 cnt = run;
        u32 tot;
        const u32 ex = block_excl_scan<RS_THREADS>(cnt, s_scan, &tot);
        s_dig_excl[d] = ex;
        // decoupled look-back for this digit (the aggregate was published above)
        u32 excl = 0;
        if (tile != 0) {
            // Walk back over the predecessors with RS_LB descriptor loads in flight (8: A/B 4 / 8 / 16 -> stage 5.19 / 4.98 / 5.08 ms): the tiles in flight publish their aggregates
            // at about the same time, so a walk is tens of steps long, and one dependent L2 round trip per step was 35 % of
            // this kernel's stall samples (ncu).
            long t = (long)tile - 1;
            bool done = false;
            while (!done) {
                u32 v[RS_LB];
#pragma unroll
                for (int q = 0; q < RS_LB; ++q) v[q] = t - q >= 0 ? *(volatile u32 *)(desc + (u64)(t - q) * 256 + d) : 0u;
                int used = 0;
#pragma unroll
                for (int q = 0; q < RS_LB; ++q) {
                    const u32 st = v[q] >> 30;
                    if (done || used != q || st == 0) continue;         // consume in order; stop at the first one that is not ready
                    excl += RS_VAL(v[q]); ++used;
                    if (st == 2) done = true;
                }
                t -= used;
            }
            atomicExch(my, RS_ST_INC | (excl + cnt));
        }
        s_gbase[d] = plan->hist[pass][d] + excl;
    }
    __syncthreads();
    // ---- reorder through shared memory so that the scatter writes runs of equal digits
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const u32 d = dig[j];
        const u32 lp = s_dig_excl[d] + s_wcnt[wid * 256 + d] + rank[j];
        rank[j] = lp;
    }
    const u64 remaining = n - tile_base;
    const u32 n_valid = remaining < (u64)TILE ? (u32)remaining : (u32)TILE;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const u64 i = tile_base + (u64)wid * 32 * ITEMS + j * 32 + lane;
        if (i < n) { s_keys[rank[j]] = key[j]; if (P::HAS_VAL) s_vals[rank[j]] = val[j]; }
    }
    __syncthreads();
    // NOTE: padding items (digit 255, highest tile indices) rank after every valid key, so valid keys occupy [0, n_valid)
    const int dst = which ^ 1;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
        const u32 lp = j * RS_THREADS + tid;
        if (lp < n_valid) {
            const Key k = s_keys[lp];
            const u32 d = P::digit(k, byte);
            const u64 g = (u64)s_gbase[d] + (lp - s_dig_excl[d]);
            P::store_key(bufs, dst, g, k);
            if (P::HAS_VAL) bufs.v[dst][g] = s_vals[lp];
        }
    }
}

template <class P>
static size_t radix_pass_smem() {
    return sizeof(typename P::Key) * RS_THREADS * P::ITEMS + (P::HAS_VAL ? 4 * RS_THREADS * P::ITEMS : 0) +
           4 * ((RS_THREADS / 32) * 256 + 256 + 256 + 32);
}

struct RadixWs {                   // device workspace for sorts of up to max_n elements
    DevBuf plan, desc;
    size_t max_n = 0;
    int alloc(size_t n) {
        max_n = n;
        MK_TRY(plan.alloc(sizeof(RadixPlan)));
        size_t tiles = n / (RS_THREADS * 8) + 2;           // smallest tile of the policies
        return desc.alloc(tiles * 256 * 4);
    }
};

// Sorts `n` elements, stable, on the scheduled bytes.  Input in buffer 0; the result ends in buffer plan->final_buf (device value).
// hist_done: the digit histograms are already in ws.plan->hist (zeroed, then filled by the kernel that produced the keys)
// What a consumer reads back (tests/test_gpu_radix_edges.py checks each point through tests/radix_harness.cu):
//   - a pass whose digit is the same for every key is skipped; final_buf = parity of plan->n_exec, the passes that ran
//   - iota_vals: the first pass that runs writes the input index as the value, so values hold the stable permutation.  When
//     NO pass runs (n_exec == 0: all keys equal on the schedule, or n == 0) the values are never written and buffer 0 keeps
//     whatever the caller left there: the permutation is the identity and the consumer takes the position itself
//     (`plan->n_exec ? v[i] : i`, pairs.cu k_mark_first, norm.cu k_nm_fill_lower)
//   - bytes outside the schedule (the whole value word of Rec16 records included) travel with their key unsorted
//   - refused before anything is enqueued: n >= 2^30 (30-bit look-back counts) or n > ws.max_n (MK_ERR_CAPACITY)
template <class P>
static int radix_sort(typename P::Bufs bufs, u64 n, const RadixSchedule &sch, RadixWs &ws, int iota_vals, int sms,
                      cudaStream_t s, u64 *launches, bool hist_done = false) {
    if (n >= (1ull << 30)) { mk_set_error("radix_sort: at most 2^30-1 elements per call"); return MK_ERR_CAPACITY; }
    if (n > ws.max_n) { mk_set_error("radix_sort: workspace too small"); return MK_ERR_CAPACITY; }
    RadixPlan *plan = ws.plan.as<RadixPlan>();
    if (!hist_done) {
        MK_CUDA(cudaMemsetAsync(plan, 0, sizeof(RadixPlan), s));
        int grid = (int)std::min<u64>((n + RS_THREADS * 8 - 1) / (RS_THREADS * 8), (u64)sms * 8);
        if (grid < 1) grid = 1;
        k_radix_hist<P><<<grid, RS_THREADS, sch.n_pass * 256 * 4, s>>>(bufs, n, sch, plan);
        *launches += 1;
    }
    k_radix_plan<<<1, 256, 0, s>>>(plan, n, sch.n_pass);
    *launches += 1;
    const int TILE = RS_THREADS * P::ITEMS;
    const u64 tiles = (n + TILE - 1) / TILE;
    const size_t smem = radix_pass_smem<P>();
    // per device, not per process: set on every call (a cheap driver call; a static flag would leave a second device unset)
    MK_CUDA(cudaFuncSetAttribute(k_radix_pass<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int p = 0; p < sch.n_pass && tiles; ++p) {
        MK_CUDA(cudaMemsetAsync(ws.desc.p, 0, tiles * 256 * 4, s));
        k_radix_pass<P><<<(unsigned)tiles, RS_THREADS, smem, s>>>(bufs, n, p, sch.byte_of[p], plan, ws.desc.as<u32>(), iota_vals);
        *launches += 1;
    }
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}
