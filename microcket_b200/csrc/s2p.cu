// s2p.cu — host side of the sam2pairs path: contexts, window pipeline, C ABI.
// Replaces the reference's main loop (src/sam2pairs/sam2pairs.cpp:23-229); see include/microcket_b200.h.
#include <algorithm>
#include <cstdarg>
#include <cstring>
#include <deque>
#include <vector>
#include "ctx.h"
#include "s2p_kernels.cuh"
#include "radix_sort.cuh"

struct mk_xchg;
extern "C" int mk_xchg_begin(mk_xchg *);
extern "C" int mk_xchg_scatter_part_device(mk_xchg *, const mk_pair *, const uint64_t *, uint32_t, void *);
extern "C" int mk_xchg_end_device(mk_xchg *, void *);
int xchg_scatter_records(mk_xchg *, const void *d_rec, u64 n, const unsigned long long *d_part, int owner, cudaStream_t);   // xchg.cu
void xchg_world_rank(const mk_xchg *, int *world, int *rank);
// multi-rank krmdup (mk_s2p_rmdup_*): off, pass 1 running, pass 1 done, keys sent, losers sent back, drop bits settled
enum { RKP_OFF = 0, RKP_PASS1, RKP_KEYED, RKP_SENT, RKP_DECIDED, RKP_SETTLED };
#define S2P_XPARTS 4096                            // windows of one mk_s2p_run_device call whose pairs can be scattered separately

static const size_t S2P_CARRY = 8u << 20;          // room in front of every window for the previous window's last group
static const u32 S2P_BATCH = 1u << 18;             // pairutil.h:48

struct S2PSlot {                                   // one in-flight window of the host streaming API
    PinBuf h_in;
    DevBuf d_in, d_text, d_pairs, d_sam;
    DevBuf d_sc;                                   // self-circle group indices of this window
    PinBuf h_state;
    cudaEvent_t ev_h2d = nullptr, ev_done = nullptr, ev_free = nullptr;   // ev_free: last reader of d_in has run
    bool free_pending = false;
    bool busy = false;                             // kernels enqueued, results not yet looked at
    size_t n_in = 0;
    // finished window whose outputs still sit in d_text / d_pairs / d_sam (pulled straight from there, or spilled)
    size_t text_len = 0, text_off = 0, pairs_n = 0, pairs_off = 0, sam_len = 0, sam_off = 0;
    u64 win_id = 0;
    bool has_output() const { return text_off < text_len || pairs_off < pairs_n || sam_off < sam_len; }
};

struct S2PCtx : mk_ctx {
    mk_s2p_cfg cfg;
    size_t W = 0, in_cap = 0; u32 cap_lines = 0, n_desc = 0, sc_cap = 0;
    u32 chr_slots = 0, chr_cap = 0, sc_cap_dev = 0;
    cudaStream_t s_comp = nullptr, s_in = nullptr, s_out = nullptr;
    u32 n_chunks_cap = 0;
    DevBuf d_cklist, d_ckcnt, d_tiletot;
    DevBuf d_params;                               // device copies of the kernels' parameter blocks (S2PParams.self)
    u32 n_sub_cap = 0;
    DevBuf d_state, d_nl, d_lmeta, d_rec, d_res, d_samdst, d_desc, d_chr, d_id2slot, d_sclist;
    DevBuf d_rmtab[2], d_rminfo; u64 rm_slots[2] = {0, 0};    // SAM-space krmdup (cfg.rmdup)
    S2PSlot slot[2];
    int grid_scan4 = 0, grid_emit = 0, grid_gs = 0, grid_parse = 0, grid_rm = 0;
    u64 launches = 0, fallback_windows = 0;
    // host streaming state
    std::vector<char> tail;                        // input not yet part of a window (a partial last line, or small pushes)
    PinBuf h_nl;                                   // a pinned '\n' (terminates a last line that lacks one)
    u64 windows = 0;
    int prev_slot = -1;
    bool finished_input = false;
    std::deque<std::vector<char>> q_text, q_sam;
    std::deque<std::vector<mk_pair>> q_pairs;
    size_t q_text_off = 0, q_sam_off = 0, q_pairs_off = 0;
    // selfCircle emulation (sam2pairs.cpp:150,172,202-210)
    u64 sc_full_rule = 0; std::vector<u64> sc_tail; u64 sc_true = 0;
    bool use_device_path = false;
    WinState last_state;
    // overlapped multi-GPU scatter (mk_s2p_attach_xchg)
    mk_xchg *xchg = nullptr; u32 xchg_res = 0; cudaStream_t s_x = nullptr; DevBuf d_xparts; u32 x_slot = 0;
    std::vector<cudaEvent_t> x_events; size_t x_ev_used = 0;
    // multi-rank krmdup: phase, pass 1's records (in d_rmtab[0], which this mode does not use as a table) and totals, the
    // owner's sort buffers, the drop bits of pass 1's lines
    int rk = RKP_OFF;
    u64 rk_cap = 0, rk_lines = 0, rk_keys = 0, rk_disc = 0;
    DevBuf d_rkcnt, d_rksort, d_rklose, d_rkdrop; RadixWs rk_rws;
    // optional per-kernel timing (bench.py roofline): events around every kernel of every window
    bool timing = false;
    std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0;
    std::vector<std::pair<int, size_t>> ev_marks;          // (kernel id, index of its start event); end = next event
    double k_ms[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; u64 k_cnt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    cudaEvent_t next_event() {
        if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
        return ev_pool[ev_used++];
    }
    S2PCtx() { kind = MK_CTX_S2P; memset(&last_state, 0, sizeof last_state); }
    ~S2PCtx() override {
        cudaSetDevice(cfg.device);
        for (auto &s : slot) { if (s.ev_h2d) cudaEventDestroy(s.ev_h2d); if (s.ev_done) cudaEventDestroy(s.ev_done); if (s.ev_free) cudaEventDestroy(s.ev_free); }
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (s_comp) cudaStreamDestroy(s_comp);
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
        if (s_x) cudaStreamDestroy(s_x);
        for (auto e : x_events) cudaEventDestroy(e);
    }
};

static u64 fnv1a(const char *s, size_t n) {
    u64 h = 0xCBF29CE484222325ull;
    for (size_t i = 0; i < n; ++i) h = (h ^ (u64)(unsigned char)s[i]) * 0x100000001B3ull;
    return h ? h : 0x9E3779B97F4A7C15ull;
}

extern "C" void mk_s2p_default_cfg(mk_s2p_cfg *c) {
    memset(c, 0, sizeof *c);
    c->mode = 1; c->min_mapped_ratio = 0.5f; c->min_mapq = 10; c->write_sam = 1; c->emu_threads = 4;   // sam2pairs.cpp:33, pairutil.h:50-53
    c->device = 0; c->emit_text = 1; c->emit_packed = 0; c->window_bytes = 0; c->lane = 0;
    c->rmdup = 0; c->rmdup_capacity = 0; c->hskip1 = 5; c->klen1 = 16; c->hskip2 = 5; c->klen2 = 16;                  // krmdup.cpp:231-234
}

static S2PParams make_params(S2PCtx *c, const char *buf, u64 *sc_list, u32 sc_cap, char *out_text, u64 text_cap, mk_pair *out_pairs, u64 pairs_cap,
                             char *out_sam, u64 sam_cap, u64 window_bytes, int running, u64 *line_off = nullptr, u64 line_off_cap = 0, u64 line_off_base = 0) {
    S2PParams p;
    memset(&p, 0, sizeof p);
    p.buf = buf; p.st = c->d_state.as<WinState>(); p.nl_pos = c->d_nl.as<u32>(); p.lmeta = c->d_lmeta.as<u8>();
    p.ck_list = c->d_cklist.as<u32>(); p.ck_cnt = c->d_ckcnt.as<u32>(); p.ck_pre = p.ck_cnt + c->n_chunks_cap; p.ck_bsum = p.ck_pre + c->n_chunks_cap; p.n_chunks_cap = c->n_chunks_cap;
    p.tile_tot = c->d_tiletot.as<uint4>(); p.tile_pre = p.tile_tot + c->n_sub_cap; p.n_sub_cap = c->n_sub_cap;
    p.seg_tot = p.tile_pre + c->n_sub_cap; p.n_seg_cap = c->n_sub_cap / EMIT_SEG + 2;
    p.rec = c->d_rec.as<LineRec>(); p.res = c->d_res.as<GroupRes>(); p.sam_dst = c->d_samdst.as<u32>();
    p.desc_scan = c->d_desc.as<u64>();
    p.chr = c->d_chr.as<ChrSlot>(); p.chr_mask = c->chr_slots - 1; p.id_to_slot = c->d_id2slot.as<int>(); p.chr_cap = c->chr_cap;
    p.sc_list = sc_list; p.sc_cap = sc_cap;
    p.out_text = out_text; p.out_text_cap = out_text ? text_cap : 0;
    p.out_pairs = out_pairs; p.out_pairs_cap = out_pairs ? pairs_cap : 0;
    p.out_sam = out_sam; p.out_sam_cap = out_sam ? sam_cap : 0;
    p.out_line_off = line_off; p.out_line_off_cap = line_off ? line_off_cap : 0; p.line_off_base = line_off_base;
    p.window_bytes = window_bytes; p.cap_lines = c->cap_lines;
    p.mode = c->cfg.mode; p.min_mapq = c->cfg.min_mapq; p.ratio = c->cfg.min_mapped_ratio; p.lane = c->cfg.lane;
    p.write_sam = c->cfg.write_sam && out_sam; p.emit_text = c->cfg.emit_text && out_text; p.emit_packed = c->cfg.emit_packed && out_pairs;
    p.running_offsets = running;
    p.xparts = (c->xchg && c->d_xparts.p && c->rk != RKP_PASS1) ? c->d_xparts.as<unsigned long long>() : nullptr;
    if (c->rk != RKP_OFF) {
        p.rk_rec = c->d_rmtab[0].as<uint4>(); p.rk_cap = c->rk_cap;
        p.rk_drop = c->d_rkdrop.as<u32>(); p.rk_lines = c->rk_lines; p.rk_cnt = c->d_rkcnt.as<unsigned long long>();
    }
    p.rm_on = c->cfg.rmdup ? 1 : 0;
    if (p.rm_on) {
        p.rm_hskip1 = c->cfg.hskip1; p.rm_klen1 = c->cfg.klen1; p.rm_hskip2 = c->cfg.hskip2; p.rm_klen2 = c->cfg.klen2;
        for (int t = 0; t < 2; ++t) { p.rm_tab[t] = c->d_rmtab[t].as<unsigned long long>(); p.rm_mask[t] = c->rm_slots[t] - 1; }
        p.rm_info = c->d_rminfo.as<u32>();
    }
    p.self = nullptr;
    return p;
}

// The parameter block also lives in device memory (slot 0..3 of d_params): out-of-line device functions take it by
// reference from there, so no kernel copies its parameters to local memory.
static int upload_params(S2PCtx *c, S2PParams &p, int slot, cudaStream_t s) {
    p.self = c->d_params.as<S2PParams>() + slot;
    MK_CUDA(cudaMemcpyAsync((void *)p.self, &p, sizeof p, cudaMemcpyHostToDevice, s));
    return MK_OK;
}

// enqueue the kernels of one window on the compute stream
static void launch_window(S2PCtx *c, const S2PParams &p, cudaStream_t s) {
    const bool t = c->timing;
    auto mark = [&](int id) { if (t) { cudaEvent_t e = c->next_event(); cudaEventRecord(e, s); c->ev_marks.emplace_back(id, c->ev_used - 1); } };
    k_win_begin<<<(c->n_desc + 255) / 256, 256, 0, s>>>(p, c->n_desc);
    mark(0);
    // chunked scan (no look-back); the look-back kernel only does work when a chunk overflowed its slot list
    k_scan_chunks<<<(c->n_chunks_cap + SC_WARPS - 1) / SC_WARPS, SC_WARPS * 32, 0, s>>>(p);
    mark(6);
    k_chunk_prefix<<<(c->n_chunks_cap + SC_PFX_BLOCK - 1) / SC_PFX_BLOCK, 256, 0, s>>>(p);
    k_chunk_compact<<<(c->n_chunks_cap + 7) / 8, 256, 0, s>>>(p);
    k_scan_lines<4, 4><<<c->grid_scan4, S2P_SCAN_THREADS, 4 * 8192, s>>>(p, 1);
    mark(1);
    if (c->rk == RKP_PASS1) {                            // multi-rank krmdup, pass 1: the key records of the window's runs, no output
        k_parse<true><<<c->grid_parse, 256, PR_SMEM, s>>>(p);
        mark(7);
        k_rm_keys<<<c->grid_rm, 256, 0, s>>>(p);
        mark(5);
        k_win_end<<<1, 1, 0, s>>>(p, c->x_slot);
        c->launches += 8;
        return;
    }
    if (p.rm_on && c->rk == RKP_SETTLED) {               // pass 2: the settled drop bits in place of the key table
        k_parse<false><<<c->grid_parse, 256, PR_SMEM, s>>>(p);
        mark(7);
        k_rm_apply<<<c->grid_gs, 256, 0, s>>>(p);
        c->launches += 1;
    } else if (p.rm_on) {                                // SAM-space krmdup: duplicate / discarded read pairs lose LM_KEEP before grouping
        k_parse<true><<<c->grid_parse, 256, PR_SMEM, s>>>(p);
        mark(7);
        k_rm_insert<<<c->grid_rm, 256, 0, s>>>(p);
        c->launches += 1;
    } else k_parse<false><<<c->grid_parse, 256, PR_SMEM, s>>>(p);
    mark(2);
    k_group<<<c->grid_gs, 256, 0, s>>>(p);
    mark(3);
    k_emit_prefix<<<c->n_sub_cap / EMIT_SEG + 2, EMIT_SEG, 0, s>>>(p);
    k_emit<<<c->grid_emit, EMIT_THREADS, 0, s>>>(p);
    mark(4);
    c->launches += 9;
    if (p.write_sam) { k_copy_sam<<<c->grid_gs, 256, 0, s>>>(p); c->launches += 1; }
    mark(5);
    k_win_end<<<1, 1, 0, s>>>(p, c->x_slot);
    c->launches += 1;
    if (p.xparts && c->xchg && p.out_pairs) {            // this window's pairs leave for their owners while the next window is parsed
        if (c->x_ev_used == c->x_events.size()) { cudaEvent_t e; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); c->x_events.push_back(e); }
        cudaEvent_t e = c->x_events[c->x_ev_used++];
        cudaEventRecord(e, s);
        cudaStreamWaitEvent(c->s_x, e, 0);
        mk_xchg_scatter_part_device(c->xchg, p.out_pairs, (const uint64_t *)(p.xparts + 2 * c->x_slot), c->xchg_res, c->s_x);
        c->x_slot = (c->x_slot + 1) % S2P_XPARTS;
    }
}

extern "C" int mk_s2p_attach_xchg(mk_ctx *x, mk_xchg *xc, uint32_t res) {
    if (!x || x->kind != MK_CTX_S2P || (xc && res == 0)) { mk_set_error("mk_s2p_attach_xchg: bad argument"); return MK_ERR_ARG; }
    S2PCtx *c = (S2PCtx *)x;
    MK_CUDA(cudaSetDevice(c->cfg.device));
    c->xchg = xc; c->xchg_res = res;
    if (xc && !c->s_x) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        MK_CUDA(cudaStreamCreateWithPriority(&c->s_x, cudaStreamNonBlocking, hi));     // its few CTAs should not queue behind a full-grid kernel
        MK_TRY(c->d_xparts.alloc((size_t)S2P_XPARTS * 16));
    }
    return MK_OK;
}

// fold the recorded events into per-kernel totals (call after the stream is idle)
static void timing_collect(S2PCtx *c) {
    for (size_t i = 0; i + 1 < c->ev_marks.size(); ++i) {
        int id = c->ev_marks[i].first;
        if (id == 5) continue;                                  // 5 closes a window
        float ms = 0;
        if (cudaEventElapsedTime(&ms, c->ev_pool[c->ev_marks[i].second], c->ev_pool[c->ev_marks[i + 1].second]) == cudaSuccess) { c->k_ms[id] += ms; c->k_cnt[id] += 1; }
    }
    c->ev_marks.clear(); c->ev_used = 0;
}

extern "C" int mk_s2p_enable_timing(mk_ctx *x, int on) {
    if (!x || x->kind != MK_CTX_S2P) { mk_set_error("not a sam2pairs context"); return MK_ERR_ARG; }
    ((S2PCtx *)x)->timing = on != 0;
    return MK_OK;
}

// ms[k], count[k] for k = 0 newline scan, 1 parse, 2 group, 3 emit, 4 copy_sam, 5 scan index (prefix + compaction + the
// look-back fallback's early exit); 6, 7 unused (accumulated since creation); arrays of 8
extern "C" int mk_s2p_kernel_times(mk_ctx *x, double *ms, uint64_t *count) {
    if (!x || x->kind != MK_CTX_S2P || !ms || !count) { mk_set_error("mk_s2p_kernel_times: bad argument"); return MK_ERR_ARG; }
    S2PCtx *c = (S2PCtx *)x;
    cudaSetDevice(c->cfg.device);
    cudaDeviceSynchronize();
    timing_collect(c);
    for (int k = 0; k < 5; ++k) { ms[k] = c->k_ms[k]; count[k] = c->k_cnt[k]; }
    ms[5] = c->k_ms[6]; count[5] = c->k_cnt[6];
    ms[6] = c->k_ms[7]; count[6] = c->k_cnt[7]; ms[7] = 0; count[7] = 0;
    return MK_OK;
}

__global__ void k_set_stream(WinState *st, u64 cursor, u64 total, u32 is_last) { st->cursor = cursor; st->total = total; st->is_last = is_last; }

// move the previous window's unprocessed tail in front of the next window's bytes and set up the cursor
__global__ void k_carry(WinState *st, const char *prev_buf, char *cur_buf, u64 carry_cap, u64 n_new, u32 is_last, int have_prev) {
    __shared__ u64 s_t, s_cur;
    if (threadIdx.x == 0) {
        u64 t = have_prev ? st->total - st->cursor : 0;
        if (t > carry_cap) { st->err |= S2P_ERR_NOPROGRESS; t = 0; }
        s_t = t; s_cur = st->cursor;
    }
    __syncthreads();
    const u64 t = s_t, from = s_cur;
    for (u64 b = threadIdx.x; b < t; b += blockDim.x) cur_buf[carry_cap - t + b] = prev_buf[from + b];
    __syncthreads();
    if (threadIdx.x == 0) { st->cursor = carry_cap - t; st->total = carry_cap + n_new; st->is_last = is_last; }
}

extern "C" int mk_s2p_create(const mk_s2p_cfg *cfg, const char *const *names, int n_chrom, mk_ctx **out) {
    if (!cfg || !out) { mk_set_error("mk_s2p_create: null argument"); return MK_ERR_ARG; }
    if (cfg->mode != 0 && cfg->mode != 1) { mk_set_error("mk_s2p_create: mode must be 0 (flash) or 1 (unc)"); return MK_ERR_ARG; }
    if (cfg->emu_threads < 2) { mk_set_error("mk_s2p_create: at least 2 threads are required"); return MK_ERR_ARG; }   // sam2pairs.cpp:36-39
    if (cfg->rmdup && (cfg->hskip1 < 0 || cfg->hskip2 < 0 || cfg->klen1 < 0 || cfg->klen2 < 0 || cfg->klen1 + cfg->klen2 < 16 || cfg->klen1 + cfg->klen2 > 32)) {
        mk_set_error("mk_s2p_create: rmdup key size must be 16..32 bases");       // krmdup.cpp:256-262
        return MK_ERR_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(cfg->device));
    S2PCtx *c = new S2PCtx();
    c->cfg = *cfg;
    c->W = cfg->window_bytes ? cfg->window_bytes : (size_t)256 << 20;
    if (c->W < (1u << 16)) c->W = 1u << 16;
    if (c->W > ((size_t)2040 << 20)) c->W = (size_t)2040 << 20;     // packed 31-bit byte counters in the emit scan
    c->W = (c->W + 15) & ~(size_t)15;
    c->in_cap = S2P_CARRY + c->W + 64;
    c->cap_lines = (u32)((S2P_CARRY + c->W) / 32 + 1024);
    c->n_sub_cap = c->cap_lines / EMIT_TILE + 4;
    c->n_desc = std::max<u32>((u32)((S2P_CARRY + c->W) / S2P_TILE_BYTES + 4), c->n_sub_cap);   // k_win_begin's grid covers both
    c->sc_cap = c->cap_lines / 2 + 16; c->sc_cap_dev = 0;
    c->n_chunks_cap = (u32)((S2P_CARRY + c->W) / SC_CHUNK + 8) & ~3u;       // multiple of 4: counts and prefixes are read as uint4
    c->chr_cap = 16384; c->chr_slots = 32768;
    int rc = MK_OK;
#define A(x) do { if (rc == MK_OK) rc = (x); } while (0)
    A(c->d_state.alloc(sizeof(WinState)));
    A(c->d_params.alloc(4 * sizeof(S2PParams)));
    A(c->d_nl.alloc((size_t)c->cap_lines * 4)); A(c->d_lmeta.alloc(c->cap_lines)); A(c->d_rec.alloc((size_t)c->cap_lines * sizeof(LineRec)));
    A(c->d_res.alloc((size_t)c->cap_lines * sizeof(GroupRes)));
    A(c->d_samdst.alloc(cfg->write_sam ? (size_t)c->cap_lines * 4 : 16));
    A(c->d_desc.alloc((size_t)c->n_desc * 8)); A(c->d_chr.alloc((size_t)c->chr_slots * sizeof(ChrSlot)));
    A(c->d_id2slot.alloc((size_t)c->chr_cap * 4));
    A(c->d_tiletot.alloc(((size_t)c->n_sub_cap * 2 + c->n_sub_cap / EMIT_SEG + 2) * sizeof(uint4)));
    A(c->d_cklist.alloc((size_t)c->n_chunks_cap * SC_CAP * 4)); A(c->d_ckcnt.alloc((size_t)c->n_chunks_cap * 2 * 4 + 160 * 4));   // counts, prefixes, 160 block sums (W <= 2040 MiB: <= 130 blocks of 1024 chunks)
    if (cfg->rmdup) {
        // two slots per expected read pair, {key, first line} = 16 bytes per slot; the lower-case identity space is rare
        const u64 cap = cfg->rmdup_capacity ? cfg->rmdup_capacity : (u64)1 << 24;
        u64 slots = 1024; while (slots < 2 * cap) slots <<= 1;
        c->rm_slots[0] = slots; c->rm_slots[1] = std::max<u64>(slots >> 4, 1024);
        for (int t = 0; t < 2; ++t) { A(c->d_rmtab[t].alloc(c->rm_slots[t] * 16)); if (rc == MK_OK && cudaMemset(c->d_rmtab[t].p, 0xFF, c->rm_slots[t] * 16) != cudaSuccess) rc = MK_ERR_CUDA; }
        A(c->d_rminfo.alloc((size_t)c->cap_lines * 4));
    }
#undef A
    if (rc != MK_OK) { delete c; return rc; }
    cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking);
    // chromosome table: pre-registered names get ids 0..n-1
    std::vector<ChrSlot> tab(c->chr_slots);
    memset(tab.data(), 0, tab.size() * sizeof(ChrSlot));
    for (auto &s : tab) s.id = -1;
    std::vector<int> id2slot(c->chr_cap, 0);
    int reg = 0;
    for (int i = 0; i < n_chrom && names; ++i) {
        size_t len = strlen(names[i]);
        if (len == 0) continue;
        u64 h = fnv1a(names[i], len);
        u32 l = (u32)std::min<size_t>(len, S2P_NAME_MAX);
        u32 s = (u32)(h ^ (h >> 29)) & (c->chr_slots - 1);
        bool dup = false;
        while (tab[s].key) { if (tab[s].key == h && tab[s].len == l && !memcmp(tab[s].name, names[i], l)) { dup = true; break; } s = (s + 1) & (c->chr_slots - 1); }
        if (dup) continue;
        tab[s].key = h; tab[s].len = (u16)l; memcpy(tab[s].name, names[i], l);
        u64 n8 = 0; for (u32 b = 0; b < l && b < 8; ++b) n8 |= (u64)(unsigned char)names[i][b] << (8 * b);
        tab[s].name8 = n8; tab[s].id = reg; id2slot[reg] = (int)s; ++reg;
    }
    WinState st; memset(&st, 0, sizeof st); st.n_chrom = (u32)reg; st.rm_allones[0] = st.rm_allones[1] = ~0ull;
    cudaMemcpy(c->d_chr.p, tab.data(), tab.size() * sizeof(ChrSlot), cudaMemcpyHostToDevice);
    cudaMemcpy(c->d_id2slot.p, id2slot.data(), id2slot.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(c->d_state.p, &st, sizeof st, cudaMemcpyHostToDevice);
    // grids: the two look-back kernels need every CTA resident
    int sms = mk_sm_count(cfg->device), occ = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_scan_lines<4, 4>, S2P_SCAN_THREADS, 4 * 8192);
    c->grid_scan4 = sms * std::max(1, std::min(occ, 4));
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_emit, EMIT_THREADS, 0);
    c->grid_emit = sms * std::max(1, occ);
    c->grid_gs = sms * 8;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_rm_insert, 256, 0);
    c->grid_rm = sms * std::max(1, occ);                   // one resident wave: the rounds are split statically
    cudaFuncSetAttribute(k_parse<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM);
    cudaFuncSetAttribute(k_parse<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM);
    if (cfg->rmdup) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_parse<true>, 256, PR_SMEM);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_parse<false>, 256, PR_SMEM);
    c->grid_parse = sms * std::max(1, occ);                 // one resident wave: every CTA then pipelines many rounds
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { mk_set_error("mk_s2p_create: %s", cudaGetErrorString(e)); delete c; return MK_ERR_CUDA; }
    *out = c;
    return MK_OK;
}

static int s2p_check(mk_ctx *x, S2PCtx **c) {
    if (!x || x->kind != MK_CTX_S2P) { mk_set_error("not a sam2pairs context"); return MK_ERR_ARG; }
    *c = (S2PCtx *)x;
    cudaSetDevice((*c)->cfg.device);
    return MK_OK;
}

static int s2p_err_check(u32 err) {
    if (!err) return MK_OK;
    if (err & S2P_ERR_LINES) mk_set_error("sam2pairs: too many lines in one window (lines shorter than 32 bytes on average); raise window capacity");
    else if (err & S2P_ERR_TEXT) mk_set_error("sam2pairs: pairs text output buffer too small");
    else if (err & S2P_ERR_PAIRS) mk_set_error("sam2pairs: packed pairs output buffer too small");
    else if (err & S2P_ERR_SAM) mk_set_error("sam2pairs: SAM passthrough output buffer too small");
    else if (err & S2P_ERR_SCLIST) mk_set_error("sam2pairs: self-circle list overflow");
    else if (err & S2P_ERR_NOPROGRESS) mk_set_error("sam2pairs: a single read group (or line) is larger than the window/carry capacity");
    else if (err & S2P_ERR_CHRTABLE) mk_set_error("sam2pairs: chromosome table full");
    else if (err & S2P_ERR_RMTABLE) mk_set_error("sam2pairs: rmdup key table full; raise cfg.rmdup_capacity (read pairs in the stream)");
    return MK_ERR_CAPACITY;
}

static void sc_absorb(S2PCtx *c, const u64 *list, u32 n, u64 groups_done_after) {
    // entries of batches that can no longer be the stream's last batch are settled with the loader/worker split rule
    const u32 T = (u32)c->cfg.emu_threads;
    const u32 share_full = S2P_BATCH / (T - 1);                       // sam2pairs.cpp:172-173 with tn = 0
    c->sc_true += n;
    for (u32 i = 0; i < n; ++i) c->sc_tail.push_back(list[i]);
    if (c->cfg.sharded) return;                                       // global indices unknown until finish_sharded
    const u64 open_batch = groups_done_after / S2P_BATCH;             // batch that may still turn out to be the last one
    size_t w = 0;
    for (size_t i = 0; i < c->sc_tail.size(); ++i) {
        u64 g = c->sc_tail[i];
        if (g / S2P_BATCH < open_batch) { if ((u32)(g % S2P_BATCH) < share_full) ++c->sc_full_rule; }
        else c->sc_tail[w++] = g;
    }
    c->sc_tail.resize(w);
}

// wait for a streaming window; its outputs stay on the device until pulled (or spilled)
static int s2p_complete(S2PCtx *c, int b) {
    S2PSlot &s = c->slot[b];
    if (!s.busy) return MK_OK;
    MK_CUDA(cudaEventSynchronize(s.ev_done));
    s.busy = false;
    WinState st = *s.h_state.as<WinState>();
    c->last_state = st;
    MK_TRY(s2p_err_check(st.err));
    s.text_len = c->cfg.emit_text ? st.w_text : 0; s.pairs_n = c->cfg.emit_packed ? st.w_emit : 0; s.sam_len = c->cfg.write_sam ? st.w_sam : 0;
    s.text_off = s.pairs_off = s.sam_off = 0;
    if (st.sc_count) {
        std::vector<u64> l(st.sc_count);
        MK_CUDA(cudaMemcpyAsync(l.data(), s.d_sc.p, (size_t)st.sc_count * 8, cudaMemcpyDeviceToHost, c->s_out));
        MK_CUDA(cudaStreamSynchronize(c->s_out));
        sc_absorb(c, l.data(), st.sc_count, st.groups_done);
    } else sc_absorb(c, nullptr, 0, st.groups_done);
    return MK_OK;
}

// move a finished window's un-pulled outputs to host queues so that the slot can be reused
static int s2p_spill(S2PCtx *c, int b) {
    S2PSlot &s = c->slot[b];
    MK_TRY(s2p_complete(c, b));
    if (s.text_off < s.text_len) {
        std::vector<char> v(s.text_len - s.text_off);
        MK_CUDA(cudaMemcpyAsync(v.data(), s.d_text.as<char>() + s.text_off, v.size(), cudaMemcpyDeviceToHost, c->s_out));
        MK_CUDA(cudaStreamSynchronize(c->s_out));
        c->q_text.emplace_back(std::move(v));
    }
    if (s.pairs_off < s.pairs_n) {
        std::vector<mk_pair> v(s.pairs_n - s.pairs_off);
        MK_CUDA(cudaMemcpyAsync(v.data(), s.d_pairs.as<mk_pair>() + s.pairs_off, v.size() * sizeof(mk_pair), cudaMemcpyDeviceToHost, c->s_out));
        MK_CUDA(cudaStreamSynchronize(c->s_out));
        c->q_pairs.emplace_back(std::move(v));
    }
    if (s.sam_off < s.sam_len) {
        std::vector<char> v(s.sam_len - s.sam_off);
        MK_CUDA(cudaMemcpyAsync(v.data(), s.d_sam.as<char>() + s.sam_off, v.size(), cudaMemcpyDeviceToHost, c->s_out));
        MK_CUDA(cudaStreamSynchronize(c->s_out));
        c->q_sam.emplace_back(std::move(v));
    }
    s.text_off = s.text_len; s.pairs_off = s.pairs_n; s.sam_off = s.sam_len;
    return MK_OK;
}

static int s2p_slot_init(S2PCtx *c, S2PSlot &s) {
    if (s.d_in.p) return MK_OK;
    MK_TRY(s.h_in.alloc(c->W + 64));
    MK_TRY(s.d_in.alloc(c->in_cap));
    MK_CUDA(cudaMemset(s.d_in.p, '\n', c->in_cap));
    MK_TRY(s.d_sc.alloc((size_t)c->sc_cap * 8));
    if (c->cfg.emit_text) MK_TRY(s.d_text.alloc(c->in_cap + 4096));
    if (c->cfg.emit_packed) MK_TRY(s.d_pairs.alloc((size_t)c->cap_lines * sizeof(mk_pair)));
    if (c->cfg.write_sam) MK_TRY(s.d_sam.alloc(c->in_cap));
    MK_TRY(s.h_state.alloc(sizeof(WinState)));
    MK_CUDA(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
    MK_CUDA(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
    MK_CUDA(cudaEventCreateWithFlags(&s.ev_free, cudaEventDisableTiming));
    if (!c->h_nl.p) { MK_TRY(c->h_nl.alloc(16)); c->h_nl.as<char>()[0] = '\n'; }
    return MK_OK;
}

// The slot for the next window, ready to be filled: its previous window (k-2) is finished and its outputs are out.
static int s2p_next_slot(S2PCtx *c, S2PSlot **out) {
    const int b = (int)(c->windows & 1);
    S2PSlot &s = c->slot[b];
    MK_TRY(s2p_slot_init(c, s));
    if (s.busy || s.has_output()) MK_TRY(s2p_spill(c, b));
    *out = &s;
    return MK_OK;
}

// Enqueue one window.  Its bytes are the first n_stage bytes of the slot's pinned buffer followed by n_direct bytes
// DMA'd straight from `direct` (caller memory that is already pinned), plus a final '\n' when add_nl.
static int s2p_submit(S2PCtx *c, size_t n_stage, const char *direct, size_t n_direct, bool add_nl, bool final_chunk) {
    const int b = (int)(c->windows & 1);
    S2PSlot &s = c->slot[b];
    const size_t n = n_stage + n_direct + (add_nl ? 1 : 0);
    s.n_in = n;
    char *dst = s.d_in.as<char>() + S2P_CARRY;
    if (s.free_pending) { MK_CUDA(cudaStreamWaitEvent(c->s_in, s.ev_free, 0)); s.free_pending = false; }
    if (n_stage) MK_CUDA(cudaMemcpyAsync(dst, s.h_in.p, n_stage, cudaMemcpyHostToDevice, c->s_in));
    if (n_direct) MK_CUDA(cudaMemcpyAsync(dst + n_stage, direct, n_direct, cudaMemcpyHostToDevice, c->s_in));
    if (add_nl) MK_CUDA(cudaMemcpyAsync(dst + n_stage + n_direct, c->h_nl.p, 1, cudaMemcpyHostToDevice, c->s_in));
    MK_CUDA(cudaEventRecord(s.ev_h2d, c->s_in));
    MK_CUDA(cudaStreamWaitEvent(c->s_comp, s.ev_h2d, 0));
    const int pb = c->prev_slot;
    const char *prev = pb >= 0 ? c->slot[pb].d_in.as<char>() : s.d_in.as<char>();
    k_carry<<<1, 1024, 0, c->s_comp>>>(c->d_state.as<WinState>(), prev, s.d_in.as<char>(), S2P_CARRY, n, final_chunk ? 1u : 0u, pb >= 0);
    c->launches += 1;
    if (pb >= 0) {                                   // window k-1's buffer may be overwritten once its tail has been carried
        MK_CUDA(cudaEventRecord(c->slot[pb].ev_free, c->s_comp));
        c->slot[pb].free_pending = true;
    }
    S2PParams p = make_params(c, s.d_in.as<char>(), s.d_sc.as<u64>(), c->sc_cap, s.d_text.as<char>(), s.d_text.n,
                              s.d_pairs.as<mk_pair>(), c->cap_lines, s.d_sam.as<char>(), s.d_sam.n, S2P_CARRY + c->W + 64, 0);
    MK_TRY(upload_params(c, p, b, c->s_comp));
    launch_window(c, p, c->s_comp);
    MK_CUDA(cudaMemcpyAsync(s.h_state.p, c->d_state.p, sizeof(WinState), cudaMemcpyDeviceToHost, c->s_comp));
    MK_CUDA(cudaEventRecord(s.ev_done, c->s_comp));
    s.busy = true; s.win_id = c->windows;
    c->prev_slot = b;
    ++c->windows;
    return MK_OK;
}

static bool host_ptr_is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

extern "C" int mk_s2p_push(mk_ctx *x, const char *bytes, size_t n, int is_last) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (c->rk != RKP_OFF) { mk_set_error("mk_s2p_push on a context in the multi-rank krmdup mode (device-resident only)"); return MK_ERR_STATE; }
    if (c->finished_input) { mk_set_error("mk_s2p_push after the last chunk"); return MK_ERR_STATE; }
    if (c->use_device_path) { mk_set_error("mk_s2p_push on a context used with mk_s2p_run_device"); return MK_ERR_STATE; }
    const bool pinned = n >= (1u << 20) && host_ptr_is_pinned(bytes);
    std::vector<char> &tail = c->tail;                   // bytes received but not yet part of a window (partial line, small pushes)
    size_t off = 0;
    while (true) {
        const size_t left = n - off, have = tail.size() + left;
        if (have == 0) break;
        if (have < c->W && !is_last) { tail.insert(tail.end(), bytes + off, bytes + off + left); off = n; break; }
        // a window of at most W bytes: the tail followed by the first `take` new bytes, cut after its last complete line
        size_t take = std::min(left, c->W - std::min(c->W, tail.size()));
        const bool whole = is_last && take == left;
        size_t cut = take;
        if (!whole) {
            const void *nl = take ? memrchr(bytes + off, '\n', take) : nullptr;
            if (nl) cut = (size_t)((const char *)nl - (bytes + off)) + 1;
            else {                                         // no line end in the new bytes: the window ends inside the tail
                tail.insert(tail.end(), bytes + off, bytes + off + take); off += take;
                const void *tn = memrchr(tail.data(), '\n', tail.size());
                if (!tn) { mk_set_error("sam2pairs: a line longer than the window (%zu bytes)", c->W); return MK_ERR_CAPACITY; }
                const size_t keep_from = (size_t)((const char *)tn - tail.data()) + 1;
                S2PSlot *sp; MK_TRY(s2p_next_slot(c, &sp));
                memcpy(sp->h_in.p, tail.data(), keep_from);
                MK_TRY(s2p_submit(c, keep_from, nullptr, 0, false, false));
                tail.erase(tail.begin(), tail.begin() + (long)keep_from);
                continue;
            }
        }
        S2PSlot *sp; MK_TRY(s2p_next_slot(c, &sp));
        char *stage = sp->h_in.as<char>();
        const size_t n_tail = tail.size();
        if (n_tail) memcpy(stage, tail.data(), n_tail);
        tail.clear();
        const bool add_nl = whole && (cut ? bytes[off + cut - 1] != '\n' : (n_tail && stage[n_tail - 1] != '\n'));   // getline accepts a last line without '\n'
        if (pinned && cut >= (1u << 20)) {
            MK_TRY(s2p_submit(c, n_tail, bytes + off, cut, add_nl, whole));   // DMA straight from the caller's pinned memory
        } else {
            memcpy(stage + n_tail, bytes + off, cut);
            size_t tot = n_tail + cut;
            if (add_nl) stage[tot++] = '\n';
            MK_TRY(s2p_submit(c, tot, nullptr, 0, false, whole));
        }
        off += cut;
        if (whole) { c->finished_input = true; break; }
    }
    if (is_last) c->finished_input = true;
    return MK_OK;
}

template <class T>
static size_t drain(std::deque<std::vector<T>> &q, size_t &qoff, T *out, size_t cap) {
    size_t n = 0;
    while (out && n < cap && !q.empty()) {
        std::vector<T> &f = q.front();
        size_t m = std::min(cap - n, f.size() - qoff);
        memcpy(out + n, f.data() + qoff, m * sizeof(T));
        n += m; qoff += m;
        if (qoff == f.size()) { q.pop_front(); qoff = 0; }
    }
    return n;
}

// slots in window order; windows still running are waited for only once the input is complete
static int s2p_ready_slots(S2PCtx *c, int order[2], int *n) {
    *n = 0;
    if (c->windows == 0) return MK_OK;
    int cand[2] = {(int)(c->windows & 1), (int)((c->windows + 1) & 1)};   // older (k-2 / k-1 ...) first
    for (int i = 0; i < 2; ++i) {
        S2PSlot &s = c->slot[cand[i]];
        if (!s.d_in.p) continue;
        if (s.busy) {
            const bool newest = s.win_id + 1 == c->windows;
            if (newest && !c->finished_input && cudaEventQuery(s.ev_done) != cudaSuccess) continue;   // let it run
            MK_TRY(s2p_complete(c, cand[i]));
        }
        order[(*n)++] = cand[i];
    }
    if (*n == 2 && c->slot[order[0]].win_id > c->slot[order[1]].win_id) std::swap(order[0], order[1]);
    return MK_OK;
}

extern "C" int mk_s2p_pull(mk_ctx *x, char *pairs_out, size_t cap, size_t *n_out, char *sam_out, size_t cap2, size_t *n_out2) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    size_t a = drain(c->q_text, c->q_text_off, pairs_out, cap), b = drain(c->q_sam, c->q_sam_off, sam_out, cap2);
    int order[2], ns = 0;
    MK_TRY(s2p_ready_slots(c, order, &ns));
    bool text_blocked = !c->q_text.empty(), sam_blocked = !c->q_sam.empty();
    for (int i = 0; i < ns; ++i) {
        S2PSlot &s = c->slot[order[i]];
        if (pairs_out && !text_blocked && s.text_off < s.text_len) {
            size_t m = std::min(cap - a, s.text_len - s.text_off);
            if (m) { MK_CUDA(cudaMemcpyAsync(pairs_out + a, s.d_text.as<char>() + s.text_off, m, cudaMemcpyDeviceToHost, c->s_out)); a += m; s.text_off += m; }
        }
        if (s.text_off < s.text_len) text_blocked = true;            // keep window order
        if (sam_out && !sam_blocked && s.sam_off < s.sam_len) {
            size_t m = std::min(cap2 - b, s.sam_len - s.sam_off);
            if (m) { MK_CUDA(cudaMemcpyAsync(sam_out + b, s.d_sam.as<char>() + s.sam_off, m, cudaMemcpyDeviceToHost, c->s_out)); b += m; s.sam_off += m; }
        }
        if (s.sam_off < s.sam_len) sam_blocked = true;
    }
    MK_CUDA(cudaStreamSynchronize(c->s_out));
    if (n_out) *n_out = a;
    if (n_out2) *n_out2 = b;
    return MK_OK;
}

extern "C" int mk_s2p_pull_packed(mk_ctx *x, mk_pair *recs, size_t cap, size_t *n) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    size_t a = drain(c->q_pairs, c->q_pairs_off, recs, cap);
    int order[2], ns = 0;
    MK_TRY(s2p_ready_slots(c, order, &ns));
    bool blocked = !c->q_pairs.empty();
    for (int i = 0; i < ns && recs && !blocked; ++i) {
        S2PSlot &s = c->slot[order[i]];
        if (s.pairs_off < s.pairs_n) {
            size_t m = std::min(cap - a, s.pairs_n - s.pairs_off);
            if (m) { MK_CUDA(cudaMemcpyAsync(recs + a, s.d_pairs.as<mk_pair>() + s.pairs_off, m * sizeof(mk_pair), cudaMemcpyDeviceToHost, c->s_out)); a += m; s.pairs_off += m; }
        }
        if (s.pairs_off < s.pairs_n) blocked = true;
    }
    MK_CUDA(cudaStreamSynchronize(c->s_out));
    if (n) *n = a;
    return MK_OK;
}

static int s2p_fill_stats(S2PCtx *c, u64 group_base, u64 total_groups, mk_s2p_stats *out) {
    WinState st;
    MK_CUDA(cudaMemcpy(&st, c->d_state.p, sizeof st, cudaMemcpyDeviceToHost));
    MK_TRY(s2p_err_check(st.err));
    memset(out, 0, sizeof *out);
    out->lowMap = (u32)st.counters[ST_LOWMAP]; out->manyHits = (u32)st.counters[ST_MANYHITS]; out->unpaired = (u32)st.counters[ST_UNPAIRED];
    out->trans = (u32)st.counters[ST_TRANS]; out->cis10K = (u32)st.counters[ST_CIS10K]; out->cis1K = (u32)st.counters[ST_CIS1K];
    out->cis0 = (u32)st.counters[ST_CIS0];
    out->selfCircle_true = st.counters[ST_SELFCIRCLE]; out->cigar_errors = st.counters[ST_CIGARERR];
    out->groups = st.groups_done; out->lines = st.lines_done;
    out->pairs = st.counters[ST_TRANS] + st.counters[ST_CIS10K] + st.counters[ST_CIS1K] + st.counters[ST_CIS0];
    // only emulated thread 0's share of the self-circles reaches the reference's log (sam2pairs.cpp:202-210)
    const u32 T = (u32)c->cfg.emu_threads;
    const u64 P = total_groups;
    const u64 full = (P / S2P_BATCH) * S2P_BATCH;
    const u32 share_full = S2P_BATCH / (T - 1), share_last = (u32)(P % S2P_BATCH) / T;
    u64 n = c->sc_full_rule;
    for (u64 g0 : c->sc_tail) {
        u64 g = g0 + group_base;
        u32 r = (u32)(g % S2P_BATCH);
        if (g < full ? r < share_full : r < share_last) ++n;
    }
    out->selfCircle = (u32)n;
    return MK_OK;
}

extern "C" int mk_s2p_finish(mk_ctx *x, mk_s2p_stats *out) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (!out) { mk_set_error("mk_s2p_finish: null stats"); return MK_ERR_ARG; }
    if (!c->use_device_path) {
        if (!c->finished_input) MK_TRY(mk_s2p_push(x, nullptr, 0, 1));
        const int o0 = (int)(c->windows & 1);
        MK_TRY(s2p_complete(c, o0)); MK_TRY(s2p_complete(c, o0 ^ 1));
    }
    MK_CUDA(cudaStreamSynchronize(c->s_comp));
    WinState st;
    MK_CUDA(cudaMemcpy(&st, c->d_state.p, sizeof st, cudaMemcpyDeviceToHost));
    return s2p_fill_stats(c, 0, st.groups_done, out);
}

extern "C" int mk_s2p_finish_sharded(mk_ctx *x, uint64_t group_base, uint64_t total_groups, mk_s2p_stats *out) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (!out) { mk_set_error("mk_s2p_finish_sharded: null stats"); return MK_ERR_ARG; }
    if (!c->use_device_path) {
        if (!c->finished_input) MK_TRY(mk_s2p_push(x, nullptr, 0, 1));
        const int o0 = (int)(c->windows & 1);
        MK_TRY(s2p_complete(c, o0)); MK_TRY(s2p_complete(c, o0 ^ 1));
    }
    MK_CUDA(cudaStreamSynchronize(c->s_comp));
    if (!c->cfg.sharded && group_base != 0) { mk_set_error("mk_s2p_finish_sharded: create the context with cfg.sharded = 1"); return MK_ERR_STATE; }
    return s2p_fill_stats(c, group_base, total_groups, out);
}

// krmdup's log of the SAM-space duplicate removal (krmdup.cpp:383-389); valid after mk_s2p_finish
extern "C" int mk_s2p_rmdup_stats(mk_ctx *x, mk_dedup_stats *out) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (!out) { mk_set_error("mk_s2p_rmdup_stats: null stats"); return MK_ERR_ARG; }
    if (!c->cfg.rmdup) { mk_set_error("mk_s2p_rmdup_stats: context created without cfg.rmdup"); return MK_ERR_STATE; }
    MK_CUDA(cudaStreamSynchronize(c->s_comp));
    if (c->rk != RKP_OFF) {                          // this rank's share: its read pairs and discards, the keys it owns
        unsigned long long h[RK_N];
        MK_CUDA(cudaDeviceSynchronize());
        MK_CUDA(cudaMemcpy(h, c->d_rkcnt.p, sizeof h, cudaMemcpyDeviceToHost));
        out->uniq = (u32)h[RK_UNIQ]; out->dup = (u32)h[RK_DUP]; out->discard = (u32)c->rk_disc; out->pairs = c->rk_keys + c->rk_disc;
        return MK_OK;
    }
    WinState st;
    MK_CUDA(cudaMemcpy(&st, c->d_state.p, sizeof st, cudaMemcpyDeviceToHost));
    out->uniq = (u32)st.rm_uniq; out->discard = (u32)st.rm_discard; out->dup = (u32)(st.rm_total - st.rm_uniq - st.rm_discard);
    out->pairs = st.rm_total;
    return MK_OK;
}

// a stream that starts over, with the chromosome table learnt so far
static int s2p_state_clear(S2PCtx *c) {
    MK_CUDA(cudaDeviceSynchronize());
    WinState st;
    MK_CUDA(cudaMemcpy(&st, c->d_state.p, sizeof st, cudaMemcpyDeviceToHost));
    u32 n_chrom = st.n_chrom;
    memset(&st, 0, sizeof st); st.n_chrom = n_chrom; st.rm_allones[0] = st.rm_allones[1] = ~0ull;
    MK_CUDA(cudaMemcpy(c->d_state.p, &st, sizeof st, cudaMemcpyHostToDevice));
    return MK_OK;
}

// Forget the stream (counters, carried group, pending output) but keep every allocation and the chromosome table:
// the context can then process another input from the start.
extern "C" int mk_s2p_reset(mk_ctx *x) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    MK_TRY(s2p_state_clear(c));
    for (int t = 0; t < 2; ++t) if (c->d_rmtab[t].p) MK_CUDA(cudaMemset(c->d_rmtab[t].p, 0xFF, c->rm_slots[t] * 16));
    if (c->d_rkcnt.p) MK_CUDA(cudaMemset(c->d_rkcnt.p, 0, c->d_rkcnt.n));
    c->rk = RKP_OFF; c->rk_lines = c->rk_keys = c->rk_disc = 0;
    for (auto &s : c->slot) { s.busy = false; s.free_pending = false; s.text_len = s.text_off = s.pairs_n = s.pairs_off = s.sam_len = s.sam_off = 0; }
    c->tail.clear(); c->windows = 0; c->prev_slot = -1; c->finished_input = false; c->use_device_path = false;
    c->q_text.clear(); c->q_sam.clear(); c->q_pairs.clear(); c->q_text_off = c->q_sam_off = c->q_pairs_off = 0;
    c->sc_full_rule = 0; c->sc_tail.clear(); c->sc_true = 0;
    return MK_OK;
}

extern "C" int mk_s2p_chrom_count(mk_ctx *x) {
    S2PCtx *c; if (s2p_check(x, &c) != MK_OK) return -1;
    WinState st;
    cudaStreamSynchronize(c->s_comp);
    if (cudaMemcpy(&st, c->d_state.p, sizeof st, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int)st.n_chrom;
}

extern "C" int mk_s2p_chrom_name(mk_ctx *x, int id, char *buf, size_t cap) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (id < 0 || (u32)id >= c->chr_cap || !buf || cap == 0) { mk_set_error("mk_s2p_chrom_name: bad argument"); return MK_ERR_ARG; }
    int slot = 0;
    MK_CUDA(cudaMemcpy(&slot, c->d_id2slot.as<int>() + id, 4, cudaMemcpyDeviceToHost));
    ChrSlot s;
    MK_CUDA(cudaMemcpy(&s, c->d_chr.as<ChrSlot>() + slot, sizeof s, cudaMemcpyDeviceToHost));
    size_t l = std::min<size_t>(s.len, cap - 1);
    memcpy(buf, s.name, l); buf[l] = 0;
    return MK_OK;
}

extern "C" uint64_t mk_launch_count(mk_ctx *x) {
    if (!x) return 0;
    if (x->kind == MK_CTX_S2P) return ((S2PCtx *)x)->launches;
    return x->launches_generic;
}

// ------------------------------------------------------------------------------------------------ device-resident run
// The windows of one device-resident call, enqueued ahead and topped up until the input is consumed (both passes of the
// multi-rank krmdup and mk_s2p_run_device)
static int s2p_device_loop(S2PCtx *c, S2PParams &p, size_t n, int is_last, cudaStream_t s, WinState &st) {
    WinState *dst = c->d_state.as<WinState>();
    k_set_stream<<<1, 1, 0, s>>>(dst, 0, n, is_last ? 1u : 0u);
    c->launches += 1;
    MK_TRY(upload_params(c, p, 2, s));
    // running output offsets restart at 0 for every call
    MK_CUDA(cudaMemsetAsync((char *)dst + offsetof(WinState, out_text), 0, 3 * sizeof(u64), s));
    // every window consumes at least W - (largest read group) bytes; enqueue an upper bound and top up if needed
    size_t done = 0;
    int guard = 0;
    while (true) {
        size_t remaining = n - done;
        size_t nwin = remaining / (c->W - c->W / 8) + 1;
        for (size_t w = 0; w < nwin; ++w) launch_window(c, p, s);
        MK_CUDA(cudaMemcpyAsync(&st, dst, sizeof st, cudaMemcpyDeviceToHost, s));
        MK_CUDA(cudaStreamSynchronize(s));
        if (c->timing) timing_collect(c);
        MK_TRY(s2p_err_check(st.err));
        if (st.sc_count) {
            std::vector<u64> l(st.sc_count);
            MK_CUDA(cudaMemcpy(l.data(), c->d_sclist.p, (size_t)st.sc_count * 8, cudaMemcpyDeviceToHost));
            sc_absorb(c, l.data(), st.sc_count, st.groups_done);
            MK_CUDA(cudaMemsetAsync((char *)dst + offsetof(WinState, sc_count), 0, 4, s));
        }
        if (st.cursor >= n) break;
        if (st.cursor == done && ++guard > 2) break;          // not last: the tail group stays unprocessed
        if (!is_last && st.we == n) break;
        done = st.cursor;
    }
    c->last_state = st;
    return MK_OK;
}

extern "C" int mk_s2p_run_device(mk_ctx *x, const char *d_sam, size_t n, int is_last, mk_s2p_dev_io *io, void *stream) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (!io) { mk_set_error("mk_s2p_run_device: null io"); return MK_ERR_ARG; }
    if (((uintptr_t)d_sam & 15) != 0) { mk_set_error("mk_s2p_run_device: d_sam must be 16-byte aligned"); return MK_ERR_ARG; }
    if (c->windows) { mk_set_error("mk_s2p_run_device on a context used with mk_s2p_push"); return MK_ERR_STATE; }
    if (c->rk != RKP_OFF && c->rk != RKP_SETTLED) { mk_set_error("mk_s2p_run_device: multi-rank krmdup pass 2 before mk_s2p_rmdup_receive"); return MK_ERR_STATE; }
    c->use_device_path = true;
    if (!c->d_sclist.p) { c->sc_cap_dev = 16u << 20; MK_TRY(c->d_sclist.alloc((size_t)c->sc_cap_dev * 8)); }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->s_comp;
    S2PParams p = make_params(c, d_sam, c->d_sclist.as<u64>(), c->sc_cap_dev, io->d_pairs_text, io->pairs_text_cap, io->d_pairs, io->pairs_cap, io->d_sam_text, io->sam_text_cap, c->W, 1, (u64 *)io->d_line_off, io->line_off_cap, io->line_off_base);
    const bool xch = c->xchg && p.xparts && p.out_pairs;
    if (xch) { MK_TRY(mk_xchg_begin(c->xchg)); c->x_ev_used = 0; }
    WinState st;
    MK_TRY(s2p_device_loop(c, p, n, is_last, s, st));
    io->pairs_text_len = st.out_text; io->n_pairs = st.out_pairs; io->sam_text_len = st.out_sam; io->consumed = st.cursor;
    if (xch) {                                              // every part is out: close the epoch on the side stream, and let `s` see it
        MK_TRY(mk_xchg_end_device(c->xchg, c->s_x));
        if (c->x_events.empty()) { cudaEvent_t e; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); c->x_events.push_back(e); }
        MK_CUDA(cudaEventRecord(c->x_events[0], c->s_x));
        MK_CUDA(cudaStreamWaitEvent(s, c->x_events[0], 0));
    }
    if (c->rk == RKP_SETTLED && is_last) {                  // pass 2 must have met every run head of pass 1, at the same lines
        unsigned long long h[RK_N];
        MK_CUDA(cudaMemcpy(h, c->d_rkcnt.p, sizeof h, cudaMemcpyDeviceToHost));
        if (st.lines_done < c->rk_lines || h[RK_FP1] != h[RK_FP2]) {
            mk_set_error("mk_s2p_run_device: pass 2 does not hold the %llu lines of pass 1 (the text differs)", (unsigned long long)c->rk_lines);
            return MK_ERR_INPUT;
        }
    }
    return MK_OK;
}

// ------------------------------------------------------------------------------------------------ multi-rank krmdup
extern "C" int mk_s2p_rmdup_keys_device(mk_ctx *x, const char *d_sam, size_t n, int is_last, size_t *consumed, void *stream) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (((uintptr_t)d_sam & 15) != 0) { mk_set_error("mk_s2p_rmdup_keys_device: d_sam must be 16-byte aligned"); return MK_ERR_ARG; }
    if (!c->cfg.rmdup) { mk_set_error("mk_s2p_rmdup_keys_device: context created without cfg.rmdup"); return MK_ERR_STATE; }
    if (c->windows || (c->rk == RKP_OFF && c->use_device_path)) { mk_set_error("mk_s2p_rmdup_keys_device on a context that has run: mk_s2p_reset first"); return MK_ERR_STATE; }
    if (c->rk != RKP_OFF && c->rk != RKP_PASS1) { mk_set_error("mk_s2p_rmdup_keys_device: pass 1 is over"); return MK_ERR_STATE; }
    if (c->rk == RKP_OFF) {
        c->rk_cap = c->cfg.rmdup_capacity ? c->cfg.rmdup_capacity : (u64)1 << 24;   // d_rmtab[0] holds 2 x that many records
        if (!c->d_rkcnt.p) MK_TRY(c->d_rkcnt.alloc(RK_N * sizeof(unsigned long long)));
        MK_CUDA(cudaMemset(c->d_rkcnt.p, 0, c->d_rkcnt.n));
        c->rk = RKP_PASS1;
    }
    c->use_device_path = true;
    if (!c->d_sclist.p) { c->sc_cap_dev = 16u << 20; MK_TRY(c->d_sclist.alloc((size_t)c->sc_cap_dev * 8)); }
    cudaStream_t s = stream ? (cudaStream_t)stream : c->s_comp;
    S2PParams p = make_params(c, d_sam, c->d_sclist.as<u64>(), c->sc_cap_dev, nullptr, 0, nullptr, 0, nullptr, 0, c->W, 1);
    WinState st;
    MK_TRY(s2p_device_loop(c, p, n, is_last, s, st));
    if (consumed) *consumed = st.cursor;
    unsigned long long h[RK_N];
    MK_CUDA(cudaMemcpy(h, c->d_rkcnt.p, sizeof h, cudaMemcpyDeviceToHost));
    if (h[RK_KEYS] + h[RK_DISC] > c->rk_cap) {
        mk_set_error("mk_s2p_rmdup_keys_device: more than cfg.rmdup_capacity = %llu read pairs in the shard", (unsigned long long)c->rk_cap);
        return MK_ERR_CAPACITY;
    }
    if (is_last) {                                           // pass 2 starts a new stream over the same lines
        c->rk_lines = st.lines_done; c->rk_keys = h[RK_KEYS]; c->rk_disc = h[RK_DISC];
        MK_TRY(s2p_state_clear(c));
        c->sc_full_rule = 0; c->sc_tail.clear(); c->sc_true = 0;
        c->rk = RKP_KEYED;
    }
    return MK_OK;
}

static int rk_step(mk_ctx *x, mk_xchg *xc, int want, const char *what, S2PCtx **out) {
    S2PCtx *c; MK_TRY(s2p_check(x, &c));
    if (!xc) { mk_set_error("%s: null exchange", what); return MK_ERR_ARG; }
    if (!c->cfg.rmdup) { mk_set_error("%s: context created without cfg.rmdup", what); return MK_ERR_STATE; }
    if (c->rk != want) {
        static const char *ph[] = {"before mk_s2p_rmdup_keys_device", "before the last pass-1 call", "before mk_s2p_rmdup_send",
                                   "before mk_s2p_rmdup_decide", "before mk_s2p_rmdup_receive", "after mk_s2p_rmdup_receive"};
        mk_set_error("%s called %s", what, ph[c->rk]);
        return MK_ERR_STATE;
    }
    *out = c;
    return MK_OK;
}

extern "C" int mk_s2p_rmdup_send(mk_ctx *x, mk_xchg *xc, void *stream) {
    S2PCtx *c; MK_TRY(rk_step(x, xc, RKP_KEYED, "mk_s2p_rmdup_send", &c));
    MK_TRY(xchg_scatter_records(xc, c->d_rmtab[0].p, c->rk_keys, nullptr, 1, (cudaStream_t)stream));
    c->rk = RKP_SENT;
    return MK_OK;
}

extern "C" int mk_s2p_rmdup_decide(mk_ctx *x, mk_xchg *xc, void *stream) {
    S2PCtx *c; MK_TRY(rk_step(x, xc, RKP_SENT, "mk_s2p_rmdup_decide", &c));
    cudaStream_t s = (cudaStream_t)stream;
    mk_pair *d_recv = nullptr; size_t n = 0;
    MK_TRY(mk_xchg_finish_device(xc, &d_recv, &n, s));                      // every rank's keys of this rank's share
    if (n >= ((size_t)1 << 30)) { mk_set_error("mk_s2p_rmdup_decide: %zu key records for one owner (at most 2^30 - 1)", n); return MK_ERR_CAPACITY; }
    if (c->d_rksort.n < n * 16) { MK_TRY(c->d_rksort.alloc(n * 16)); MK_TRY(c->d_rklose.alloc(n * 16)); }
    if (!c->rk_rws.plan.p || c->rk_rws.max_n < n) MK_TRY(c->rk_rws.alloc(n));
    // (tag, key, ord), LSD: ord's line and rank bytes, the key, the tag byte
    RadixSchedule sch; sch.n_pass = 15;
    for (int b = 0; b < 6; ++b) sch.byte_of[b] = 8 + b;
    for (int b = 0; b < 8; ++b) sch.byte_of[6 + b] = b;
    sch.byte_of[14] = 15;
    Rec16::Bufs b; b.k[0] = (uint4 *)d_recv; b.k[1] = c->d_rksort.as<uint4>(); b.v[0] = b.v[1] = nullptr;
    const int sms = mk_sm_count(c->cfg.device);
    MK_TRY(radix_sort<Rec16>(b, n, sch, c->rk_rws, 0, sms, s, &c->launches));
    unsigned long long *cnt = c->d_rkcnt.as<unsigned long long>();
    const int grid = (int)std::max<u64>(1, std::min<u64>((n + 255) / 256, (u64)sms * 8));
    k_rm_decide<<<grid, 256, 0, s>>>(b.k[0], b.k[1], &c->rk_rws.plan.as<RadixPlan>()->final_buf, n, c->d_rklose.as<uint4>(), cnt);
    c->launches += 1;
    MK_CUDA(cudaGetLastError());
    MK_TRY(mk_xchg_begin(xc));                                                // the losers go back to their ranks
    MK_TRY(xchg_scatter_records(xc, c->d_rklose.p, 0, cnt + RK_LOSE, 2, s));
    MK_TRY(mk_xchg_end_device(xc, s));
    c->rk = RKP_DECIDED;
    return MK_OK;
}

extern "C" int mk_s2p_rmdup_receive(mk_ctx *x, mk_xchg *xc, void *stream) {
    S2PCtx *c; MK_TRY(rk_step(x, xc, RKP_DECIDED, "mk_s2p_rmdup_receive", &c));
    cudaStream_t s = (cudaStream_t)stream;
    mk_pair *d_recv = nullptr; size_t n = 0;
    MK_TRY(mk_xchg_finish_device(xc, &d_recv, &n, s));                      // this rank's losers, from every owner
    int world = 1, rank = 0;
    xchg_world_rank(xc, &world, &rank);
    const size_t words = c->rk_lines / 32 + 1;
    if (c->d_rkdrop.n < words * 4) MK_TRY(c->d_rkdrop.alloc(words * 4));
    MK_CUDA(cudaMemsetAsync(c->d_rkdrop.p, 0, words * 4, s));
    unsigned long long *cnt = c->d_rkcnt.as<unsigned long long>();
    const int sms = mk_sm_count(c->cfg.device);
    auto grid = [&](u64 m) { return (int)std::max<u64>(1, std::min<u64>((m + 255) / 256, (u64)sms * 8)); };
    k_rm_settle<<<grid(c->rk_disc), 256, 0, s>>>(c->d_rmtab[0].as<uint4>() + (c->rk_cap - c->rk_disc), c->rk_disc, (u32)rank, 0, c->rk_lines, c->d_rkdrop.as<u32>(), cnt);
    k_rm_settle<<<grid(n), 256, 0, s>>>((const uint4 *)d_recv, n, (u32)rank, 1, c->rk_lines, c->d_rkdrop.as<u32>(), cnt);
    c->launches += 2;
    unsigned long long bad = 0;
    MK_CUDA(cudaMemcpyAsync(&bad, cnt + RK_BAD, 8, cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    if (bad) { mk_set_error("mk_s2p_rmdup_receive: %llu returned records name another rank or a line past pass 1", bad); return MK_ERR_STATE; }
    c->rk = RKP_SETTLED;
    return MK_OK;
}
