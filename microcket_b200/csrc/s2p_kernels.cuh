// s2p_kernels.cuh — sm_100a kernels of the sam2pairs path.
//
// One *window* of SAM text (<= 2040 MiB, device resident) goes through
//   k_win_begin    set up the window from the device-side cursor, clear the per-tile sums
//   k_scan_chunks  K1: byte-parallel newline index, one warp per 16 KiB chunk, no inter-CTA dependency   (replaces getline, pairutil.h:152)
//   k_chunk_prefix / k_chunk_compact   the chunks' newline lists -> the dense nl_pos[] (k_scan_lines: look-back fallback for windows
//                  with more than 512 newlines in a chunk; also the FASTQ path's scan)
//   k_parse        K2: one thread per line: first six fields, filter, CIGAR walk         (pairutil.h:63-126,155-161; unc2pairs.h:34-36)
//   k_rm_insert    (cfg.rmdup only) krmdup's duplicate removal taken on the SAM: duplicate read pairs lose LM_KEEP    (src/preprocess/krmdup.cpp:103-212)
//                  over several ranks (mk_s2p_rmdup_*): k_rm_keys in pass 1, k_rm_decide / k_rm_settle between the passes,
//                  k_rm_apply in its place in pass 2
//   k_group        K3: group heads among kept records + per-group resolution             (pairutil.h:163-173; flash2pairs.h; unc2pairs.h)
//   k_emit_prefix / k_emit   K4: prefixes of the per-tile output sizes, .pairs text + packed records + line offsets   (unc2pairs.h:310-348)
//   k_copy_sam     K5: SAM passthrough of the kept lines of emitted groups               (unc2pairs.h:351-356)
//   k_win_end      advance the cursor to the window's last (unprocessed) read group
// All window geometry lives in device memory (WinState), so consecutive windows are
// enqueued back to back without a host round trip.
#pragma once
#include <type_traits>
#include "mk_common.cuh"

#define S2P_TILE_BYTES 32768
#define S2P_SCAN_THREADS 256
#define S2P_NAME_MAX 42

enum { ST_NONE = 0, ST_LOWMAP, ST_MANYHITS, ST_UNPAIRED, ST_SELFCIRCLE, ST_TRANS, ST_CIS10K, ST_CIS1K, ST_CIS0, ST_CIGARERR, ST_NCOUNTER };

// line meta bits
#define LM_KEEP 1u
#define LM_EQ 2u
#define LM_HEAD 4u
#define LM_PROC 8u
#define LM_EMIT 16u

struct __align__(16) LineRec {       // 48 B, written by K2 for kept lines
    u32 pos, right0, left1, right1;
    u32 leftClip, rightClip, mappable, line_len;
    u16 flag, qname_len, chr_slot; u8 segCnt /* 0 = cigar error, 3 = more than 2 */, pad0;
    u32 qname_off;                   // offset of the QNAME's first byte from the line start
    u32 pad1;
};

struct __align__(16) GroupRes {      // 32 B, written by K3 for group heads
    u32 posA, posB;
    u16 chrA, chrB;                  // chromosome ids
    u8 status, strands; u16 rid_len;   // length of the read id (QNAME of the group's last kept record)
    u32 rid_off, last_line, text_len, sam_len;   // rid_off: offset of that QNAME from the window start
};

struct __align__(64) ChrSlot {       // open-addressing table keyed by a 64-bit hash of the name
    unsigned long long key;          // 0 = empty
    unsigned long long name8;        // first 8 bytes of the name, zero padded (fast exact check for short names)
    int id;                          // -1 until published
    u16 len; char name[S2P_NAME_MAX];
};

struct WinState {
    // stream / buffer geometry
    u64 cursor, total;               // next window start; bytes available
    u64 ws, we;                      // this window
    u32 n_lines, carry_line, first_tile, is_last;
    u32 err, scan_ovf;               // scan_ovf: a 16 KiB chunk held more newlines than its slot list (the look-back scan redoes the window)
    // per-window emit totals
    u32 w_groups, w_emit, w_text, w_sam;
    // running output offsets (device-resident multi-window runs)
    u64 out_text, out_pairs, out_sam;
    // stream totals
    u64 groups_done, lines_done;
    unsigned long long counters[ST_NCOUNTER];
    u32 sc_count, n_chrom;
    u32 tickets[4];                  // dynamic tile tickets of look-back kernels, reset per window
    // SAM-space krmdup (cfg.rmdup): QNAME runs counted so far end before this global line index; log counters; first
    // occurrence (global line index) of the all-ones key, which is the tables' empty marker
    u64 rm_counted;
    unsigned long long rm_total, rm_uniq, rm_discard, rm_allones[2];
};

#define S2P_ERR_LINES 1u
#define S2P_ERR_TEXT 2u
#define S2P_ERR_PAIRS 4u
#define S2P_ERR_SAM 8u
#define S2P_ERR_SCLIST 16u
#define S2P_ERR_NOPROGRESS 32u
#define S2P_ERR_CHRTABLE 64u
#define S2P_ERR_RMTABLE 128u

struct S2PParams {
    const char *buf;          // SAM text base (16-byte aligned)
    WinState *st;
    u32 *nl_pos;              // newline offsets relative to ws
    u32 *ck_list, *ck_cnt, *ck_pre, *ck_bsum;   // chunked scan: per-chunk newline lists (SC_CAP slots each), counts, in-block exclusive prefixes, block sums
    u32 n_chunks_cap;
    u8 *lmeta;
    LineRec *rec;
    GroupRes *res;
    u32 *sam_dst;
    u64 *desc_scan;
    uint4 *seg_tot; u32 n_seg_cap;              // per EMIT_SEG tiles: (groups, emitted, text bytes, passthrough bytes), also summed by K3
    uint4 *tile_tot, *tile_pre; u32 n_sub_cap;  // per EMIT_TILE lines: (groups | emitted << 16, text bytes, passthrough bytes) summed by K3; exclusive prefixes (groups, emitted, text, passthrough)
    ChrSlot *chr; u32 chr_mask; int *id_to_slot; u32 chr_cap;
    u64 *sc_list; u32 sc_cap;
    char *out_text; u64 out_text_cap;
    mk_pair *out_pairs; u64 out_pairs_cap;
    u64 *out_line_off; u64 out_line_off_cap, line_off_base;   // optional: offset (in out_text) of every emitted pair's line, plus the end of the last one
    char *out_sam; u64 out_sam_cap;
    u64 window_bytes; u32 cap_lines;
    int mode, min_mapq, write_sam, emit_text, emit_packed; float ratio; u16 lane;
    int running_offsets;      // 1: append at st->out_* (device-resident runs); 0: every window writes at 0
    // SAM-space krmdup: key tables ({key, first global line index} per slot; [1] = the T bucket's lower-case identity space),
    // per-line key / status of the window's QNAME runs
    int rm_on, rm_hskip1, rm_klen1, rm_hskip2, rm_klen2;
    unsigned long long *rm_tab[2]; u64 rm_mask[2];
    u32 *rm_info;   // rm_info: K2's (flag | SEQ offset << 16) per line
    // multi-rank krmdup (mk_s2p_rmdup_*): pass 1 writes {key, ord} records from the front of rk_rec and discarded run heads
    // from its back; pass 2 reads the settled drop bits of the first rk_lines lines.  rk_cnt: RK_* counters
    uint4 *rk_rec; u64 rk_cap;
    const u32 *rk_drop; u64 rk_lines;
    unsigned long long *rk_cnt;
    unsigned long long *xparts;   // optional: per launched window (end, count) of its packed pairs, for the overlapped multi-GPU scatter
    const S2PParams *self;    // device copy of this struct: what out-of-line callees are handed, so that the kernels' parameter block is never copied to local memory
};

// ------------------------------------------------------------------------------------------------ begin / end
static __global__ void k_win_begin(S2PParams p, u32 n_desc) {
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.n_sub_cap) p.tile_tot[i] = make_uint4(0, 0, 0, 0);
    if (i < p.n_seg_cap) p.seg_tot[i] = make_uint4(0, 0, 0, 0);
    if (i < n_desc) p.desc_scan[i] = 0;                        // look-back descriptors of the fallback scan
    if (i == 0) {
        WinState *s = p.st;
        s->ws = s->cursor;
        u64 we = s->cursor + p.window_bytes;
        s->we = we < s->total ? we : s->total;
        s->n_lines = 0; s->carry_line = 0xFFFFFFFFu; s->scan_ovf = 0;
        s->first_tile = (u32)(s->ws / S2P_TILE_BYTES);
        s->w_groups = s->w_emit = s->w_text = s->w_sam = 0;
        s->tickets[0] = s->tickets[1] = s->tickets[2] = s->tickets[3] = 0;
        if (!p.running_offsets) { s->out_text = s->out_pairs = s->out_sam = 0; s->sc_count = 0; }
    }
}

static __global__ void k_win_end(S2PParams p, u32 xslot) {
    WinState *s = p.st;
    u64 ws = s->ws, we = s->we;
    u32 n = s->n_lines;
    u64 next;
    const bool carried = s->carry_line != 0xFFFFFFFFu;
    const bool final_win = (we == s->total) && s->is_last;
    u32 cut = carried ? s->carry_line : n;                    // first line that is not consumed (no kept record: every complete line is)
    if (p.rm_on && !final_win && n) {
        // SAM-space krmdup works on whole QNAME runs (dropped lines included): the next window starts at a run's first line,
        // and the window's last run (possibly cut by the window end) is always seen again
        if (!carried) cut = n - 1;
        while (cut > 0 && (p.lmeta[cut] & LM_EQ)) --cut;
        u32 hl = n - 1;
        while (hl > 0 && (p.lmeta[hl] & LM_EQ)) --hl;
        s->rm_counted = s->lines_done + hl;
    } else if (p.rm_on) s->rm_counted = s->lines_done + n;
    if (carried || cut != n) s->carry_line = cut;
    next = ws + (cut ? (u64)p.nl_pos[cut - 1] + 1 : 0);
    if (final_win) next = s->total;                        // the stream's last group is never processed (pairutil.h:176)
    else if (next == ws && we > ws && we - ws >= p.window_bytes) s->err |= S2P_ERR_NOPROGRESS;  // one group (or line) fills the window
    s->cursor = next;
    s->lines_done += final_win ? n : cut;
    s->groups_done += s->w_groups;
    s->out_text += s->w_text; s->out_pairs += s->w_emit; s->out_sam += s->w_sam;
    if (p.out_line_off && s->out_pairs < p.out_line_off_cap) p.out_line_off[s->out_pairs] = p.line_off_base + s->out_text;   // end of the last line so far
    if (p.xparts) { p.xparts[2 * xslot] = s->out_pairs; p.xparts[2 * xslot + 1] = s->w_emit; }
}

// ------------------------------------------------------------------------------------------------ K1: newline index
// Tile = 32 KiB at absolute 32 KiB boundaries of the buffer.  Loads are coalesced 128-bit streaming
// loads; the 16 newline flags of every 16-byte word go through shared memory so that each thread then
// owns 128 CONTIGUOUS bytes (8 words), which makes ranks a single block scan.
// Shared by the SAM and FASTQ paths: positions (relative to ws) of every '\n' in [ws, we).
//
// Per 16-byte word the four SWAR results are merged WITHOUT gathering: bit (8*j + k) of the word's flag mask is set
// iff byte j of 32-bit lane k is '\n' (3 ALU ops per lane + 6 to merge).  The permuted order only matters for the rare
// word that holds two newlines.  Shared-memory buffers are double-buffered so a tile costs three barriers, and the
// next tile's loads are issued before the current tile's scan so HBM stays busy across the barriers.
__device__ __forceinline__ u32 nl_y(u32 x) {
    u32 t = ((x ^ 0x0A0A0A0Au) & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(t | x) & 0x80808080u;
}
__device__ __forceinline__ u32 nl_flags16(const uint4 &w) { return (nl_y(w.x) >> 7) | (nl_y(w.y) >> 6) | (nl_y(w.z) >> 5) | (nl_y(w.w) >> 4); }
__device__ __forceinline__ u32 perm_bit_of_byte(u32 q) { return 8u * (q & 3u) + (q >> 2); }       // byte q (0..15) -> bit
__device__ __forceinline__ u32 byte_of_perm_bit(u32 b) { return ((b & 7u) << 2) | (b >> 3); }     // bit -> byte

// Tiles go round-robin over a fully resident grid (tile = first + blockIdx + k * gridDim); a tile is S2P_NT sub-tiles of
// 32 KiB = 128 KiB, so the grid-wide dependency of the look-back (every wave waits for its slowest CTA) and the three
// block barriers are paid once per 128 KiB, and the sub-tiles' loads are software-pipelined so HBM stays busy.
// (Measured on B200: 32 KiB tiles 2.0 TB/s; atomic tickets and a wave-parallel prefix were both slower.)
template <int S2P_NT>
__device__ __forceinline__ void scan_lines_body(const char *buf, const u64 ws, const u64 we,
                                                u32 *nl_pos, const u32 cap_lines, u64 *desc, u32 *n_lines_out, u32 *err_out, u32 err_bit) {
    extern __shared__ __align__(16) u32 s_z_dyn[];                     // S2P_NT * 2048 words (dynamic: 64 KiB for NT = 8)
    u32 (*s_z)[S2P_TILE_BYTES / 16] = (u32 (*)[S2P_TILE_BYTES / 16])s_z_dyn;
    __shared__ u32 s_wtot[2][S2P_NT][S2P_SCAN_THREADS / 32];
    __shared__ u32 s_base[2];
    constexpr u64 S2P_SUPER = (u64)S2P_NT * S2P_TILE_BYTES;
    if (we <= ws) return;
    const int first_tile = (int)(ws / S2P_SUPER), last_tile = (int)((we - 1) / S2P_SUPER);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    u64 *dsc = desc - first_tile;
    uint4 w[8];
    auto load_sub = [&](u64 sbase) {                                   // one 32 KiB sub-tile into registers
        const uint4 *src = (const uint4 *)(buf + sbase);
        const bool interior = sbase >= ws && sbase + S2P_TILE_BYTES <= we;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (interior) w[j] = ld_stream_v4(src + j * S2P_SCAN_THREADS + tid);
            else {
                const u64 off = sbase + ((u64)(j * S2P_SCAN_THREADS + tid) << 4);
                w[j] = (off < we && off + 16 > ws) ? ld_stream_v4(src + j * S2P_SCAN_THREADS + tid) : make_uint4(0, 0, 0, 0);
            }
        }
    };
    int tile = first_tile + (int)blockIdx.x;
    if (tile <= last_tile) load_sub((u64)tile * S2P_SUPER);
    for (int pb = 0; tile <= last_tile; tile += gridDim.x, pb ^= 1) {
        const u64 tbase = (u64)tile * S2P_SUPER;
#pragma unroll 1
        for (int k = 0; k < S2P_NT; ++k) {                              // rolled: the kernel must fit the instruction cache
            const u64 sbase = tbase + (u64)k * S2P_TILE_BYTES;
            const bool interior = sbase >= ws && sbase + S2P_TILE_BYTES <= we;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u32 z = nl_flags16(w[j]);
                if (!interior && z) {                                 // window edges: drop flags of bytes outside [ws, we)
                    const u64 off = sbase + ((u64)(j * S2P_SCAN_THREADS + tid) << 4);
                    u32 keep = 0;
#pragma unroll 1
                    for (u32 q = 0; q < 16; ++q) if (off + q >= ws && off + q < we) keep |= 1u << perm_bit_of_byte(q);
                    z &= keep;
                }
                s_z[k][j * S2P_SCAN_THREADS + tid] = z;
            }
            // next sub-tile (of this tile, or the first one of this CTA's next tile) while the flags are being used
            if (k + 1 < S2P_NT) load_sub(sbase + S2P_TILE_BYTES);
            else if (tile + (int)gridDim.x <= last_tile) load_sub((u64)(tile + gridDim.x) * S2P_SUPER);
        }
        __syncthreads();
        u32 cnt[S2P_NT], inc[S2P_NT];
#pragma unroll
        for (int k = 0; k < S2P_NT; ++k) {
            const uint4 za = ((const uint4 *)s_z[k])[2 * tid], zb = ((const uint4 *)s_z[k])[2 * tid + 1];   // bytes [tid*128, +128) of sub-tile k
            cnt[k] = __popc(za.x) + __popc(za.y) + __popc(za.z) + __popc(za.w) + __popc(zb.x) + __popc(zb.y) + __popc(zb.z) + __popc(zb.w);
            inc[k] = warp_incl_scan(cnt[k], lane);
            if (lane == 31) s_wtot[pb][k][wid] = inc[k];
        }
        __syncthreads();
        u32 pre[S2P_NT], total = 0;                                     // exclusive prefix of this thread's block in sub-tile k, inside the tile
#pragma unroll
        for (int k = 0; k < S2P_NT; ++k) {
            u32 before = 0, sub = 0;
#pragma unroll
            for (int q = 0; q < S2P_SCAN_THREADS / 32; ++q) { const u32 v = s_wtot[pb][k][q]; sub += v; if (q < wid) before += v; }
            pre[k] = total + before + inc[k] - cnt[k];
            total += sub;
        }
        if (wid == 0) {
            const u64 b = lookback_exclusive(dsc, tile, first_tile, total, lane);
            if (lane == 0) {
                s_base[pb] = (u32)b;
                if (tile == last_tile) {
                    u64 nl = b + total;
                    if (nl > cap_lines) { atomicOr(err_out, err_bit); nl = cap_lines; }
                    *n_lines_out = (u32)nl;
                }
            }
        }
        __syncthreads();
        const u32 base = s_base[pb];
#pragma unroll
        for (int k = 0; k < S2P_NT; ++k) {                              // (cnt / pre are registers: static indices)
            if (!cnt[k]) continue;
            u32 idx = base + pre[k];
            const u32 rel = (u32)(tbase + (u64)k * S2P_TILE_BYTES + (u64)tid * 128 - ws);   // may wrap for bytes before ws: those have no flags
#pragma unroll 1
            for (int i = 0; i < 8; ++i) {
                u32 z = s_z[k][8 * tid + i];
                if (!z) continue;
                if (z & (z - 1)) {                                    // several newlines in one 16-byte word: restore byte order
#pragma unroll 1
                    u32 m = 0;
                    while (z) { const u32 b = __ffs(z) - 1; z &= z - 1; m |= 1u << byte_of_perm_bit(b); }
                    while (m) { const u32 q = __ffs(m) - 1; m &= m - 1; if (idx < cap_lines) nl_pos[idx] = rel + i * 16 + q; ++idx; }
                } else {
                    if (idx < cap_lines) nl_pos[idx] = rel + i * 16 + byte_of_perm_bit(__ffs(z) - 1);
                    ++idx;
                }
            }
        }
        __syncthreads();                                               // s_z is rewritten by the next tile
    }
}

template <int NT, int MINB = 3>
static __global__ void __launch_bounds__(S2P_SCAN_THREADS, MINB) k_scan_lines(S2PParams p, int only_if_ovf) {
    WinState *st = p.st;
    if (only_if_ovf && !st->scan_ovf) return;          // fallback of the chunked scan: runs only for windows with very short lines
    scan_lines_body<NT>(p.buf, st->ws, st->we, p.nl_pos, p.cap_lines, p.desc_scan, &st->n_lines, &st->err, S2P_ERR_LINES);
}

// ------------------------------------------------------------------------------------------------ K1 (default): chunked newline index
// No inter-CTA dependency and no barrier: every WARP owns one 16 KiB chunk (absolute 16 KiB boundaries of the buffer), streams it
// with coalesced 128-bit loads (lane l reads word 32 * it + l), and appends the positions of its newlines, in byte order, to the
// chunk's own slot list; ranks inside the warp come from one ballot.  k_chunk_prefix then turns the 64 Ki chunk counts of a window
// into exclusive prefixes (one CTA) and k_chunk_compact copies the lists to the dense nl_pos[] the other kernels index.  The
// look-back scan above was held at ~0.5 of the HBM peak by its grid-wide dependency (every wave waits for its slowest CTA) and by
// 73 instructions per 16-byte word; this one needs ~40.  A chunk with more than SC_CAP newlines (average line < 32 B) raises
// scan_ovf and the look-back kernel redoes that window, so any input is still handled.
#define SC_CHUNK 16384u
#define SC_CAP 512u
#define SC_UNROLL 8
#define SC_WARPS 8

__device__ __forceinline__ u32 nl_raw(u32 x) {          // bit 7 of byte k set iff that byte is '\n'; other bits are garbage (mask with 0x80808080)
    const u32 t = x ^ 0x0A0A0A0Au;
    return (t - 0x01010101u) & ~t & ~(t << 7);            // borrow false positives (a 0x0B right above a newline) have bit 0 set
}

static __global__ void __launch_bounds__(SC_WARPS * 32, 4) k_scan_chunks(S2PParams p) {
    const WinState *st = p.st;
    const u64 ws = st->ws, we = st->we;
    if (we <= ws) return;
    const u32 lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    const u64 first_chunk = ws / SC_CHUNK, last_chunk = (we - 1) / SC_CHUNK;
    const u64 lc = (u64)blockIdx.x * SC_WARPS + wid;               // chunk index inside the window
    const u64 chunk = first_chunk + lc;
    if (chunk > last_chunk || lc >= p.n_chunks_cap) return;
    const u64 cbase = chunk * SC_CHUNK;
    const bool edge = cbase < ws || cbase + SC_CHUNK > we;
    const uint4 *src = (const uint4 *)(p.buf + cbase) + lane;
    u32 *list = p.ck_list + lc * SC_CAP;
    const u32 rel0 = (u32)(cbase - ws) + lane * 16u;                 // wraps for bytes before ws: those are filtered below
    const u32 lt = (1u << lane) - 1u;
    u32 n = 0;
#pragma unroll 1
    for (u32 it = 0; it < SC_CHUNK / 512u; it += SC_UNROLL) {
        uint4 w[SC_UNROLL];
        if (!edge) {
#pragma unroll
            for (int u = 0; u < SC_UNROLL; ++u) w[u] = ld_stream_v4(src + (it + u) * 32u);
        } else {
#pragma unroll
            for (int u = 0; u < SC_UNROLL; ++u) {
                const u64 off = cbase + (u64)((it + u) * 32u + lane) * 16u;
                w[u] = (off < we && off + 16 > ws) ? ld_stream_v4(src + (it + u) * 32u) : make_uint4(0, 0, 0, 0);
            }
        }
#pragma unroll
        for (int u = 0; u < SC_UNROLL; ++u) {
            const u32 e0 = nl_raw(w[u].x), e1 = nl_raw(w[u].y), e2 = nl_raw(w[u].z), e3 = nl_raw(w[u].w);
            // bit (8 * j + k) <- byte j of 32-bit lane k (the permuted order of nl_flags16); built on every row so that a row
            // with newlines costs one more ballot, two popcounts and the store
            u32 z = ((e0 >> 7) & 0x01010101u) | ((e1 >> 6) & 0x02020202u) | ((e2 >> 5) & 0x04040404u) | ((e3 >> 4) & 0x08080808u);
            if (edge && z) {
                const u64 off = cbase + (u64)((it + u) * 32u + lane) * 16u;
                u32 keep = 0;
#pragma unroll 1
                for (u32 q = 0; q < 16; ++q) if (off + q >= ws && off + q < we) keep |= 1u << perm_bit_of_byte(q);
                z &= keep;
            }
            const u32 bal = __ballot_sync(0xFFFFFFFFu, z != 0);
            if (bal == 0) continue;                                  // warp-uniform
            const u32 multi = __ballot_sync(0xFFFFFFFFu, (z & (z - 1u)) != 0);
            const u32 rel = rel0 + (it + u) * 512u;
            if (multi == 0) {                                        // at most one newline per 16-byte word: ranks from the ballot
                if (z) {
                    const u32 idx = n + __popc(bal & lt);
                    if (idx < SC_CAP) list[idx] = rel + byte_of_perm_bit(__ffs(z) - 1);
                }
                n += __popc(bal);
                continue;
            }
            const u32 c = __popc(z);
            const u32 inc = warp_incl_scan(c, (int)lane);
            const u32 tot = __shfl_sync(0xFFFFFFFFu, inc, 31);
            if (c) {                                                 // restore byte order inside the word
                u32 m = 0, idx = n + inc - c;
#pragma unroll 1
                while (z) { const u32 b = __ffs(z) - 1; z &= z - 1; m |= 1u << byte_of_perm_bit(b); }
#pragma unroll 1
                while (m) { const u32 q = __ffs(m) - 1; m &= m - 1; if (idx < SC_CAP) list[idx] = rel + q; ++idx; }
            }
            n += tot;
        }
    }
    if (lane == 0) p.ck_cnt[lc] = n;
}

// Chunk counts -> positions in nl_pos[], in two small kernels without a serial pass:
//   k_chunk_prefix  one CTA per 1024 chunks: exclusive prefix inside the block (one uint4 of counts per thread) + the block's sum
//   k_chunk_compact one warp per chunk: base = sum of the earlier blocks' sums (<= 128, one REDUX) + the in-block prefix;
//                   copies the chunk's slot list into the dense nl_pos[]; the last chunk's warp publishes n_lines
#define SC_PFX_BLOCK 1024u                                              // chunks per k_chunk_prefix CTA
static __global__ void __launch_bounds__(256) k_chunk_prefix(S2PParams p) {
    __shared__ u32 s_w[8];
    WinState *st = p.st;
    const u64 ws = st->ws, we = st->we;
    if (we <= ws) return;
    const u64 nc64 = (we - 1) / SC_CHUNK - ws / SC_CHUNK + 1;
    const u32 nc = (u32)(nc64 < p.n_chunks_cap ? nc64 : p.n_chunks_cap);
    const u32 tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    const u32 i = blockIdx.x * (SC_PFX_BLOCK / 4) + tid;             // uint4 index
    if (blockIdx.x * SC_PFX_BLOCK >= nc) return;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (4u * i < nc) {
        v = ((const uint4 *)p.ck_cnt)[i];
        if (4u * i + 3u >= nc) { if (4u * i + 1u >= nc) v.y = 0; if (4u * i + 2u >= nc) v.z = 0; v.w = 0; }   // stale counts past the window
    }
    if ((v.x > SC_CAP) | (v.y > SC_CAP) | (v.z > SC_CAP) | (v.w > SC_CAP) | (nc64 > p.n_chunks_cap)) st->scan_ovf = 1u;
    const u32 sum = v.x + v.y + v.z + v.w;
    const u32 inc = warp_incl_scan(sum, (int)lane);
    if (lane == 31) s_w[wid] = inc;
    __syncthreads();
    u32 before = 0, total = 0;
#pragma unroll
    for (u32 q = 0; q < 8; ++q) { const u32 x = s_w[q]; total += x; if (q < wid) before += x; }
    uint4 o; o.x = before + inc - sum; o.y = o.x + v.x; o.z = o.y + v.y; o.w = o.z + v.z;
    if (4u * i < nc) ((uint4 *)p.ck_pre)[i] = o;
    if (tid == 0) p.ck_bsum[blockIdx.x] = total;
}

static __global__ void __launch_bounds__(256) k_chunk_compact(S2PParams p) {
    WinState *st = p.st;
    const u64 lc = (u64)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (lc >= p.n_chunks_cap) return;
    const u32 lane = threadIdx.x & 31u;
    const u32 *list = p.ck_list + lc * SC_CAP;
    // every load is issued before the first use: one memory round trip for chunks of up to 64 lines
    const u32 ovf = st->scan_ovf;
    const u64 ws = st->ws, we = st->we;
    const u32 cnt = p.ck_cnt[lc], pre = p.ck_pre[lc];
    const u32 blk = (u32)(lc / SC_PFX_BLOCK);
    u32 bs = 0;
#pragma unroll
    for (u32 q = 0; q < 5; ++q) { const u32 b = lane + 32u * q; const u32 x = p.ck_bsum[b]; if (b < blk) bs += x; }   // ck_bsum has 160 slots
    const u32 a = list[lane], b2 = list[lane + 32];                    // in bounds (SC_CAP >= 64); stale past cnt
    if (ovf || we <= ws) return;
    const u64 nc = (we - 1) / SC_CHUNK - ws / SC_CHUNK + 1;
    if (lc >= nc) return;
    const u32 base = __reduce_add_sync(0xFFFFFFFFu, bs) + pre;
    if (lc == nc - 1 && lane == 0) {
        u32 nl = base + cnt;
        if (nl > p.cap_lines) { atomicOr(&st->err, S2P_ERR_LINES); nl = p.cap_lines; }
        st->n_lines = nl;
    }
    if (lane < cnt && base + lane < p.cap_lines) p.nl_pos[base + lane] = a;
    if (lane + 32 < cnt && base + lane + 32 < p.cap_lines) p.nl_pos[base + lane + 32] = b2;
    for (u32 i = lane + 64; i < cnt; i += 32) if (base + i < p.cap_lines) p.nl_pos[base + i] = list[i];
}

// ------------------------------------------------------------------------------------------------ chromosome table
__device__ __forceinline__ u64 hash_step(u64 h, int c) { return (h ^ (u64)c) * 0x100000001B3ull; }

// Returns the slot of the name; inserts it when unseen (lock-free; ids are published by the inserter).
static __device__ __noinline__ int chr_lookup_insert_slow(const S2PParams &p, u64 h, u64 name8, const char *buf, u64 name_off, u32 len) {
    if (h == 0) h = 0x9E3779B97F4A7C15ull;
    const u32 l = len < S2P_NAME_MAX ? len : S2P_NAME_MAX;
    u32 s = (u32)(h ^ (h >> 29)) & p.chr_mask;
    for (u32 probe = 0; probe <= p.chr_mask; ++probe, s = (s + 1) & p.chr_mask) {
        ChrSlot *sl = &p.chr[s];
        unsigned long long k = *(volatile unsigned long long *)&sl->key;
        if (k == 0) {
            unsigned long long old = atomicCAS(&sl->key, 0ull, (unsigned long long)h);
            if (old == 0) {
                sl->len = (u16)l; sl->name8 = name8;
                for (u32 i = 0; i < l; ++i) sl->name[i] = buf[name_off + i];
                int id = (int)atomicAdd(&p.st->n_chrom, 1u);
                if ((u32)id < p.chr_cap) p.id_to_slot[id] = (int)s; else atomicOr(&p.st->err, S2P_ERR_CHRTABLE);
                __threadfence();
                *(volatile int *)&sl->id = id;
                return (int)s;
            }
            k = old;
        }
        if (k == h) {
            int id = *(volatile int *)&sl->id;
            if (id < 0) return (int)s;                       // being inserted by a concurrent thread: identity by hash
            __threadfence();
            bool same = sl->len == l && sl->name8 == name8;
            if (same && l > 8) for (u32 i = 8; same && i < l; ++i) same = sl->name[i] == buf[name_off + i];
            if (same) return (int)s;
        }
    }
    atomicOr(&p.st->err, S2P_ERR_CHRTABLE);
    return 0;
}

// Hot path: the name is already in the table (published by an earlier launch or earlier in this one) and is short.
// Plain cached loads are enough here: a stale view can only look "absent", which falls through to the exact slow path.
__device__ __forceinline__ int chr_lookup_insert(const S2PParams &p, u64 h, u64 name8, const char *buf, u64 name_off, u32 len) {
    const u64 hh = h ? h : 0x9E3779B97F4A7C15ull;
    const ChrSlot *sl = &p.chr[(u32)(hh ^ (hh >> 29)) & p.chr_mask];
    if (len <= 8 && sl->key == hh && sl->id >= 0 && sl->len == len && sl->name8 == name8) return (int)(sl - p.chr);
    return chr_lookup_insert_slow(*p.self, h, name8, buf, name_off, len);
}

// ------------------------------------------------------------------------------------------------ K2: parse
template <class R>
__device__ __forceinline__ u32 parse_uint_tok(R &r, int &c) {
    while (is_blank(c)) c = r.next();
    u32 v = 0; bool bad = false; int n = 0;
    while (!is_ws(c)) { u32 d = (u32)(c - '0'); bad |= d > 9u; v = v * 10u + d; ++n; c = r.next(); }
    return (bad || n == 0) ? 0u : v;
}

// One SAM line: first six fields, record filter, CIGAR walk.  `r` is positioned at the line's first byte; when
// cmp_prev, `q` is positioned at the previous line's first byte and the two QNAMEs are compared on the fly.
// Returns the line's meta bits; `rec` is filled for kept lines.
template <class R>
__device__ __forceinline__ u32 parse_line(const S2PParams &p, R &r, R &q, const bool cmp_prev, const u64 line_abs, LineRec &rec) {
    int c = r.next();
    if (c == '@') return 0;                                   // header line (QNAME cannot contain '@')
    while (is_blank(c)) c = r.next();
    const u32 qoff = (u32)(r.pos - 1 - line_abs);
    u32 meta = 0;
    if (cmp_prev) {
        int d = q.next();
        while (is_blank(d)) d = q.next();
        bool eq = true;
        while (!is_ws(c)) { eq &= (c == d); if (!is_ws(d)) d = q.next(); c = r.next(); }
        eq &= is_ws(d);
        if (eq) meta |= LM_EQ;
    } else {
        while (!is_ws(c)) c = r.next();
    }
    const u32 qlen = (u32)(r.pos - 1 - line_abs) - qoff;
    const u32 flag = parse_uint_tok(r, c);
    while (is_blank(c)) c = r.next();
    const u64 name_off = r.pos - 1;
    u64 h = 0xCBF29CE484222325ull, name8 = 0;
    u32 name_len = 0;
    while (!is_ws(c)) { h = hash_step(h, c); if (name_len < 8) name8 |= (u64)c << (8 * name_len); ++name_len; c = r.next(); }
    const u32 pos = parse_uint_tok(r, c);
    const u32 mapq = parse_uint_tok(r, c);
    if (mapq < (u32)p.min_mapq || (flag & 0x700u)) return meta;   // pairutil.h:157-161
    meta |= LM_KEEP;
    // CIGAR walk (pairutil.h:63-126)
    while (is_blank(c)) c = r.next();
    u32 val = 0, idx = 0, leftClip = 0, rightClip = 0, mappable = 0;
    u32 cur = pos, right0 = 0, left1 = 0, right1 = 0, last_right = 0;
    bool err = false;
    while (!is_ws(c)) {
        u32 d = (u32)(c - '0');
        if (d <= 9u) { val = val * 10u + d; c = r.next(); continue; }
        const int nxt = r.next();                       // one byte of look-ahead: is this op the last character?
        if (c == 'H' || c == 'S') {
            if (is_ws(nxt)) rightClip = val;
            else if (idx == 0) leftClip = val;          // overwrites: 5H30S100M leaves leftClip = 30
            else err = true;
        } else if (c == 'M' || c == 'D') {
            if (c == 'M') mappable += val;
            cur += val; last_right = cur - 1;
            if (idx == 0) right0 = last_right; else if (idx == 1) right1 = last_right;
        } else if (c == 'N') {
            cur += val; ++idx; last_right = 0;
            if (idx == 1) left1 = cur;
        } else if (c != 'I') err = true;
        val = 0; c = nxt;
    }
    rec.pos = pos; rec.right0 = right0; rec.left1 = left1; rec.right1 = right1;
    rec.leftClip = leftClip; rec.rightClip = rightClip; rec.mappable = mappable; rec.line_len = 0;
    rec.flag = (u16)flag; rec.qname_len = (u16)qlen;
    rec.chr_slot = (u16)chr_lookup_insert(p, h, name8, p.buf, name_off, name_len);
    const u32 segCnt = idx + 1;
    if (last_right == 0) err = true;                             // pairutil.h:119
    rec.segCnt = err ? 0 : (u8)(segCnt > 2 ? 3 : segCnt);
    rec.pad0 = 0; rec.qname_off = qoff; rec.pad1 = 0;
    return meta;
}

__device__ __forceinline__ u32 lt21_y(u32 x) {                       // 0x80 in every byte < 0x21
    const u32 t = (x & 0x7F7F7F7Fu) + 0x5F5F5F5Fu;
    return ~(t | x) & 0x80808080u;
}
static __device__ __noinline__ bool qname_equal_abs(const S2PParams &p, u64 pa, u64 pb);
static __device__ __forceinline__ bool qname_equal_slow(const S2PParams &p, u64 ws, u32 a, u32 b);

// ---- word-at-a-time fast path -------------------------------------------------------------------------------------
// Well-formed lines (single tabs between the first six fields, nothing else below 0x21, digits where numbers belong,
// RNAME <= 8 bytes) are tokenised with SWAR on 16-byte words instead of byte loops; anything else returns false and goes
// through parse_line, so the result is identical by construction.
__device__ __forceinline__ u32 lt21_mask16(const uint4 &w) {         // bit q set iff byte q of the word is < 0x21 (byte order)
    return gather_flags4(lt21_y(w.x)) | (gather_flags4(lt21_y(w.y)) << 4) | (gather_flags4(lt21_y(w.z)) << 8) | (gather_flags4(lt21_y(w.w)) << 12);
}
// Fetchers: aligned 16- and 8-byte loads from global memory, or from the shared-memory copy of a tile where it covers them
struct GlobalFetch {
    const char *buf; u64 A;                                             // A: 16-byte aligned base of the relative accessors
    __device__ __forceinline__ uint4 ld16r(u32 r) const { return __ldg((const uint4 *)(buf + A + r)); }
    __device__ __forceinline__ u64 ld8r(u32 r) const { return __ldg((const u64 *)(buf + A + r)); }
    __device__ __forceinline__ int byter(u32 r) const { return (int)(unsigned char)buf[A + r]; }
    __device__ __forceinline__ uint4 ld16(u64 a) const { return __ldg((const uint4 *)(buf + a)); }
    __device__ __forceinline__ u64 ld8(u64 a) const { return __ldg((const u64 *)(buf + a)); }
    __device__ __forceinline__ int byte(u64 a) const { return (int)(unsigned char)buf[a]; }
};
template <class F>
__device__ __forceinline__ u64 fetch8r(const F &f, u32 r) {           // 8 bytes at any offset relative to f.A
    const u32 a8 = r & ~7u, sh = (r & 7u) * 8;
    const u64 lo = f.ld8r(a8);
    if (sh == 0) return lo;
    return (lo >> sh) | (f.ld8r(a8 + 8) << (64 - sh));
}
template <class F>
__device__ __forceinline__ u64 fetch8(const F &f, u64 abs) {          // 8 bytes at any offset, from aligned loads
    const u64 a8 = abs & ~(u64)7;
    const u32 sh = (u32)(abs & 7) * 8;
    const u64 lo = f.ld8(a8);
    if (sh == 0) return lo;
    return (lo >> sh) | (f.ld8(a8 + 8) << (64 - sh));
}
// QNAME of the line at `a` (length t0, already tokenised) equal to the first token of the line at `pa`?
template <class F>
__device__ __forceinline__ bool qname_eq_fetch(const F &f, u64 a, u64 pa, u32 t0) {
    bool eq = true;
    for (u32 k = 0; k < t0 && eq; k += 8) {
        u64 x = fetch8(f, a + k), y = fetch8(f, pa + k);
        if (t0 - k < 8) { const u64 m = (1ull << (8 * (t0 - k))) - 1; x &= m; y &= m; }
        eq = x == y;
    }
    return eq && is_ws(f.byte(pa + t0));
}
__device__ __forceinline__ u32 pop_lowest128(u32 &m0, u32 &m1, u32 &m2, u32 &m3) {
    if (m0) { const u32 b = __ffs(m0) - 1; m0 &= m0 - 1; return b; }
    if (m1) { const u32 b = __ffs(m1) - 1; m1 &= m1 - 1; return 32 + b; }
    if (m2) { const u32 b = __ffs(m2) - 1; m2 &= m2 - 1; return 64 + b; }
    if (m3) { const u32 b = __ffs(m3) - 1; m3 &= m3 - 1; return 96 + b; }
    return 255;
}
// decimal field of `len` (1..10) characters starting at abs; false if a non-digit is found
template <class F>
__device__ __forceinline__ bool dec_field(const F &buf, u32 abs, u32 len, u32 &out) {
    u64 x = fetch8r(buf, abs);
    u32 v = 0; bool ok = true;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if ((u32)k < len) { const u32 d = (u32)((x >> (8 * k)) & 0xFF) - '0'; ok &= d <= 9u; v = v * 10u + d; }
    }
    if (len > 8) {
        x = fetch8r(buf, abs + 8);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            if ((u32)(8 + k) < len) { const u32 d = (u32)((x >> (8 * k)) & 0xFF) - '0'; ok &= d <= 9u; v = v * 10u + d; }
        }
    }
    out = v;
    return ok;
}

// first byte < 0x21 in the 8 bytes of x (0..7), or 8 when there is none
__device__ __forceinline__ u32 first_ws8(u64 x) {
    const u32 lo = lt21_y((u32)x), hi = lt21_y((u32)(x >> 32));
    if (lo) return (u32)(__ffs(lo) - 1) >> 3;
    if (hi) return 4u + ((u32)(__ffs(hi) - 1) >> 3);
    return 8u;
}
// (A field-by-field tokeniser — QNAME's end from 16-byte words, every later field from the eight bytes at its start — needs a
// third fewer instructions but chains every fetch to the previous field's end: measured 3.68 ms against 3.01 ms for the mask
// of all seven staged words below, whose loads and SWAR tests are independent.  This kernel is bound by per-thread latency.)
struct FastTok { u32 t0; u64 q[5]; bool ok; };                       // QNAME length and its first 40 bytes (zero padded)

template <class F, bool WANT_Q, bool RM, class RT>
__device__ __forceinline__ bool parse_line_fast(const S2PParams &p, const F &f, const u64 a, const u64 limit, FastTok &tok, RT &rec, u32 &meta, u32 &rminfo) {
    tok.ok = false;
    if (a + 144 > limit) return false;
    const u64 A = a & ~(u64)15;
    const u32 s = (u32)(a - A);
    uint4 w[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) w[j] = f.ld16r(16 * j);
    if ((char)((w[0].x >> 0) & 0xFF) == '@' && s == 0) return false;   // cheap early-out; the exact test is below
    u32 m0 = lt21_mask16(w[0]) | (lt21_mask16(w[1]) << 16), m1 = lt21_mask16(w[2]) | (lt21_mask16(w[3]) << 16);
    u32 m2 = lt21_mask16(w[4]) | (lt21_mask16(w[5]) << 16), m3 = lt21_mask16(w[6]);
    if (s) {                                                          // bit j <-> byte a + j
        m0 = __funnelshift_r(m0, m1, s); m1 = __funnelshift_r(m1, m2, s); m2 = __funnelshift_r(m2, m3, s); m3 >>= s;
    }
    const u32 t0 = pop_lowest128(m0, m1, m2, m3), t1 = pop_lowest128(m0, m1, m2, m3), t2 = pop_lowest128(m0, m1, m2, m3);
    const u32 t3 = pop_lowest128(m0, m1, m2, m3), t4 = pop_lowest128(m0, m1, m2, m3), t5 = pop_lowest128(m0, m1, m2, m3);
    if (t5 >= 112 - s) return false;                                  // six separators inside the words we looked at
    // every separator must be a single TAB, every field non-empty
    if (t0 == 0 || t1 == t0 + 1 || t2 == t1 + 1 || t3 == t2 + 1 || t4 == t3 + 1 || t5 == t4 + 1) return false;
    if (f.byter(s + t0) != '\t' || f.byter(s + t1) != '\t' || f.byter(s + t2) != '\t' || f.byter(s + t3) != '\t' || f.byter(s + t4) != '\t' ||
        f.byter(s + t5) != '\t') return false;
    if (f.byter(s) == '@') return false;
    const u32 l_flag = t1 - t0 - 1, l_name = t2 - t1 - 1, l_pos = t3 - t2 - 1, l_mapq = t4 - t3 - 1;
    if (l_flag > 5 || l_name > 8 || l_pos > 10 || l_mapq > 3) return false;
    u32 flag, pos, mapq;
    if (!dec_field(f, s + t0 + 1, l_flag, flag)) return false;
    if (!dec_field(f, s + t2 + 1, l_pos, pos)) return false;
    if (!dec_field(f, s + t3 + 1, l_mapq, mapq)) return false;
    u32 rm_so = 0, qlen = 0;
    if (RM) {                                                          // SAM-space krmdup: where SEQ (field 10) starts, when the prefix shows it
        const u32 t6 = pop_lowest128(m0, m1, m2, m3), t7 = pop_lowest128(m0, m1, m2, m3), t8 = pop_lowest128(m0, m1, m2, m3);
        if (flag <= 0xFFFu) {
            // SEQ's offset when the staged prefix reaches it, else the offset of field 7 (three short tab searches are left)
            if (t8 < 112 - s && f.byter(s + t6) == '\t' && f.byter(s + t7) == '\t' && f.byter(s + t8) == '\t') rm_so = (t8 + 1) | 128u;
            else rm_so = t5 + 1;
        }
        rminfo = flag | (rm_so << 12);                                 // rm_so = 0: k_rm_keys finds FLAG and SEQ itself
    }
    tok.t0 = t0;
    if (WANT_Q) {                                                      // QNAME words for the neighbour-lane comparison
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            u64 x = (u32)(8 * k) < t0 ? fetch8r(f, s + 8 * k) : 0;
            if (t0 < (u32)(8 * k + 8) && t0 > (u32)(8 * k)) x &= (1ull << (8 * (t0 - 8 * k))) - 1;
            tok.q[k] = x;
        }
    }
    tok.ok = t0 <= 40;
    meta = 0;
    if (mapq < (u32)p.min_mapq || (flag & 0x700u)) {                  // pairutil.h:157-161
        if (RM && rm_so && !(flag & 0x900u)) {                         // a dropped PRIMARY record still carries its read: SEQ length from the CIGAR
            const u32 lc = t5 - t4 - 1;
            u32 v = 0; u64 y = 0;
            for (u32 k = 0; k < lc; ++k) {
                if ((k & 7) == 0) y = fetch8r(f, s + t4 + 1 + k);
                const int c = (int)(y & 0xFF); y >>= 8;
                const u32 d = (u32)(c - '0');
                if (d <= 9u) { v = v * 10u + d; continue; }
                if (c == 'M' || c == 'I' || c == 'S' || c == '=' || c == 'X') qlen += v;
                v = 0;
            }
            if (qlen < 4096u) rminfo |= qlen << 20;
        }
        return true;
    }
    meta = LM_KEEP;
    // RNAME: FNV-1a over its bytes, same as the byte loop
    u64 name8 = fetch8r(f, s + t1 + 1);
    if (l_name < 8) name8 &= (1ull << (8 * l_name)) - 1;
    u64 h = 0xCBF29CE484222325ull;
#pragma unroll
    for (int k = 0; k < 8; ++k) if ((u32)k < l_name) h = hash_step(h, (int)((name8 >> (8 * k)) & 0xFF));
    // CIGAR walk (pairutil.h:63-126), 8 characters per fetch
    u32 val = 0, idx = 0, leftClip = 0, rightClip = 0, mappable = 0;
    u32 cur = pos, right0 = 0, left1 = 0, right1 = 0, last_right = 0;
    bool err = false;
    const u32 l_cig = t5 - t4 - 1;
    u64 x = 0;
    for (u32 k = 0; k < l_cig; ++k) {
        if ((k & 7) == 0) x = fetch8r(f, s + t4 + 1 + k);
        const int c = (int)(x & 0xFF); x >>= 8;
        const u32 d = (u32)(c - '0');
        if (d <= 9u) { val = val * 10u + d; continue; }
        if (c == 'H' || c == 'S') {
            if (k + 1 == l_cig) rightClip = val;
            else if (idx == 0) leftClip = val;
            else err = true;
        } else if (c == 'M' || c == 'D') {
            if (c == 'M') mappable += val;
            cur += val; last_right = cur - 1;
            if (idx == 0) right0 = last_right; else if (idx == 1) right1 = last_right;
        } else if (c == 'N') {
            cur += val; ++idx; last_right = 0;
            if (idx == 1) left1 = cur;
        } else if (c != 'I') err = true;
        if (RM && (c == 'M' || c == 'I' || c == 'S')) qlen += val;     // bases present in SEQ (SAM spec 1.4.6)
        val = 0;
    }
    if (RM && rm_so && !err && qlen < 4096u) rminfo |= qlen << 20;
    rec.pos = pos; rec.right0 = right0; rec.left1 = left1; rec.right1 = right1;
    rec.leftClip = leftClip; rec.rightClip = rightClip; rec.mappable = mappable; rec.line_len = 0;
    rec.flag = (u16)flag; rec.qname_len = (u16)t0;
    rec.chr_slot = (u16)chr_lookup_insert(p, h, name8, p.buf, a + t1 + 1, l_name);
    const u32 segCnt = idx + 1;
    if (last_right == 0) err = true;
    rec.segCnt = err ? 0 : (u8)(segCnt > 2 ? 3 : segCnt);
    rec.pad0 = 0; rec.qname_off = 0; rec.pad1 = 0;
    return true;
}

// the generic byte-loop parser, out of line: it is the rare path and would otherwise triple the hot loop's code size
static __device__ __noinline__ u32 parse_line_slow_abs(const S2PParams &p, u64 a, bool has_prev, u64 pa, LineRec &rec) {
    ByteReader r, q;
    r.init(p.buf, a);
    if (has_prev) q.init(p.buf, pa);
    return parse_line(p, r, q, has_prev, a, rec);
}
static __device__ __forceinline__ u32 parse_line_slow(const S2PParams &p, u64 ws, u32 i, u64 a, LineRec &rec) {
    return parse_line_slow_abs(*p.self, a, i > 0, ws + (i > 1 ? p.nl_pos[i - 2] + 1 : 0), rec);
}

// ---- K2 staging: every thread's line prefix (7 x 16 bytes from the line's 16-byte aligned base) is copied global -> shared
// with cp.async (LDGSTS: no register staging, no store instructions) into the thread's own 144-byte row, one round AHEAD
// of the round being parsed, so the DRAM latency of a round's scattered 112-byte reads is covered by the previous round's
// parsing.  (The first version loaded into registers, transposed into shared-memory word columns and parsed in the same
// round: ncu showed 4.3 long-scoreboard stalls per issue at 24 resident warps.)  Row stride 144 = 9 x 16 bytes: the eight
// lanes of a quarter-warp start 36 words apart, so 16-byte row reads are conflict-free; bytes 112..127 of a row are a zero
// pad that is never rewritten, so eight bytes at ANY offset below 112 are three 32-bit loads and two funnel shifts with
// no bounds test.
#define PR_ROW 144
// PR_STAGES = 2 stages a round AHEAD of the round being parsed (double buffer, 74 KB per CTA: three CTAs per SM);
// PR_STAGES = 1 stages and parses in the same round and lets four CTAs (32 warps) share the SM.  Measured on B200, 19.8 GB:
// 3.35 ms with the read-ahead, 3.00 ms with the extra warps (five CTAs: 3.00 ms again) — this kernel wants warps more than it
// wants prefetch, so one stage is the default.
#ifndef PR_OCC
#define PR_OCC 4
#endif
#ifndef PR_STAGES
#define PR_STAGES 1
#endif
#ifndef PR_LDG
#define PR_LDG 0
#endif
__device__ __forceinline__ void cp_async16(u32 saddr, const void *g) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
struct RowFetch {
    const char *row;                                                    // this line's 144-byte row in shared memory
    __device__ __forceinline__ uint4 ld16r(u32 r) const { return *(const uint4 *)(row + r); }      // r = 16 j
    __device__ __forceinline__ int byter(u32 r) const { return (int)(unsigned char)row[r]; }
    __device__ __forceinline__ u64 f8(u32 r) const {                   // r + 8 <= 120
        const u32 *q = (const u32 *)(row + (r & ~3u)); const u32 sh = (r & 3u) * 8u;
        const u32 a = q[0], b = q[1], c = q[2];
        return (u64)__funnelshift_r(a, b, sh) | ((u64)__funnelshift_r(b, c, sh) << 32);
    }
};
__device__ __forceinline__ u64 fetch8r(const RowFetch &f, u32 r) { return f.f8(r); }

// Every WARP runs its own pipeline over chunks of 32 consecutive lines (chunk = warp index + k x warps in the grid): no block
// barrier anywhere — a lane's left neighbour is in the same warp, and lane 0 compares its QNAME with the previous chunk's
// last line through global memory (L2: another warp has just staged those bytes).  ncu on the block-synchronous version:
// 15 % of the stall samples on the two barriers per round (threads of a CTA finish their lines at very different times:
// CIGAR length, the rare slow path).
template <bool RM>
static __global__ void __launch_bounds__(256, PR_STAGES == 1 ? PR_OCC : 3) k_parse(S2PParams p) {
    extern __shared__ __align__(16) char s_rows[];                     // [PR_STAGES][256][PR_ROW]
    __shared__ u32 s_st[PR_STAGES][256];                               // the staged line's start (relative to ws), or ~0 when not staged
    const WinState *st = p.st;
    const u32 n_lines = st->n_lines;
    const u64 ws = st->ws;
    const u64 limit = st->total;
    const int tid = threadIdx.x;
    const u32 lane = tid & 31u;
#pragma unroll
    for (int b = 0; b < PR_STAGES; ++b) *(uint4 *)(s_rows + ((size_t)b * 256 + tid) * PR_ROW + 112) = make_uint4(0, 0, 0, 0);
    __syncwarp();
    const u32 n_round = (n_lines + 31u) & ~31u;                       // whole warps stay in the loop
    const u32 stride = gridDim.x * 256u;                               // lines between two chunks of one warp
    u32 i = (blockIdx.x * 8u + (tid >> 5)) * 32u + lane;
    // The newline in front of line k is what gives its start.  It is fetched two rounds ahead with NOTHING depending on the
    // loaded value until the round that uses it (the index is clamped instead of the value selected), so its latency is
    // never waited for: kind 0 = no such line, 1 = line 0 (starts at the window start), 2 = start is the loaded value + 1.
    auto nl_kind = [&](u32 k, bool in_range) -> u32 { return (in_range && k < n_lines) ? (k ? 2u : 1u) : 0u; };
    auto nl_load = [&](u32 k, u32 kind) -> u32 {
        u32 v;
        asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p.nl_pos + (kind == 2u ? k - 1u : 0u)));
        return v;
    };
    auto stage = [&](int b, u32 raw, u32 kind) {                       // issue the copies of one line's prefix
        u32 staged = 0xFFFFFFFFu;
        const u32 start = kind == 2u ? raw + 1u : 0u;
        if (kind) {
            const u64 a = ws + start;
            if (a + 144 <= limit) {
                staged = start;
                const char *g = p.buf + (a & ~(u64)15);
#if PR_LDG
                // seven independent 128-bit loads, then seven 128-bit shared stores (four wavefronts each with the 144-byte row
                // stride); cp.async writes every lane's 16 bytes as a wavefront of its own: 28 per instruction (ncu)
                uint4 w[7];
#pragma unroll
                for (int j = 0; j < 7; ++j) w[j] = __ldg((const uint4 *)g + j);
                uint4 *row = (uint4 *)(s_rows + ((size_t)b * 256 + tid) * PR_ROW);
#pragma unroll
                for (int j = 0; j < 7; ++j) row[j] = w[j];
#else
                const u32 sa = smem_u32(s_rows + ((size_t)b * 256 + tid) * PR_ROW);
#pragma unroll
                for (int j = 0; j < 7; ++j) cp_async16(sa + 16 * j, g + 16 * j);
#endif
            }
        }
        s_st[b][tid] = staged;
        cp_async_commit();
    };
    u32 k_cur = nl_kind(i, i < n_round), k_nxt = nl_kind(i + stride, i + stride < n_round);
    u32 r_cur = nl_load(i, k_cur), r_nxt = nl_load(i + stride, k_nxt);
    if (PR_STAGES > 1 && i < n_round) stage(0, r_cur, k_cur);
    int b = 0;
    for (; i < n_round; i += stride, b ^= (PR_STAGES - 1)) {
        const bool active = i < n_lines;
        // next round's copies go out first, then the newline of the round after it is fetched
        const bool more = i + stride < n_round;
        if (PR_STAGES == 1) stage(0, r_cur, k_cur);                    // one stage: this round's own copies
        else if (more) stage(b ^ 1, r_nxt, k_nxt);
        const u32 k_nn = nl_kind(i + 2 * stride, more && i + 2 * stride < n_round);
        const u32 r_nn = nl_load(i + 2 * stride, k_nn);
        if (more && PR_STAGES > 1) cp_async_wait<1>(); else cp_async_wait<0>();
        __syncwarp();                                                  // neighbours read each other's rows
        if (active) {
            if (p.write_sam) p.sam_dst[i] = 0xFFFFFFFFu;
            const u64 a = ws + (u64)(k_cur == 2u ? r_cur + 1u : 0u);
            RowFetch lf; lf.row = s_rows + ((size_t)b * 256 + tid) * PR_ROW;
            const bool staged = s_st[b][tid] != 0xFFFFFFFFu;
            LineRec rec; u32 meta = 0;
            FastTok tok;
            u32 rminfo = 0;                                            // SEQ offset unknown
            if (staged && parse_line_fast<RowFetch, false, RM>(p, lf, a, limit, tok, rec, meta, rminfo)) {
                if (i > 0) {
                    // QNAME equal to the previous line's?  That line's prefix sits in the neighbouring row.
                    const u32 pst = lane > 0 ? s_st[b][tid - 1] : 0xFFFFFFFFu;
                    const u32 sp = (u32)((ws + pst) & 15u);            // the previous line's first byte inside its row
                    bool eq;
                    if (pst != 0xFFFFFFFFu && sp + tok.t0 + 1 <= 112) {
                        RowFetch lp; lp.row = lf.row - PR_ROW;
                        if (is_blank(lp.byter(sp))) eq = qname_equal_slow(p, ws, i, i - 1);   // operator>> skips leading blanks
                        else {
                            const u32 so = (u32)(a & 15u);
                            eq = true;
                            for (u32 k = 0; k < tok.t0 && eq; k += 8) {
                                u64 x = fetch8r(lf, so + k), y = fetch8r(lp, sp + k);
                                if (tok.t0 - k < 8) { const u64 m = (1ull << (8 * (tok.t0 - k))) - 1; x &= m; y &= m; }
                                eq = x == y;
                            }
                            eq = eq && is_ws(lp.byter(sp + tok.t0));
                        }
                    } else {                                           // first lane of the warp, or a line the staging skipped
                        const u64 pa = ws + (i > 1 ? p.nl_pos[i - 2] + 1 : 0);
                        if (is_blank((int)(unsigned char)p.buf[pa])) eq = qname_equal_slow(p, ws, i, i - 1);
                        else { GlobalFetch gf; gf.buf = p.buf; gf.A = 0; eq = qname_eq_fetch(gf, a, pa, tok.t0); }
                    }
                    if (eq) meta |= LM_EQ;
                }
            } else meta = parse_line_slow(p, ws, i, a, rec);
            if (meta & LM_KEEP) p.rec[i] = rec;
            p.lmeta[i] = (u8)meta;
            if (RM) p.rm_info[i] = rminfo;
        }
        __syncwarp();                                                  // this round's rows are the target of the next round's copies
        k_cur = k_nxt; r_cur = r_nxt; k_nxt = k_nn; r_nxt = r_nn;
    }
}
#define PR_SMEM (PR_STAGES * 256 * PR_ROW)

// ------------------------------------------------------------------------------------------------ K3: groups
struct Seg { u32 pos, right0, left1, right1, leftClip, rightClip, mappable; int segCnt; bool minus; u16 chr; };

template <class RT>
__device__ __forceinline__ Seg seg_of(const RT &r) {
    Seg s; s.pos = r.pos; s.right0 = r.right0; s.left1 = r.left1; s.right1 = r.right1;
    s.leftClip = r.leftClip; s.rightClip = r.rightClip; s.mappable = r.mappable; s.segCnt = r.segCnt;
    s.minus = (r.flag & 16u) != 0; s.chr = r.chr_slot;
    return s;
}
// pairutil.h:180-188.  fp32 on purpose: __fmul_rn keeps the product un-fused and un-contracted.
__device__ __forceinline__ bool integrity1(const Seg &s, float ratio) {
    int total = (int)s.mappable;
    if ((int)s.leftClip > 20) total += (int)s.leftClip;
    if ((int)s.rightClip > 20) total += (int)s.rightClip;
    return (float)(int)s.mappable >= __fmul_rn((float)total, ratio);
}
// pairutil.h:190-208, including the s1.rightClip test of line 200
__device__ __forceinline__ bool integrity2(const Seg &a, const Seg &b, float ratio) {
    int ta = (int)a.mappable, tb = (int)b.mappable;
    if ((int)a.leftClip > 20) ta += (int)a.leftClip;
    if ((int)a.rightClip > 20) ta += (int)a.rightClip;
    if ((int)b.leftClip > 20) tb += (int)b.leftClip;
    if ((int)a.rightClip > 20) tb += (int)b.rightClip;
    int big = ta > tb ? ta : tb;
    return (float)(int)(a.mappable + b.mappable) >= __fmul_rn((float)big, ratio);
}
// the mate test of unc2pairs.h:191-308 (positions compared as signed int like the reference)
__device__ __forceinline__ bool mates(const Seg &lone, const Seg &c) {
    if (lone.chr != c.chr) return false;
    if (!lone.minus) return c.minus && (int)lone.pos < (int)c.pos && (int)c.right0 - (int)lone.pos <= 1000;
    return !c.minus && (int)c.pos < (int)lone.pos && (int)lone.right0 - (int)c.pos <= 1000;
}
__device__ __forceinline__ u32 distal_end(const Seg &s) { return (int)s.leftClip > (int)s.rightClip ? s.right0 : s.pos; }

// Exact comparison of the first tokens (QNAMEs) of lines a and b, 8 bytes at a time.  Bytes below 0x21 that are not
// white space, and leading blanks, are left to the byte loop so that the result is operator>>'s in every case.
static __device__ __noinline__ bool qname_equal_bytes(const S2PParams &p, u64 pa, u64 pb) {
    ByteReader x, y;
    x.init(p.buf, pa); y.init(p.buf, pb);
    int c = x.next(), d = y.next();
    while (is_blank(c)) c = x.next();
    while (is_blank(d)) d = y.next();
    while (!is_ws(c) && !is_ws(d)) { if (c != d) return false; c = x.next(); d = y.next(); }
    return is_ws(c) && is_ws(d);
}
static __device__ __forceinline__ bool qname_equal_slow(const S2PParams &p, u64 ws, u32 a, u32 b) {
    return qname_equal_abs(*p.self, ws + (a ? p.nl_pos[a - 1] + 1 : 0), ws + (b ? p.nl_pos[b - 1] + 1 : 0));
}
// first tokens of the lines that start at absolute offsets pa and pb
static __device__ __noinline__ bool qname_equal_abs(const S2PParams &p, u64 pa, u64 pb) {
    GlobalFetch gf; gf.buf = p.buf; gf.A = 0;
    for (u32 k = 0;; k += 8) {
        const u64 x = fetch8(gf, pa + k), y = fetch8(gf, pb + k);
        const u32 tx = first_ws8(x), ty = first_ws8(y);
        if (tx == 8 && ty == 8) { if (x != y) return false; continue; }
        // a token ends inside this word: both must end at the same byte, on real white space, after equal bytes
        const u32 t = tx < ty ? tx : ty;
        const int cx = tx < 8 ? (int)((x >> (8 * tx)) & 0xFF) : 'x', cy = ty < 8 ? (int)((y >> (8 * ty)) & 0xFF) : 'x';
        if ((tx < 8 && !is_ws(cx)) || (ty < 8 && !is_ws(cy)) || (k == 0 && t == 0)) return qname_equal_bytes(p, pa, pb);
        if (tx != ty) return false;
        const u64 m = t ? ((1ull << (8 * t)) - 1) : 0;
        return (x & m) == (y & m);
    }
}

// ------------------------------------------------------------------------------------------------ SAM-space krmdup
// The reference removes PCR duplicates from the FASTQ BEFORE alignment (src/preprocess/krmdup.cpp): key = bases
// [hskip, hskip + klen) of each mate, 2 bits per base (:168-193); the first pair with a key in file order is kept, later ones
// and pairs with a short mate or a non-ACGT base in a key window are dropped (:103-111,159-198,201-212); the pairs whose first
// key base is not exactly 'A' / 'C' / 'G' share the fourth set (:134-141).  The aligner keeps the read order and SEQ holds the
// read's bases (reverse-complemented when flag & 16), so the same decision can be taken on the SAM: a QNAME run (consecutive
// lines with equal QNAME, dropped ones included) is one read pair, its PRIMARY records (flag & 0x900 == 0) carry the full
// reads.  flag & 64 -> mate 1, flag & 128 -> mate 2, neither (a stitched read) -> mate 1 = the read, mate 2 = its reverse
// complement.  Runs the reference would not have let through lose LM_KEEP before K3 sees them, so everything downstream
// (grouping, counters, the 2^18-batch self-circle rule, the dropped last group) is what sam2pairs does on the SAM of the
// deduplicated FASTQ.  A run without a primary record for a mate counts as discarded.
#define RM_EMPTY 0xFFFFFFFFFFFFFFFFull
// per-line status (rm_stat): which mates the line's SEQ provides and whether their key windows are valid
#define RL_M1 1u
#define RL_M2 2u
#define RL_OK1 4u
#define RL_OK2 8u
#define RL_TAG 16u
#define RL_HDR 32u

__device__ __forceinline__ u64 rm_tabmask(u64 w) {                      // bit 7 of every byte that is '\t' (exact)
    const u64 x = w ^ 0x0909090909090909ull;
    return ~(((x & 0x7F7F7F7F7F7F7F7Full) + 0x7F7F7F7F7F7F7F7Full) | x) & 0x8080808080808080ull;
}
// first '\t' in [from, end) or end; aligned 16-byte loads (the buffer is 16-byte aligned and padded)
__device__ __forceinline__ u64 rm_next_tab(const char *buf, u64 from, u64 end) {
    u64 pos = from & ~15ull;
    uint4 w = __ldg((const uint4 *)(buf + pos));
    u64 lo = rm_tabmask((u64)w.x | ((u64)w.y << 32)), hi = rm_tabmask((u64)w.z | ((u64)w.w << 32));
    const u32 sk = (u32)(from - pos);                                   // bytes before `from` do not count
    if (sk >= 8) { lo = 0; hi &= ~0ull << (8 * (sk - 8)); } else lo &= ~0ull << (8 * sk);
    while (true) {
        if (lo | hi) {
            const u64 t = pos + (lo ? ((u32)(__ffsll((long long)lo) - 1) >> 3) : 8u + ((u32)(__ffsll((long long)hi) - 1) >> 3));
            return t < end ? t : end;
        }
        do {                                                            // four SIMD compares per 16 bytes until a word holds a tab
            pos += 16;
            if (pos >= end) return end;
            w = __ldg((const uint4 *)(buf + pos));
        } while (!(__vcmpeq4(w.x, 0x09090909u) | __vcmpeq4(w.y, 0x09090909u) | __vcmpeq4(w.z, 0x09090909u) | __vcmpeq4(w.w, 0x09090909u)));
        lo = rm_tabmask((u64)w.x | ((u64)w.y << 32)); hi = rm_tabmask((u64)w.z | ((u64)w.w << 32));
    }
}
// 8 bases in memory order -> their 2-bit codes, base k at bits 2k (krmdup.cpp:171-177: A 1, T 2, C 0, G 3, either case; from
// (c >> 1) & 3 = A 0, C 1, T 2, G 3); ok is cleared when one of the first nb bytes is not a base
__device__ __forceinline__ u32 rm_codes8(u64 w, int nb, bool &ok) {
    const u32 ul = (u32)w & 0xDFDFDFDFu, uh = (u32)(w >> 32) & 0xDFDFDFDFu;
    const u32 vl = __vcmpeq4(ul, 0x41414141u) | __vcmpeq4(ul, 0x43434343u) | __vcmpeq4(ul, 0x47474747u) | __vcmpeq4(ul, 0x54545454u);
    const u32 vh = __vcmpeq4(uh, 0x41414141u) | __vcmpeq4(uh, 0x43434343u) | __vcmpeq4(uh, 0x47474747u) | __vcmpeq4(uh, 0x54545454u);
    const u64 need = nb >= 8 ? ~0ull : ((1ull << (8 * nb)) - 1);
    ok = ok && ((((u64)vl | ((u64)vh << 32)) & need) == need);
    const u64 x = (w >> 1) & 0x0303030303030303ull;
    u64 c = (x ^ ((~x >> 1) & 0x0101010101010101ull)) & need;
    c = (c | (c >> 6)) & 0x000F000F000F000Full;
    c = (c | (c >> 12)) & 0x000000FF000000FFull;
    c = (c | (c >> 24)) & 0xFFFFull;
    return (u32)c;
}
// bases [hskip, hskip + klen) of the mate that is SEQ (rev = false) or its reverse complement; false = discard.
// The klen bytes are fetched in memory order, eight at a time: for the reverse complement that IS the key's order once
// every code is complemented (code ^ 3); for the forward mate the 2-bit groups are reversed.
// lower_first: the mate's first key base is a lower-case a / c / g (krmdup.cpp:134-141: T bucket, own identity space)
__device__ __forceinline__ bool rm_half(const char *buf, u64 seq, u32 L, bool rev, int hskip, int klen, u64 &bits, bool &lower_first) {
    bits = 0; lower_first = false;
    if (L < (u32)(hskip + klen)) return false;
    if (klen == 0) return true;
    GlobalFetch gf; gf.buf = buf; gf.A = 0;
    const u64 start = rev ? seq + L - (u32)(hskip + klen) : seq + (u32)hskip;
    u64 le = 0; bool ok = true;
    for (int o = 0; o < klen; o += 8) le |= (u64)rm_codes8(fetch8(gf, start + (u32)o), klen - o, ok) << (2 * o);
    const u32 c0 = (u32)(unsigned char)buf[rev ? start + (u32)klen - 1 : start];
    if (rev) bits = le ^ (klen >= 32 ? ~0ull : ((1ull << (2 * klen)) - 1));
    else {
        u64 r = __brevll(le);
        r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
        bits = r >> (64 - 2 * klen);
    }
    lower_first = (c0 & 0x20u) && ((bits >> (2 * klen - 2)) & 3u) != 2u;
    return ok;
}
__device__ __forceinline__ u64 rm_hash(u64 k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}
// slot of `key`, inserted when absent (claimed = this call put it there); ~0 when the table is full
__device__ __forceinline__ u64 rm_slot(unsigned long long *tab, u64 mask, u64 key, bool &claimed) {
    u64 s = rm_hash(key) & mask;
    claimed = false;
    for (u64 probe = 0; probe <= mask; ++probe, s = (s + 1) & mask) {
        unsigned long long cur = *(volatile unsigned long long *)&tab[2 * s];
        if (cur == RM_EMPTY) {
            cur = atomicCAS(&tab[2 * s], RM_EMPTY, (unsigned long long)key);
            if (cur == RM_EMPTY) { claimed = true; return s; }
        }
        if (cur == key) return s;
    }
    return ~0ull;
}
// the lines of the run that starts at line h stop counting as kept
__device__ __forceinline__ void rm_drop_run(const S2PParams &p, u32 h, u32 n) {
    u32 j = h;
    do { const u32 m = p.lmeta[j]; if (m & LM_KEEP) p.lmeta[j] = (u8)(m & ~LM_KEEP); ++j; } while (j < n && (p.lmeta[j] & LM_EQ));
}

// the key bits the SEQ of line i gives to mate 1 and / or mate 2 (primary records only)
static __device__ __forceinline__ void rm_line_keys(const S2PParams &p, const u64 ws, const u32 i, u32 &stat, u64 &key, u64 &key2) {
    const u32 info = p.rm_info[i];                                      // K2: flag | offset << 12 | (offset is SEQ's, not field 7's) << 19 | SEQ length by the CIGAR << 20
    const u64 a = ws + (i ? (u64)p.nl_pos[i - 1] + 1 : 0), e = ws + p.nl_pos[i];
    u32 flag = info & 0xFFFu;
    const u32 so = (info >> 12) & 0x7Fu, ql = info >> 20;
    u64 seq = a + so;
    bool primary = true;
    stat = 0; key = 0; key2 = 0;
    if (so && !(info & (1u << 19)) && !(flag & 0x900u)) {               // from field 7 (RNEXT): PNEXT, TLEN, SEQ
        u64 t = seq;
        for (int k = 0; k < 3 && t < e; ++k) { t = rm_next_tab(p.buf, t, e); if (t < e) ++t; }
        seq = t;
    }
    if (so == 0) {                                                      // K2 did not parse the line: FLAG = field 2, SEQ = field 10
        if (p.buf[a] == '@') { stat = RL_HDR; primary = false; }
        else {
            const u64 t1 = rm_next_tab(p.buf, a, e);
            u64 t = t1 < e ? rm_next_tab(p.buf, t1 + 1, e) : e;
            flag = 0;
            for (u64 q = t1 + 1; q < t; ++q) flag = flag * 10u + (u32)((unsigned char)p.buf[q] - '0');
            for (int k = 2; k < 9 && t < e; ++k) t = rm_next_tab(p.buf, t + 1, e);
            seq = t < e ? t + 1 : e;
        }
    }
    if (primary && !(flag & 0x900u)) {
        // SEQ length: the CIGAR's when the byte behind it ends the field (no scan over the bases), else counted
        u32 L;
        if (so && ql && seq + ql <= e && (seq + ql == e || p.buf[seq + ql] == '\t') && p.buf[seq + ql - 1] != '\t') L = ql;
        else L = seq < e ? (u32)(rm_next_tab(p.buf, seq, e) - seq) : 0u;
        const bool m1 = (flag & 64u) || !(flag & 192u), m2 = !(flag & 64u);   // 128 only -> mate 2; neither (stitched) -> both
        const bool rev = (flag & 16u) != 0;
        bool lf = false, l2;
        if (m1) { stat |= RL_M1; if (rm_half(p.buf, seq, L, rev, p.rm_hskip1, p.rm_klen1, key, lf)) stat |= RL_OK1; if (lf) stat |= RL_TAG; }
        if (m2) { stat |= RL_M2; if (rm_half(p.buf, seq, L, (flag & 192u) ? rev : !rev, p.rm_hskip2, p.rm_klen2, key2, l2)) stat |= RL_OK2; }
    }
}
// the same for a line of another CTA's tile (a run that crosses a tile boundary: one in ~100); out of line to keep the kernel small
static __device__ __noinline__ void rm_line_keys_far(const S2PParams &p, u64 ws, u32 i, u32 &stat, u64 &key, u64 &key2) { rm_line_keys(p, ws, i, stat, key, key2); }

// One kernel, 256 consecutive lines per CTA round.  Every thread first works out what ITS line contributes (staged in shared
// memory); then the thread of a run's first line combines the run's mates into the pair's key and settles the run on the spot.
// The table keeps, per key, the smallest global line index seen so far (atomicMin), and the value it held before tells
// everything: nothing or this very line (a re-parsed run) -> this run is the first occurrence so far; a larger index ->
// likewise, and the run that index belongs to (necessarily of this window: earlier windows hold smaller indices) is a
// duplicate after all, so ITS lines are dropped here - every index is handed back to exactly one later, smaller insert;
// a smaller index -> this run is the duplicate.  No second pass over the table.  Uniq = keys ever claimed.
// A run cut by the window end is decided in the next window; until then its lines do not count as kept, so that the group
// before it stays the window's last (carried) group: it may yet turn out to be the stream's last one (pairutil.h:176).
// The read pair of the run that starts at line i: its mates' key bits b1 / b2 and have = RL_M* | RL_OK* | RL_TAG.  Lines of
// the CTA's round (i0 + t, t < 256) come from the staged s_*[t], later ones from global memory.  Returns the line after the run.
static __device__ __forceinline__ u32 rm_run_combine(const S2PParams &p, u64 ws, u32 n, u32 i0, u32 i, u32 sl, u64 k1, u64 k2, const u8 *s_meta,
                                                     const u8 *s_stat, const unsigned long long *s_k1, const unsigned long long *s_k2,
                                                     u32 &have, u64 &b1, u64 &b2) {
    have = 0; b1 = 0; b2 = 0;
    u32 j = i;
    while (true) {
        if (sl & ~have & RL_M1) { b1 = k1; have |= RL_M1 | (sl & (RL_OK1 | RL_TAG)); }
        if (sl & ~have & RL_M2) { b2 = k2; have |= RL_M2 | (sl & RL_OK2); }
        ++j;
        if (j >= n) break;
        const u32 t = j - i0;
        if (t < 256u) { if (!(s_meta[t] & LM_EQ)) break; sl = s_stat[t]; k1 = s_k1[t]; k2 = s_k2[t]; }
        else { if (!(p.lmeta[j] & LM_EQ)) break; rm_line_keys_far(*p.self, ws, j, sl, k1, k2); }
    }
    return j;
}

static __global__ void __launch_bounds__(256) k_rm_insert(S2PParams p) {
    __shared__ unsigned long long s_k1[256], s_k2[256];
    __shared__ u8 s_stat[256], s_meta[256];
    WinState *st = p.st;
    const u32 n = st->n_lines;
    const u64 ws = st->ws, g0 = st->lines_done, counted = st->rm_counted;
    const bool final_win = (st->we == st->total) && st->is_last;
    const u32 tid = threadIdx.x;
    u32 c_tot = 0, c_uniq = 0, c_disc = 0;
    for (u32 i0 = blockIdx.x * 256u; i0 < n; i0 += gridDim.x * 256u) {
        const u32 i = i0 + tid;
        u32 m_i = 0, sl = 0; u64 k1 = 0, k2 = 0;
        if (i < n) { m_i = p.lmeta[i]; rm_line_keys(p, ws, i, sl, k1, k2); }
        __syncthreads();                                                // the previous round's entries have been consumed
        s_meta[tid] = (u8)m_i; s_stat[tid] = (u8)sl; s_k1[tid] = k1; s_k2[tid] = k2;
        __syncthreads();
        if (i < n && !(m_i & LM_EQ) && !(sl & RL_HDR)) {
            u32 have; u64 b1, b2;
            const u32 j = rm_run_combine(p, ws, n, i0, i, sl, k1, k2, s_meta, s_stat, s_k1, s_k2, have, b1, b2);
            bool keep = false;
            if (j >= n && !final_win) ;                                  // undecided
            else if ((have & (RL_OK1 | RL_OK2)) == (RL_OK1 | RL_OK2)) {
                const u64 key = (b1 << (2 * p.rm_klen2)) | b2, me = g0 + i;
                const u32 tag = (have & RL_TAG) ? 1u : 0u;
                unsigned long long old = 0; bool claimed = false, full = false;
                if (key == RM_EMPTY) { old = atomicMin(&st->rm_allones[tag], (unsigned long long)me); claimed = old == RM_EMPTY; }
                else {
                    const u64 s = rm_slot(p.rm_tab[tag], p.rm_mask[tag], key, claimed);
                    if (s == ~0ull) { atomicOr(&st->err, S2P_ERR_RMTABLE); full = true; }
                    else old = atomicMin(&p.rm_tab[tag][2 * s + 1], (unsigned long long)me);
                }
                if (!full) {
                    keep = old >= me;                                    // RM_EMPTY (all ones) included
                    if (old != RM_EMPTY && old > me && old - g0 < n) rm_drop_run(p, (u32)(old - g0), n);
                    if (claimed) ++c_uniq;
                    if (me >= counted) ++c_tot;
                }
            } else if (g0 + i >= counted) { ++c_tot; ++c_disc; }
            if (!keep) rm_drop_run(p, i, n);
        }
    }
    c_tot = __reduce_add_sync(0xFFFFFFFFu, c_tot); c_uniq = __reduce_add_sync(0xFFFFFFFFu, c_uniq); c_disc = __reduce_add_sync(0xFFFFFFFFu, c_disc);
    if ((threadIdx.x & 31u) == 0) {
        if (c_tot) atomicAdd(&st->rm_total, (unsigned long long)c_tot);
        if (c_uniq) atomicAdd(&st->rm_uniq, (unsigned long long)c_uniq);
        if (c_disc) atomicAdd(&st->rm_discard, (unsigned long long)c_disc);
    }
}

// ---- the same rule over several ranks (mk_s2p_rmdup_*).  Shard line index = global line index of the single-GPU kernels.
// A record is {key, ord}, ord = tag << 63 | rank << 40 | line of the run head: the smallest ord of a (tag, key) is the
// first occurrence in (rank, line) order.  The rank is stamped by the exchange on the way to the key's owner.
#define RK_KEYS 0      /* rk_cnt[]: records written from the front of rk_rec */
#define RK_DISC 1      /* discarded run heads written from the back */
#define RK_FP1 2       /* fingerprint of pass 1's run heads */
#define RK_FP2 3       /* the same over pass 2's run heads below rk_lines */
#define RK_UNIQ 4      /* owner: (tag, key) segments */
#define RK_DUP 5       /* owner: records after a segment's first */
#define RK_LOSE 6      /* owner: the losers' part (end, count) for the way back: 6, 7 */
#define RK_BAD 8       /* receive: losers that name another rank or a line past pass 1 */
#define RK_N 9
#define RK_LINE_MASK ((1ull << 40) - 1)
// what pass 2 must see again at a run head: its line index and the line's first bytes
static __device__ __forceinline__ unsigned long long rk_fp(const S2PParams &p, u64 ws, u32 i, u64 me) {
    const u64 a = ws + (i ? (u64)p.nl_pos[i - 1] + 1 : 0);
    const u32 len = p.nl_pos[i] - (u32)(a - ws);
    GlobalFetch gf; gf.buf = p.buf; gf.A = 0;
    u64 x = fetch8(gf, a);
    if (len < 8) x &= (1ull << (8 * len)) - 1;
    return rm_hash(x ^ rm_hash(me + 1));
}

// Pass 1: one record per run head that the single-GPU kernel would settle (same staging, same run rule); a discarded run
// (short mate, non-ACGT key base, no primary record for a mate) only leaves its line index, at the back.
static __global__ void __launch_bounds__(256) k_rm_keys(S2PParams p) {
    __shared__ unsigned long long s_k1[256], s_k2[256];
    __shared__ u8 s_stat[256], s_meta[256];
    WinState *st = p.st;
    const u32 n = st->n_lines;
    const u64 ws = st->ws, g0 = st->lines_done, counted = st->rm_counted;
    const bool final_win = (st->we == st->total) && st->is_last;
    const u32 tid = threadIdx.x, lane = tid & 31u;
    unsigned long long fp = 0;
    for (u32 i0 = blockIdx.x * 256u; i0 < n; i0 += gridDim.x * 256u) {
        const u32 i = i0 + tid;
        u32 m_i = 0, sl = 0; u64 k1 = 0, k2 = 0;
        if (i < n) { m_i = p.lmeta[i]; rm_line_keys(p, ws, i, sl, k1, k2); }
        __syncthreads();
        s_meta[tid] = (u8)m_i; s_stat[tid] = (u8)sl; s_k1[tid] = k1; s_k2[tid] = k2;
        __syncthreads();
        bool is_key = false, is_disc = false;
        uint4 rec = make_uint4(0, 0, 0, 0);
        const u64 me = g0 + i;
        if (i < n && !(m_i & LM_EQ) && !(sl & RL_HDR)) {
            u32 have; u64 b1, b2;
            const u32 j = rm_run_combine(p, ws, n, i0, i, sl, k1, k2, s_meta, s_stat, s_k1, s_k2, have, b1, b2);
            if ((j < n || final_win) && me >= counted) {                // settled here, and not in an earlier window
                const u64 ord = ((have & RL_TAG) ? 1ull << 63 : 0ull) | me;
                if ((have & (RL_OK1 | RL_OK2)) == (RL_OK1 | RL_OK2)) {
                    const u64 key = (b1 << (2 * p.rm_klen2)) | b2;
                    rec = make_uint4((u32)key, (u32)(key >> 32), (u32)ord, (u32)(ord >> 32));
                    is_key = true;
                } else { rec = make_uint4(0, 0, (u32)me, (u32)(me >> 32)); is_disc = true; }
                fp += rk_fp(p, ws, i, me);
            }
        }
        // one reservation per warp and kind
        const u32 bk = __ballot_sync(0xFFFFFFFFu, is_key), bd = __ballot_sync(0xFFFFFFFFu, is_disc);
        unsigned long long base_k = 0, base_d = 0;
        if (lane == 0 && bk) base_k = atomicAdd(&p.rk_cnt[RK_KEYS], (unsigned long long)__popc(bk));
        if (lane == 0 && bd) base_d = atomicAdd(&p.rk_cnt[RK_DISC], (unsigned long long)__popc(bd));
        base_k = __shfl_sync(0xFFFFFFFFu, base_k, 0); base_d = __shfl_sync(0xFFFFFFFFu, base_d, 0);
        const u32 below = (1u << lane) - 1u;
        if (is_key) { const u64 k = base_k + __popc(bk & below); if (k < p.rk_cap) p.rk_rec[k] = rec; }
        if (is_disc) { const u64 d = base_d + __popc(bd & below); if (d < p.rk_cap) p.rk_rec[p.rk_cap - 1 - d] = rec; }
    }
    for (int o = 16; o; o >>= 1) fp += __shfl_xor_sync(0xFFFFFFFFu, fp, o);
    if (lane == 0 && fp) atomicAdd(&p.rk_cnt[RK_FP1], fp);
}

// Pass 2, in place of k_rm_insert: a run loses LM_KEEP when its head's drop bit is set, or when the window end cuts it (it
// is seen again in the next window, as in k_rm_insert).  Lines from rk_lines on belong to no settled run (the shard-boundary
// group appended behind the shard) and are kept.
static __global__ void __launch_bounds__(256) k_rm_apply(S2PParams p) {
    const WinState *st = p.st;
    const u32 n = st->n_lines;
    const u64 ws = st->ws, g0 = st->lines_done, counted = st->rm_counted;
    const bool final_win = (st->we == st->total) && st->is_last;
    unsigned long long fp = 0;
    for (u32 i = blockIdx.x * 256u + threadIdx.x; i < n; i += gridDim.x * 256u) {
        if (p.lmeta[i] & LM_EQ) continue;
        if (p.buf[ws + (i ? (u64)p.nl_pos[i - 1] + 1 : 0)] == '@') continue;   // a header line is no run (RL_HDR)
        u32 j = i + 1;
        while (j < n && (p.lmeta[j] & LM_EQ)) ++j;
        const u64 me = g0 + i;
        bool drop = false;
        if (j >= n && !final_win) drop = true;
        else if (me < p.rk_lines) {
            drop = (p.rk_drop[me >> 5] >> (me & 31u)) & 1u;
            if (me >= counted) fp += rk_fp(p, ws, i, me);
        }
        if (drop) rm_drop_run(p, i, n);
    }
    for (int o = 16; o; o >>= 1) fp += __shfl_xor_sync(0xFFFFFFFFu, fp, o);
    if ((threadIdx.x & 31u) == 0 && fp) atomicAdd(&p.rk_cnt[RK_FP2], fp);
}

// Owner: the received records sorted by (tag, key, ord).  The first of each (tag, key) segment is the first occurrence;
// every other one is a loser and goes back to its rank.
static __global__ void __launch_bounds__(256) k_rm_decide(const uint4 *b0, const uint4 *b1, const unsigned *final_buf, u64 n, uint4 *lose,
                                                          unsigned long long *cnt) {
    const uint4 *r = *final_buf ? b1 : b0;
    const u32 lane = threadIdx.x & 31u;
    u32 c_uniq = 0, c_dup = 0;
    const u64 n_round = (n + 31) & ~(u64)31;
    for (u64 i = (u64)blockIdx.x * 256u + threadIdx.x; i < n_round; i += (u64)gridDim.x * 256u) {
        bool loser = false;
        uint4 x = make_uint4(0, 0, 0, 0);
        if (i < n) {
            x = r[i];
            if (i > 0) { const uint4 y = r[i - 1]; loser = x.x == y.x && x.y == y.y && (x.w >> 31) == (y.w >> 31); }
            if (loser) ++c_dup; else ++c_uniq;
        }
        const u32 b = __ballot_sync(0xFFFFFFFFu, loser);
        unsigned long long base = 0;
        if (lane == 0 && b) { base = atomicAdd(&cnt[RK_LOSE], (unsigned long long)__popc(b)); atomicAdd(&cnt[RK_LOSE + 1], (unsigned long long)__popc(b)); }
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (loser) lose[base + __popc(b & ((1u << lane) - 1u))] = x;
    }
    c_uniq = __reduce_add_sync(0xFFFFFFFFu, c_uniq); c_dup = __reduce_add_sync(0xFFFFFFFFu, c_dup);
    if (lane == 0) { if (c_uniq) atomicAdd(&cnt[RK_UNIQ], (unsigned long long)c_uniq); if (c_dup) atomicAdd(&cnt[RK_DUP], (unsigned long long)c_dup); }
}

// Origin: the drop bit of every run head in `rec` (losers back from the owners, or this rank's own discards)
static __global__ void __launch_bounds__(256) k_rm_settle(const uint4 *rec, u64 n, u32 rank, int check_rank, u64 lines, u32 *drop,
                                                          unsigned long long *cnt) {
    for (u64 i = (u64)blockIdx.x * 256u + threadIdx.x; i < n; i += (u64)gridDim.x * 256u) {
        const uint4 x = rec[i];
        const u64 ord = (u64)x.w << 32 | x.z, line = ord & RK_LINE_MASK;
        if (line >= lines || (check_rank && ((ord >> 40) & 63u) != rank)) { atomicAdd(&cnt[RK_BAD], 1ull); continue; }
        atomicOr(&drop[line >> 5], 1u << (line & 31u));
    }
}

// EQ of line q: its QNAME equals line q-1's (evaluated by K2)
__device__ __forceinline__ bool line_eq(const S2PParams &, u64, u32, u32 mq) { return (mq & LM_EQ) != 0; }
__device__ __forceinline__ u32 line_len_of(const S2PParams &p, u32 q) { return p.nl_pos[q] - (q ? p.nl_pos[q - 1] + 1 : 0); }

// bytewise order of two chromosome names (std::string::compare)
static __device__ __noinline__ int chr_name_cmp_slow(const ChrSlot *a, const ChrSlot *b) {
    u32 la = a->len, lb = b->len, m = la < lb ? la : lb;
    for (u32 i = 0; i < m; ++i) {
        int d = (int)(u8)a->name[i] - (int)(u8)b->name[i];
        if (d) return d;
    }
    return la < lb ? -1 : (la > lb ? 1 : 0);
}
// names of up to 8 bytes (name8 = the bytes, little endian, zero padded) compare as big-endian integers
__device__ __forceinline__ int chr_name_cmp(const S2PParams &p, u16 sa, u16 sb) {
    if (sa == sb) return 0;
    const ChrSlot *a = &p.chr[sa], *b = &p.chr[sb];
    if (a->len <= 8 && b->len <= 8) {
        const u64 x = a->name8, y = b->name8;
        const u32 xh = __byte_perm((u32)x, 0, 0x0123), xl = __byte_perm((u32)(x >> 32), 0, 0x0123);
        const u32 yh = __byte_perm((u32)y, 0, 0x0123), yl = __byte_perm((u32)(y >> 32), 0, 0x0123);
        return xh != yh ? (xh < yh ? -1 : 1) : (xl != yl ? (xl < yl ? -1 : 1) : 0);   // zero padding: a proper prefix sorts first
    }
    return chr_name_cmp_slow(a, b);
}

__device__ __forceinline__ u32 dec_digits(u32 v) {
    return v >= 1000000000u ? 10 : v >= 100000000u ? 9 : v >= 10000000u ? 8 : v >= 1000000u ? 7 : v >= 100000u ? 6 :
           v >= 10000u ? 5 : v >= 1000u ? 4 : v >= 100u ? 3 : v >= 10u ? 2 : 1;
}

// Resolution of one read group from the records of its kept lines (flash2pairs.h:25-154, unc2pairs.h:29-358): n kept records,
// n1 / n2 of them flagged first / second in pair; f0, f1 = the first two kept records, a1, b1 / a2, b2 = the first two R1 / R2
// records (pointers beyond the counts are never dereferenced).  Shared by the multi-kernel path and the single-pass tile path.
struct Resolved { u32 p1, p2; u16 sA, sB; u8 status, strands; bool have; };
template <class RT>
__device__ __forceinline__ Resolved resolve_group(const S2PParams &p, u32 n, u32 n1, u32 n2, const RT *f0, const RT *f1,
                                                  const RT *a1, const RT *b1, const RT *a2, const RT *b2) {
    Resolved o; o.p1 = o.p2 = 0; o.sA = o.sB = 0; o.status = ST_NONE; o.strands = 0; o.have = false;
    u32 p1 = 0, p2 = 0; u16 c1 = 0, c2 = 0; bool m1 = false, m2 = false; bool have = false, ordered = false;
    const float ratio = p.ratio;
    if (p.mode == 0) {                   // flash2pairs.h:25-154
        if (n == 1) {
            Seg a = seg_of(*f0);
            if (a.segCnt == 0) o.status = ST_CIGARERR;
            else if (a.segCnt > 2) o.status = ST_MANYHITS;
            else if (!integrity1(a, ratio)) o.status = ST_LOWMAP;
            else {
                p1 = a.pos; p2 = a.segCnt == 2 ? a.right1 : a.right0;
                u32 d = p2 - p1;
                o.status = d >= 10000u ? ST_CIS10K : (d >= 1000u ? ST_CIS1K : ST_CIS0);
                c1 = c2 = a.chr; m1 = false; m2 = true; have = true; ordered = true;   // always "+ -", never swapped
            }
        } else if (n == 2) {
            Seg a = seg_of(*f0), b = seg_of(*f1);
            if (a.segCnt == 0 || b.segCnt == 0) o.status = ST_CIGARERR;
            else if (a.segCnt != 1 || b.segCnt != 1) o.status = ST_MANYHITS;
            else if (!integrity2(a, b, ratio)) o.status = ST_LOWMAP;
            else {
                p1 = (int)a.leftClip > (int)a.rightClip ? a.right0 : a.pos;
                p2 = (int)b.leftClip > (int)b.rightClip ? b.right0 : b.pos;
                c1 = a.chr; c2 = b.chr; m1 = a.minus; m2 = b.minus; have = true;
            }
        } else o.status = ST_MANYHITS;
    } else {                             // unc2pairs.h:29-358
        if (n1 == 0 || n2 == 0 || n1 + n2 > 3) o.status = ST_NONE;        // silent drops, unc2pairs.h:52-59
        else if (n1 == 1 && n2 == 1) {
            Seg a = seg_of(*a1), b = seg_of(*a2);
            if (a.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity1(a, ratio)) o.status = ST_LOWMAP;
            else if (b.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity1(b, ratio)) o.status = ST_LOWMAP;
            else if (a.segCnt + b.segCnt > 3) o.status = ST_MANYHITS;
            else {
                c1 = a.chr; c2 = b.chr; m1 = a.minus; m2 = b.minus; have = true;
                if (a.segCnt == 1 && b.segCnt == 1) {
                    p1 = a.minus ? a.right0 : a.pos; p2 = b.minus ? b.right0 : b.pos;
                } else if (a.segCnt == 2) {                                   // unc2pairs.h:146-167
                    if (!a.minus) {
                        if (b.minus && a.chr == b.chr && (int)a.left1 < (int)b.pos && (int)b.right0 - (int)a.left1 <= 1000) { p1 = a.pos; p2 = b.right0; }
                        else { o.status = ST_UNPAIRED; have = false; }
                    } else {
                        if (!b.minus && a.chr == b.chr && (int)b.pos < (int)a.pos && (int)a.right0 - (int)b.pos <= 1000) { p1 = a.right1; p2 = b.pos; }
                        else { o.status = ST_UNPAIRED; have = false; }
                    }
                } else {                                                      // unc2pairs.h:168-189
                    if (!a.minus) {
                        if (b.minus && a.chr == b.chr && (int)a.pos < (int)b.pos && (int)b.right0 - (int)a.pos <= 1000) { p1 = a.pos; p2 = b.right1; }
                        else { o.status = ST_UNPAIRED; have = false; }
                    } else {
                        if (!b.minus && a.chr == b.chr && (int)b.left1 < (int)a.pos && (int)a.right0 - (int)b.left1 <= 1000) { p1 = a.right0; p2 = b.pos; }
                        else { o.status = ST_UNPAIRED; have = false; }
                    }
                }
            }
        } else if (n1 == 1) {            // 1 + 2
            Seg a = seg_of(*a1), b = seg_of(*a2), c = seg_of(*b2);
            if (a.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity1(a, ratio)) o.status = ST_LOWMAP;
            else if (b.segCnt == 0 || c.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity2(b, c, ratio)) o.status = ST_LOWMAP;
            else if (a.segCnt != 1 || b.segCnt != 1 || c.segCnt != 1) o.status = ST_MANYHITS;
            else {
                c1 = a.chr; m1 = a.minus; p1 = a.minus ? a.right0 : a.pos;
                if (mates(a, b)) { c2 = c.chr; m2 = c.minus; p2 = distal_end(c); have = true; }
                else if (mates(a, c)) { c2 = b.chr; m2 = b.minus; p2 = distal_end(b); have = true; }
                else o.status = ST_UNPAIRED;
            }
        } else {                         // 2 + 1
            Seg a = seg_of(*a1), b = seg_of(*b1), c = seg_of(*a2);
            if (a.segCnt == 0 || b.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity2(a, b, ratio)) o.status = ST_LOWMAP;
            else if (c.segCnt == 0) o.status = ST_CIGARERR;
            else if (!integrity1(c, ratio)) o.status = ST_LOWMAP;
            else if (a.segCnt != 1 || b.segCnt != 1 || c.segCnt != 1) o.status = ST_MANYHITS;
            else {
                c2 = c.chr; m2 = c.minus; p2 = c.minus ? c.right0 : c.pos;
                if (mates(c, a)) { c1 = b.chr; m1 = b.minus; p1 = distal_end(b); have = true; }
                else if (mates(c, b)) { c1 = a.chr; m1 = a.minus; p1 = distal_end(a); have = true; }
                else o.status = ST_UNPAIRED;
            }
        }
    }
    if (have) {
        u16 sA = c1, sB = c2;
        if (!ordered) {                  // unc2pairs.h:310-348
            int cc = chr_name_cmp(p, c1, c2);
            if (!(cc < 0 || (cc == 0 && p1 < p2))) {
                u32 t = p1; p1 = p2; p2 = t; sA = c2; sB = c1; bool tm = m1; m1 = m2; m2 = tm;
            }
            if (cc == 0) {
                u32 d = p2 - p1;
                o.status = d <= 10u ? ST_SELFCIRCLE : (d >= 10000u ? ST_CIS10K : (d >= 1000u ? ST_CIS1K : ST_CIS0));
            } else o.status = ST_TRANS;
        }
        o.p1 = p1; o.p2 = p2; o.sA = sA; o.sB = sB; o.strands = (u8)((m1 ? 1 : 0) | (m2 ? 2 : 0)); o.have = true;
    }
    return o;
}

#define EMIT_THREADS 256
#define EMIT_ITEMS 1
#define EMIT_TILE (EMIT_THREADS * EMIT_ITEMS)
#define EMIT_STAGE 20480
#define GROUP_CHUNK 2048u

// A warp takes 128 consecutive lines.  Their KEEP / EQ flags (and those of the lines around them) are gathered with five
// coalesced byte loads per lane and ten ballots; from the masks every lane classifies its four lines by bit arithmetic: not a
// group head, head of a group of exactly 1 / 2 / 3 consecutive kept lines whose neighbours are kept too (the common case), or
// "needs the general walk" (dropped lines inside or next to the group, more than three records, the window's last group).
// The heads are then COMPACTED by class into per-warp lists and resolved class by class, 32 at a time: all lanes of a batch
// run the same case of the reference's analysis.  ncu on the one-thread-per-line version: 8.8, then (after the masks) 11 of
// 32 lanes active per instruction — a single-record group, a two-record group and a non-head line in neighbouring lanes
// serialise three code paths.  The general walk below is the definition; the fast classes are shortcuts to its result.
struct GroupSums { u32 vA, vT, vS; };
__device__ __forceinline__ void group_finish(const S2PParams &p, u32 i, u32 mi, u32 n, u32 n1, u32 n2, const u32 *first, const u32 *r1, const u32 *r2,
                                             u32 sam_len, u32 prev, u32 *s_cnt, GroupSums &sum) {
    GroupRes g; g.posA = g.posB = 0; g.chrA = g.chrB = 0; g.strands = 0;
    {
        const LineRec *rp = &p.rec[prev];
        g.rid_len = rp->qname_len; g.rid_off = (prev ? p.nl_pos[prev - 1] + 1 : 0) + rp->qname_off;
    }
    g.last_line = prev; g.text_len = 0; g.sam_len = sam_len;
    const Resolved rs = resolve_group(p, n, n1, n2, &p.rec[first[0]], &p.rec[first[1]], &p.rec[r1[0]], &p.rec[r1[1]], &p.rec[r2[0]], &p.rec[r2[1]]);
    g.status = rs.status;
    u32 meta = mi | LM_HEAD | LM_PROC;
    if (rs.have) {
        g.posA = rs.p1; g.posB = rs.p2; g.strands = rs.strands;
        const ChrSlot *ca = &p.chr[rs.sA], *cb = &p.chr[rs.sB];
        g.chrA = (u16)ca->id; g.chrB = (u16)cb->id;
        if (g.status != ST_SELFCIRCLE) {
            meta |= LM_EMIT;
            g.text_len = (u32)g.rid_len + ca->len + cb->len + dec_digits(rs.p1) + dec_digits(rs.p2) + 9u;
        }
    }
    if (!(meta & LM_EMIT)) g.sam_len = 0;
    if (g.status != ST_NONE) atomicAdd(&s_cnt[g.status], 1u);
    p.res[i] = g;
    p.lmeta[i] = (u8)meta;
    sum.vA += 1u | ((meta & LM_EMIT) ? 1u << 16 : 0u);
    if (meta & LM_EMIT) { sum.vT += g.text_len; if (p.write_sam) sum.vS += g.sam_len; }
}

// bits [32 r + b, 32 r + b + 32) of a 160-bit mask held in five words, r a compile-time constant and b in [0, 34): only
// static register indices (a dynamically indexed array would live in local memory)
template <u32 R>
__device__ __forceinline__ u32 mask_window(const u32 (&w)[5], u32 b) {
    const u32 w2 = R + 2 < 5 ? w[R + 2 < 5 ? R + 2 : 4] : 0u;
    return b < 32u ? __funnelshift_r(w[R], w[R + 1], b) : __funnelshift_r(w[R + 1], w2, b - 32u);
}

#define GROUP_WARP_LINES 128u
#ifndef GROUP_OCC
#define GROUP_OCC 6
#endif
static __global__ void __launch_bounds__(256, GROUP_OCC) k_group(S2PParams p) {
    __shared__ u32 s_cnt[ST_NCOUNTER];
    __shared__ u8 s_list[8][4][GROUP_WARP_LINES];                    // per warp, per class: offsets (0..127) of the heads inside the warp's chunk
    __shared__ u32 s_chunk;
    WinState *st = p.st;
    if (threadIdx.x < ST_NCOUNTER) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u32 n_lines = st->n_lines;
    const u64 ws = st->ws;
    const u32 lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    const u32 lt = (1u << lane) - 1u;
    // CTAs claim chunks of GROUP_CHUNK lines with a ticket: groups cost very different amounts of work, and with a static split
    // the kernel's last 10 % were CTAs waiting for their slowest warp
    while (true) {
      if (threadIdx.x == 0) s_chunk = atomicAdd(&st->tickets[1], 1u);
      __syncthreads();
      const u32 chunk0 = s_chunk * GROUP_CHUNK;
      __syncthreads();
      if (chunk0 >= n_lines) break;
      for (u32 B = chunk0 + wid * GROUP_WARP_LINES; B < chunk0 + GROUP_CHUNK && B < n_lines; B += 8u * GROUP_WARP_LINES) {
        // ---- masks: bit j <-> line B - 1 + j, j in [0, 160)
        u32 keepw[5], eqw[5];
#pragma unroll
        for (u32 k = 0; k < 5; ++k) {
            const u32 q = B + 32u * k + lane;                          // line q - 1 (q = 0 only for the window's very first slot)
            const u32 m = (q >= 1u && q - 1u < n_lines) ? p.lmeta[q - 1u] : 0u;
            keepw[k] = __ballot_sync(0xFFFFFFFFu, m & LM_KEEP);
            eqw[k] = __ballot_sync(0xFFFFFFFFu, m & LM_EQ);
        }
        // ---- classify this lane's four lines, compact the heads by class (list entry: offset | EQ flag << 7)
        u32 cnt[4] = {0, 0, 0, 0};
        auto classify = [&](auto rc) {
            constexpr u32 r = decltype(rc)::value;
            const u32 off = lane + 32u * r, i = B + off;               // this line's bit is 32 r + lane + 1
            const u32 self = mask_window<r>(keepw, lane + 1u), eq_self = mask_window<r>(eqw, lane + 1u);   // KEEP / EQ from this line on
            u32 cls = 0xFFu;                                            // none
            if (i < n_lines && (self & 1u)) {
                const bool prev_kept = i == 0 || ((keepw[r] >> lane) & 1u);
                if (!prev_kept) cls = 3;                                // general walk decides whether it is a head
                else if (i != 0 && (eq_self & 1u)) cls = 0xFFu;         // same read id as the kept line before it: not a head
                else {
                    const u32 after_eq = mask_window<r>(eqw, lane + 2u);   // EQ of the following lines
                    const u32 gn = (u32)__ffs((int)~after_eq);          // group size: 1 + consecutive lines with this read id behind the head
                    const u32 need = (2u << (gn & 31u)) - 1u;           // the members and the terminating line must all be kept
                    cls = (after_eq != 0xFFFFFFFFu && gn <= 3u && (self & need) == need) ? gn - 1u : 3u;
                }
            }
#pragma unroll
            for (u32 t = 0; t < 4; ++t) {
                const u32 bal = __ballot_sync(0xFFFFFFFFu, cls == t);
                if (cls == t) s_list[wid][t][cnt[t] + __popc(bal & lt)] = (u8)(off | ((eq_self & 1u) << 7));
                cnt[t] += __popc(bal);
            }
        };
        classify(std::integral_constant<u32, 0>{}); classify(std::integral_constant<u32, 1>{});
        classify(std::integral_constant<u32, 2>{}); classify(std::integral_constant<u32, 3>{});
        __syncwarp();
        GroupSums sum; sum.vA = sum.vT = sum.vS = 0;
        // ---- classes 0..2: groups of gn = 1, 2, 3 consecutive kept lines, resolved 32 at a time
#pragma unroll 1
        for (u32 t = 0; t < 3; ++t) {
            const u32 gn = t + 1u;
            for (u32 b0 = 0; b0 < cnt[t]; b0 += 32u) {
                if (b0 + lane >= cnt[t]) continue;
                const u32 ent = s_list[wid][t][b0 + lane], i = B + (ent & 127u);
                const u32 mi = LM_KEEP | ((ent & 128u) ? LM_EQ : 0u);
                u32 first[2] = {i, i + 1u}, r1[2] = {0, 0}, r2[2] = {0, 0}, n1 = 0, n2 = 0;
                u32 fl[3];
#pragma unroll
                for (u32 k = 0; k < 3; ++k) fl[k] = k < gn ? p.rec[i + k].flag : 0u;
#pragma unroll
                for (u32 k = 0; k < 3; ++k) {
                    if (k < gn) { if (fl[k] & 64u) { if (n1 < 2) r1[n1] = i + k; ++n1; } else if (fl[k] & 128u) { if (n2 < 2) r2[n2] = i + k; ++n2; } }
                }
                const u32 prev = i + gn - 1u;
                const u32 sam_len = p.nl_pos[prev] + 1u - (i ? p.nl_pos[i - 1] + 1u : 0u);   // consecutive lines: one span
                group_finish(p, i, mi, gn, n1, n2, first, r1, r2, sam_len, prev, s_cnt, sum);
            }
        }
        // ---- class 3: the general walk (pairutil.h:163-173: currId != lastId among kept records)
        for (u32 b0 = 0; b0 < cnt[3]; b0 += 32u) {
            if (b0 + lane >= cnt[3]) continue;
            const u32 ent = s_list[wid][3][b0 + lane], i = B + (ent & 127u);
            const u32 mi = LM_KEEP | ((ent & 128u) ? LM_EQ : 0u);
            bool head;
            {
                bool chain = line_eq(p, ws, i, mi);
                long jj = (long)i - 1;
                while (jj >= 0) { u32 mj = p.lmeta[jj]; if (mj & LM_KEEP) break; chain = chain && line_eq(p, ws, (u32)jj, mj); --jj; }
                if (jj < 0) head = true;
                else if (chain) head = false;
                else if (jj == (long)i - 1) head = true;
                else head = !qname_equal_slow(p, ws, i, (u32)jj);
            }
            if (!head) continue;
            // collect the group's kept records
            u32 first[2] = {i, 0}, r1[2] = {0, 0}, r2[2] = {0, 0};
            u32 n = 0, n1 = 0, n2 = 0, sam_len = 0, prev = i;
            u32 k = i;
            bool chain = true, off_end = false;
            while (true) {
                const LineRec *rk = &p.rec[k];                          // k is a member
                u32 fl = rk->flag;
                if (n < 2) first[n] = k;
                ++n;
                if (fl & 64u) { if (n1 < 2) r1[n1] = k; ++n1; } else if (fl & 128u) { if (n2 < 2) r2[n2] = k; ++n2; }
                sam_len += line_len_of(p, k) + 1;
                prev = k;
                u32 q = k + 1; chain = true;                            // next kept line
                while (q < n_lines) { u32 mq = p.lmeta[q]; chain = chain && line_eq(p, ws, q, mq); if (mq & LM_KEEP) break; ++q; }
                if (q >= n_lines) { off_end = true; break; }
                bool same = chain ? true : (q == prev + 1 ? false : qname_equal_slow(p, ws, q, prev));
                if (!same) break;
                k = q;
            }
            if (off_end) {                       // the window's last group: carried to the next window (or dropped at EOF)
                st->carry_line = i;
                p.lmeta[i] = (u8)(mi | LM_HEAD);
                continue;
            }
            group_finish(p, i, mi, n, n1, n2, first, r1, r2, sam_len, prev, s_cnt, sum);
        }
        __syncwarp();                                                  // the lists are rewritten by the warp's next chunk
        // sizes per EMIT_TILE lines for K4 (the warp's 128 lines lie in one 256-line tile): one reduction per warp
        const u32 vA = __reduce_add_sync(0xFFFFFFFFu, sum.vA), vT = __reduce_add_sync(0xFFFFFFFFu, sum.vT), vS = __reduce_add_sync(0xFFFFFFFFu, sum.vS);
        if (lane == 0 && vA) {
            u32 *tt = (u32 *)&p.tile_tot[B / EMIT_TILE];
            atomicAdd(tt, vA);
            if (vT) atomicAdd(tt + 1, vT);
            if (vS) atomicAdd(tt + 2, vS);
            u32 *sg = (u32 *)&p.seg_tot[B / (EMIT_TILE * 128u)];         // EMIT_SEG tiles per segment (k_emit_prefix)
            atomicAdd(sg, vA & 0xFFFFu); atomicAdd(sg + 1, vA >> 16);
            if (vT) atomicAdd(sg + 2, vT);
            if (vS) atomicAdd(sg + 3, vS);
        }
      }
    }
    __syncthreads();
    if (threadIdx.x < ST_NCOUNTER && s_cnt[threadIdx.x]) atomicAdd(&st->counters[threadIdx.x], (unsigned long long)s_cnt[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------ K4: emit

__device__ __forceinline__ u32 put_uint(char *dst, u32 v) {
    u32 n = dec_digits(v);
    for (int i = (int)n - 1; i >= 0; --i) { dst[i] = (char)('0' + v % 10u); v /= 10u; }
    return n;
}

// rid \t chrA \t posA \t chrB \t posB \t sA \t sB \n   (unc2pairs.h:327-347)
__device__ __forceinline__ char *put_bytes8(char *out, u64 x, u32 n) {       // the low n (<= 8) bytes of x
#pragma unroll
    for (int b = 0; b < 8; ++b) if ((u32)b < n) out[b] = (char)(x >> (8 * b));
    return out + n;
}
__device__ __forceinline__ char *put_name(char *out, const ChrSlot *c) {
    const u32 l = c->len;
    if (l <= 8) return put_bytes8(out, c->name8, l);
    for (u32 i = 0; i < l; ++i) out[i] = c->name[i];
    return out + l;
}
struct RidInfo { u64 abs; u32 len; };                                          // where the group's read id sits in the SAM text
__device__ __forceinline__ RidInfo rid_info(const S2PParams &p, u64 ws, const GroupRes &g) {
    RidInfo r; r.len = g.rid_len; r.abs = ws + g.rid_off;
    return r;
}
__device__ __forceinline__ void write_pair_line_slots(const S2PParams &p, const RidInfo &rid, const ChrSlot *ca, const ChrSlot *cb,
                                                      u32 posA, u32 posB, u32 strands, char *out) {
    GlobalFetch gf; gf.buf = p.buf; gf.A = 0;
    for (u32 k = 0; k < rid.len; k += 8) { const u32 n = rid.len - k < 8 ? rid.len - k : 8; out = put_bytes8(out, fetch8(gf, rid.abs + k), n); }
    *out++ = '\t';
    out = put_name(out, ca);
    *out++ = '\t';
    out += put_uint(out, posA);
    *out++ = '\t';
    out = put_name(out, cb);
    *out++ = '\t';
    out += put_uint(out, posB);
    *out++ = '\t'; *out++ = (strands & 1) ? '-' : '+'; *out++ = '\t'; *out++ = (strands & 2) ? '-' : '+'; *out++ = '\n';
}
__device__ __forceinline__ void write_pair_line(const S2PParams &p, const RidInfo &rid, const GroupRes &g, char *out) {
    write_pair_line_slots(p, rid, &p.chr[p.id_to_slot[g.chrA]], &p.chr[p.id_to_slot[g.chrB]], g.posA, g.posB, g.strands, out);
}

// ---------------------------------------------------------------------------------------------- lean text writer
// A line is a sequence of pieces of at most four bytes.  They are collected in a 64-bit accumulator and OR-ed into the
// (zeroed) shared-memory stage as aligned 32-bit words: the first and last word of a line are shared with the neighbouring
// lines, which other lanes write, and OR makes that safe without any byte-level special case.
// (red.shared on a 32-bit shared address: a generic-pointer atomicOr compiles to the slow generic ATOM path)
__device__ __forceinline__ void sts_or(u32 saddr, u32 v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }
struct TextW { u32 w; u32 lo, hi, fill; };                            // w: shared-memory byte address of the current word
__device__ __forceinline__ void tw_init(TextW &t, char *dst) {
    const u32 sa = smem_u32(dst);
    t.w = sa & ~3u; t.fill = sa & 3u; t.lo = t.hi = 0;
}
__device__ __forceinline__ void tw_put(TextW &t, u32 x, u32 n) {     // the low n (0..4) bytes of x; the bytes above them must be zero
    const u32 sh = t.fill * 8u;
    t.lo |= x << sh; t.hi |= __funnelshift_l(x, 0u, sh);
    t.fill += n;
    if (t.fill >= 4u) { sts_or(t.w, t.lo); t.w += 4u; t.lo = t.hi; t.hi = 0; t.fill -= 4u; }
}
__device__ __forceinline__ void tw_end(TextW &t) { if (t.fill) sts_or(t.w, t.lo); }
// four decimal digits of v (< 10000) as characters, most significant in the lowest byte
__device__ __forceinline__ u32 dig4(u32 v) {
    const u32 hi2 = (v * 5243u) >> 19, lo2 = v - hi2 * 100u;           // v / 100 for v < 10000
    const u32 a = (hi2 * 103u) >> 10, b = (lo2 * 103u) >> 10;          // x / 10 for x < 100
    return (a | ((hi2 - a * 10u) << 8) | (b << 16) | ((lo2 - b * 10u) << 24)) + 0x30303030u;
}
// the nd decimal characters of v, left-aligned in three words (first character in the lowest byte of d0)
__device__ __forceinline__ void dec_chars(u32 v, u32 nd, u32 &d0, u32 &d1, u32 &d2) {
    const u32 q1 = v / 10000u, r1 = v - q1 * 10000u, q2 = q1 / 10000u, r2 = q1 - q2 * 10000u;
    const u32 w0 = dig4(q2), w1 = dig4(r2), w2 = dig4(r1);             // "00dddddddddd": twelve characters, 12 - nd leading zeros
    const u32 k = 12u - nd, i = k >> 2, sh = (k & 3u) * 8u;
    const u32 a = i == 0 ? w0 : (i == 1 ? w1 : w2), b = i == 0 ? w1 : (i == 1 ? w2 : 0u), c = i == 0 ? w2 : 0u;
    d0 = __funnelshift_r(a, b, sh); d1 = __funnelshift_r(b, c, sh); d2 = c >> sh;
}
__device__ __forceinline__ u32 piece_len(u32 total, u32 j) { return total > 4u * j ? (total - 4u * j > 4u ? 4u : total - 4u * j) : 0u; }
// rid \t chrA \t posA \t chrB \t posB \t sA \t sB \n   (unc2pairs.h:327-347) into the zeroed stage; the read id comes back out of
// L2.  Chromosome names of up to 8 bytes (ChrSlot.name8); longer ones take the byte-wise writer.
__device__ __forceinline__ void fs_write_pair_line(const char *buf, u64 rid_abs, u32 rid_len, const ChrSlot *ca, const ChrSlot *cb,
                                                   u32 posA, u32 posB, u32 strands, char *out) {
    TextW t; tw_init(t, out);
    {
        // the first 48 bytes of the read id: seven aligned 8-byte loads issued together (they come from L2 or DRAM), then
        // realigned in registers; longer ids continue with one dependent load per 8 bytes
        const u64 a8 = rid_abs & ~(u64)7; const u32 sh = (u32)(rid_abs & 7u) * 8u;
        const u64 *src = (const u64 *)(buf + a8);
        const u32 span = rid_len + (sh >> 3);
        u64 r[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) r[j] = (u32)(8 * j) < span ? __ldg(src + j) : 0ull;
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            if ((u32)(8 * j) < rid_len) {
                const u64 x = sh ? (r[j] >> sh) | (r[j + 1] << (64u - sh)) : r[j];
                const u32 n = rid_len - 8u * j < 8u ? rid_len - 8u * j : 8u;
                u32 xl = (u32)x, xh = (u32)(x >> 32);
                if (n < 8u) { if (n <= 4u) { xh = 0; if (n < 4u) xl &= (1u << (8u * n)) - 1u; } else xh &= (1u << (8u * (n - 4u))) - 1u; }
                tw_put(t, xl, n < 4u ? n : 4u);
                tw_put(t, xh, n > 4u ? n - 4u : 0u);
            }
        }
        if (rid_len > 48u) {
            u64 cur = r[6];
#pragma unroll 1
            for (u32 k = 48; k < rid_len; k += 8) {
                const u64 nxt = __ldg(src + (k >> 3) + 1);
                const u64 x = sh ? (cur >> sh) | (nxt << (64u - sh)) : cur;
                cur = nxt;
                const u32 n = rid_len - k < 8u ? rid_len - k : 8u;
                u32 xl = (u32)x, xh = (u32)(x >> 32);
                if (n < 8u) { if (n <= 4u) { xh = 0; if (n < 4u) xl &= (1u << (8u * n)) - 1u; } else xh &= (1u << (8u * (n - 4u))) - 1u; }
                tw_put(t, xl, n < 4u ? n : 4u);
                tw_put(t, xh, n > 4u ? n - 4u : 0u);
            }
        }
    }
    // the fourteen pieces behind the read id, through ONE tw_put site (code size)
    const u32 la = ca->len, lb = cb->len;
    const u64 na = ca->name8, nb = cb->name8;
    const u32 nda = dec_digits(posA), ndb = dec_digits(posB);
    u32 a0, a1, a2, b0, b1, b2;
    dec_chars(posA, nda, a0, a1, a2); dec_chars(posB, ndb, b0, b1, b2);
    // "\t" name "\t" as up to ten bytes in three words
    const u64 ta = (u64)'\t' | (na << 8) | (la < 7u ? (u64)'\t' << (8u * (la + 1u)) : 0ull), tb = (u64)'\t' | (nb << 8) | (lb < 7u ? (u64)'\t' << (8u * (lb + 1u)) : 0ull);
    const u32 ta2 = (u32)(na >> 56) | (la == 7u ? (u32)'\t' : 0u) | (la == 8u ? (u32)'\t' << 8 : 0u);
    const u32 tb2 = (u32)(nb >> 56) | (lb == 7u ? (u32)'\t' : 0u) | (lb == 8u ? (u32)'\t' << 8 : 0u);
    const u32 tail = (u32)'\t' | ((strands & 1u) ? (u32)'-' << 8 : (u32)'+' << 8) | ((u32)'\t' << 16) | ((strands & 2u) ? (u32)'-' << 24 : (u32)'+' << 24);
#pragma unroll 1
    for (u32 step = 0; step < 14u; ++step) {
        u32 x, n;
        switch (step) {
        case 0: x = (u32)ta; n = piece_len(la + 2u, 0); break;
        case 1: x = (u32)(ta >> 32); n = piece_len(la + 2u, 1); break;
        case 2: x = ta2; n = piece_len(la + 2u, 2); break;
        case 3: x = a0; n = piece_len(nda, 0); break;
        case 4: x = a1; n = piece_len(nda, 1); break;
        case 5: x = a2; n = piece_len(nda, 2); break;
        case 6: x = (u32)tb; n = piece_len(lb + 2u, 0); break;
        case 7: x = (u32)(tb >> 32); n = piece_len(lb + 2u, 1); break;
        case 8: x = tb2; n = piece_len(lb + 2u, 2); break;
        case 9: x = b0; n = piece_len(ndb, 0); break;
        case 10: x = b1; n = piece_len(ndb, 1); break;
        case 11: x = b2; n = piece_len(ndb, 2); break;
        case 12: x = tail; n = 4u; break;
        default: x = (u32)'\n'; n = 1u; break;
        }
        tw_put(t, x, n);
    }
    tw_end(t);
}
// byte-wise writer: long chromosome names, or a round whose text does not fit the stage (rare).  or_mode: the destination is the
// zeroed shared-memory stage that neighbouring lines are OR-ed into, so every byte is OR-ed into its word as well.
__device__ __forceinline__ void put_byte_mode(char *out, char c, bool or_mode) {
    if (or_mode) { const u32 sa = smem_u32(out); sts_or(sa & ~3u, (u32)(unsigned char)c << (8u * (sa & 3u))); }
    else *out = c;
}
static __device__ __noinline__ void fs_write_pair_line_bytes(const char *buf, u64 rid_abs, u32 rid_len, const ChrSlot *ca, const ChrSlot *cb,
                                                              u32 posA, u32 posB, u32 strands, char *out, bool or_mode) {
    for (u32 k = 0; k < rid_len; ++k) put_byte_mode(out++, buf[rid_abs + k], or_mode);
    put_byte_mode(out++, '\t', or_mode);
    for (u32 k = 0; k < ca->len; ++k) put_byte_mode(out++, ca->name[k], or_mode);
    put_byte_mode(out++, '\t', or_mode);
    for (int pass = 0; pass < 2; ++pass) {
        u32 v = pass ? posB : posA;
        const u32 n = dec_digits(v);
        for (int i = (int)n - 1; i >= 0; --i) { put_byte_mode(out + i, (char)('0' + v % 10u), or_mode); v /= 10u; }
        out += n;
        put_byte_mode(out++, '\t', or_mode);
        if (pass == 0) { for (u32 k = 0; k < cb->len; ++k) put_byte_mode(out++, cb->name[k], or_mode); put_byte_mode(out++, '\t', or_mode); }
    }
    put_byte_mode(out++, (strands & 1) ? '-' : '+', or_mode); put_byte_mode(out++, '\t', or_mode);
    put_byte_mode(out++, (strands & 2) ? '-' : '+', or_mode); put_byte_mode(out++, '\n', or_mode);
}

// Tiles of EMIT_TILE (256) lines.  K3 has already summed every tile's sizes (tile_tot), k_emit_prefix turns them into exclusive prefixes
// (one CTA, a few microseconds), so a tile here depends on no other tile: no look-back, no grid-wide dependency, and the
// small tiles leave no idle tail (the look-back version needed 2048-line tiles to amortise its chain: 5.1 tiles per CTA
// per 2 GiB window, i.e. a sixth round that was 90 % idle).

// One CTA per SEGMENT of EMIT_SEG tiles: its base is the sum of the earlier segments' totals (K3 accumulates those too, at
// most a few hundred values), then one block scan of the segment's own tiles.  (One CTA scanning all 17 800 tiles of a
// 2040 MiB window took 24 us on the critical path of every window.)
#define EMIT_SEG 128u
static __global__ void __launch_bounds__(EMIT_SEG) k_emit_prefix(S2PParams p) {
    __shared__ u32 s_w[4][EMIT_SEG / 32];
    __shared__ u32 s_base[4];
    WinState *st = p.st;
    const u32 n_sub = (st->n_lines + EMIT_TILE - 1) / EMIT_TILE;
    const u32 n_seg = (n_sub + EMIT_SEG - 1) / EMIT_SEG;
    const u32 seg = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    if (seg >= n_seg && !(seg == 0 && n_seg == 0)) return;
    // ---- base: totals of the segments before this one
    u32 G = 0, E = 0, T = 0, S = 0;
    for (u32 j = tid; j < seg; j += EMIT_SEG) { const uint4 v = p.seg_tot[j]; G += v.x; E += v.y; T += v.z; S += v.w; }
    G = __reduce_add_sync(0xFFFFFFFFu, G); E = __reduce_add_sync(0xFFFFFFFFu, E); T = __reduce_add_sync(0xFFFFFFFFu, T); S = __reduce_add_sync(0xFFFFFFFFu, S);
    if (lane == 0) { s_w[0][wid] = G; s_w[1][wid] = E; s_w[2][wid] = T; s_w[3][wid] = S; }
    __syncthreads();
    if (tid < 4) { u32 t = 0; for (u32 w = 0; w < EMIT_SEG / 32; ++w) t += s_w[tid][w]; s_base[tid] = t; }
    __syncthreads();
    // ---- this segment's tiles
    const u32 i = seg * EMIT_SEG + tid;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (i < n_sub) v = p.tile_tot[i];
    const u32 vG = v.x & 0xFFFFu, vE = v.x >> 16, vT = v.y, vS = v.z;
    const u32 iG = warp_incl_scan(vG, (int)lane), iE = warp_incl_scan(vE, (int)lane), iT = warp_incl_scan(vT, (int)lane), iS = warp_incl_scan(vS, (int)lane);
    __syncthreads();                                                    // s_w is reused
    if (lane == 31) { s_w[0][wid] = iG; s_w[1][wid] = iE; s_w[2][wid] = iT; s_w[3][wid] = iS; }
    __syncthreads();
    u32 bG = s_base[0], bE = s_base[1], bT = s_base[2], bS = s_base[3];
    for (u32 w = 0; w < wid; ++w) { bG += s_w[0][w]; bE += s_w[1][w]; bT += s_w[2][w]; bS += s_w[3][w]; }
    if (i < n_sub) p.tile_pre[i] = make_uint4(bG + iG - vG, bE + iE - vE, bT + iT - vT, bS + iS - vS);
    if (seg + 1 == n_seg && tid == EMIT_SEG - 1) { st->w_groups = bG + iG; st->w_emit = bE + iE; st->w_text = bT + iT; st->w_sam = bS + iS; }
    if (n_seg == 0 && tid == 0) { st->w_groups = st->w_emit = st->w_text = st->w_sam = 0; }
}

// the nd (1..10) decimal characters of v as byte stores, without a division chain
__device__ __forceinline__ char *put_uint_fast(char *out, u32 v, u32 nd) {
    u32 d0, d1, d2;
    dec_chars(v, nd, d0, d1, d2);
#pragma unroll
    for (int b = 0; b < 4; ++b) if ((u32)b < nd) out[b] = (char)(d0 >> (8 * b));
#pragma unroll
    for (int b = 0; b < 4; ++b) if ((u32)(4 + b) < nd) out[4 + b] = (char)(d1 >> (8 * b));
#pragma unroll
    for (int b = 0; b < 2; ++b) if ((u32)(8 + b) < nd) out[8 + b] = (char)(d2 >> (8 * b));
    return out + nd;
}

// One line per thread, tiles of 256 lines.  Every global load of a tile's round — line flags, the group's resolution, and the
// read id's bytes out of the SAM text (seven aligned 8-byte words, realigned in registers) — is issued before the first
// byte is formatted: ncu had the read-id fetch, one dependent load per 8 bytes inside the formatting loop, at 25 % of this
// kernel's stall samples.  64 registers and a 20 KiB stage leave room for five CTAs per SM (was three).
#ifndef EMIT_OCC
#define EMIT_OCC 5
#endif
static __global__ void __launch_bounds__(EMIT_THREADS, EMIT_OCC) k_emit(S2PParams p) {
    __shared__ __align__(16) char s_stage[EMIT_STAGE + 16];
    __shared__ u32 s_w[2][3][EMIT_THREADS / 32];
    WinState *st = p.st;
    const u32 n_lines = st->n_lines;
    const u64 ws = st->ws;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n_tiles = (int)((n_lines + EMIT_TILE - 1) / EMIT_TILE);
    const u64 base_text = st->out_text, base_pairs = st->out_pairs, base_sam = st->out_sam, base_groups = st->groups_done;
    int pb = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, pb ^= 1) {
        const uint4 tbase = p.tile_pre[tile];                           // (groups, emitted, text, passthrough) before this tile
        const u32 i = (u32)tile * EMIT_TILE + tid;
        // ---- loads
        const u32 m = i < n_lines ? p.lmeta[i] : 0;
        const bool proc = (m & LM_HEAD) && (m & LM_PROC), emit = proc && (m & LM_EMIT);
        GroupRes g; g.text_len = 0; g.sam_len = 0; g.rid_len = 0; g.rid_off = 0; g.status = ST_NONE;
        if (proc) g = p.res[i];
        const bool want_text = emit && p.emit_text;
        const u64 rid_abs = ws + g.rid_off;
        const u32 rsh = (u32)(rid_abs & 7u) * 8u;
        u64 rw[7];
        {
            const u64 *src = (const u64 *)(p.buf + (rid_abs & ~(u64)7));
            const u32 span = g.rid_len + (rsh >> 3);
#pragma unroll
            for (int j = 0; j < 7; ++j) rw[j] = (want_text && (u32)(8 * j) < span) ? __ldg(src + j) : 0ull;
        }
        const ChrSlot *ca = nullptr, *cb = nullptr;
        if (want_text) { ca = &p.chr[p.id_to_slot[g.chrA]]; cb = &p.chr[p.id_to_slot[g.chrB]]; }
        // ---- sizes: (groups | emitted << 16, text bytes, passthrough bytes), scanned over the tile
        const u32 vA = (proc ? 1u : 0u) | (emit ? 1u << 16 : 0u), vT = emit ? g.text_len : 0u, vS = (emit && p.write_sam) ? g.sam_len : 0u;
        const u32 iA = warp_incl_scan(vA, lane), iT = warp_incl_scan(vT, lane), iS = warp_incl_scan(vS, lane);
        if (lane == 31) { s_w[pb][0][wid] = iA; s_w[pb][1][wid] = iT; s_w[pb][2][wid] = iS; }
        __syncthreads();
        u32 lA = iA - vA, lT = iT - vT, lS = iS - vS, totT = 0;
#pragma unroll
        for (int q = 0; q < EMIT_THREADS / 32; ++q) {
            const u32 xa = s_w[pb][0][q], xt = s_w[pb][1][q], xs = s_w[pb][2][q];
            totT += xt;
            if (q < wid) { lA += xa; lT += xt; lS += xs; }
        }
        const u32 g_idx = tbase.x + (lA & 0xFFFFu), e_idx = tbase.y + (lA >> 16);
        const u64 t_off = base_text + tbase.z;                           // first text byte of the tile
        const u64 s_run = base_sam + tbase.w + lS;
        const bool text_fits = t_off + totT <= p.out_text_cap;
        const bool staged = totT <= EMIT_STAGE;
        const u32 phase = (u32)((u64)(p.out_text + t_off) & 15u);       // stage with the destination's 16-byte phase
        if (p.emit_text && totT && !text_fits && tid == 0) atomicOr(&st->err, S2P_ERR_TEXT);
        // ---- outputs
        if (proc) {
            if (g.status == ST_SELFCIRCLE) {                             // for the thread-0-share emulation on the host
                u32 slot = atomicAdd(&st->sc_count, 1u);
                if (slot < p.sc_cap) p.sc_list[slot] = base_groups + g_idx; else atomicOr(&st->err, S2P_ERR_SCLIST);
            }
            if (emit) {
                const u64 o = base_pairs + e_idx;
                if (p.emit_packed) {
                    if (o < p.out_pairs_cap) {
                        mk_pair r; r.pos1 = g.posA; r.pos2 = g.posB; r.chr1 = g.chrA; r.chr2 = g.chrB; r.strands = g.strands;
                        r.cls = (u8)(g.status - ST_TRANS); r.lane = p.lane;
                        p.out_pairs[o] = r;
                    } else atomicOr(&st->err, S2P_ERR_PAIRS);
                }
                if (p.out_line_off && p.emit_text && o < p.out_line_off_cap) p.out_line_off[o] = p.line_off_base + t_off + lT;
                if (p.emit_text && text_fits) {
                    // rid \t chrA \t posA \t chrB \t posB \t sA \t sB \n   (unc2pairs.h:327-347)
                    char *out = staged ? s_stage + phase + lT : p.out_text + t_off + lT;
#pragma unroll
                    for (int j = 0; j < 6; ++j) {
                        if ((u32)(8 * j) < g.rid_len) {
                            const u64 x = rsh ? (rw[j] >> rsh) | (rw[j + 1] << (64u - rsh)) : rw[j];
                            const u32 nb = g.rid_len - 8u * j < 8u ? g.rid_len - 8u * j : 8u;
                            out = put_bytes8(out, x, nb);
                        }
                    }
                    for (u32 k = 48; k < g.rid_len; ++k) *out++ = p.buf[rid_abs + k];    // read ids beyond 48 bytes: rare
                    *out++ = '\t';
                    out = put_name(out, ca);
                    *out++ = '\t';
                    out = put_uint_fast(out, g.posA, dec_digits(g.posA));
                    *out++ = '\t';
                    out = put_name(out, cb);
                    *out++ = '\t';
                    out = put_uint_fast(out, g.posB, dec_digits(g.posB));
                    *out++ = '\t'; *out++ = (g.strands & 1) ? '-' : '+'; *out++ = '\t'; *out++ = (g.strands & 2) ? '-' : '+'; *out++ = '\n';
                }
                if (p.write_sam) {                                       // destination of every kept line of the group; K5 copies
                    if (s_run + g.sam_len > p.out_sam_cap) atomicOr(&st->err, S2P_ERR_SAM);
                    else {
                        u64 o2 = s_run; u32 ql = i;
                        while (true) {
                            p.sam_dst[ql] = (u32)(o2 - base_sam);
                            o2 += line_len_of(p, ql) + 1;
                            if (ql == g.last_line) break;
                            ++ql; while (!(p.lmeta[ql] & LM_KEEP)) ++ql;
                        }
                    }
                }
            }
        }
        if (p.emit_text && totT && text_fits && staged) {
            __syncthreads();
            char *dst = p.out_text + t_off;
            const u32 head = phase ? (16u - phase < totT ? 16u - phase : totT) : 0u;
            if ((u32)tid < head) dst[tid] = s_stage[phase + tid];
            const u32 body = (totT - head) >> 4;
            for (u32 w = tid; w < body; w += EMIT_THREADS)
                st_stream_v4((uint4 *)(dst + head + ((u64)w << 4)), *(const uint4 *)(s_stage + phase + head + (w << 4)));
            const u32 tail0 = head + (body << 4);
            if (tail0 + tid < totT) dst[tail0 + tid] = s_stage[phase + tail0 + tid];
            __syncthreads();                                             // the stage is reused by the next tile
        }
    }
}

// ------------------------------------------------------------------------------------------------ K5: SAM passthrough
// The lines of emitted groups are copied verbatim (with their '\n').  A CTA takes 256 lines: their (source, destination,
// length) are gathered with coalesced loads into shared memory first, so that the copy loop itself has no dependent
// metadata loads; then each warp copies its lines two at a time (both lines' loads are issued before the first store).
// Source and destination have unrelated alignments, so the copy runs on the DESTINATION's 16-byte grid: a lane builds one
// aligned 16-byte chunk from two aligned 128-bit source loads (word offset chosen by a warp-uniform switch, byte offset by
// four funnel shifts) and stores it with one 128-bit streaming store; the ragged head and tail of a line go out bytewise.
struct SamCopy { const char *src; char *dst; u32 len, h, body, q, sh; const uint4 *sa; };
__device__ __forceinline__ SamCopy sam_copy_setup(const char *src, char *dst, u32 len) {
    SamCopy c; c.src = src; c.dst = dst; c.len = len;
    const u32 head = (16u - (u32)((uintptr_t)dst & 15u)) & 15u;      // bytes before the destination's first 16-byte boundary
    c.h = head < len ? head : len;
    c.body = (len - c.h) >> 4;                                       // whole aligned 16-byte chunks
    const char *sb = src + c.h;
    c.q = ((u32)((uintptr_t)sb & 15u)) >> 2; c.sh = (u32)((uintptr_t)sb & 3u) * 8u;
    c.sa = (const uint4 *)((uintptr_t)sb & ~(uintptr_t)15);
    return c;
}
__device__ __forceinline__ uint4 sam_copy_chunk(const SamCopy &c, const uint4 &a, const uint4 &b) {
    u32 w0, w1, w2, w3, w4;                                          // the five source words the chunk is cut from (q is warp-uniform)
    switch (c.q) {
    case 0: w0 = a.x; w1 = a.y; w2 = a.z; w3 = a.w; w4 = b.x; break;
    case 1: w0 = a.y; w1 = a.z; w2 = a.w; w3 = b.x; w4 = b.y; break;
    case 2: w0 = a.z; w1 = a.w; w2 = b.x; w3 = b.y; w4 = b.z; break;
    default: w0 = a.w; w1 = b.x; w2 = b.y; w3 = b.z; w4 = b.w; break;
    }
    return make_uint4(__funnelshift_r(w0, w1, c.sh), __funnelshift_r(w1, w2, c.sh), __funnelshift_r(w2, w3, c.sh), __funnelshift_r(w3, w4, c.sh));
}
static __global__ void __launch_bounds__(256) k_copy_sam(S2PParams p) {
    __shared__ u32 s_src[256], s_dst[256], s_len[256];
    const WinState *st = p.st;
    const u32 n_lines = st->n_lines;
    const u64 ws = st->ws, base = st->out_sam;
    const u32 tid = threadIdx.x, lane = tid & 31u, wid = tid >> 5;
    const u32 n_tiles = (n_lines + 255u) / 256u;
    for (u32 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const u32 i = tile * 256u + tid;
        u32 len = 0, start = 0, d = 0;
        if (i < n_lines && (p.lmeta[i] & LM_KEEP)) {
            d = p.sam_dst[i];
            if (d != 0xFFFFFFFFu) { start = i ? p.nl_pos[i - 1] + 1 : 0; len = p.nl_pos[i] - start + 1; }
        }
        __syncthreads();                                                 // the previous tile's entries have been consumed
        s_src[tid] = start; s_dst[tid] = d; s_len[tid] = len;
        __syncthreads();
#pragma unroll 1
        for (u32 l = wid; l < 256u; l += 16u) {                          // this warp's lines, two at a time
            const u32 la = s_len[l], lb = s_len[l + 8u];
            if (!la && !lb) continue;
            const SamCopy A = sam_copy_setup(p.buf + ws + s_src[l], p.out_sam + base + s_dst[l], la);
            const SamCopy B = sam_copy_setup(p.buf + ws + s_src[l + 8u], p.out_sam + base + s_dst[l + 8u], lb);
            const u32 rounds = ((A.body > B.body ? A.body : B.body) + 31u) >> 5;
            for (u32 r = 0; r < rounds; ++r) {
                const u32 c = r * 32u + lane;
                uint4 a0, a1, b0, b1;
                const bool ga = c < A.body, gb = c < B.body;
                // the second word is only read when the source is not 16-byte aligned: it then starts inside the chunk's own bytes
                if (ga) { a0 = __ldg(A.sa + c); a1 = (A.q | A.sh) ? __ldg(A.sa + c + 1) : a0; }
                if (gb) { b0 = __ldg(B.sa + c); b1 = (B.q | B.sh) ? __ldg(B.sa + c + 1) : b0; }
                if (ga) st_stream_v4((uint4 *)(A.dst + A.h) + c, sam_copy_chunk(A, a0, a1));
                if (gb) st_stream_v4((uint4 *)(B.dst + B.h) + c, sam_copy_chunk(B, b0, b1));
            }
            if (lane < A.h) A.dst[lane] = A.src[lane];
            if (lane < B.h) B.dst[lane] = B.src[lane];
            const u32 ta = A.h + (A.body << 4), tb = B.h + (B.body << 4);
            if (ta + lane < A.len) A.dst[ta + lane] = A.src[ta + lane];
            if (tb + lane < B.len) B.dst[tb + lane] = B.src[tb + lane];
        }
    }
}
