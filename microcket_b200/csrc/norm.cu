// norm.cu — balancing of contact matrices: the VC, VC_SQRT and KR normalisation vectors `juicer_tools pre` stores in a `.hic`
// (microcket:525-529), per chromosome, from its intra-chromosomal matrix; and the GW_VC / GW_KR (whole-genome matrix) and
// INTER_VC / INTER_KR (inter-chromosomal entries only) vectors, one balancing problem over every bin.  Restated from juicer's
// published behaviour (Knight & Ruiz 2013 `bnewt` for KR, juicer's sum factor); PARITY UNPINNED like the rest of the
// container (DESIGN.md §5).
//
// The COO of one resolution (sorted by (bin1, bin2), upper triangle: what mk_pairs_bin_device / mk_hist_coo_device return)
// becomes ONE symmetric CSR of the entries in the call's scope, built once and reused by every product:
//   row r = [mirrored half: (column bin1 < r), bin1 ascending][upper half: (column bin2 >= r), bin2 ascending]
// The scope is INTRA (both bins in one chromosome), GENOME (every entry) or INTER (the two bins in different chromosomes).
// Row r's entries in the COO are one run sorted by column; its INTRA entries are a prefix of the run (up to the end of r's
// chromosome), its INTER entries the rest.  The upper half is therefore already CSR by bin1 in the COO; the mirrored half
// comes from one stable radix sort on bin2 (radix_sort.cuh, values = entry index) of the scope's off-diagonal entries.
// Entries are (u32 column, u32 count), row pointers 64-bit.
//
// A segment is one balancing problem: a chromosome for INTRA, every bin for GENOME and INTER (segment 0).  The commands, the
// results and the row skip of the element-wise kernels are indexed by segment through a bin -> segment table.
//
//   k_nm_classify     validation, scope test, where every row's entries in the scope start / end in the COO, sort keys
//   k_nm_lower_runs   where every row's mirrored entries start / end in the sorted keys
//   k_nm_row_ptr      row pointers (ticketed tiles, decoupled look-back)
//   k_nm_fill_upper / k_nm_fill_lower   the CSR entries
//   k_nm_spmv         y = A u: one warp per row, every lane sums a fixed stride of the row in order, then a fixed
//                     butterfly: no floating-point atomics, so the vectors are bitwise reproducible from run to run
//   k_nm_pre          per row, the vector that goes into the next product, from its chromosome's command
//   k_nm_post         the vector updates and reductions after a product, one CTA per chromosome (INTRA), in one launch
//   k_nm_gpost        the same for the one segment of GENOME / INTER, over fixed slices of NM_GS rows, in 1 or 3 launches;
//                     both run the same per-row phases (nm_row_sums ... nm_cg_update) and scalar decisions (nm_alpha ...)
//   k_nm_finish       1 / x (KR) or sqrt (VC_SQRT) into the output vectors; k_nm_scale: the sum factors
//
// KR runs for all segments in lockstep: every step is k_nm_pre -> k_nm_spmv -> k_nm_post (k_nm_gpost), and the per-segment
// scalars come back in ONE small copy; the host advances every segment's state machine (plain C++ below) and sends the next
// step's commands in one copy.  Each unfinished segment needs exactly one product per step: A (x∘p) inside CG, A x after
// an outer update.  Finished segments' rows are skipped by the product.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <vector>
#include "mk_common.cuh"
#include "radix_sort.cuh"

#define NM_T 256                 // element-wise kernels and the product
#define NM_RT 1024               // per-chromosome kernels: one CTA per chromosome (32 warps: the block reductions rely on it)
#define NP_T 256                 // row pointer scan
#define NP_ITEMS 16
#define NM_GS 2048               // rows per slice of a GENOME / INTER segment: fixed, so the bits depend neither on the card nor on the grid

// Knight-Ruiz parameters (bnewt defaults, as juicer uses them)
#define KR_TOL 1e-6
#define KR_DELTA 0.1
#define KR_DELTA_HI 3.0
#define KR_ETAMAX 0.1
#define KR_G 0.9
#define KR_MAX_OUTER 100
#define KR_MAX_INNER 10000       // CG steps in one outer step; bnewt has no bound, an unbounded loop would stall every chromosome

enum { OP_IDLE = 0, OP_ONES, OP_KR_INIT, OP_KR_OUTER, OP_CG_FIRST, OP_CG_NEXT, OP_SUMF };
enum { ST_CG_CONT = 0, ST_CG_BREAK = 1, ST_FAIL = 2 };
enum { NM_INTRA = 0, NM_GENOME = MK_NORM_SCOPE_GW, NM_INTER = MK_NORM_SCOPE_INTER };

struct NormCmd { int op, pad; double beta, rho; };             // host -> device, one per chromosome and step
struct NormRes { double a, b, c; int flag, pad; };             // device -> host
struct NormPart { double a, b, c, d; };                         // a phase's totals over one CTA's rows (in k_nm_gpost: one slice's)
static_assert(sizeof(NormRes) == sizeof(NormPart), "k_nm_gpost's result sits behind its final partials, copied in one piece");

struct NormVecs { double *x, *v, *rk, *y, *z, *p, *w, *u, *au, *rs; u8 *kept; };   // rs: row sums (au is every product's output)

// ---------------------------------------------------------------- CSR build
__device__ __forceinline__ u32 nm_chr_end(const u32 *chr_of_bin, const u32 *chr_off, u32 bin) { return chr_off[chr_of_bin[bin] + 1]; }

template <int SC>
__device__ __forceinline__ bool nm_in_scope(const u32 *chr_of_bin, const u32 *chr_off, u32 a, u32 b) {
    return SC == NM_GENOME || ((b < nm_chr_end(chr_of_bin, chr_off, a)) == (SC == NM_INTRA));
}

// err bit 0: bin1 > bin2, bit 1: a bin past the end, bit 2: not sorted by (bin1, bin2)
template <int SC>
__global__ void __launch_bounds__(NM_T) k_nm_classify(const u32 *b1, const u32 *b2, u64 nnz, u32 nb, const u32 *chr_of_bin, const u32 *chr_off,
                                                     u32 *row_start, u32 *up_end, u64 *keys, u32 *err, unsigned long long *n_low) {
    u32 e = 0, low = 0;
    for (u64 i = (u64)blockIdx.x * NM_T + threadIdx.x; i < nnz; i += (u64)gridDim.x * NM_T) {
        const u32 a = b1[i], b = b2[i];
        bool bad = false;
        if (a > b) { e |= 1u; bad = true; }
        if (b >= nb) { e |= 2u; bad = true; }
        if (i && (b1[i - 1] > a || (b1[i - 1] == a && b2[i - 1] >= b))) e |= 4u;
        if (bad) { keys[i] = nb; continue; }
        const bool in = nm_in_scope<SC>(chr_of_bin, chr_off, a, b);
        // a row's entries in the scope are one piece of its run in the COO (columns ascend, the chromosome ends at chr_end):
        // INTRA a prefix, INTER a suffix, GENOME the whole run
        if (in && (i == 0 || b1[i - 1] != a || (SC == NM_INTER && b2[i - 1] < nm_chr_end(chr_of_bin, chr_off, a)))) row_start[a] = (u32)i;
        if (in && (i + 1 == nnz || b1[i + 1] != a || (SC == NM_INTRA && b2[i + 1] >= nm_chr_end(chr_of_bin, chr_off, a)))) up_end[a] = (u32)(i + 1);
        const bool mirror = in && a != b;
        keys[i] = mirror ? (u64)b : (u64)nb;                    // everything else sorts behind the mirrored entries
        low += mirror;
    }
    for (int d = 16; d; d >>= 1) { e |= __shfl_xor_sync(0xffffffffu, e, d); low += __shfl_xor_sync(0xffffffffu, low, d); }
    if ((threadIdx.x & 31) == 0) { if (e) atomicOr(err, e); if (low) atomicAdd(n_low, (unsigned long long)low); }
}

__global__ void __launch_bounds__(NM_T) k_nm_lower_runs(const RadixPlan *plan, const u64 *k0, const u64 *k1, const unsigned long long *n_low,
                                                       u32 *low_start, u32 *low_end) {
    const u64 *k = plan->final_buf ? k1 : k0;
    const u64 m = *n_low;
    for (u64 j = (u64)blockIdx.x * NM_T + threadIdx.x; j < m; j += (u64)gridDim.x * NM_T) {
        const u64 r = k[j];
        if (j == 0 || k[j - 1] != r) low_start[r] = (u32)j;
        if (j + 1 == m || k[j + 1] != r) low_end[r] = (u32)(j + 1);
    }
}

__device__ __forceinline__ u32 nm_row_len(u32 r, const u32 *row_start, const u32 *up_end, const u32 *low_start, const u32 *low_end) {
    return (up_end[r] - row_start[r]) + (low_end[r] - low_start[r]);
}

__global__ void __launch_bounds__(NP_T) k_nm_row_ptr(u32 nb, const u32 *row_start, const u32 *up_end, const u32 *low_start, const u32 *low_end,
                                                    u64 *row_ptr, u64 *desc, u32 *ticket) {
    __shared__ u32 s_scan[NP_T / 32 + 1];
    __shared__ u64 s_base;
    __shared__ u32 s_tile;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const u64 n_tiles = ((u64)nb + NP_T * NP_ITEMS - 1) / (NP_T * NP_ITEMS);
    while (true) {
        if (tid == 0) s_tile = atomicAdd(ticket, 1u);
        __syncthreads();
        const u64 tile = s_tile;
        if (tile >= n_tiles) break;
        const u64 base = tile * NP_T * NP_ITEMS + (u64)tid * NP_ITEMS;
        u32 len[NP_ITEMS], sum = 0;
#pragma unroll
        for (int k = 0; k < NP_ITEMS; ++k) { len[k] = base + k < nb ? nm_row_len((u32)(base + k), row_start, up_end, low_start, low_end) : 0u; sum += len[k]; }
        u32 tot;
        const u32 ex = block_excl_scan<NP_T>(sum, s_scan, &tot);
        if (wid == 0) {
            const u64 b = lookback_exclusive(desc, (int)tile, 0, tot, lane);
            if (lane == 0) { s_base = b; if (tile == n_tiles - 1) row_ptr[nb] = b + tot; }
        }
        __syncthreads();
        u64 o = s_base + ex;
#pragma unroll
        for (int k = 0; k < NP_ITEMS; ++k) if (base + k < nb) { row_ptr[base + k] = o; o += len[k]; }
        __syncthreads();
    }
}

template <int SC>
__global__ void __launch_bounds__(NM_T) k_nm_fill_upper(const u32 *b1, const u32 *b2, const u32 *cnt, u64 nnz, const u32 *chr_of_bin, const u32 *chr_off,
                                                       const u64 *row_ptr, const u32 *row_start, const u32 *low_start, const u32 *low_end, uint2 *ents) {
    for (u64 i = (u64)blockIdx.x * NM_T + threadIdx.x; i < nnz; i += (u64)gridDim.x * NM_T) {
        const u32 a = b1[i], b = b2[i];
        if (!nm_in_scope<SC>(chr_of_bin, chr_off, a, b)) continue;
        ents[row_ptr[a] + (low_end[a] - low_start[a]) + (i - row_start[a])] = make_uint2(b, cnt[i]);
    }
}

__global__ void __launch_bounds__(NM_T) k_nm_fill_lower(const RadixPlan *plan, const u64 *k0, const u64 *k1, const u32 *v0, const u32 *v1,
                                                       const unsigned long long *n_low, const u32 *b1, const u32 *cnt, const u64 *row_ptr,
                                                       const u32 *low_start, uint2 *ents) {
    const u64 *k = plan->final_buf ? k1 : k0;
    const u32 *v = plan->final_buf ? v1 : v0;
    const u64 m = *n_low;
    for (u64 j = (u64)blockIdx.x * NM_T + threadIdx.x; j < m; j += (u64)gridDim.x * NM_T) {
        // no pass ran (every key equal: all entries mirror into one column): the values were never written, the order is the input's
        const u32 r = (u32)k[j], idx = plan->n_exec ? v[j] : (u32)j;
        ents[row_ptr[r] + (j - low_start[r])] = make_uint2(b1[idx], cnt[idx]);
    }
}

// ---------------------------------------------------------------- product
__global__ void __launch_bounds__(NM_T) k_nm_spmv(const u64 *row_ptr, const uint2 *ents, u32 nb, const u32 *seg_of_bin, const NormCmd *cmd,
                                                 const double *u, double *y) {
    const int lane = threadIdx.x & 31;
    const u64 warps = (u64)gridDim.x * (NM_T / 32);
    for (u64 r = (u64)blockIdx.x * (NM_T / 32) + (threadIdx.x >> 5); r < nb; r += warps) {
        if (cmd[seg_of_bin[r]].op == OP_IDLE) continue;
        const u64 beg = row_ptr[r], end = row_ptr[r + 1];
        double acc = 0.0;
        u64 k = beg + lane;
        for (; k + 96 < end; k += 128) {                                 // four loads in flight, summed in row order
            uint2 e[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) e[q] = __ldg(ents + k + 32 * q);
#pragma unroll
            for (int q = 0; q < 4; ++q) acc += (double)e[q].y * u[e[q].x];
        }
        for (; k < end; k += 32) { const uint2 e = __ldg(ents + k); acc += (double)e.y * u[e.x]; }
#pragma unroll
        for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (lane == 0) y[r] = acc;
    }
}

// ---------------------------------------------------------------- per-row commands before a product
__global__ void __launch_bounds__(NM_T) k_nm_pre(u32 nb, const u32 *seg_of_bin, const NormCmd *cmd, NormVecs V, const double *nvec) {
    for (u64 r = (u64)blockIdx.x * NM_T + threadIdx.x; r < nb; r += (u64)gridDim.x * NM_T) {
        const NormCmd c = cmd[seg_of_bin[r]];
        const bool kp = V.kept[r];
        switch (c.op) {
        case OP_ONES: V.u[r] = 1.0; break;
        case OP_KR_INIT: V.x[r] = kp ? 1.0 : 0.0; V.u[r] = V.x[r]; break;
        case OP_KR_OUTER: if (kp) V.x[r] *= V.y[r]; V.u[r] = V.x[r]; break;
        case OP_CG_FIRST: {
            const double z = kp ? V.rk[r] / V.v[r] : 0.0;
            V.y[r] = 1.0; V.z[r] = z; V.p[r] = z; V.u[r] = V.x[r] * z; break;
        }
        case OP_CG_NEXT: { const double p = V.z[r] + c.beta * V.p[r]; V.p[r] = p; V.u[r] = V.x[r] * p; break; }
        case OP_SUMF: { const double n = nvec[r]; V.u[r] = (n > 0.0 && isfinite(n)) ? 1.0 / n : 0.0; break; }
        default: break;
        }
    }
}

// ---------------------------------------------------------------- updates and reductions after a product
// A phase walks rows [r0, r1) with a stride of NT from threadIdx.x, in order, updates V, and reduces its per-thread partials
// over the CTA's NT threads with a fixed tree (nm_bred): the same bits on every run.  It returns the CTA's totals, several of
// them as a NormPart.
enum { RED_SUM = 0, RED_MIN, RED_MAX };
template <int OP> __device__ __forceinline__ double nm_op(double a, double b) { return OP == RED_SUM ? a + b : OP == RED_MIN ? fmin(a, b) : fmax(a, b); }
template <int OP> __device__ __forceinline__ double nm_pad() { return OP == RED_SUM ? 0.0 : OP == RED_MIN ? INFINITY : -INFINITY; }

// NW <= 32 warps: each warp's butterfly, then one over the warps' results in warp 0.  sh: 33 doubles
template <int OP, int NW>
__device__ __forceinline__ double nm_bred(double v, double *sh) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d; d >>= 1) v = nm_op<OP>(v, __shfl_xor_sync(0xffffffffu, v, d));
    if (lane == 0) sh[wid] = v;
    __syncthreads();
    if (wid == 0) {
        double t = lane < NW ? sh[lane] : nm_pad<OP>();
#pragma unroll
        for (int d = 16; d; d >>= 1) t = nm_op<OP>(t, __shfl_xor_sync(0xffffffffu, t, d));
        if (lane == 0) sh[32] = t;
    }
    __syncthreads();
    const double r = sh[32];
    __syncthreads();
    return r;
}

// row sums (OP_ONES) -> {raw total, rows kept by KR}
template <int NT>
__device__ __forceinline__ NormPart nm_row_sums(const NormVecs &V, u32 r0, u32 r1, double *sh) {
    double s = 0.0, k = 0.0;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) { const double a = V.au[r]; s += a; k += a > 0.0; V.rs[r] = a; V.kept[r] = a > 0.0; }
    return NormPart{nm_bred<RED_SUM, NT / 32>(s, sh), nm_bred<RED_SUM, NT / 32>(k, sh), 0.0, 0.0};
}

// the sum factor's u·(A u) (OP_SUMF)
template <int NT>
__device__ __forceinline__ double nm_sumf(const NormVecs &V, u32 r0, u32 r1, double *sh) {
    double s = 0.0;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) s += V.u[r] * V.au[r];
    return nm_bred<RED_SUM, NT / 32>(s, sh);
}

// after A x (OP_KR_INIT / OP_KR_OUTER): v = x (A x), rk = 1 - v -> {rk·rk, min x, > 0 when an x or v is not finite}
template <int NT>
__device__ __forceinline__ NormPart nm_outer(const NormVecs &V, u32 r0, u32 r1, double *sh) {
    double s = 0.0, xmin = INFINITY; int bad = 0;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) {
        if (!V.kept[r]) continue;
        const double x = V.x[r], v = x * V.au[r], rk = 1.0 - v;
        V.v[r] = v; V.rk[r] = rk;
        s += rk * rk; xmin = fmin(xmin, x); bad |= !isfinite(x) || !isfinite(v);
    }
    return NormPart{nm_bred<RED_SUM, NT / 32>(s, sh), nm_bred<RED_MIN, NT / 32>(xmin, sh), nm_bred<RED_SUM, NT / 32>((double)bad, sh), 0.0};
}

// a CG step's product A (x p): w -> {p·w, rk·Z}
template <int NT>
__device__ __forceinline__ NormPart nm_cg_product(const NormVecs &V, u32 r0, u32 r1, double *sh) {
    double pw = 0.0, rz = 0.0;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) {
        if (!V.kept[r]) continue;
        const double p = V.p[r], w = V.x[r] * V.au[r] + V.v[r] * p;
        V.w[r] = w; pw += p * w; rz += V.rk[r] * V.z[r];
    }
    return NormPart{nm_bred<RED_SUM, NT / 32>(pw, sh), nm_bred<RED_SUM, NT / 32>(rz, sh), 0.0, 0.0};
}

// the box test of y + alpha p -> {min, max, step to the lower edge, step to the upper edge}
template <int NT>
__device__ __forceinline__ NormPart nm_box(const NormVecs &V, u32 r0, u32 r1, double alpha, double *sh) {
    double ymin = INFINITY, ymax = -INFINITY, glo = INFINITY, ghi = INFINITY;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) {
        if (!V.kept[r]) continue;
        const double y = V.y[r], ap = alpha * V.p[r], yn = y + ap;
        ymin = fmin(ymin, yn); ymax = fmax(ymax, yn);
        if (ap < 0.0) glo = fmin(glo, (KR_DELTA - y) / ap);
        if (yn > KR_DELTA_HI) ghi = fmin(ghi, (KR_DELTA_HI - y) / ap);
    }
    return NormPart{nm_bred<RED_MIN, NT / 32>(ymin, sh), nm_bred<RED_MAX, NT / 32>(ymax, sh), nm_bred<RED_MIN, NT / 32>(glo, sh),
                    nm_bred<RED_MIN, NT / 32>(ghi, sh)};
}

// the step that leaves the box stops at its edge
template <int NT>
__device__ __forceinline__ void nm_edge(const NormVecs &V, u32 r0, u32 r1, double gamma, double alpha) {
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) if (V.kept[r]) V.y[r] = V.y[r] + gamma * (alpha * V.p[r]);
}

// the step inside the box: y, rk, Z -> the new rk·Z
template <int NT>
__device__ __forceinline__ double nm_cg_update(const NormVecs &V, u32 r0, u32 r1, double alpha, double *sh) {
    double s = 0.0;
    for (u32 r = r0 + threadIdx.x; r < r1; r += NT) {
        if (!V.kept[r]) continue;
        const double rk = V.rk[r] - alpha * V.w[r], z = rk / V.v[r];
        V.y[r] = V.y[r] + alpha * V.p[r]; V.rk[r] = rk; V.z[r] = z; s += rk * z;
    }
    return nm_bred<RED_SUM, NT / 32>(s, sh);
}

// A CG step's scalars from nm_cg_product's totals: rho is the step's rk·Z at OP_CG_FIRST, else the last update's.
// false: alpha is not finite, the segment fails.
__device__ __forceinline__ bool nm_alpha(const NormCmd &cm, const NormPart &pr, double &rho, double &alpha) {
    rho = cm.op == OP_CG_FIRST ? pr.b : cm.rho; alpha = rho / pr.a;
    return isfinite(alpha);
}
// from nm_box's totals: the step leaves the box (stop at its edge, end the inner loop), and the edge's gamma
__device__ __forceinline__ bool nm_leaves_box(double ymin, double ymax) { return ymin <= KR_DELTA || ymax >= KR_DELTA_HI; }
__device__ __forceinline__ double nm_gamma(double ymin, double glo, double ghi) { return ymin <= KR_DELTA ? glo : ghi; }

// one CTA per chromosome, every phase of the step in one launch
__global__ void __launch_bounds__(NM_RT) k_nm_post(const u32 *chr_off, const NormCmd *cmd, NormVecs V, NormRes *res) {
    __shared__ double sh[33];
    const int c = blockIdx.x;
    const NormCmd cm = cmd[c];
    if (cm.op == OP_IDLE) return;
    const u32 r0 = chr_off[c], r1 = chr_off[c + 1];
    NormRes out = {0.0, 0.0, 0.0, 0, 0};
    if (cm.op == OP_ONES) {
        const NormPart t = nm_row_sums<NM_RT>(V, r0, r1, sh);
        out.a = t.a; out.b = t.b;
    } else if (cm.op == OP_SUMF) {
        out.a = nm_sumf<NM_RT>(V, r0, r1, sh);
    } else if (cm.op == OP_KR_INIT || cm.op == OP_KR_OUTER) {
        const NormPart t = nm_outer<NM_RT>(V, r0, r1, sh);
        out.a = t.a; out.b = t.b; out.flag = t.c > 0.0;
    } else {
        double rho, alpha;
        const bool ok = nm_alpha(cm, nm_cg_product<NM_RT>(V, r0, r1, sh), rho, alpha);
        out.a = rho; out.c = alpha;
        if (!ok) out.flag = ST_FAIL;
        else {
            const NormPart box = nm_box<NM_RT>(V, r0, r1, alpha, sh);
            if (nm_leaves_box(box.a, box.b)) { nm_edge<NM_RT>(V, r0, r1, nm_gamma(box.a, box.c, box.d), alpha); out.flag = ST_CG_BREAK; }
            else { out.b = nm_cg_update<NM_RT>(V, r0, r1, alpha, sh); out.flag = ST_CG_CONT; }
        }
    }
    if (threadIdx.x == 0) res[c] = out;
}

// ---------------------------------------------------------------- the same phases for the one segment of GENOME / INTER
// One CTA per segment would stream every vector of 617 669 rows (hg38 at 5 kb) through one SM.  The rows are cut into slices
// of NM_GS; a CTA runs the phase on slices blockIdx.x, + gridDim.x, ... and writes one NormPart per slice.  A CG step's
// dependent reductions are three launches: phase 0 nm_cg_product, phase 1 nm_box, phase 2 nm_edge or nm_cg_update.  In
// phases 1 and 2 every CTA recomputes the totals of the earlier phases from their partials (nm_gred: in slice order, then a
// fixed tree), so every CTA takes the same decision and the bits depend on the slice width only, not on the grid.  The other
// ops need phase 0 only.  The final partials (pf) and phase 2's scalars (res) go to the host in one copy; nm_gres sums them
// there in slice order.
template <int OP>
__device__ __forceinline__ double nm_gred(const NormPart *p, u32 ns, int f, double *sh) {
    double s = nm_pad<OP>();
    for (u32 i = threadIdx.x; i < ns; i += NM_T) s = nm_op<OP>(s, (&p[i].a)[f]);
    return nm_bred<OP, NM_T / 32>(s, sh);
}

// part: [phase 0: ns][phase 1: ns][final: ns][NormRes]
__global__ void __launch_bounds__(NM_T) k_nm_gpost(int phase, u32 nb, const NormCmd *cmd, NormVecs V, NormPart *part) {
    __shared__ double sh[33];
    const NormCmd cm = cmd[0];
    if (cm.op == OP_IDLE) return;
    const u32 ns = (nb + NM_GS - 1) / NM_GS;
    NormPart *p0 = part, *p1 = part + ns, *pf = part + 2 * (size_t)ns;
    NormRes *res = (NormRes *)(pf + ns);
    const bool cg = cm.op == OP_CG_FIRST || cm.op == OP_CG_NEXT;
    double rho = 0.0, alpha = 0.0, gamma = 0.0;
    bool brk = false;
    if (phase > 0) {
        const NormPart pr = {nm_gred<RED_SUM>(p0, ns, 0, sh), nm_gred<RED_SUM>(p0, ns, 1, sh), 0.0, 0.0};
        if (!nm_alpha(cm, pr, rho, alpha)) {
            if (phase == 2 && blockIdx.x == 0 && threadIdx.x == 0) *res = NormRes{rho, 0.0, alpha, ST_FAIL, 0};
            return;
        }
    }
    if (phase == 2) {
        const NormPart box = {nm_gred<RED_MIN>(p1, ns, 0, sh), nm_gred<RED_MAX>(p1, ns, 1, sh), nm_gred<RED_MIN>(p1, ns, 2, sh),
                              nm_gred<RED_MIN>(p1, ns, 3, sh)};
        brk = nm_leaves_box(box.a, box.b);
        gamma = nm_gamma(box.a, box.c, box.d);
        if (blockIdx.x == 0 && threadIdx.x == 0) *res = NormRes{rho, 0.0, alpha, brk ? ST_CG_BREAK : ST_CG_CONT, 0};
    }
    for (u32 sl = blockIdx.x; sl < ns; sl += gridDim.x) {
        const u32 r0 = sl * NM_GS, r1 = min(nb, r0 + NM_GS);
        NormPart o = {0.0, 0.0, 0.0, 0.0};
        if (phase == 0 && cm.op == OP_ONES) o = nm_row_sums<NM_T>(V, r0, r1, sh);
        else if (phase == 0 && cm.op == OP_SUMF) o.a = nm_sumf<NM_T>(V, r0, r1, sh);
        else if (phase == 0 && !cg) o = nm_outer<NM_T>(V, r0, r1, sh);
        else if (phase == 0) o = nm_cg_product<NM_T>(V, r0, r1, sh);
        else if (phase == 1) o = nm_box<NM_T>(V, r0, r1, alpha, sh);
        else if (brk) nm_edge<NM_T>(V, r0, r1, gamma, alpha);
        else o.a = nm_cg_update<NM_T>(V, r0, r1, alpha, sh);
        if (threadIdx.x == 0) (phase == 0 && cg ? p0 : phase == 1 ? p1 : pf)[sl] = o;
    }
}

// the host side of k_nm_gpost: segment 0's NormRes from the final partials, summed in slice order
static void nm_gres(int op, const NormPart *pf, u32 ns, NormRes *out) {
    if (op == OP_CG_FIRST || op == OP_CG_NEXT) {
        *out = *(const NormRes *)(pf + ns);
        if (out->flag == ST_CG_CONT) { double s = 0.0; for (u32 i = 0; i < ns; ++i) s += pf[i].a; out->b = s; }
        return;
    }
    NormRes r = {0.0, op == OP_ONES ? 0.0 : INFINITY, 0.0, 0, 0};
    for (u32 i = 0; i < ns; ++i) {
        r.a += pf[i].a;
        if (op == OP_ONES) r.b += pf[i].b;
        else { r.b = std::min(r.b, pf[i].b); r.flag |= pf[i].c > 0.0; }
    }
    *out = r;
}

// kind 0: VC (row sums), 1: VC_SQRT, 2: KR (1 / x on kept rows of balanced segments, NaN elsewhere)
__global__ void __launch_bounds__(NM_T) k_nm_finish(int kind, u32 nb, const u32 *seg_of_bin, const u8 *kr_ok, NormVecs V, double *out) {
    for (u64 r = (u64)blockIdx.x * NM_T + threadIdx.x; r < nb; r += (u64)gridDim.x * NM_T) {
        const double s = V.rs[r];
        if (kind == 0) out[r] = s;
        else if (kind == 1) out[r] = sqrt(s);
        else out[r] = (kr_ok[seg_of_bin[r]] && V.kept[r]) ? 1.0 / V.x[r] : (double)NAN;
    }
}

__global__ void __launch_bounds__(NM_T) k_nm_scale(u32 nb, const u32 *seg_of_bin, const double *f, double *n) {
    for (u64 r = (u64)blockIdx.x * NM_T + threadIdx.x; r < nb; r += (u64)gridDim.x * NM_T) n[r] *= f[seg_of_bin[r]];
}

// ---------------------------------------------------------------- host side
struct mk_norm {
    int device = 0, sms = 148, n_chrom = 0, scope = NM_INTRA;   // scope: the current call's
    u32 res = 0, nb = 0, ns = 0;                                 // ns: slices of a GENOME / INTER segment
    size_t max_nnz = 0;
    std::vector<u32> chr_off;                               // n_chrom + 1 bin offsets
    DevBuf d_chr_of_bin, d_chr_off, d_row_ptr, d_runs /* row_start | up_end | low_start | low_end */, d_ents;
    DevBuf d_keys[2], d_vals[2], d_desc, d_small /* err, n_low, ticket */, d_vecs, d_kept, d_cmd, d_res, d_f, d_krok;
    DevBuf d_seg0 /* nb zeros: every bin in segment 0 */, d_gpart /* k_nm_gpost's partials and result */;
    RadixWs rws;
    PinBuf h_cmd, h_res, h_f, h_gpart;
    u64 launches = 0;
    bool timing = false;
    double ms[8] = {0}; u64 count[8] = {0};
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    ~mk_norm() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); }
    NormVecs vecs() const {
        double *b = d_vecs.as<double>();
        NormVecs V;
        V.x = b; V.v = b + nb; V.rk = b + 2 * (size_t)nb; V.y = b + 3 * (size_t)nb; V.z = b + 4 * (size_t)nb; V.p = b + 5 * (size_t)nb;
        V.w = b + 6 * (size_t)nb; V.u = b + 7 * (size_t)nb; V.au = b + 8 * (size_t)nb; V.rs = b + 9 * (size_t)nb; V.kept = d_kept.as<u8>();
        return V;
    }
    int grid(u64 n, int per) const { return (int)std::max<u64>(1, std::min<u64>((n + per - 1) / per, (u64)sms * 16)); }
    int n_seg() const { return scope == NM_INTRA ? n_chrom : 1; }
    const u32 *seg_of_bin() const { return scope == NM_INTRA ? d_chr_of_bin.as<u32>() : d_seg0.as<u32>(); }
};

extern "C" int mk_norm_create(int device, const uint32_t *chrom_len, int n_chrom, uint32_t res, size_t max_nnz, mk_norm **out) {
    if (!out || !chrom_len || n_chrom <= 0 || res == 0) { mk_set_error("mk_norm_create: bad argument"); return MK_ERR_ARG; }
    if (max_nnz >= (1ull << 30)) { mk_set_error("mk_norm_create: max_nnz %zu: at most 2^30 - 1 entries (one radix sort call)", max_nnz); return MK_ERR_CAPACITY; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { mk_set_error("no CUDA device: microcket_b200 has no CPU fallback"); return MK_ERR_CUDA; }
    MK_CUDA(cudaSetDevice(device));
    std::vector<u32> off(n_chrom + 1, 0);
    u64 nb = 0;
    for (int c = 0; c < n_chrom; ++c) { nb += chrom_len[c] / res + 1; if (nb >= (1ull << 31)) { mk_set_error("mk_norm_create: more than 2^31 bins"); return MK_ERR_CAPACITY; } off[c + 1] = (u32)nb; }
    mk_norm *h = new mk_norm();
    h->device = device; h->sms = mk_sm_count(device); h->n_chrom = n_chrom; h->res = res; h->nb = (u32)nb; h->max_nnz = max_nnz; h->chr_off = off;
    h->ns = (u32)((nb + NM_GS - 1) / NM_GS);
    std::vector<u32> cob(nb);
    for (int c = 0; c < n_chrom; ++c) for (u32 r = off[c]; r < off[c + 1]; ++r) cob[r] = (u32)c;
    const size_t m = std::max<size_t>(max_nnz, 1);
    int rc = MK_OK;
    auto A = [&](DevBuf &b, size_t bytes) { if (rc == MK_OK) rc = b.alloc(bytes); };
    A(h->d_chr_of_bin, nb * 4); A(h->d_chr_off, (n_chrom + 1) * 4); A(h->d_row_ptr, (nb + 1) * 8); A(h->d_runs, 4 * nb * 4);
    A(h->d_ents, 2 * m * 8); A(h->d_keys[0], m * 8); A(h->d_keys[1], m * 8); A(h->d_vals[0], m * 4); A(h->d_vals[1], m * 4);
    A(h->d_desc, ((nb + NP_T * NP_ITEMS - 1) / (NP_T * NP_ITEMS) + 2) * 8); A(h->d_small, 64);
    A(h->d_vecs, 10 * nb * 8); A(h->d_kept, nb); A(h->d_cmd, n_chrom * sizeof(NormCmd)); A(h->d_res, n_chrom * sizeof(NormRes));
    A(h->d_f, n_chrom * 8); A(h->d_krok, n_chrom); A(h->d_seg0, nb * 4); A(h->d_gpart, (3 * (size_t)h->ns + 1) * sizeof(NormPart));
    if (rc == MK_OK) rc = h->rws.alloc(m);
    if (rc == MK_OK) rc = h->h_cmd.alloc(n_chrom * sizeof(NormCmd));
    if (rc == MK_OK) rc = h->h_res.alloc(n_chrom * sizeof(NormRes));
    if (rc == MK_OK) rc = h->h_f.alloc(n_chrom * 8);
    if (rc == MK_OK) rc = h->h_gpart.alloc(((size_t)h->ns + 1) * sizeof(NormPart));
    if (rc == MK_OK && cudaMemset(h->d_seg0.p, 0, nb * 4) != cudaSuccess) { mk_set_error("mk_norm_create: cudaMemset"); rc = MK_ERR_CUDA; }
    if (rc == MK_OK && (cudaMemcpy(h->d_chr_of_bin.p, cob.data(), nb * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
                        cudaMemcpy(h->d_chr_off.p, off.data(), (n_chrom + 1) * 4, cudaMemcpyHostToDevice) != cudaSuccess)) { mk_set_error("mk_norm_create: table upload failed"); rc = MK_ERR_CUDA; }
    for (int k = 0; k < 4 && rc == MK_OK; ++k) if (cudaEventCreate(&h->ev[k]) != cudaSuccess) { mk_set_error("mk_norm_create: cudaEventCreate"); rc = MK_ERR_CUDA; }
    if (rc != MK_OK) { delete h; return rc; }
    *out = h;
    return MK_OK;
}

extern "C" void mk_norm_destroy(mk_norm *h) { if (h) { cudaSetDevice(h->device); delete h; } }
extern "C" uint64_t mk_norm_launch_count(mk_norm *h) { return h ? h->launches : 0; }
extern "C" int mk_norm_enable_timing(mk_norm *h, int on) {
    if (!h) { mk_set_error("mk_norm_enable_timing: null"); return MK_ERR_ARG; }
    h->timing = on != 0;
    for (int k = 0; k < 8; ++k) { h->ms[k] = 0; h->count[k] = 0; }
    return MK_OK;
}
extern "C" int mk_norm_kernel_times(mk_norm *h, double *ms, uint64_t *count) {
    if (!h || !ms || !count) { mk_set_error("mk_norm_kernel_times: bad argument"); return MK_ERR_ARG; }
    for (int k = 0; k < 8; ++k) { ms[k] = h->ms[k]; count[k] = h->count[k]; }
    return MK_OK;
}

static double nm_elapsed(cudaEvent_t a, cudaEvent_t b) { float t = 0; cudaEventElapsedTime(&t, a, b); return t; }

// symmetric CSR of the entries in h->scope
static int nm_build(mk_norm *h, const char *who, const u32 *b1, const u32 *b2, const u32 *cnt, u64 nnz, cudaStream_t s) {
    const u32 nb = h->nb;
    u32 *runs = h->d_runs.as<u32>();
    u32 *row_start = runs, *up_end = runs + nb, *low_start = runs + 2 * (size_t)nb, *low_end = runs + 3 * (size_t)nb;
    u32 *err = h->d_small.as<u32>();
    unsigned long long *n_low = (unsigned long long *)(h->d_small.as<char>() + 8);
    u32 *ticket = (u32 *)(h->d_small.as<char>() + 16);
    const u32 *cob = h->d_chr_of_bin.as<u32>(), *coff = h->d_chr_off.as<u32>();
    if (h->timing) MK_CUDA(cudaEventRecord(h->ev[0], s));
    MK_CUDA(cudaMemsetAsync(runs, 0, 4 * (size_t)nb * 4, s));
    MK_CUDA(cudaMemsetAsync(h->d_small.p, 0, 64, s));
    MK_CUDA(cudaMemsetAsync(h->d_kept.p, 0, nb, s));
    if (nnz) {
        auto classify = h->scope == NM_GENOME ? k_nm_classify<NM_GENOME> : h->scope == NM_INTER ? k_nm_classify<NM_INTER> : k_nm_classify<NM_INTRA>;
        classify<<<h->grid(nnz, NM_T), NM_T, 0, s>>>(b1, b2, nnz, nb, cob, coff, row_start, up_end, h->d_keys[0].as<u64>(), err, n_low);
        h->launches += 1;
        u32 e = 0;
        MK_CUDA(cudaMemcpyAsync(&e, err, 4, cudaMemcpyDeviceToHost, s));
        MK_CUDA(cudaStreamSynchronize(s));
        MK_CUDA(cudaGetLastError());
        if (e & 1u) { mk_set_error("%s: an entry with bin1 > bin2 (the COO must be an upper triangle)", who); return MK_ERR_ARG; }
        if (e & 2u) { mk_set_error("%s: a bin at or beyond the %u bins of resolution %u", who, nb, h->res); return MK_ERR_ARG; }
        if (e & 4u) { mk_set_error("%s: the COO is not sorted by (bin1, bin2)", who); return MK_ERR_ARG; }
        RadixSchedule sch; sch.n_pass = 0;
        for (u64 v = nb; v; v >>= 8) { sch.byte_of[sch.n_pass] = sch.n_pass; ++sch.n_pass; }   // keys <= nb
        KV64::Bufs kb; kb.k[0] = h->d_keys[0].as<u64>(); kb.k[1] = h->d_keys[1].as<u64>(); kb.v[0] = h->d_vals[0].as<u32>(); kb.v[1] = h->d_vals[1].as<u32>();
        MK_TRY(radix_sort<KV64>(kb, nnz, sch, h->rws, 1, h->sms, s, &h->launches));
        const RadixPlan *plan = h->rws.plan.as<RadixPlan>();
        k_nm_lower_runs<<<h->grid(nnz, NM_T), NM_T, 0, s>>>(plan, kb.k[0], kb.k[1], n_low, low_start, low_end);
        h->launches += 1;
    }
    const u64 n_tiles = ((u64)nb + NP_T * NP_ITEMS - 1) / (NP_T * NP_ITEMS);
    MK_CUDA(cudaMemsetAsync(h->d_desc.p, 0, (n_tiles + 1) * 8, s));
    k_nm_row_ptr<<<(int)std::min<u64>((u64)h->sms * 8, n_tiles), NP_T, 0, s>>>(nb, row_start, up_end, low_start, low_end, h->d_row_ptr.as<u64>(), h->d_desc.as<u64>(), ticket);
    h->launches += 1;
    if (nnz) {
        auto fill_upper = h->scope == NM_GENOME ? k_nm_fill_upper<NM_GENOME> : h->scope == NM_INTER ? k_nm_fill_upper<NM_INTER> : k_nm_fill_upper<NM_INTRA>;
        fill_upper<<<h->grid(nnz, NM_T), NM_T, 0, s>>>(b1, b2, cnt, nnz, cob, coff, h->d_row_ptr.as<u64>(), row_start, low_start, low_end, h->d_ents.as<uint2>());
        k_nm_fill_lower<<<h->grid(nnz, NM_T), NM_T, 0, s>>>(h->rws.plan.as<RadixPlan>(), h->d_keys[0].as<u64>(), h->d_keys[1].as<u64>(), h->d_vals[0].as<u32>(),
                                                             h->d_vals[1].as<u32>(), n_low, b1, cnt, h->d_row_ptr.as<u64>(), low_start, h->d_ents.as<uint2>());
        h->launches += 2;
    }
    if (h->timing) {
        MK_CUDA(cudaEventRecord(h->ev[1], s));
        MK_CUDA(cudaEventSynchronize(h->ev[1]));
        h->ms[0] += nm_elapsed(h->ev[0], h->ev[1]); h->count[0] += 1;
    }
    MK_CUDA(cudaGetLastError());
    return MK_OK;
}

// One step for every segment: commands up, pre -> product -> post, results down.  nvec: the vector of OP_SUMF.
// Timing slots: in_kr ? (1 product, 2 pre + post) : (4 product, 5 pre + post).
static int nm_step(mk_norm *h, const double *nvec, bool in_kr, cudaStream_t s) {
    const NormVecs V = h->vecs();
    const u32 *seg = h->seg_of_bin();
    const NormCmd *cmd = h->d_cmd.as<NormCmd>();
    const int op0 = h->h_cmd.as<NormCmd>()[0].op;
    MK_CUDA(cudaMemcpyAsync(h->d_cmd.p, h->h_cmd.p, h->n_seg() * sizeof(NormCmd), cudaMemcpyHostToDevice, s));
    if (h->timing) MK_CUDA(cudaEventRecord(h->ev[0], s));
    k_nm_pre<<<h->grid(h->nb, NM_T), NM_T, 0, s>>>(h->nb, seg, cmd, V, nvec);
    if (h->timing) MK_CUDA(cudaEventRecord(h->ev[1], s));
    k_nm_spmv<<<h->grid(h->nb, NM_T / 32), NM_T, 0, s>>>(h->d_row_ptr.as<u64>(), h->d_ents.as<uint2>(), h->nb, seg, cmd, V.u, V.au);
    if (h->timing) MK_CUDA(cudaEventRecord(h->ev[2], s));
    if (h->scope == NM_INTRA) {
        k_nm_post<<<h->n_chrom, NM_RT, 0, s>>>(h->d_chr_off.as<u32>(), cmd, V, h->d_res.as<NormRes>());
        h->launches += 3;
    } else {
        const int phases = op0 == OP_CG_FIRST || op0 == OP_CG_NEXT ? 3 : 1;
        for (int ph = 0; ph < phases; ++ph) k_nm_gpost<<<h->grid(h->ns, 1), NM_T, 0, s>>>(ph, h->nb, cmd, V, h->d_gpart.as<NormPart>());
        h->launches += 2 + phases;
    }
    if (h->timing) MK_CUDA(cudaEventRecord(h->ev[3], s));
    if (h->scope == NM_INTRA) MK_CUDA(cudaMemcpyAsync(h->h_res.p, h->d_res.p, h->n_chrom * sizeof(NormRes), cudaMemcpyDeviceToHost, s));
    else MK_CUDA(cudaMemcpyAsync(h->h_gpart.p, h->d_gpart.as<NormPart>() + 2 * (size_t)h->ns, ((size_t)h->ns + 1) * sizeof(NormPart), cudaMemcpyDeviceToHost, s));
    MK_CUDA(cudaStreamSynchronize(s));
    MK_CUDA(cudaGetLastError());
    if (h->scope != NM_INTRA && op0 != OP_IDLE) nm_gres(op0, h->h_gpart.as<NormPart>(), h->ns, h->h_res.as<NormRes>());
    if (h->timing) {
        const int a = in_kr ? 1 : 4;
        h->ms[a] += nm_elapsed(h->ev[1], h->ev[2]); h->count[a] += 1;
        h->ms[a + 1] += nm_elapsed(h->ev[0], h->ev[1]) + nm_elapsed(h->ev[2], h->ev[3]); h->count[a + 1] += 1;
    }
    return MK_OK;
}

struct KrState {                 // bnewt's scalars of one chromosome
    int op = OP_IDLE, outer = 0, inner = 0;
    double rho_km1 = 0, rho_km2 = 0, rout = 0, rold = 0, eta = KR_ETAMAX, innertol = 0;
    bool done = false, failed = false;
};

// Knight-Ruiz for every segment with kept rows, in lockstep; kr_ok[c] = 1 for the balanced ones
static int nm_kr(mk_norm *h, const std::vector<double> &kept_rows, std::vector<u8> &kr_ok, mk_norm_stats *st, cudaStream_t s) {
    const int nc = h->n_seg();
    const double rt = KR_TOL * KR_TOL, stop_tol = 0.5 * KR_TOL;
    std::vector<KrState> k(nc);
    int active = 0;
    for (int c = 0; c < nc; ++c) if (kept_rows[c] > 0) { k[c].op = OP_KR_INIT; ++active; }
    NormCmd *cmd = h->h_cmd.as<NormCmd>();
    const NormRes *res = h->h_res.as<NormRes>();
    const auto t0 = std::chrono::steady_clock::now();
    u32 steps = 0;
    while (active) {
        for (int c = 0; c < nc; ++c) { cmd[c].op = k[c].op; cmd[c].pad = 0; cmd[c].beta = k[c].rho_km2 != 0 ? k[c].rho_km1 / k[c].rho_km2 : 0.0; cmd[c].rho = k[c].rho_km1; }
        MK_TRY(nm_step(h, nullptr, true, s));
        ++steps;
        for (int c = 0; c < nc; ++c) {
            KrState &q = k[c];
            if (q.op == OP_IDLE) continue;
            const NormRes &r = res[c];
            bool fail = false;
            if (q.op == OP_KR_INIT || q.op == OP_KR_OUTER) {
                if (q.op == OP_KR_OUTER && (r.flag || !(r.b > 0.0))) fail = true;            // some x_i <= 0 or not finite
                else {
                    q.rho_km1 = q.rout = r.a;
                    if (q.op == OP_KR_INIT) q.rold = q.rout;
                    else {
                        const double rat = q.rout / q.rold, eta_o = q.eta;
                        q.rold = q.rout; q.eta = KR_G * rat;
                        if (KR_G * eta_o * eta_o > 0.1) q.eta = std::max(q.eta, KR_G * eta_o * eta_o);
                        q.eta = std::max(std::min(q.eta, KR_ETAMAX), stop_tol / std::sqrt(q.rout));
                    }
                    if (!std::isfinite(q.rout)) fail = true;
                    else if (!(q.rout > rt)) q.done = true;
                    else if (q.outer == KR_MAX_OUTER) fail = true;                       // not converged after 100 outer steps
                    else {
                        // a new outer step; its inner loop always starts: eta <= 0.1 and rout > rt put innertol below rout
                        ++q.outer; q.inner = 1; q.innertol = std::max(q.eta * q.eta * q.rout, rt); q.op = OP_CG_FIRST;
                    }
                }
            } else if (r.flag == ST_FAIL) fail = true;
            else if (r.flag == ST_CG_BREAK) q.op = OP_KR_OUTER;
            else {
                q.rho_km2 = r.a; q.rho_km1 = r.b;
                if (!std::isfinite(q.rho_km1)) fail = true;
                else if (q.rho_km1 > q.innertol) { if (++q.inner > KR_MAX_INNER) fail = true; else q.op = OP_CG_NEXT; }
                else q.op = OP_KR_OUTER;
            }
            if (fail) q.failed = true;
            if (q.done || q.failed) { q.op = OP_IDLE; --active; }
        }
    }
    if (h->timing) {
        h->ms[3] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        h->count[3] += steps;
    }
    st->kr_matvecs = steps;
    for (int c = 0; c < nc; ++c) {
        if (kept_rows[c] <= 0) continue;
        st->kr_outer_max = std::max<u32>(st->kr_outer_max, (u32)k[c].outer);
        if (k[c].failed) st->kr_failed += 1;
        else { kr_ok[c] = 1; st->kr_residual_max = std::max(st->kr_residual_max, std::sqrt(k[c].rout)); }
    }
    return MK_OK;
}

// One call in h->scope: CSR, row sums, KR, the requested vectors with their sum factors.  status: n_seg() values.
static int nm_run(mk_norm *h, const char *who, const u32 *d_bin1, const u32 *d_bin2, const u32 *d_cnt, size_t nnz, int types,
                  double *d_vc, double *d_vc_sqrt, double *d_kr, uint8_t *status, mk_norm_stats *stats, cudaStream_t s) {
    if (nnz > h->max_nnz) { mk_set_error("%s: %zu entries, capacity %zu", who, nnz, h->max_nnz); return MK_ERR_CAPACITY; }
    MK_CUDA(cudaSetDevice(h->device));
    const int nc = h->n_seg();
    const u32 nb = h->nb;
    mk_norm_stats st; st.kr_outer_max = 0; st.kr_matvecs = 0; st.kr_failed = 0; st.kr_residual_max = 0.0;
    MK_TRY(nm_build(h, who, d_bin1, d_bin2, d_cnt, nnz, s));
    // row sums: VC, the raw totals of the sum factors, the rows KR keeps
    NormCmd *cmd = h->h_cmd.as<NormCmd>();
    const NormRes *res = h->h_res.as<NormRes>();
    for (int c = 0; c < nc; ++c) cmd[c] = NormCmd{OP_ONES, 0, 0.0, 0.0};
    MK_TRY(nm_step(h, nullptr, false, s));
    std::vector<double> raw(nc), kept_rows(nc);
    for (int c = 0; c < nc; ++c) { raw[c] = res[c].a; kept_rows[c] = res[c].b; }
    std::vector<u8> kr_ok(nc, 0);
    if (types & MK_NORM_KR) MK_TRY(nm_kr(h, kept_rows, kr_ok, &st, s));
    MK_CUDA(cudaMemcpyAsync(h->d_krok.p, kr_ok.data(), nc, cudaMemcpyHostToDevice, s));
    const NormVecs V = h->vecs();
    const u32 *seg = h->seg_of_bin();
    const int kinds[3] = {MK_NORM_VC, MK_NORM_VC_SQRT, MK_NORM_KR};
    double *outs[3] = {d_vc, d_vc_sqrt, d_kr};
    for (int t = 0; t < 3; ++t) {
        if (!(types & kinds[t])) continue;
        if (h->timing) MK_CUDA(cudaEventRecord(h->ev[0], s));
        k_nm_finish<<<h->grid(nb, NM_T), NM_T, 0, s>>>(t, nb, seg, h->d_krok.as<u8>(), V, outs[t]);
        if (h->timing) MK_CUDA(cudaEventRecord(h->ev[1], s));
        h->launches += 1;
        if (h->timing) { MK_CUDA(cudaEventSynchronize(h->ev[1])); h->ms[5] += nm_elapsed(h->ev[0], h->ev[1]); h->count[5] += 1; }
        // sum factor: n <- n sqrt(nrm / raw), nrm = sum over valid entries of c / (n_x n_y) (both halves = upper x 2 off the diagonal)
        for (int c = 0; c < nc; ++c) cmd[c] = NormCmd{(raw[c] > 0 && (t < 2 || kr_ok[c])) ? OP_SUMF : OP_IDLE, 0, 0.0, 0.0};
        MK_TRY(nm_step(h, outs[t], false, s));
        double *f = h->h_f.as<double>();
        for (int c = 0; c < nc; ++c) f[c] = cmd[c].op == OP_SUMF ? std::sqrt(res[c].a / raw[c]) : 1.0;
        MK_CUDA(cudaMemcpyAsync(h->d_f.p, f, nc * 8, cudaMemcpyHostToDevice, s));
        k_nm_scale<<<h->grid(nb, NM_T), NM_T, 0, s>>>(nb, seg, h->d_f.as<double>(), outs[t]);
        h->launches += 1;
    }
    MK_CUDA(cudaStreamSynchronize(s));
    MK_CUDA(cudaGetLastError());
    if (status) for (int c = 0; c < nc; ++c) status[c] = raw[c] <= 0 ? 1 : ((types & MK_NORM_KR) && !kr_ok[c]) ? 2 : 0;
    if (stats) *stats = st;
    return MK_OK;
}

extern "C" int mk_norm_device(mk_norm *h, const uint32_t *d_bin1, const uint32_t *d_bin2, const uint32_t *d_cnt, size_t nnz, int types,
                              double *d_vc, double *d_vc_sqrt, double *d_kr, uint8_t *chrom_status, mk_norm_stats *stats, void *stream) {
    if (!h || (nnz && (!d_bin1 || !d_bin2 || !d_cnt)) || (types & ~(MK_NORM_VC | MK_NORM_VC_SQRT | MK_NORM_KR)) ||
        ((types & MK_NORM_VC) && !d_vc) || ((types & MK_NORM_VC_SQRT) && !d_vc_sqrt) || ((types & MK_NORM_KR) && !d_kr)) {
        mk_set_error("mk_norm_device: bad argument"); return MK_ERR_ARG;
    }
    h->scope = NM_INTRA;
    return nm_run(h, "mk_norm_device", d_bin1, d_bin2, d_cnt, nnz, types, d_vc, d_vc_sqrt, d_kr, chrom_status, stats, (cudaStream_t)stream);
}

extern "C" int mk_norm_genome_device(mk_norm *h, const uint32_t *d_bin1, const uint32_t *d_bin2, const uint32_t *d_cnt, size_t nnz, int scope,
                                     int types, double *d_vc, double *d_kr, uint8_t *status, mk_norm_stats *stats, void *stream) {
    // no VC_SQRT: juicer has no genome-wide or inter-chromosomal form of it
    if (!h || (nnz && (!d_bin1 || !d_bin2 || !d_cnt)) || (scope != MK_NORM_SCOPE_GW && scope != MK_NORM_SCOPE_INTER) ||
        (types & ~(MK_NORM_VC | MK_NORM_KR)) || ((types & MK_NORM_VC) && !d_vc) || ((types & MK_NORM_KR) && !d_kr)) {
        mk_set_error("mk_norm_genome_device: bad argument"); return MK_ERR_ARG;
    }
    h->scope = scope;
    return nm_run(h, "mk_norm_genome_device", d_bin1, d_bin2, d_cnt, nnz, types, d_vc, nullptr, d_kr, status, stats, (cudaStream_t)stream);
}
