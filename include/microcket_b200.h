/*
 * microcket_b200.h — C ABI of libmicrocket_b200.so, the B200-native (sm_100a)
 * implementation of Microcket's post-alignment hot path.
 *
 * The reference (hellosunking/Microcket v1.4) has no in-process API for this
 * path: its boundary is process + argv + stdio (SURVEY.md §8b).  Each group of
 * entry points below therefore replaces one reference *program*; the drop-in
 * executables built from microcket_b200/csrc/cli_*.cpp are thin argv/stdio
 * shells over these calls (see INTEGRATION.md).
 *
 *   mk_s2p_*    replaces  src/sam2pairs/sam2pairs.cpp:23-229 (main: argv
 *               :33-54, batch loop :143-190, log :195-219) with
 *               pairutil.h:63-208, flash2pairs.h:17-155, unc2pairs.h:16-358
 *   mk_dedup_*  replaces  src/preprocess/krmdup.cpp:278-397 (main) with
 *               load_batch :88-149 and do_rmdup :151-227; also
 *               src/preprocess/krmdup.pipe.cpp (same algorithm, stdout)
 *   mk_pairs_*  coordinate-keyed duplicate removal + binning of packed pairs;
 *               replaces the `juicer_tools pre` call at microcket:525-529 up
 *               to COO counts (no reference source exists: parity unpinned)
 *
 * Conventions: plain C types only; caller-owned host buffers; callee-owned
 * device memory; return 0 = ok, negative = error (text from mk_last_error(),
 * thread-local).  A context is bound to one GPU and is not thread-safe;
 * distinct contexts are independent.  Every compute entry point needs a CUDA
 * device: there is no CPU fallback.
 */
#ifndef MICROCKET_B200_H
#define MICROCKET_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MK_OK             0
#define MK_ERR_ARG       -1
#define MK_ERR_CUDA      -2
#define MK_ERR_NOMEM     -3
#define MK_ERR_CAPACITY  -4   /* an internal per-window capacity was exceeded (lines, output bytes, carry) */
#define MK_ERR_STATE     -5
#define MK_ERR_INPUT     -6   /* malformed input the reference itself is undefined on */

typedef struct mk_ctx mk_ctx;

const char *mk_last_error(void);
int  mk_version(void);
int  mk_device_count(void);          /* CUDA devices visible; 0 when there is no GPU (no error) */
void mk_destroy(mk_ctx *);
int  mk_copy_device(void *d_dst, const void *d_src, size_t nbytes);   /* synchronous device-to-device copy between raw pointers */
/* raw device / pinned host memory and synchronous copies, for host programs built without the CUDA toolkit (the CLIs) */
int  mk_dev_alloc(int device, size_t nbytes, void **d_ptr);
void mk_dev_free(void *d_ptr);
int  mk_host_alloc(size_t nbytes, void **h_ptr);
void mk_host_free(void *h_ptr);
int  mk_copy_to_device(void *d_dst, const void *h_src, size_t nbytes);
int  mk_copy_to_host(void *h_dst, const void *d_src, size_t nbytes);

/* ------------------------------------------------------------------ packed pair record (16 B) */
typedef struct {
    uint32_t pos1, pos2;   /* 1-based 5' ends, after the reference's ordering rule (unc2pairs.h:310-348) */
    uint16_t chr1, chr2;   /* chromosome ids: index into the table given to / learnt by the context */
    uint8_t  strands;      /* bit0: strand1 == '-', bit1: strand2 == '-' */
    uint8_t  cls;          /* 0 trans, 1 cis10K, 2 cis1K, 3 cis0 (sam2pairs.cpp:211-218 classes) */
    uint16_t lane;         /* sequencing lane / replicate id for `-b` style per-lane dedup (microcket:428-451) */
} mk_pair;

/* ------------------------------------------------------------------ sam2pairs */
typedef struct {
    int   mode;              /* 0 = flash (stitched reads), 1 = unc (paired reads): argv[2], sam2pairs.cpp:57-67 */
    float min_mapped_ratio;  /* argv[5], default 0.5 (pairutil.h:52) — compared in fp32 like the reference */
    int   min_mapq;          /* argv[6], default 10 (pairutil.h:50) */
    int   write_sam;         /* argv[7]: pass through the kept lines of every emitted group */
    int   emu_threads;       /* argv[4] (T >= 2): reproduces the reference's selfCircle log value, which only
                                counts thread 0's share of each 2^18-group batch (sam2pairs.cpp:150,172,202-210) */
    int   device;            /* CUDA device ordinal */
    int   emit_text;         /* produce .pairs text lines (stdout of the reference) */
    int   emit_packed;       /* produce mk_pair records for the fused dedup/binning path */
    size_t window_bytes;     /* bytes of SAM text per device window; 0 = default (256 MiB) */
    uint16_t lane;           /* stamped into mk_pair.lane */
    int   sharded;           /* 1: this context sees one shard of a larger stream; the selfCircle log value is
                                settled in mk_s2p_finish_sharded once the global group indices are known */
    /* SAM-space krmdup (SURVEY 8f-4): the duplicate removal src/preprocess/krmdup.cpp does on the FASTQ before alignment,
     * taken on the SAM instead.  A read pair = a run of consecutive lines with one QNAME; its key = bases [hskip, hskip+klen)
     * of each mate (krmdup.cpp:168-193) read from the SEQ column of the primary records (reverse-complemented back when
     * flag & 16; a stitched read stands for mate 1, its reverse complement for mate 2).  First occurrence in file order
     * wins over the whole stream (krmdup.cpp:201-212); later ones, short mates and non-ACGT key bases are removed BEFORE
     * grouping, so text / log / packed pairs are those of sam2pairs on the alignment of krmdup's output.  The fields must
     * be tab separated (SAM spec).  mk_s2p_rmdup_stats gives krmdup's log. */
    int   rmdup;
    uint64_t rmdup_capacity; /* read pairs the key table is sized for (the whole stream); 0 = 16 M.  16 bytes x 2 slots per pair */
    int   hskip1, klen1, hskip2, klen2;   /* krmdup -k -s -K -S; defaults 5,16,5,16 */
} mk_s2p_cfg;

typedef struct {
    uint32_t lowMap, manyHits, unpaired, selfCircle, trans, cis10K, cis1K, cis0; /* log order, sam2pairs.cpp:211-218 */
    uint64_t selfCircle_true;  /* every self-circle, not only emulated thread 0's */
    uint64_t groups;           /* read groups processed (the stream's last group is not, pairutil.h:176) */
    uint64_t lines;            /* SAM lines seen (headers included) */
    uint64_t cigar_errors;     /* groups dropped where the reference's cigar2segment returns false (UB there) */
    uint64_t pairs;            /* pair lines emitted */
} mk_s2p_stats;

void mk_s2p_default_cfg(mk_s2p_cfg *);
/* chrom_names may be NULL/0: names are then learnt from the RNAME column (any name is accepted,
 * order is bytewise like std::string::compare).  Pre-registered names get ids 0..n-1. */
int  mk_s2p_create(const mk_s2p_cfg *, const char *const *chrom_names, int n_chrom, mk_ctx **);
/* Host streaming API (what the sam2pairs CLI uses).  `sam_bytes` may be split anywhere; the
 * library carries partial lines and the trailing read group over to the next call.  Pageable memory is copied before
 * the call returns.  Memory that is already pinned (cudaHostAlloc / cudaHostRegister) is DMA'd straight from the
 * caller's buffer, asynchronously: it must stay valid and unchanged until mk_s2p_finish (or mk_s2p_reset) returns. */
int  mk_s2p_push(mk_ctx *, const char *sam_bytes, size_t n, int is_last);
/* Drains produced output; *n_out == 0 and *n_out2 == 0 when nothing is pending.  Either buffer may be NULL. */
int  mk_s2p_pull(mk_ctx *, char *pairs_out, size_t cap, size_t *n_out,
                 char *sam_out, size_t cap2, size_t *n_out2);
int  mk_s2p_pull_packed(mk_ctx *, mk_pair *recs, size_t cap, size_t *n);
int  mk_s2p_finish(mk_ctx *, mk_s2p_stats *);
/* Sharded finish: this context processed groups [group_base, group_base + stats.groups) of a stream of
 * total_groups processed groups (multi-GPU: bases from an all-gather of per-rank group counts). */
int  mk_s2p_finish_sharded(mk_ctx *, uint64_t group_base, uint64_t total_groups, mk_s2p_stats *);
struct mk_dedup_stats_s;
/* cfg.rmdup: Total / Uniq / Dup / Discard of krmdup's log (krmdup.cpp:383-389) for the stream; after mk_s2p_finish */
int  mk_s2p_rmdup_stats(mk_ctx *, struct mk_dedup_stats_s *);
/* Start over on a new input with the same configuration, allocations and chromosome table. */
int  mk_s2p_reset(mk_ctx *);
/* Chromosome table after (or during) a run: id → name. */
int  mk_s2p_chrom_count(mk_ctx *);
int  mk_s2p_chrom_name(mk_ctx *, int id, char *buf, size_t cap);

/* Device-resident API: SAM text already in HBM (d_sam: device pointer, 16-byte aligned, readable up to
 * the next 16-byte boundary past n).  Outputs stay on the device in caller-provided buffers.
 * The text must end with '\n'.  When is_last == 0 the trailing read group is not processed and
 * *consumed tells where it starts.  `stream` is a cudaStream_t (0 = default stream). */
typedef struct {
    char    *d_pairs_text;  size_t pairs_text_cap;   /* may be NULL when emit_text == 0 */
    mk_pair *d_pairs;       size_t pairs_cap;        /* may be NULL when emit_packed == 0 */
    char    *d_sam_text;    size_t sam_text_cap;     /* may be NULL when write_sam == 0 */
    uint64_t *d_line_off;   size_t line_off_cap;     /* optional (NULL): d_line_off[e] = offset in d_pairs_text of emitted pair e's
                                                        line, d_line_off[n_pairs] = pairs_text_len; needs cap >= n_pairs + 1.
                                                        Input of mk_pairs_sort_text_device / mk_pairs_filter_text_device */
    uint64_t line_off_base;                          /* added to every recorded offset (a caller that appends the text of several
                                                        calls to one buffer passes the bytes already there) */
    /* results (host values, valid after the call returns) */
    size_t   pairs_text_len, n_pairs, sam_text_len, consumed;
} mk_s2p_dev_io;
int  mk_s2p_run_device(mk_ctx *, const char *d_sam, size_t n, int is_last, mk_s2p_dev_io *io, void *stream);
/* Multi-GPU: every window's packed pairs are sent to their owners (mk_xchg_*, partition resolution `res`) on a side stream
 * while the next window is parsed; when mk_s2p_run_device returns, the epoch is closed and the caller only has to call
 * mk_xchg_finish_device.  NULL detaches. */
struct mk_xchg;
int  mk_s2p_attach_xchg(mk_ctx *, struct mk_xchg *, uint32_t res);
/* number of kernel launches issued by this context so far (for bench accounting) */
uint64_t mk_launch_count(mk_ctx *);
/* Optional per-kernel device timing with CUDA events on the launching stream (bench.py's roofline figure).
 * ms[k] / count[k]; arrays of 8.  k = 0 newline scan, 1 parse, 2 group, 3 emit, 4 SAM passthrough, 5 scan index (chunk
 * prefix + compaction), 6 the SAM-space krmdup kernel (cfg.rmdup), 7 unused. */
int  mk_s2p_enable_timing(mk_ctx *, int on);
int  mk_s2p_kernel_times(mk_ctx *, double *ms, uint64_t *count);

/* ------------------------------------------------------------------ krmdup */
typedef struct {
    int hskip1, klen1, hskip2, klen2;  /* -k -s -K -S; defaults 5,16,5,16 (krmdup.cpp:231-234); 16 <= klen1+klen2 <= 32 */
    int device;
    size_t window_bytes;               /* bytes of FASTQ per device window; 0 = default */
    int async_pull;                    /* 1: mk_dedup_pull only ENQUEUES its device-to-host copies, so that they run while the next
                                          mk_dedup_push copies its window in (PCIe both ways at once).  The bytes a pull reported are
                                          in the caller's buffers once the NEXT mk_dedup_pull, or mk_dedup_finish, has returned; the
                                          buffers should be pinned.  0 (default): they are there when the pull returns. */
} mk_dedup_cfg;
typedef struct mk_dedup_stats_s { uint32_t uniq, dup, discard; uint64_t pairs; } mk_dedup_stats;   /* krmdup.cpp:383-389 */

void mk_dedup_default_cfg(mk_dedup_cfg *);
int  mk_dedup_create(const mk_dedup_cfg *, mk_ctx **);
/* Pageable memory is copied before the call returns.  Memory that is already pinned (cudaHostAlloc / cudaHostRegister) is
 * DMA'd straight from the caller's buffer and its unconsumed tail (krmdup works in whole 65 536-pair batches) is left
 * there until the next call: it must stay valid and unchanged until mk_dedup_finish returns. */
int  mk_dedup_push(mk_ctx *, const char *fq_bytes, size_t n, int is_last);
/* read1/read2 records of kept pairs in the reference's file order (per 65 536-pair batch: buckets A,C,G,T;
 * krmdup.cpp:216-226).  For krmdup.pipe interleave the two streams record by record. */
int  mk_dedup_pull(mk_ctx *, char *r1_out, size_t cap1, size_t *n1, char *r2_out, size_t cap2, size_t *n2);
int  mk_dedup_finish(mk_ctx *, mk_dedup_stats *);
int  mk_dedup_reset(mk_ctx *);   /* a new krmdup process on the same allocations: empty key sets, zero counters */
/* Device-resident key path: 64-bit krmdup keys (or any 64-bit keys) already in HBM.
 * keep[i] = 1 iff key i is the first occurrence in index order.  d_keep: n bytes on the device. */
int  mk_dedup_keys_device(int device, const uint64_t *d_keys, size_t n, uint8_t *d_keep,
                          uint64_t *n_unique, void *stream);

/* ------------------------------------------------------------------ packed pairs: dedup + binning */
typedef struct mk_pairs_ws mk_pairs_ws;   /* reusable device workspace */
int  mk_pairs_ws_create(int device, size_t max_pairs, mk_pairs_ws **);
void mk_pairs_ws_destroy(mk_pairs_ws *);
/* Coordinate-keyed duplicate removal over (lane, chr1,pos1,strand1, chr2,pos2,strand2): first in index
 * order wins.  d_pairs is compacted in place to the kept pairs, SORTED by key; *n_kept returns the count. */
int  mk_pairs_dedup_device(mk_pairs_ws *, mk_pair *d_pairs, size_t n, size_t *n_kept, void *stream);
/* Contact counts at one resolution: bin = chrom_bin_offset[chr] + pos / res with offsets the running sum of
 * (len / res + 1) in the given chromosome order; COO triplets sorted by (bin1, bin2), bin1 <= bin2.
 * chrom_id_map (host, may be NULL) maps mk_pair chromosome ids to indices of chrom_len. */
int  mk_pairs_bin_device(mk_pairs_ws *, const mk_pair *d_pairs, size_t n,
                         const uint32_t *chrom_len, int n_chrom, const uint16_t *chrom_id_map, int n_map,
                         uint32_t res, uint32_t *d_bin1, uint32_t *d_bin2, uint32_t *d_cnt, size_t cap,
                         size_t *nnz, void *stream);
/* Both steps with ONE sort: pairs are packed as (bin1, bin2, lane, pos1 % res, pos2 % res, strands) integers, so equal
 * pairs are adjacent (dedup) and every (bin1,bin2) cell is contiguous (binning).  d_pairs is replaced by the kept pairs
 * in that order; the COO counts are those of the kept pairs.  max_lane = largest mk_pair.lane present (0 if unused). */
int  mk_pairs_dedup_bin_device(mk_pairs_ws *, mk_pair *d_pairs, size_t n,
                               const uint32_t *chrom_len, int n_chrom, const uint16_t *chrom_id_map, int n_map,
                               uint32_t res, uint16_t max_lane, uint32_t *d_bin1, uint32_t *d_bin2, uint32_t *d_cnt, size_t cap,
                               size_t *n_kept, size_t *nnz, void *stream);
/* The same call, also reporting WHICH input pairs survive (what a deduplicated .pairs file needs, SURVEY.md §8a D3: the
 * first occurrence in input order wins, like the reference's unordered_set probe, krmdup.cpp:201-212):
 *   d_keep      n bytes (device, may be NULL): keep[i] = 1 iff input pair i is the first of its key
 *   d_kept_idx  n x u32 (device, may be NULL): input index of every kept pair, in the key order of the kept pairs
 * Pairs that cannot be keyed (chromosome id outside the table, position past the chromosome end, lane > max_lane) are
 * left out of both outputs and counted: mk_pairs_dropped() returns the count of the last call. */
int  mk_pairs_dedup_bin_indexed_device(mk_pairs_ws *, mk_pair *d_pairs, size_t n,
                               const uint32_t *chrom_len, int n_chrom, const uint16_t *chrom_id_map, int n_map,
                               uint32_t res, uint16_t max_lane, uint32_t *d_bin1, uint32_t *d_bin2, uint32_t *d_cnt, size_t cap,
                               uint8_t *d_keep, uint32_t *d_kept_idx, size_t *n_kept, size_t *nnz, void *stream);
uint64_t mk_pairs_dropped(mk_pairs_ws *);
/* .pairs text of the kept pairs in the order the driver's `LANG=C sort -k2,2d -k4,4d -k3,3n -k5,5n` (microcket:480,484,502,
 * 506,514) produces: chromosome names under sort's dictionary rule (chrom_rank[id], from mk_pairs_chrom_ranks), positions
 * numerically, ties by whole-line bytewise comparison (GNU sort's last resort).  d_pairs / d_pairs_text / d_line_off are the
 * outputs of one mk_s2p_run_device call (emission order); d_keep (may be NULL = all) is mk_pairs_dedup_bin_indexed_device's
 * mask.  max_pos: largest position present (chromosome length bound; 0 = 32 bits).  Replaces that sort process. */
int  mk_pairs_sort_text_device(mk_pairs_ws *, const mk_pair *d_pairs, size_t n, const uint8_t *d_keep,
                               const char *d_pairs_text, const uint64_t *d_line_off, const uint16_t *chrom_rank, int n_ids,
                               uint32_t max_pos, char *d_out, size_t out_cap, size_t *out_len, size_t *n_lines, void *stream);
/* The lines of the kept pairs in input order (deduplicated, unsorted). */
int  mk_pairs_filter_text_device(mk_pairs_ws *, size_t n, const uint8_t *d_keep, const char *d_pairs_text,
                                 const uint64_t *d_line_off, char *d_out, size_t out_cap, size_t *out_len, void *stream);
/* A `.pairs` file's text (anno/4DN.DCIC.header:2 columns; d_text 16-byte aligned, ending with '\n', < 4 GiB per call) to
 * packed pairs on the device: d_out[i] = line i.  Header lines ('#'), malformed lines and chromosome names outside
 * chrom_names get chromosome id 0xFFFF, which the dedup / binning / histogram calls leave out and count. */
int  mk_pairs_parse_text_device(mk_pairs_ws *, const char *d_text, size_t n_bytes, const char *const *chrom_names, int n_chrom,
                                mk_pair *d_out, size_t cap, size_t *n_lines, size_t *n_skipped, void *stream);
/* rank[i] of names[i] under `sort -d` in the C locale (only blanks and alphanumerics compare); equal keys share a rank */
int  mk_pairs_chrom_ranks(const char *const *names, int n, uint16_t *rank);
/* Multi-GPU: group pairs by owner rank = mix(chr1, chr2, pos1 / res) mod world into d_out (segments in rank order;
 * counts[r] pairs for rank r).  The caller moves the segments with an all-to-all (NCCL via torch.distributed in
 * bench.py); afterwards equal keys and equal (bin1,bin2) cells at `res` are on one rank. */
int  mk_pairs_partition_device(mk_pairs_ws *, const mk_pair *d_pairs, size_t n, int world, uint32_t res, mk_pair *d_out,
                               uint64_t *counts, void *stream);
uint32_t mk_pairs_owner(uint32_t chr1, uint32_t chr2, uint32_t pos1, uint32_t res, uint32_t world);
/* Host-buffer form of the two calls above (pairs2bins CLI, end-to-end measurements): `pairs` is replaced by the kept
 * pairs in key order when do_dedup != 0; COO triplets are written to bin1/bin2/cnt when res != 0. */
int  mk_pairs_dedup_bin_host(mk_pairs_ws *, mk_pair *pairs, size_t n, int do_dedup,
                             const uint32_t *chrom_len, int n_chrom, const uint16_t *chrom_id_map, int n_map, uint32_t res,
                             uint32_t *bin1, uint32_t *bin2, uint32_t *cnt, size_t cap, size_t *n_kept, size_t *nnz);
uint64_t mk_pairs_launch_count(mk_pairs_ws *);

/* ------------------------------------------------------------------ dense multi-resolution histogram */
/* Contact counts of every requested resolution from ONE read of the packed pairs (the `-r` list of microcket:98,176-180 as
 * consumed by `juicer_tools pre`, microcket:525-529): per resolution an upper-triangle u32 matrix in HBM, the diagonals
 * privatised in shared memory, off-diagonal cells as global atomics.  For resolutions whose triangle fits in memory
 * (mk_hist_cells; hg38 at 100 kb: 1.9 GB); finer ones use mk_pairs_bin_device.  d_cells (may be NULL, or hold NULLs):
 * caller-owned, ZEROED matrices — e.g. torch tensors that an NCCL reduce sums across GPUs before mk_hist_coo_device. */
typedef struct mk_hist mk_hist;
int  mk_hist_cells(const uint32_t *chrom_len, int n_chrom, uint32_t res, uint64_t *n_bins, uint64_t *n_cells);
int  mk_hist_create(int device, const uint32_t *chrom_len, int n_chrom, const uint32_t *res, int n_res,
                    uint32_t *const *d_cells, mk_hist **);
void mk_hist_destroy(mk_hist *);
int  mk_hist_reset(mk_hist *, void *stream);                       /* zero every matrix */
/* Adds n pairs to every matrix (may be called once per window).  Pairs with an unknown chromosome id or a position past
 * the chromosome end are left out of EVERY resolution and counted (mk_hist_dropped). */
int  mk_hist_add_device(mk_hist *, const mk_pair *d_pairs, size_t n, const uint16_t *chrom_id_map, int n_map, void *stream);
int  mk_hist_matrix(mk_hist *, int res_idx, uint32_t **d_cells, uint64_t *n_cells, uint64_t *n_bins);
/* Non-zero cells of one resolution as COO triplets sorted by (bin1, bin2), bin1 <= bin2; *total = sum of the counts. */
int  mk_hist_coo_device(mk_hist *, int res_idx, uint32_t *d_bin1, uint32_t *d_bin2, uint32_t *d_cnt, size_t cap,
                        size_t *nnz, uint64_t *total, void *stream);
uint64_t mk_hist_dropped(mk_hist *);
uint64_t mk_hist_launch_count(mk_hist *);

/* ------------------------------------------------------------------ matrix balancing (normalisation vectors) */
/* The VC, VC_SQRT and KR vectors `juicer_tools pre` stores in a .hic (microcket:525-529), per chromosome, from its
 * intra-chromosomal matrix A (symmetric, diagonal counted once; bins as in the COO: len / res + 1 per chromosome).
 *   VC       n_i = sum_j A_ij; VC_SQRT = sqrt(VC); empty rows 0
 *   KR       Knight-Ruiz bnewt (tol 1e-6, delta 0.1, Delta 3, etamax 0.1, g 0.9) on the rows with a nonzero sum, n_i = 1 / x_i;
 *            NaN on the rows left out.  A chromosome FAILS when it has not converged after 100 outer steps, some x_i is <= 0
 *            or not finite, or its matrix has no doubly-stochastic scaling; a failed chromosome's KR entries are all NaN.
 * Every vector is then multiplied per chromosome by juicer's sum factor sqrt(sum c/(n_x n_y) / sum c) over the entries with
 * valid norms (off-diagonal entries twice), so that the normalised matrix sums to the raw one.  No floating-point atomics:
 * the same input gives the same bits.  PARITY UNPINNED (juicer_tools is absent; DESIGN.md §5). */
typedef struct mk_norm mk_norm;
#define MK_NORM_VC       1
#define MK_NORM_VC_SQRT  2
#define MK_NORM_KR       4
typedef struct {
    uint32_t kr_outer_max;      /* most outer (Newton) steps any chromosome (segment) took */
    uint32_t kr_matvecs;        /* lockstep KR steps = products over all unfinished chromosomes at once */
    uint32_t kr_failed;         /* chromosomes whose KR failed */
    double   kr_residual_max;   /* largest ||1 - x (A x)||_2 of the balanced chromosomes */
} mk_norm_stats;
/* One object per resolution; max_nnz: the most COO entries a call may pass (below 2^30: one radix sort call). */
int  mk_norm_create(int device, const uint32_t *chrom_len, int n_chrom, uint32_t res, size_t max_nnz, mk_norm **);
void mk_norm_destroy(mk_norm *);
/* One resolution's COO as mk_pairs_bin_device / mk_hist_coo_device return it (device, sorted by (bin1, bin2), bin1 <= bin2).
 * types: MK_NORM_* bits; d_vc / d_vc_sqrt / d_kr: n_bins doubles each on the device, global bin order (may be NULL when the
 * type is not requested).  chrom_status (host, n_chrom, may be NULL): 0 ok, 1 no intra contacts (no vector of any type),
 * 2 KR failed.  Refused: nnz > max_nnz (MK_ERR_CAPACITY); bin1 > bin2, a bin past the resolution's bins, an unsorted COO
 * (MK_ERR_ARG). */
int  mk_norm_device(mk_norm *, const uint32_t *d_bin1, const uint32_t *d_bin2, const uint32_t *d_cnt, size_t nnz, int types,
                    double *d_vc, double *d_vc_sqrt, double *d_kr, uint8_t *chrom_status, mk_norm_stats *, void *stream);
/* The genome-wide vectors over every bin at once (juicer's GW_VC / GW_KR and INTER_VC / INTER_KR), same COO and object:
 * scope MK_NORM_SCOPE_GW balances the whole-genome matrix (every entry), MK_NORM_SCOPE_INTER its inter-chromosomal entries only
 * (bins in different chromosomes).  One balancing problem over all n_bins rows with the definitions above (KR on the rows
 * with a nonzero sum, one sum factor for the whole genome).  types: MK_NORM_VC and / or MK_NORM_KR (there is no GW / INTER
 * VC_SQRT); d_vc / d_kr: n_bins doubles each on the device, global bin order.  *status (host, may be NULL): 0 ok, 1 the
 * matrix has no entries (no vector of any type), 2 KR failed (no KR vector; VC is still written).  Refused like
 * mk_norm_device, and also for MK_NORM_VC_SQRT, an unknown type bit or an unknown scope (MK_ERR_ARG). */
#define MK_NORM_SCOPE_GW     1
#define MK_NORM_SCOPE_INTER  2
int  mk_norm_genome_device(mk_norm *, const uint32_t *d_bin1, const uint32_t *d_bin2, const uint32_t *d_cnt, size_t nnz, int scope,
                           int types, double *d_vc, double *d_kr, uint8_t *status, mk_norm_stats *, void *stream);
uint64_t mk_norm_launch_count(mk_norm *);
/* Optional timing (tools/norm_bench.py): CUDA events on the stream, host clock for the KR loop.  ms[k] / count[k], arrays of 8:
 * 0 CSR build, 1 products inside KR, 2 KR vector kernels (pre + post), 3 KR loop wall time incl. the host round trips
 * (count = steps), 4 products outside KR (row sums, sum factors), 5 other vector kernels, 6-7 unused. */
int  mk_norm_enable_timing(mk_norm *, int on);
int  mk_norm_kernel_times(mk_norm *, double *ms, uint64_t *count);

/* ------------------------------------------------------------------ BGZF inflate (bgzipped .pairs, BAM) */
/* BGZF (SAMv1 §4.1) is a chain of gzip members, each an independent raw-deflate stream of at most 64 KiB of output whose
 * header gives its compressed size (BSIZE) and whose trailer gives its CRC-32 and output size (ISIZE): mk_bgzf_scan finds
 * the members on the host, mk_bgzf_inflate_device inflates them side by side in HBM (one warp per member). */
typedef struct {
    uint64_t in_off;    /* the member's first byte in the compressed buffer */
    uint64_t out_off;   /* where its output goes in the output buffer: the running sum of ISIZE */
    uint32_t in_len;    /* BSIZE + 1: header, deflate data and trailer */
    uint32_t isize;     /* output bytes (<= 65536) */
} mk_bgzf_member;
/* Walks the member headers at the start of buf (host memory): one entry per WHOLE member, at most cap of them.  Stops at the
 * first incomplete member (or the end of buf, or cap); *n_bytes = bytes the whole members take (may be NULL), *n_out = sum of
 * their ISIZE (may be NULL).  A member that is not BGZF (1f 8b 08 with FLG.FEXTRA, a BC subfield with SLEN 2 among any others,
 * BSIZE covering header and trailer, ISIZE <= 65536) is refused with MK_ERR_INPUT and a message naming its byte offset;
 * plain gzip (no BC subfield) is refused so. */
int  mk_bgzf_scan(const void *buf, size_t n, mk_bgzf_member *members, size_t cap, size_t *n_members, size_t *n_bytes, uint64_t *n_out);
/* A reusable device object for calls of up to max_members members (member table and error word; no allocation per call). */
typedef struct mk_bgzf mk_bgzf;
int  mk_bgzf_create(int device, size_t max_members, mk_bgzf **);
void mk_bgzf_destroy(mk_bgzf *);
/* Inflates members[0..n) (host array, as mk_bgzf_scan returns them) of the compressed bytes at d_in (device) to
 * d_out + out_off (device); checks every member's CRC-32 and ISIZE on the device, and returns when the output is complete.
 * Any input bytes are safe: no read outside a member's in_len bytes, no write outside [out_off, out_off + isize).
 * Damaged members (bad block type, code set or symbol, a distance before the member's start, output past or short of
 * ISIZE, a stream that does not end right before the trailer, a CRC or ISIZE mismatch) give MK_ERR_INPUT naming the first
 * failing member in file order and the reason.  Refused before any launch (MK_ERR_ARG): out_cap below the sum of ISIZE,
 * a member whose output leaves [0, out_cap) or whose sizes break the format's limits; n > max_members (MK_ERR_CAPACITY).
 * Byte-identical to zlib on every member zlib accepts; no floating point, no atomics on the output. */
int  mk_bgzf_inflate_device(mk_bgzf *, const void *d_in, const mk_bgzf_member *members, size_t n, void *d_out, size_t out_cap, void *stream);
/* What the last successful call wrote, for text consumers: the number of '\n' bytes, and the offset from d_out of the last
 * one (-1 when there is none). */
int  mk_bgzf_text_stats(mk_bgzf *, uint64_t *newlines, int64_t *last_newline);
uint64_t mk_bgzf_launch_count(mk_bgzf *);

/* ------------------------------------------------------------------ BGZF deflate (bgzip, .pairs.gz output) */
/* The other direction: input bytes in HBM -> BGZF members in HBM, one CTA per member.  Member k holds input bytes
 * [k * 65280, min(n, (k + 1) * 65280)), the cut bgzip makes, and bgzip's header bytes (XLEN 6, one BC subfield).  Levels 1-9
 * (and -1, the default) all write the same bytes: a greedy parse with one match candidate per position and per-member
 * Huffman codes, the smallest of a stored, fixed or dynamic block.  Level 0 writes stored members only.  The bytes depend
 * only on the input and on "level 0 or not": not on the card, the grid, the stream, the input address, or on where a
 * caller cuts its input into calls, as long as the cuts fall on multiples of 65280.  They are this project's own (not
 * htslib's bgzip bytes); zlib, gzip, htslib and mk_bgzf_inflate_device read them back. */
/* Worst-case output bytes for n input bytes (every member stored: n + 31 per member); no EOF member. */
size_t mk_bgzf_deflate_bound(size_t n);
/* A reusable device object for calls of up to max_bytes input bytes (staging, member sizes, scratch; no allocation per call). */
typedef struct mk_bgzf_enc mk_bgzf_enc;
int  mk_bgzf_enc_create(int device, size_t max_bytes, mk_bgzf_enc **);
void mk_bgzf_enc_destroy(mk_bgzf_enc *);
/* Compresses n bytes at d_in (device) into members written back to back at d_out (device); returns when they are complete.
 * *out_len: their bytes; *n_members: their number; members (host, may be NULL): the table mk_bgzf_scan returns on the output.
 * No EOF member is written: the caller appends it (28 bytes, 1f 8b 08 04 00 00 00 00 00 ff 06 00 42 43 02 00 1b 00 03 00 then
 * eight zeros).  Refused before any launch: a null object, pointer or count pointer, level outside -1..9, out_cap below
 * mk_bgzf_deflate_bound(n), a members table smaller than the member count (MK_ERR_ARG); n > max_bytes (MK_ERR_CAPACITY). */
int  mk_bgzf_deflate_device(mk_bgzf_enc *, const void *d_in, size_t n, int level, void *d_out, size_t out_cap, size_t *out_len,
                            mk_bgzf_member *members, size_t members_cap, size_t *n_members, void *stream);
uint64_t mk_bgzf_enc_launch_count(mk_bgzf_enc *);

/* ------------------------------------------------------------------ multi-GPU exchange over NVLink peer memory */
/* One object per rank (one process per GPU, or several ranks in one process).  Owner bucketing and the all-to-all are ONE
 * kernel: owner = mix(chr1, chr2, pos1 / res) mod world (mk_pairs_owner); every rank writes its pairs straight into the
 * owners' receive buffers through peer pointers and publishes an epoch flag there; the consumer waits on the device.
 * Bootstrap: every rank calls mk_xchg_handle, the 128-byte handles are all-gathered by whatever the host program has
 * (torch.distributed, MPI, a file), then mk_xchg_connect.  Ranks inside one process use mk_xchg_connect_local.
 * Choose res = least common multiple of the binning resolutions (5 Mb for microcket:98's default list): every duplicate and
 * every cell of every resolution then has one owner, and nothing else has to cross GPUs.  Arrival order is not
 * deterministic: which of several IDENTICAL packed pairs survives the dedup is not defined across ranks. */
typedef struct mk_xchg mk_xchg;
int  mk_xchg_create(int device, int world, int rank, size_t cap_pairs /* most pairs this rank can own per exchange */, mk_xchg **);
void mk_xchg_destroy(mk_xchg *);
int  mk_xchg_handle(mk_xchg *, void *handle128);
int  mk_xchg_connect(mk_xchg *, const void *all_handles /* world x 128 bytes, rank order */);
int  mk_xchg_connect_local(mk_xchg *const *all /* rank order */, int world);
/* enqueue: this rank's n pairs go to their owners (returns at once; d_pairs may be reused when the stream has passed it) */
int  mk_xchg_scatter_device(mk_xchg *, const mk_pair *d_pairs, size_t n, uint32_t res, void *stream);
/* The same exchange in pieces, overlapped with the producer: mk_xchg_begin, any number of parts (each = the d_part[1] pairs
 * that END at index d_part[0] of d_base, both values on the DEVICE), mk_xchg_end_device; all on one stream.
 * mk_s2p_attach_xchg makes mk_s2p_run_device do exactly this, one part per window, on a side stream of its own. */
int  mk_xchg_begin(mk_xchg *);
int  mk_xchg_scatter_part_device(mk_xchg *, const mk_pair *d_base, const uint64_t *d_part, uint32_t res, void *stream);
int  mk_xchg_end_device(mk_xchg *, void *stream);
/* wait on the device until all ranks have delivered; *d_recv / *n_recv: the pairs this rank owns (inside the object's
 * buffer, valid until the scatter after next; may be modified in place, e.g. by mk_pairs_dedup_bin_device) */
int  mk_xchg_finish_device(mk_xchg *, mk_pair **d_recv, size_t *n_recv, void *stream);
uint64_t mk_xchg_launch_count(mk_xchg *);

/* ------------------------------------------------------------------ synthetic inputs (tests / bench) */
/* Same bytes on host and device for a given (seed, mode, genome, first, count).  mode: 0 flash, 1 unc,
 * 2 interleaved FASTQ.  genome: 0 hg38, 1 mm10.  Returns bytes written in *n_out (or needed when buf == NULL). */
int  mk_synth_host(uint64_t seed, int mode, int genome, uint64_t first, uint64_t count,
                   char *buf, size_t cap, size_t *n_out);
int  mk_synth_device(int device, uint64_t seed, int mode, int genome, uint64_t first, uint64_t count,
                     char *d_buf, size_t cap, size_t *n_out, void *stream);

/* The same generators with the workload mixture exposed (BASELINE configs[2..4], SURVEY.md §8d): per-1024 weights, -1 =
 * default.  dup_per_1024 > 0: a read group (or FASTQ pair) re-uses the fragment of group `hash % dup_universe` — a PCR
 * duplicate with its own read id; set dup_universe to the job's total group count so duplicates cross shards. */
typedef struct {
    int      dup_per_1024;
    uint64_t dup_universe;
    int      chimeric_per_1024;    /* groups with a split alignment (default: unc 256, flash 358) */
    int      noise_per_1024;       /* low MAPQ / unmapped / secondary / odd clips / introns (default 51) */
    int      selfcircle_per_1024;  /* default 5 */
} mk_synth_opts;
void mk_synth_default_opts(mk_synth_opts *);
int  mk_synth_host_ex(uint64_t seed, int mode, int genome, const mk_synth_opts *, uint64_t first, uint64_t count,
                      char *buf, size_t cap, size_t *n_out);
int  mk_synth_device_ex(int device, uint64_t seed, int mode, int genome, const mk_synth_opts *, uint64_t first, uint64_t count,
                        char *d_buf, size_t cap, size_t *n_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif
