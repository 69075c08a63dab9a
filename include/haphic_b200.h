/*
 * haphic_b200 -- C ABI of the B200-native `haphic cluster` hot path.
 *
 * This is the drop-in boundary: a plain C interface (pointers + sizes, no torch / C++ types)
 * that a maintainer of zengxiaofei/HapHiC would bind with ctypes from
 * scripts/HapHiC_cluster.py (see INTEGRATION.md).  The reference has no FFI of its own -- the
 * whole path is in-process Python -- so every entry point below names the reference function
 * (file:line in scripts/HapHiC_cluster.py, v1.0.7) whose work it replaces.
 *
 * Conventions
 *   - every function returns HH_OK (0) or an HH_ERR_* code; hh_last_error() gives the message
 *     (thread-local);
 *   - objects are opaque handles owned by the library until the matching *_destroy;
 *   - `mem` arguments say where a caller buffer lives: HH_MEM_HOST (pageable or pinned host
 *     memory) or HH_MEM_DEVICE (device memory of the context's GPU, e.g. a torch tensor's
 *     data_ptr());  all *_fetch_* outputs are HOST buffers sized by the caller from the
 *     preceding *_info call;
 *   - all calls are synchronous on return unless stated otherwise;
 *   - there is NO CPU fallback: without a CUDA device hh_ctx_create fails.
 *
 * Contig identifiers are dense int32 ids in FASTA order; the host keeps the name <-> id map
 * (fa_dict, HapHiC_cluster.py:87-113).  Where the reference orders by contig NAME
 * (`sorted(((ref, pos+1), (mref, mpos+1)))`, 1629) the caller passes `name_rank`.
 */
#ifndef HAPHIC_B200_H
#define HAPHIC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HH_VERSION 100

enum {
    HH_OK = 0,
    HH_ERR_CUDA = 1,      /* CUDA runtime / launch failure            */
    HH_ERR_ARG = 2,       /* invalid argument                         */
    HH_ERR_CAPACITY = 3,  /* a bounded device structure overflowed    */
    HH_ERR_NOMEM = 4,     /* device allocation failed                 */
    HH_ERR_STATE = 5,     /* call sequence violated                   */
    HH_ERR_UNSUPPORTED = 6
};

enum { HH_MEM_HOST = 0, HH_MEM_DEVICE = 1 };

typedef struct hh_ctx hh_ctx;       /* one GPU + one stream                                   */
typedef struct hh_links hh_links;   /* link counters of one run (full/flank/HT/per-fragment)  */
typedef struct hh_matrix hh_matrix; /* contig x contig link matrix, MCL-ready                 */
typedef struct hh_mcl hh_mcl;       /* Markov-cluster state: M0, pre-expanded M1, iterates     */

int hh_version(void);
const char* hh_last_error(void);

/* ---- context ------------------------------------------------------------------------- */
int hh_ctx_create(int device, hh_ctx** out);
int hh_ctx_destroy(hh_ctx* ctx);
int hh_ctx_sync(hh_ctx* ctx);
/* the cudaStream_t every kernel of this context is launched on (for CUDA-event timing) */
void* hh_ctx_stream(hh_ctx* ctx);
int hh_ctx_device(hh_ctx* ctx);
int hh_ctx_sm_count(hh_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t hh_ctx_launches(hh_ctx* ctx);

/* ---- link counting: parse_alignments_for_ctgs, HapHiC_cluster.py:1596-1655 ----------------
 * One record per read pair: int32 {ctg_a, pos_a, ctg_b, pos_b}, positions 0-based exactly as
 * the generators yield them (1562-1593).  Records with ctg_a == ctg_b are dropped
 * (pairs_generator_inter_ctgs, 1582; BAM filter `refid != mrefid`, 2862), records naming an
 * id outside [0, n_ctg) are skipped (1625).
 *   ctg_len[n_ctg]   contig lengths (frag_len_dict)
 *   name_rank[n_ctg] rank of each contig under Python str ordering of the names (1629)
 *   in_nx[n_ctg]     1 if the contig is in Nx_ctg_set (stat_fragments, 273-288)
 *   flank_bp         args.flank * 1000 (1603); 0 = whole contig (is_flank, 299-307)
 *   capacity_hint    expected number of distinct contig pairs (0 = let the table grow)
 */
int hh_links_create(hh_ctx* ctx, int32_t n_ctg, const int64_t* ctg_len, const int32_t* name_rank,
                    const uint8_t* in_nx, int64_t flank_bp, int64_t capacity_hint, hh_links** out);
/* Fragment mode -- parse_alignments, HapHiC_cluster.py:1658-1752 (some contig longer than bin_size): records
 * still name CONTIGS, the table is keyed by FRAGMENT pairs.  Contig c owns the fragment ids
 * [frag_base[c], frag_base[c+1]); more than one fragment means the contig is split into bins of `bin_size` bp
 * (bin = ceil(coord / bin_size), convert_frags 1662-1670).  Pairs inside one unsplit contig or one bin are
 * dropped (1699, 1715); ends are ordered by contig name then coordinate (1707) and, when a bin is involved,
 * re-ordered by fragment name rank (1719-1720).  Counts the flank links between fragments and the
 * per-fragment totals (1723-1726); its full/HT counters refer to fragment pairs and have no counterpart in the
 * reference -- full_link_dict / HT_link_dict / clm of that run come from a second, contig-level table fed
 * with the same records (hh_links_create with in_nx = 0). */
int hh_links_create_frags(hh_ctx* ctx, int32_t n_ctg, const int32_t* ctg_rank, const int32_t* frag_base,
                          int32_t n_frag, const int64_t* frag_len, const int32_t* frag_rank,
                          const uint8_t* frag_in_nx, int64_t bin_size, int64_t flank_bp, int64_t capacity_hint,
                          hh_links** out);
/* stream `n_rec` more records; `stream_offset` is the index of rec[0] in the whole read stream
 * (first-seen order of dict keys is reproduced from it; use the running total on one GPU, the
 * shard offset when the stream is split over ranks).  May be called repeatedly. */
int hh_links_add(hh_links* lk, const int32_t* rec, int64_t n_rec, int64_t stream_offset, int mem);
/* asynchronous variant for device-resident records: returns after enqueueing (no growth check:
 * the caller guarantees capacity_hint was sufficient; overflow is reported by hh_links_finish) */
int hh_links_add_async(hh_links* lk, const int32_t* rec_dev, int64_t n_rec, int64_t stream_offset);

typedef struct {
    int64_t n_records;   /* records seen                                        */
    int64_t n_used;      /* records counted (passed the id / inter-contig tests) */
    int64_t nnz_full;    /* len(full_link_dict)                                  */
    int64_t nnz_flank;   /* len(flank_link_dict)                                 */
    int64_t table_slots; /* hash-table capacity at the end                       */
} hh_links_info;

/* close the stream: orders the distinct pairs by first appearance (dict insertion order) */
int hh_links_finish(hh_links* lk, hh_links_info* info);

/* full_link_dict / flank_link_dict / HT_link_dict as parallel arrays of nnz_full entries in
 * full_link_dict insertion order (1649).  key_i/key_j: contig ids with name(key_i) < name(key_j).
 * first_full / first_flank: stream index of the record that created the key in the respective
 * dict (first_flank = 0xFFFFFFFF when flank == 0).  ht[4*e + 2*ti + tj]: HT_link_dict counts,
 * ti/tj = 1 for the `_T` half (`coord*2 > len`, 404-416).  Any pointer may be NULL. */
int hh_links_fetch(hh_links* lk, int32_t* key_i, int32_t* key_j, uint32_t* full, uint32_t* flank,
                   uint32_t* first_full, uint32_t* first_flank, uint32_t* ht);
/* ctg_link_dict (1638-1639): per-contig flank-link totals, [n_ctg] */
int hh_links_fetch_ctg(hh_links* lk, int64_t* ctg_links);
/* multi-GPU: export the finished table as device arrays / merge a peer's export into this
 * table (a finished table is re-opened; call hh_links_finish again afterwards).  An export is 9 uint32 per entry: {i, j, full, flank, first_full,
 * first_flank, HT, TH, TT}.  ctg totals travel separately (int64 [n_ctg]). */
int hh_links_export(hh_links* lk, uint32_t* entries_dev, int64_t* ctg_links_dev);
int hh_links_merge(hh_links* lk, const uint32_t* entries_dev, int64_t n_entries, const int64_t* ctg_links_dev,
                   int64_t n_records, int64_t n_used);
/* Routed multi-GPU counting (SURVEY.md 8e "route each pair to its owner"): every contig pair is owned by one rank
 * (hash of the unordered contig pair), so the partition tables are disjoint and nothing is reduced afterwards.
 *   hh_links_route:  split this rank's shard of the stream (device records, global index of rec[0] = stream_offset)
 *     into `world` destination groups: rec_out_dev [n_rec][4] / pos_out_dev [n_rec] receive records and their stream
 *     indices grouped by owner, counts[world] (host) the group sizes.  Records that can never be used (same contig,
 *     ids outside the FASTA) are dropped here.  The caller exchanges the groups (all-to-all).
 *   hh_links_add_routed: count records with explicit stream indices (any order).
 *   hh_links_finish_partition: compact list of this rank's partition (unordered); hh_links_export hands it out.
 *   hh_links_adopt: the table becomes the union of all partitions (entries = concatenated exports [n][9],
 *     ctg_links / n_records / n_used summed over ranks, stream_end = length of the whole stream).  The index,
 *     the matrix and hh_links_fetch (which restores dict insertion order on first use) work as after hh_links_finish. */
int hh_links_route(hh_links* lk, const int32_t* rec_dev, int64_t n_rec, int64_t stream_offset, int world,
                   int32_t* rec_out_dev, uint32_t* pos_out_dev, int64_t* counts);
int hh_links_add_routed(hh_links* lk, const int32_t* rec_dev, const uint32_t* pos_dev, int64_t n_rec);
int hh_links_finish_partition(hh_links* lk, hh_links_info* info);
int hh_links_adopt(hh_links* lk, const uint32_t* entries_dev, int64_t n_entries, const int64_t* ctg_links_dev,
                   int64_t n_records, int64_t n_used, int64_t stream_end);
int hh_links_destroy(hh_links* lk);

/* ---- dict_to_matrix, HapHiC_cluster.py:310-373 ------------------------------------------------
 * Two steps because the reference appends kept-but-unlinked fragments in Python set order
 * (355-359), which only the host can reproduce:
 *   hh_links_linked_index: first-seen index of every fragment that occurs in flank_link_dict
 *     restricted to `keep` (327-349); index[c] = -1 otherwise; *n_linked = len(frags_in_dict).
 *   hh_matrix_from_links: builds the symmetric fp32 matrix, with self loops = 1 when add_self_loops (351-364);
 *     `tail[n_tail]` lists the kept-but-unlinked contig ids in the order they get the following
 *     indices.  normalize_by_nlinks != 0 applies links / sqrt(tot_i * tot_j) first (718-724).
 */
int hh_links_linked_index(hh_links* lk, const uint8_t* keep, int32_t* index, int32_t* n_linked);
int hh_matrix_from_links(hh_links* lk, const uint8_t* keep, const int32_t* tail, int32_t n_tail,
                         int normalize_by_nlinks, int add_self_loops, hh_matrix** out);
/* rank-sum statistic of filter_fragments, HapHiC_cluster.py:864-892, on a matrix WITHOUT self loops: for every
 * fragment, sort its row by links descending (ties by matrix index, a stable list.sort(reverse=True)), take
 * the first topN fragments and sum min(rank_a(b), rank_b(a)) over their pairs.  rank_sum[n] (host) is
 * indexed by matrix index.  topN <= 32. */
int hh_matrix_rank_sums(hh_matrix* m, int topN, int64_t* rank_sum);
/* the same matrix from a host CSC (symmetric, self loops included) -- the entry point when host
 * code edited the link dict (allele-aware removal, UL boosts, phasing weights: 2911-2928) */
int hh_matrix_from_csc(hh_ctx* ctx, int32_t n, const int64_t* indptr, const int32_t* indices,
                       const float* data, hh_matrix** out);
int hh_matrix_info(hh_matrix* m, int32_t* n, int64_t* nnz);
/* canonical CSC (row-sorted) of the raw link matrix, host buffers: indptr[n+1], indices/data[nnz] */
int hh_matrix_fetch_csc(hh_matrix* m, int64_t* indptr, int32_t* indices, float* data);
int hh_matrix_destroy(hh_matrix* m);

/* ---- Markov clustering: run_mcl_clustering / mcl / prune, HapHiC_cluster.py:1987-2062, 2132-2162
 * hh_mcl_create does 2144 (column-L1 normalise, M0) and 2146-2149 (pre-expansion M1 = M0^e, kept
 * resident and shared by the whole inflation sweep).  [col_lo, col_hi) is the block of columns
 * this context owns (0, n for one GPU): M1 and every iterate are computed for owned columns only.
 */
int hh_mcl_create(hh_matrix* m, int expansion, int32_t col_lo, int32_t col_hi, hh_mcl** out);
/* The same with the engine of the pre-expansion (2146-2149) chosen by the caller:
 *   HH_PREEXP_SPARSE  Gustavson SpGEMM on a shared-memory column accumulator (the reference's sparse mode,
 *                     mkl_matrix_power 2017-2023);
 *   HH_PREEXP_DENSE   the product as a symmetric dense GEMM on the tensor cores (tcgen05 / TMEM / TMA; 16-bit operand
 *                     planes that reproduce the fp32 product to 2^-23, fp32 accumulation) -- the reference's dense mode
 *                     (`--dense_matrix`, numpy.linalg.matrix_power 2035 / 2149);
 *   HH_PREEXP_AUTO    whichever is estimated cheaper for this matrix (hh_mcl_create; env HH_MCL_PREEXP overrides).
 * Both engines give M1 within fp32 rounding of the exact product; every later step is shared. */
enum { HH_PREEXP_AUTO = 0, HH_PREEXP_SPARSE = 1, HH_PREEXP_DENSE = 2 };
int hh_mcl_create_ex(hh_matrix* m, int expansion, int32_t col_lo, int32_t col_hi, int preexp_mode, hh_mcl** out);
typedef struct {
    int32_t mode;          /* HH_PREEXP_SPARSE or HH_PREEXP_DENSE: what ran                              */
    int32_t a_planes;      /* dense: 16-bit planes of the count operand (1: integer counts, 3: weights)    */
    int32_t passes;        /* dense: tensor-core passes per k-block                                        */
    int32_t cta_group;     /* dense: 2 = CTA pairs (256 x 256 tiles), 1 = single CTAs (128 x 128)          */
    int32_t stages;        /* dense: shared-memory pipeline stages                                         */
    int32_t chunk_kb;      /* dense: 64-wide k-blocks accumulated in TMEM between two register drains      */
    float total_ms;        /* device time of the pre-expansion                                             */
    float densify_ms;      /* dense: operand planes from the CSC                                           */
    float gemm_ms;         /* dense: the GEMM kernel                                                       */
    float clip_ms;         /* dense: sparse correction for link counts above `clip` (0 when there are none) */
    double flops;          /* dense: tensor-core flops issued                                              */
    int64_t products;      /* sparse: Gustavson products (dense: products of the clip correction)          */
    float clip;            /* dense: counts enter the GEMM as min(count, clip): 2048 (f16 plane) / 256 (bf16) */
    int32_t b_planes;      /* dense: planes of the M0 operand (2: f16 hi + lo, 22 bits; 3: exact bf16)      */
    int32_t fmt_a, fmt_b;  /* dense: operand formats, 0 = bf16, 1 = f16                                    */
    int32_t k_chunks;      /* dense: launches the K range was cut into (operand planes of one chunk at a time) */
} hh_preexp_info;
int hh_mcl_preexp_info(hh_mcl* mc, hh_preexp_info* info);
/* normalize_ms / preexp_ms: device time of the two kernels hh_mcl_create ran */
int hh_mcl_info(hh_mcl* mc, int32_t* n, int64_t* nnz_m0, int64_t* preexp_products, float* normalize_ms,
                float* preexp_ms);
/* M0 as canonical CSC / owned block of M1 as dense column-major fp32 [n * (col_hi-col_lo)] */
int hh_mcl_fetch_m0(hh_mcl* mc, int64_t* indptr, int32_t* indices, float* data);
int hh_mcl_fetch_m1(hh_mcl* mc, float* dense);

typedef struct {
    int32_t rounds;          /* iterations executed ("after N rounds", 2047-2060)          */
    int32_t converged;       /* 1 if the convergence test (2044-2055) fired                 */
    int64_t nnz;             /* stored entries of the returned matrix                       */
    int64_t products;        /* sum over iterations of Gustavson products (flops / 2)       */
    int64_t bytes;           /* sum over iterations of algorithmic bytes (SURVEY.md 8d)     */
} hh_mcl_result;

/* one mcl() call (2026-2062) on one GPU owning all columns.  iter_nnz / iter_products /
 * iter_delta / iter_ms: optional host arrays of max_iter entries receiving per-iteration statistics
 * (iter_ms = device time of the iteration's column kernel, CUDA events on the context stream). */
int hh_mcl_run(hh_mcl* mc, double inflation, int max_iter, double pruning, hh_mcl_result* res,
               int64_t* iter_nnz, int64_t* iter_products, float* iter_delta, float* iter_ms);
/* the matrix hh_mcl_run (or the last hh_mcl_step + hh_mcl_commit) left, canonical CSC, host */
int hh_mcl_fetch_result(hh_mcl* mc, int64_t* indptr, int32_t* indices, float* data);

/* step-wise interface for column-sharded multi-GPU runs (one rank per GPU):
 *   begin -> { step -> pack -> [host: all-gather] -> unpack(peer blocks) -> commit } ...
 * hh_mcl_step computes iteration `it` (0-based; it == 0 streams the dense M1, 2030) for the owned
 * columns and returns their stats; *delta is max(|M - L| - 1e-5|L|) over owned columns (2045);
 * *kernel_ms the device time of the column kernel.
 * hh_mcl_pack writes the owned block as {len[col_hi-col_lo] int32} and packed {idx int32, val
 * fp32}[nnz_owned] into caller-provided DEVICE buffers; hh_mcl_unpack installs a peer's block. */
int hh_mcl_begin(hh_mcl* mc, double inflation, double pruning);
int hh_mcl_step(hh_mcl* mc, int it, int64_t* nnz_owned, int64_t* products, float* delta, float* kernel_ms);
int hh_mcl_pack(hh_mcl* mc, int32_t* len_dev, int32_t* idx_dev, float* val_dev);
int hh_mcl_unpack(hh_mcl* mc, int32_t col_lo, int32_t col_hi, const int32_t* len_dev,
                  const int32_t* idx_dev, const float* val_dev, int64_t nnz_block);
int hh_mcl_commit(hh_mcl* mc);
/* change the block of columns the following steps compute (between hh_mcl_commit and hh_mcl_step, after iteration 0;
 * reset by hh_mcl_begin).  Column shards switch to (0, n) once the iterate is tiny: no exchange is needed any more
 * because every rank then computes the identical full iterate. */
int hh_mcl_set_block(hh_mcl* mc, int32_t col_lo, int32_t col_hi);
int hh_mcl_destroy(hh_mcl* mc);

/* ---- assembly correction (`--correct_nrounds`): correct_assembly, HapHiC_cluster.py:943-1297 ------------------------
 * Coverage of a contig is int32 over len // res + 1 bins (1312); contig c owns bins [bin_off[c], bin_off[c+1]) of one array
 * and every fragment split from it is a sub-range of those bins (the reference slices numpy views, 1158 / 1180).  The
 * intra-contig read pairs are kept as links {bucket, lo, hi} (lo <= hi, 0-based); a bucket is an id the host gives to a key
 * string of ctg_link_pos_dict (initially bucket = contig id).
 *   hh_correct_create:  res = --correct_resolution.
 *   hh_correct_add:     parse_pairs_for_correction / parse_bam_for_correction (1300-1398): records {id_a, pos_a, id_b, pos_b}
 *     with id_a == id_b in [0, n_ctg) add 1 to the bins [lo // res, hi // res] and append a link; other records are ignored.
 *     A same-contig position outside [0, contig length) is an error.  Not allowed after the first detect / split / fetch.
 *   hh_correct_info / hh_correct_fetch: bin count, link count; coverage [n_bins], bin_off [n_ctg + 1] and links [n_links][3]
 *     (host buffers, any may be NULL).  Dropped links keep their slot with bucket -1.
 *   hh_correct_detect:  detect_break_points (943-1014) on the fragments seg_off[s] (first bin), seg_nbins[s], seg_len[s] (bp):
 *     n_bp[s] breakpoints each, packed in fragment order into bp_bin / bp_cov (bin relative to the fragment, its coverage;
 *     the breakpoint is bin * res) up to max_bp entries; *total_bp = their number.
 *   hh_correct_detect_segments: the same on a caller's host coverage array (stateless).
 *   hh_correct_split:   one non-last round of break_and_update_ctgs (1074-1121) for n_frag broken fragments: fragment f holds
 *     the links of bucket frag_bucket[f] (-1: none) and starts at bin frag_off[f]; shift_pos[list_off[f] .. list_off[f+1])
 *     is pos_shift_list (its breakpoints descending, then 0) and piece_bucket[] the bucket of the key pos_shift gives each
 *     entry.  frag_zero[f] = 0 (one non-zero breakpoint): links whose closed span overlaps [bp, bp + res] leave the coverage.
 *     The other links move to the bucket of their piece with shifted coordinates; links across pieces are dropped.
 *   hh_correct_set_pieces / hh_correct_remap: convert_ctg of the second pass (1405-1411).  Contig c's pieces are
 *     [piece_off[c], piece_off[c+1]) with ascending 0-based starts (the first 0) and their ids in the corrected fa_dict;
 *     remap rewrites every {id, pos} in place to {piece id, pos - piece start}; ids outside [0, n_ctg) become -1. */
typedef struct hh_correct hh_correct;
int hh_correct_create(hh_ctx* ctx, int32_t n_ctg, const int64_t* ctg_len, int32_t res, hh_correct** out);
int hh_correct_add(hh_correct* hc, const int32_t* rec, int64_t n_rec, int mem);
int hh_correct_info(hh_correct* hc, int64_t* n_bins, int64_t* n_links);
int hh_correct_fetch(hh_correct* hc, int32_t* cov, int64_t* bin_off, int32_t* links);
int hh_correct_detect(hh_correct* hc, int32_t n_seg, const int64_t* seg_off, const int32_t* seg_nbins, const int64_t* seg_len,
                      double median_cov_ratio, double region_len_ratio, int64_t min_region_cutoff, int32_t* n_bp,
                      int32_t* bp_bin, int32_t* bp_cov, int64_t max_bp, int64_t* total_bp);
int hh_correct_detect_segments(hh_ctx* ctx, const int32_t* cov, int64_t n_cov, int32_t res, int32_t n_seg,
                               const int64_t* seg_off, const int32_t* seg_nbins, const int64_t* seg_len,
                               double median_cov_ratio, double region_len_ratio, int64_t min_region_cutoff, int32_t* n_bp,
                               int32_t* bp_bin, int32_t* bp_cov, int64_t max_bp, int64_t* total_bp);
int hh_correct_split(hh_correct* hc, int32_t n_frag, const int32_t* frag_bucket, const int64_t* frag_off,
                     const uint8_t* frag_zero, const int32_t* list_off, const int32_t* shift_pos, const int32_t* piece_bucket,
                     int32_t n_buckets);
int hh_correct_set_pieces(hh_correct* hc, int32_t n_piece, const int32_t* piece_off, const int32_t* piece_start,
                          const int32_t* piece_id);
int hh_correct_remap(hh_correct* hc, int32_t* rec, int64_t n_rec, int mem);
int hh_correct_destroy(hh_correct* hc);

/* ---- host-side I/O around the path (native, no CUDA) ------------------------------------------------
 * .pairs / .pairs.gz reader: pairs_generator / pairs_generator_inter_ctgs, HapHiC_cluster.py:1539-1583.  Skips blank
 * and '#' lines, takes `cols[1], int(cols[2])-1, cols[3], int(cols[4])-1`, writes the two BED lines per pair
 * to `bed_path` (may be NULL) and returns int32 records {id_a, pos_a, id_b, pos_b} (id -1 = name not in the table);
 * with inter_only pairs whose two names are equal are dropped (1582).  names_blob = n_names NUL-terminated names.
 * The text is cut at line boundaries and parsed on `threads` host threads (0 = all cores, at most 16); bgzipped
 * input is inflated block-parallel, other gzip streams by zlib. */
typedef struct hh_pairs_reader hh_pairs_reader;
int hh_pairs_open(const char* path, const char* names_blob, int32_t n_names, const char* bed_path, int inter_only,
                  int threads, hh_pairs_reader** out);
int hh_pairs_next(hh_pairs_reader* r, int32_t* rec, int64_t max_records, int64_t* n_out);   /* *n_out == 0: end of file */
int hh_pairs_close(hh_pairs_reader* r);
/* the inverse, for fixtures and benchmarks: n_rec records {id_a, pos_a, id_b, pos_b} (0-based positions) as 4DN .pairs text
 * `r{first_index + i}\tname_a\tpos_a+1\tname_b\tpos_b+1\t+\t-`; append != 0 continues an existing file without the header */
int hh_pairs_write(const char* path, const char* names_blob, int32_t n_names, const int32_t* rec, int64_t n_rec, int64_t first_index,
                   int append, int threads);
/* BAM input (bam_generator, HapHiC_cluster.py:1586-1593, with the htslib filters `flag.read1 [&& refid != mrefid]` of
 * 2855 / 2862): BGZF blocks are inflated on `threads` host threads; one record per read1 alignment,
 * (id(reference_name), reference_start, id(next_reference_name), next_reference_start), ids through the BAM header's
 * reference names (-1 = not in the FASTA / unmapped).  hh_bam_header_text gives the SAM header (sorting order check,
 * check_sorting_order 1347-1359); the pointer stays valid until hh_bam_close. */
typedef struct hh_bam_reader hh_bam_reader;
int hh_bam_open(const char* path, const char* names_blob, int32_t n_names, int inter_only, int threads, hh_bam_reader** out);
int hh_bam_header_text(hh_bam_reader* r, const char** text, int64_t* len);
int hh_bam_next(hh_bam_reader* r, int32_t* rec, int64_t max_records, int64_t* n_out);
int hh_bam_close(hh_bam_reader* r);

/* paired_links.clm straight from the record stream (update_clm_dict 395-401 + output_clm 376-392): for every contig
 * pair with >= 2 links, in dict insertion order, four lines (orientations ++ +- -+ --)
 * `{ci}{s} {cj}{s}\t{2*links}\t{every ascending distance printed twice}`.  rec = n_rec int32 records
 * {id_a, pos_a, id_b, pos_b} in stream order (same-contig records and ids outside [0, n_names) are skipped),
 * ctg_len / name_rank per contig id.  Grouping, the per-pair sorts and the text formatting run on `threads` host
 * threads (0 = all cores, at most 16). */
int hh_clm_from_records(const char* path, const char* names_blob, int32_t n_names, const int32_t* rec, int64_t n_rec,
                        const int64_t* ctg_len, const int32_t* name_rank, int threads);
/* full_links.pkl / HT_links.pkl (output_pickle, 710-715) written from the fetched arrays, without materialising the
 * Python dicts: the file loads (pickle.load) as `defaultdict(int, {(name_i, name_j): value})` in entry order.
 * Give values_i64 or values_f64 for one entry per pair, or ht[n_entries][4] = {HH, HT, TH, TT} for HT_link_dict, whose
 * keys are (name_i + '_H'|'_T', name_j + '_H'|'_T') for the non-zero counters (update_HT_link_dict, 404-416). */
int hh_pickle_links(const char* path, const char* names_blob, int32_t n_names, const int32_t* key_i, const int32_t* key_j,
                    int64_t n_entries, const int64_t* values_i64, const double* values_f64, const uint32_t* ht);

#ifdef __cplusplus
}
#endif
#endif /* HAPHIC_B200_H */
