/*
 * mgatk2_b200 — C ABI of the B200-native per-cell chrM pileup hot path.
 *
 * This is the drop-in boundary for the three-call seam inside the reference's
 * MtDNAPipeline.run() (reference src/core/pipeline.py:80-81,102-103):
 *
 *     BAMReader.collect_reads_by_barcode()           src/processing/readers.py:63-201
 *     CellProcessor.process_cells_progressive()      src/processing/processors.py:87-144
 *       -> process_barcode_worker()                  src/processing/processors.py:20-55
 *       -> PileupGenerator.generate_pileup()         src/processing/pileup.py:18-126
 *       -> PileupGenerator.filter_strand_bias()      src/processing/pileup.py:128-154
 *     per-cell depth statistics / reference allele   src/file_io/writers.py:187-197,345-349,493-500
 *
 * The reference has no FFI for this path (it is pure Python); the entry points
 * below are what a ctypes/cffi binding inside those three functions would call
 * (see INTEGRATION.md for the reference-side stub).
 *
 * Conventions
 *   - plain C, no C++/torch types; all pointers are caller-owned;
 *   - "_device" entry points take DEVICE pointers and a cudaStream_t passed as
 *     void*; they only enqueue work (no host synchronisation);
 *   - "_host" entry points take HOST pointers, do H2D, the kernels, D2H and
 *     synchronise before returning;
 *   - every entry point returns an mgatk_status; 0 is success. No exceptions
 *     cross the boundary. mgatk_last_error() gives a human readable string.
 *   - one handle per GPU; handles are independent (no global mutable state);
 *     a handle must be used from one thread at a time.
 */
#ifndef MGATK2_B200_H
#define MGATK2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGATK_ABI_VERSION 2

/* ---- status codes -------------------------------------------------------- */
typedef enum mgatk_status {
    MGATK_OK = 0,
    MGATK_ERR_BAD_ARG = 1,       /* null pointer, negative size, bad enum           */
    MGATK_ERR_CUDA = 2,          /* a CUDA runtime call failed (see last_error)     */
    MGATK_ERR_WORKSPACE = 3,     /* caller workspace smaller than workspace_bytes() */
    MGATK_ERR_UNSORTED = 4,      /* records are not sorted by reference_start       */
    MGATK_ERR_EXTENT = 5,        /* a read exceeds params.max_read_extent           */
    MGATK_ERR_OVERFLOW_CAP = 6,  /* more >65535 entries than overflow_capacity      */
    MGATK_ERR_NO_DEVICE = 7,     /* no usable CUDA device                           */
    MGATK_ERR_RANGE = 8,         /* n_cells / n_records / blob outside limits       */
    MGATK_ERR_STREAM_SATURATED = 9 /* streaming: more cells with entries beyond 65535 than carry-plane sets */
} mgatk_status;

/* ---- dedup strategies (reference src/cli/utils.py:164-169) ---------------- */
#define MGATK_DEDUP_FRAGMENT_LENGTH 0 /* alignment_and_fragment_length: (start, strand, |tlen|) */
#define MGATK_DEDUP_POSITION_ONLY   1 /* alignment_start: (start, strand)                       */
#define MGATK_DEDUP_NONE            2 /* none: skip                                             */

/* ---- output plane order -------------------------------------------------- */
/* planes[cell][plane][pos_padded], uint16, saturated at 65535 exactly like the
 * reference's HDF5 writer (src/file_io/writers.py:205-218); values above 65535
 * are additionally listed exactly in the overflow list so that the unsaturated
 * text layout (src/file_io/writers.py:442-462) stays bit-exact. */
#define MGATK_PLANE_A_FWD 0
#define MGATK_PLANE_A_REV 1
#define MGATK_PLANE_C_FWD 2
#define MGATK_PLANE_C_REV 3
#define MGATK_PLANE_G_FWD 4
#define MGATK_PLANE_G_REV 5
#define MGATK_PLANE_T_FWD 6
#define MGATK_PLANE_T_REV 7
#define MGATK_PLANE_TN5_FWD 8
#define MGATK_PLANE_TN5_REV 9
#define MGATK_PLANE_COVERAGE 10
#define MGATK_N_PLANES 11

/* positions are padded to a multiple of 64 so every flush is a full 128-byte store */
#define MGATK_POS_PAD(P) ((((int64_t)(P)) + 63) / 64 * 64)

/* ---- parameters (reference src/core/config.py:8-23,111-114) --------------- */
typedef struct mgatk_params {
    int32_t min_baseq;           /* QualityThresholds.min_baseq   (int8 compare, pileup.py:80) */
    int32_t min_mapq;            /* QualityThresholds.min_mapq    (pileup.py:33)               */
    int32_t min_distance_from_end; /* QualityThresholds.min_distance_from_end (pileup.py:67-72) */
    int32_t dedup_mode;          /* MGATK_DEDUP_*                 (readers.py:118-150)         */
    double  max_strand_bias;     /* QualityThresholds.max_strand_bias (pileup.py:143-145)      */
    int32_t min_reads_per_cell;  /* PipelineConfig.min_reads_per_cell (processors.py:22)       */
    int32_t mito_length;         /* PipelineConfig.mito_length, 16569                          */
    int32_t n_cells;             /* whitelist length; bc_idx in [0,n_cells) or -1              */
    int32_t max_read_extent;     /* upper bound on max(reference span, l_seq) over the batch;
                                    verified on the device (MGATK_ERR_EXTENT)                  */
    int32_t flags;               /* MGATK_FLAG_*                                               */
} mgatk_params;

/* generate_pileup() without filter_strand_bias(): no strand-bias zeroing and Tn5 counts are
 * kept at positions without coverage, i.e. the dict PileupGenerator.generate_pileup returns
 * (pileup.py:100-124) before pileup.py:128-154 is applied. */
#define MGATK_FLAG_RAW_PILEUP 1

/* Streaming over several batches (BASELINE configs[4]: inputs larger than HBM). The records of a coordinate-sorted
 * BAM are cut into batches on reference_start borders (all duplicates of a read share its start, so dedup needs no
 * state across batches, readers.py:118-150); the planes stay resident and every batch ADDS its raw counts:
 *     mgatk_stream_begin_device(...)                            zero planes / QC / counters
 *     mgatk_pileup_device(..., flags | MGATK_FLAG_ACCUMULATE)   once per batch, in file order
 *     mgatk_stream_finish_device(...)                           cell gate, strand-bias filter, coverage, Tn5 gating,
 *                                                               depth statistics, base totals, medians
 * The result equals the one-batch result bit for bit, whatever the depth: a cell whose plane entry passes 65535 while the
 * batches add up (bulk mode, deep piles) gets a set of 32-bit carry planes inside the handle (64 sets, allocated by
 * mgatk_stream_begin_device; one stream per handle at a time), folded back in by mgatk_stream_finish_device.
 * MGATK_ERR_STREAM_SATURATED only when every set is taken. */
#define MGATK_FLAG_ACCUMULATE 2

/* ---- one batch of records, structure-of-arrays, BAM (coordinate) order ---- */
/* One entry per record returned by fetch(chrM) (readers.py:87-93), i.e. also
 * unmapped-placed / secondary / supplementary records and records without a
 * (whitelisted) barcode: the flag and whitelist tests are stage 1 on the GPU.
 * blob: for record i, starting at byte 16*blob_off[i]:
 *        n_cigar[i] uint32 BAM cigar words (len<<4|op), then (l_seq+1)/2 bytes of
 *        4-bit packed SEQ (BAM nibble order), then l_seq bytes of raw phred QUAL —
 *        the same contiguous cigar|seq|qual region a BAM record carries. */
typedef struct mgatk_batch {
    int64_t n_records;
    const int32_t  *pos;      /* reference_start, 0-based                              */
    const int32_t  *tlen;     /* template_length (signed)                              */
    const uint16_t *flag;     /* BAM FLAG                                              */
    const uint8_t  *mapq;     /* mapping_quality                                       */
    const int32_t  *bc_idx;   /* whitelist index of the barcode tag, -1 = absent/unknown */
    const uint16_t *l_seq;    /* len(query_sequence)                                   */
    const uint16_t *n_cigar;  /* number of cigar operations                            */
    const uint32_t *blob_off; /* offset of the record's blob in 16-byte units          */
    const uint8_t  *blob;     /* cigar|seq|qual blobs, each 16-byte aligned            */
    int64_t blob_bytes;       /* total size of blob (multiple of 16)                   */
} mgatk_batch;

/* ---- per-cell QC row, 32 bytes (processors.py:33-39, writers.py:187-197) --- */
typedef struct mgatk_cell_qc {
    uint32_t n_reads;     /* len(reads) after dedup                (processors.py:33)   */
    uint32_t n_paired;    /* reads with flag&1                     (processors.py:34)   */
    uint64_t sum_depth;   /* sum of depth over covered positions   (writers.py:192)     */
    uint32_t covered;     /* positions with depth>0                (processors.py:38)   */
    uint32_t max_depth;   /* unsaturated                           (writers.py:191)     */
    uint32_t median_lo;   /* the two middle order statistics of the covered depths;    */
    uint32_t median_hi;   /* np.median == (lo+hi)/2                (writers.py:190)     */
} mgatk_cell_qc;

/* ---- global counters (readers.py:193-199) --------------------------------- */
typedef struct mgatk_stats {
    uint64_t total_reads;      /* every fetched record                                  */
    uint64_t stage1_reads;     /* passed flag + barcode filter                          */
    uint64_t filtered_reads;   /* survivors of dedup (== stats["filtered_reads"])       */
    uint64_t dup_with_length;  /* stats["duplicate_reads_with_length"]                  */
    uint64_t dup_position_only;/* stats["duplicate_reads_position_only"]                */
    uint64_t n_empty_seq;      /* dedup survivors with l_seq==0 (reference raises)      */
    uint64_t n_overflow;       /* entries written to the overflow list                  */
    uint64_t error_bits;       /* bit0 unsorted, bit1 extent, bit2 overflow capacity, bit3 stream saturated,
                                  bit4 a deletion out of range (mgatk_deletion_scan_device) */
} mgatk_stats;

/* exact value of one saturated plane entry */
typedef struct mgatk_overflow {
    int32_t  cell;
    uint32_t plane_pos;  /* plane<<24 | position */
    uint32_t value;
} mgatk_overflow;

/* ---- outputs -------------------------------------------------------------- */
typedef struct mgatk_outputs {
    uint16_t        *planes;       /* [n_cells][MGATK_N_PLANES][MGATK_POS_PAD(P)]; fully written */
    mgatk_cell_qc   *cell_qc;      /* [n_cells]                                                 */
    mgatk_stats     *stats;        /* [1]                                                       */
    int64_t         *base_totals;  /* [P][4] sum over cells of fwd+rev after filtering
                                      (reference allele vote, writers.py:220-222,345-349)      */
    mgatk_overflow  *overflow;     /* [overflow_capacity], may be NULL if capacity 0           */
    int64_t          overflow_capacity;
} mgatk_outputs;

typedef struct mgatk_handle mgatk_handle;

/* library / ABI */
int         mgatk_abi_version(void);
const char *mgatk_status_string(int status);

/* handle: binds to CUDA device `device`; owns nothing but small scratch and the
 * buffers used by the _host entry point */
int         mgatk_create(mgatk_handle **out, int device);
int         mgatk_destroy(mgatk_handle *h);
const char *mgatk_last_error(const mgatk_handle *h);

/* size of the device workspace the _device entry point needs for a batch shape; max_read_extent as in mgatk_params
 * (it selects the slot layout: 32 bytes per read up to an extent of 56, 16 + 16 * ceil(extent / 32) bytes beyond, at
 * most 144). -1 when the shape is outside the limits. */
int64_t     mgatk_workspace_bytes(int64_t n_records, int32_t n_cells, int32_t max_read_extent);

/* Stages 1-6 on device-resident buffers; enqueues on `stream`, never blocks.
 * After the stream has drained, mgatk_check_stats turns a host copy of
 * stats (its error_bits) into a status code. */
int mgatk_pileup_device(mgatk_handle *h, const mgatk_params *params,
                        const mgatk_batch *batch_dev, const mgatk_outputs *out_dev,
                        void *workspace_dev, int64_t workspace_bytes, void *stream);

int mgatk_check_stats(const mgatk_stats *stats_host);

/* streaming: see MGATK_FLAG_ACCUMULATE. params->flags of the finish call selects raw / filtered output. */
int mgatk_stream_begin_device(mgatk_handle *h, const mgatk_params *params, const mgatk_outputs *out_dev, void *stream);
int mgatk_stream_finish_device(mgatk_handle *h, const mgatk_params *params, const mgatk_outputs *out_dev, void *stream);

/* PileupGenerator.filter_strand_bias (pileup.py:128-154) on raw planes, in place:
 * planes_dev is [n_cells][MGATK_N_PLANES][MGATK_POS_PAD(P)] as written with MGATK_FLAG_RAW_PILEUP
 * (values above 65535 are not representable here; use the 32-bit variant below for those). */
int mgatk_filter_strand_bias_device(mgatk_handle *h, uint16_t *planes_dev, int32_t n_cells, int32_t mito_length,
                                    double max_strand_bias, void *stream);
/* The same rule on 32-bit planes (same shape): exact for any depth. This is what PileupGenerator.filter_strand_bias
 * is given when a caller hands over the dict generate_pileup() returned (pileup.py:128: plain Python ints there). */
int mgatk_filter_strand_bias_u32_device(mgatk_handle *h, uint32_t *planes_dev, int32_t n_cells, int32_t mito_length,
                                        double max_strand_bias, void *stream);

/* Same, but batch and outputs are HOST buffers (pinned for full speed): H2D copy,
 * kernels, D2H copy, synchronise. Device buffers are cached inside the handle. */
int mgatk_pileup_host(mgatk_handle *h, const mgatk_params *params,
                      const mgatk_batch *batch_host, const mgatk_outputs *out_host);

/* The same call in two halves, for callers with more than one batch (one BAM per sample or per
 * cell, as in the reference's `call` command, cli/options.py:310,421): submit enqueues the upload, the kernels and the
 * download on three streams and returns; wait blocks until out_host of that ticket is complete
 * (overflow list included) and returns the batch's status. Up to TWO tickets may be in flight:
 * the upload of batch k+1 then runs while batch k computes and downloads (PCIe is full duplex),
 * which is what bounds throughput with host buffers. batch_host / out_host must stay valid and
 * untouched until wait returns; pinned memory is needed for the copies to overlap. Tickets may be
 * waited for in any order. mgatk_pileup_host == submit + wait. */
int mgatk_pileup_host_submit(mgatk_handle *h, const mgatk_params *params, const mgatk_batch *batch_host,
                             const mgatk_outputs *out_host, int64_t *ticket);
int mgatk_pileup_host_wait(mgatk_handle *h, int64_t ticket);

/* ---- variant statistics (DESIGN §8, "Variant statistics") ------------------
 * A cross-cell reduction over the filtered planes of a result, for the heteroplasmy statistics of Signac's
 * IdentifyVariants. Every count is exact: a plane entry of 65535 takes its value from the overflow list
 * (stats->n_overflow entries of result->overflow; an entry of 65535 without a list entry is 65535). The reference
 * allele ref[p] is the vote of result->base_totals: the first of A,C,G,T with the largest total, N when none is
 * positive. For every position p with ref[p] != N and every b in A,C,G,T other than ref[p] there is one variant
 * p ref>b; per selected cell, f / r are the b forward / reverse counts, a = f + r and d the coverage entry.
 * out is laid out [P][4] by alt letter; the slot alt == ref and every slot of an N position have valid = 0 and all
 * sums 0. */
typedef struct mgatk_variant_sums {
    uint64_t sum_fwd, sum_rev, sum_cov;  /* sum of f, r, d over the selected cells                                  */
    uint64_t sum_ff, sum_rr, sum_fr;     /* over the cells with a > 0: sum of f*f, r*r, f*r                          */
    uint64_t max_alt, max_cov;           /* (a, d) of the largest a/d over cells with d > 0 (exact cross-multiplied
                                            compare; ties keep the lowest cell index); 0, 0 when no cell has d > 0   */
    double   dev_sum, dev_sq;            /* sum of u and u*u, u = a/d - mean for cells with d >= L, else 0;
                                            mean = (sum_fwd + sum_rev) / sum_cov, 0 when sum_cov = 0                 */
    uint32_t n_covered;                  /* cells with d > 0                                                         */
    uint32_t n_detected;                 /* cells with a > 0 (= the cells of sum_ff, sum_rr, sum_fr)                 */
    uint32_t n_conf_detected;            /* cells with f >= 2 and r >= 2                                             */
    uint32_t n_strand;                   /* cells with a > 0 (the n of the strand correlation)                       */
    uint32_t n_over[4];                  /* cells with d > 0 and 100 a >= k d, k = 5, 10, 20, 95                     */
    uint32_t n_low;                      /* cells with d < L (L = low_coverage_threshold)                            */
    int32_t  ref;                        /* reference allele 0..3 = A,C,G,T; -1 = N                                  */
    int32_t  valid;                      /* 1: a variant; 0: alt == ref or ref = N                                    */
    int32_t  reserved;                   /* 0 */
} mgatk_variant_sums;                    /* 128 bytes */

/* Variant sums of the result `result_dev` (planes [n_cells][11][MGATK_POS_PAD(P)], stats, overflow, base_totals; all
 * device pointers) over the cells with cell_mask_dev[c] != 0 (u8[n_cells]; NULL = all cells), into
 * out_dev[P][4]. Integer fields do not depend on the launch configuration; dev_sum / dev_sq are reduced in a fixed
 * order, so a call gives the same bits every time. Enqueues on `stream`; the overflow lookup table lives in the
 * handle, so calls on one handle must be ordered (one stream). */
int mgatk_variant_stats_device(mgatk_handle *h, const mgatk_params *params, const mgatk_outputs *result_dev,
                               const uint8_t *cell_mask_dev, int32_t low_coverage_threshold,
                               mgatk_variant_sums *out_dev, void *stream);
/* Exact per-cell counts of n_variants variants (variants_dev: int32 pos * 4 + alt, pos in [0, P), alt 0..3 = A,C,G,T)
 * for every cell: out_dev[n_variants][3][n_cells] = alt forward, alt reverse, coverage. An id outside [0, 4 P) gives
 * rows of zeros. Enqueues on `stream`; same handle rule as above. */
int mgatk_variant_cells_device(mgatk_handle *h, const mgatk_params *params, const mgatk_outputs *result_dev,
                               const int32_t *variants_dev, int32_t n_variants, uint32_t *out_dev, void *stream);

/* ---- clones (DESIGN §8, "Clones") -----------------------------------------
 * Cells grouped into clones by the heteroplasmy of called variants: Signac's AlleleFreq + FindClonotypes, with an
 * exact kNN search and deterministic Louvain. x[c][v] = (f + r) / d (0 when d = 0) from the counts of
 * mgatk_variant_cells_device; every float operation is an IEEE fp64 multiply, add, square root or divide (no FMA):
 *     dot(i, j) = sum over v ascending of acc = acc + x[i][v] * x[j][v], from acc = 0
 *     inv[i] = 1 / sqrt(dot(i, i)) (0 when dot(i, i) = 0),   cos(i, j) = (dot(i, j) * inv[i]) * inv[j]
 * N(i) is row i itself with similarity 1.0, then the k_eff - 1 other rows with the largest cos(i, j), ties to the lower
 * row index (k_eff = min(k, n_rows)). */
#define MGATK_CLONE_K_MAX 64
#define MGATK_CLONE_MAX_ROWS (1 << 24)            /* n_rows                                            */
#define MGATK_CLONE_MAX_VARIANTS 4096             /* n_variants                                        */
#define MGATK_CLONE_MAX_ELEMENTS ((int64_t)1 << 31) /* n_rows * (n_variants rounded up to 32): x scratch */

/* kNN of the graph rows. counts_dev: uint32 [n_variants][3][n_cells] (alt forward, alt reverse, coverage) as the
 * variant-cells entry writes it; rows_dev: int32 [n_rows] distinct cell indices in [0, n_cells), each with x > 0 for at
 * least one variant (the graph rows). A row that breaks this (no detection, or a cell index outside [0, n_cells),
 * read as zero counts) has cosine 0 with every row, so the result stays defined and deterministic. Writes nbr_out int32 [n_rows][k_eff] (row
 * indices into rows_dev, N(i) in order) and sim_out fp64 [n_rows][k_eff]. The result does not depend on the launch
 * configuration. MGATK_ERR_BAD_ARG: k outside [2, MGATK_CLONE_K_MAX], a negative size, a null pointer, n_variants = 0
 * or n_rows > n_cells with rows; MGATK_ERR_RANGE: beyond the MGATK_CLONE_MAX_* limits. x and inv live in handle
 * scratch: calls on one handle must be ordered (one stream). */
int mgatk_clone_knn_device(mgatk_handle *h, const uint32_t *counts_dev, const int32_t *rows_dev, int32_t n_rows,
                           int32_t n_cells, int32_t n_variants, int32_t k, int32_t *nbr_out, double *sim_out, void *stream);
/* Shared-nearest-neighbour weight of every directed kNN edge: w_out[i][t] = s / (2 k_eff - s), s = |N(i) ∩ N(j)|,
 * j = nbr_dev[i][t] (fp64 divide). nbr_dev is [n][k_eff] as the kNN entry writes it. MGATK_ERR_BAD_ARG: negative n,
 * k_eff outside [1, min(MGATK_CLONE_K_MAX, n)], a null pointer; MGATK_ERR_RANGE: n above MGATK_CLONE_MAX_ROWS. */
int mgatk_clone_snn_device(mgatk_handle *h, const int32_t *nbr_dev, int32_t n, int32_t k_eff, double *w_out, void *stream);
/* Deterministic Louvain on the host (no CUDA call, no handle): a symmetric weighted graph in CSR form (indptr int64
 * [n + 1] from 0, indices int32 ascending within a row, weights fp64 >= 0, diagonal allowed) at `resolution` > 0.
 * labels_out int32 [n]: clone numbers 1..K by size descending, ties to the smallest member; *n_levels_out: levels whose
 * first phase moved a node. The rules are those of DESIGN §8 "Clones". MGATK_ERR_BAD_ARG for a malformed graph or
 * resolution, MGATK_ERR_RANGE for 2^31 or more entries or when memory runs out. */
int mgatk_louvain_host(int32_t n, const int64_t *indptr, const int32_t *indices, const double *weights, double resolution,
                       int32_t *labels_out, int32_t *n_levels_out);

/* ---- clone markers (DESIGN §8, "Clone markers") ------------------------------
 * Seurat's FindAllMarkers test on the heteroplasmy of variants: a two-sided Wilcoxon rank-sum test per variant, each
 * group of cells against the other cells of the population. x = (f + r) / d as for the clones (0 when d = 0); the
 * population is the cells with a label in [1, n_groups], N their number; rank(c) is the 1-based mid-rank of x[v][c]
 * among the population. The device gives exact integers; the host forms U, the tie-corrected normal approximation and
 * p from them. */
#define MGATK_MARKER_MAX_CELLS (1 << 21)          /* n_cells: N^3 stays below 2^63                       */

/* Wilcoxon rank sums of x = (f + r) / d per variant: counts_dev uint32 [n_variants][3][n_cells] as
 * mgatk_variant_cells_device writes it, labels_dev int32 [n_cells] (1..n_groups: a group; anything else: not in
 * the test). rank2_out uint64 [n_variants][n_groups] = sum over the group's cells of 2 * mid-rank, ties_out uint64
 * [n_variants] = sum over runs of equal x of t^3 - t. Every output entry is written; integer results, so they do not
 * depend on the launch configuration. Scratch lives in the handle (calls on one handle ordered, freed by
 * mgatk_destroy). MGATK_ERR_BAD_ARG: a null pointer with a non-zero size, a negative size, n_groups < 1;
 * MGATK_ERR_RANGE: n_cells above MGATK_MARKER_MAX_CELLS, n_variants above MGATK_CLONE_MAX_VARIANTS, n_groups above
 * n_cells (n_cells > 0). n_variants = 0 or n_cells = 0: MGATK_OK (outputs zero when n_cells = 0). */
int mgatk_marker_ranks_device(mgatk_handle *h, const uint32_t *counts_dev, const int32_t *labels_dev, int32_t n_cells,
                              int32_t n_variants, int32_t n_groups, uint64_t *rank2_out, uint64_t *ties_out, void *stream);

/* ---- deletions (DESIGN §8, "Deletions") ---------------------------------------
 * Large mtDNA deletions from the reads themselves, as mgatk-del does: soft-clip breakpoints and, per cell, the reads that
 * show a junction against the reads that span a breakpoint. The reads are those the pileup counts: stage 1
 * (flag & 0x904 == 0, 0 <= bc_idx < n_cells), dedup per params->dedup_mode and barcode with the first record of a key in
 * file order surviving, then mapq >= min_mapq (after dedup). Per read: a0 = pos, a1 = pos + span - 1 (span = sum of
 * M/D/N/=/X; span 0 takes no part), sl / sr = the S ops before the first / after the last M/=/X op (0 when longer than
 * SEQ or without such an op). A deletion is (l, r): l the last kept position before the deleted segment, r the first one
 * after it, 0 <= l, l + 1 < r < P (HGVS m.{l+2}_{r}del). Per read and deletion, at most one class:
 *     clip_left   a1 = l and sr >= min_clip          clip_right   a0 = r and sl >= min_clip
 *     gap         a D or N op over exactly [l + 1, r)
 *     wt          one M/=/X block covers l and l + 1, or r - 1 and r
 * Discovery histograms over all reads and cells: end_clip[p] reads with sr >= min_clip and a1 = p; start_clip[p] reads
 * with sl >= min_clip and a0 = p; end_seq[p][j][b] / start_seq[p][j][b] the base b (A, C, G, T; other codes are not
 * counted) of those reads at SEQ[l_seq - sr + j] / SEQ[sl - 1 - j], j < min(MGATK_DEL_KMER, clip). */
#define MGATK_DEL_KMER 16
#define MGATK_DEL_MAX 1024                        /* n_deletions */

/* One part of a coordinate-sorted input (parts cut on reference_start borders add up: dedup keys only repeat within a
 * run of equal starts). left_dev / right_dev: int32 [n_deletions] device arrays of l and r. Every output is ADDED to, so
 * the caller zeroes them once and calls once per part:
 *     counts_out     uint32 [n_deletions][4][n_cells]: clip_left, clip_right, gap, wt
 *     clip_hist_out  uint64 [2][P]: end_clip, start_clip; NULL = no discovery
 *     clip_seq_out   uint64 [2][P][MGATK_DEL_KMER][4]: end_seq, start_seq; NULL exactly when clip_hist_out is
 *     error_bits_out uint64 [1], OR-ed with the bits of mgatk_stats.error_bits: 1 records not sorted by reference_start,
 *                    2 a stage-1 read longer than params->max_read_extent (l_seq of every one, the reference span of every
 *                    one whose CIGAR is read: those near a breakpoint, or all with discovery), 16 a deletion outside
 *                    0 <= l, l + 1 < r < P (it matches nothing). mgatk_check_stats maps them to MGATK_ERR_UNSORTED,
 *                    MGATK_ERR_EXTENT and MGATK_ERR_RANGE once the stream has drained.
 * params supplies min_mapq, dedup_mode, n_cells, mito_length (P) and max_read_extent. Integer results: they do not depend
 * on the launch configuration. Enqueues on `stream`; scratch (about 36 bytes per record) lives in the handle, so calls on
 * one handle must be ordered; mgatk_destroy frees it. MGATK_ERR_BAD_ARG: a null pointer where data is needed, a negative
 * size, min_clip < 1, dedup_mode outside 0..2, max_read_extent < 1, a blob not 16-byte aligned, only one of clip_hist_out
 * and clip_seq_out; MGATK_ERR_EXTENT: max_read_extent above 2^20; MGATK_ERR_RANGE: n_deletions above MGATK_DEL_MAX,
 * mito_length of 2^24 or more, 2^31 - 256 records or more. No records, or no deletions without discovery: MGATK_OK and
 * nothing is enqueued. */
int mgatk_deletion_scan_device(mgatk_handle *h, const mgatk_params *params, const mgatk_batch *batch_dev,
                               int32_t min_clip, const int32_t *left_dev, const int32_t *right_dev, int32_t n_deletions,
                               uint32_t *counts_out, uint64_t *clip_hist_out, uint64_t *clip_seq_out,
                               uint64_t *error_bits_out, void *stream);

/* number of kernel launches issued by the last mgatk_pileup_* call on this handle */
int64_t mgatk_last_launch_count(const mgatk_handle *h);

/* device time (ms, CUDA events on the launch stream) of each stage of the last
 * _host call; names/ms arrays of length *n (n<=16). For profiling only. */
int mgatk_last_stage_times(const mgatk_handle *h, const char **names, float *ms, int *n);

#ifdef __cplusplus
}
#endif
#endif /* MGATK2_B200_H */
