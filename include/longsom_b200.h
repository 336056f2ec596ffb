/*
 * longsom_b200.h -- C-ABI of the B200-native LongSom SNV hot path.
 *
 * The reference (cbg-ethz/LongSom) has no in-process FFI for this path: its
 * boundary is "python CLI in, TSV out" (workflow/rules/SNVCalling.smk:50-60,
 * 143-156,178-189; CellClustering.smk:86-103; CellTypeReannotation.smk:141-151,
 * 378-394).  The drop-in CLIs under workflow/scripts/ keep that boundary; this
 * header is the layer below them: what a ctypes / cgo / JNI stub binds.  Every
 * entry point names the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes; the caller owns every host buffer it passes;
 *   - every function returns LS_OK (0) or a negative LS_E_* code and never
 *     throws; ls_last_error(ctx) holds a human-readable message;
 *   - one ls_ctx == one CUDA device + one stream; a ctx is not thread-safe,
 *     different ctxs are independent;
 *   - there is NO CPU fallback: without a CUDA device ls_ctx_create fails with
 *     LS_E_CUDA.
 */
#ifndef LONGSOM_B200_H
#define LONGSOM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LS_ABI_VERSION 1

/* error codes */
#define LS_OK 0
#define LS_E_CUDA (-1)     /* CUDA runtime error (no device, OOM, launch failure) */
#define LS_E_ARG (-2)      /* invalid argument (null pointer, unsorted input, ...) */
#define LS_E_STATE (-3)    /* call order violated (run before upload, ...) */
#define LS_E_CAPACITY (-4) /* caller buffer too small */

/* Allele classes, in the reference's dictionary order
 * (BaseCellCounter.py:228 keys A,C,T,G,D,I,N,O; printed order A:C:T:G:I:D,
 * BaseCellCounter.py:300).  Index = class id used throughout this ABI. */
#define LS_CLASS_A 0
#define LS_CLASS_C 1
#define LS_CLASS_T 2
#define LS_CLASS_G 3
#define LS_CLASS_I 4
#define LS_CLASS_D 5
#define LS_CLASS_N 6
#define LS_CLASS_O 7
#define LS_CLASS_NA 8 /* '>' '<' IUPAC '=' : ignored (EasyReadPileup :177-178) */

/* Per-site record of ls_pileup_count: 26 uint32 words.
 *   [0] DP  [1] NC  [2..7] CC  [8..13] BCf  [14..19] BCr  [20..25] BQ
 * each 6-vector in printed allele order A,C,T,G,I,D; BC = BCf + BCr.
 * (BaseCellCounter.py:291-308) */
#define LS_SITE_WORDS 26
#define LS_SITE_DP 0
#define LS_SITE_NC 1
#define LS_SITE_CC 2
#define LS_SITE_BCF 8
#define LS_SITE_BCR 14
#define LS_SITE_BQ 20

/* Read batches: per-read query bases start at multiples of LS_BASE_ALIGN. */
#define LS_BASE_ALIGN 16

typedef struct ls_ctx ls_ctx;

/* Structure-of-arrays batch of decoded BAM records, coordinate sorted by
 * (tid, pos) exactly as the BAM file orders them.  This is what the host
 * decoder produces in place of pysam's per-column Python objects
 * (BaseCellCounter.py:190-191,214-216,225,238-249). */
typedef struct ls_read_batch {
  int64_t n_reads;
  int64_t n_cigar;           /* total CIGAR ops */
  int64_t n_bases;           /* length of qual[] (padded), seq4 holds n_bases/2 bytes */
  const int32_t *tid;        /* [n_reads] contig index */
  const int32_t *pos;        /* [n_reads] 0-based leftmost reference position */
  const uint16_t *flag;      /* [n_reads] BAM FLAG */
  const uint8_t *mapq;       /* [n_reads] */
  const int32_t *cell;       /* [n_reads] dense barcode id (CB tag, text before the first '-',
                                BaseCellCounter.py:241-246); -1 = no CB tag */
  const uint32_t *cigar_off; /* [n_reads+1] */
  const uint32_t *cigar;     /* [n_cigar] BAM encoding len<<4|op, ops MIDNSHP=X */
  const uint64_t *base_off;  /* [n_reads+1] first query base of read i in seq4/qual, multiple of
                                LS_BASE_ALIGN; l_qseq(i) is NOT base_off[i+1]-base_off[i] (padding) */
  const int32_t *l_qseq;     /* [n_reads] query length */
  const uint8_t *seq4;       /* BAM nibble codes "=ACMGRSVTWYHKDBN"; base j of the batch is the high
                                nibble of seq4[j>>1] when j is even, the low nibble when odd */
  const uint8_t *qual;       /* [n_bases] phred */
} ls_read_batch;

/* Genomic windows = the reference's unit of work (MakeWindows, BaseCellCounter.py:81-113;
 * one pysam pileup() call per window, :190-191).  0-based half-open, sorted by
 * (tid, start), non-overlapping.  ref holds the reference bases (ASCII, any case) of every
 * window back to back; window w occupies ref[ref_off[w] .. ref_off[w] + end-start). */
typedef struct ls_windows {
  int64_t n_windows;
  const int32_t *tid;
  const int32_t *start;
  const int32_t *end;
  const uint64_t *ref_off; /* [n_windows+1] */
  const uint8_t *ref;
} ls_windows;

/* Thresholds of BaseCellCounter.run_interval (BaseCellCounter.py:182, CLI :334-339). */
typedef struct ls_count_params {
  int32_t min_bq;    /* --min_bq  (pileup min_base_quality) */
  int32_t min_mq;    /* --min_mq  (pileup min_mapping_quality) */
  int32_t min_dp;    /* --min_dp  (:211,:221,:282) */
  int32_t min_cc;    /* --min_cc  (:294) */
  int32_t min_ac;    /* --min_ac  (:221) */
  int32_t max_depth; /* pileup max_depth, 200000 in the reference (:191); 0 = unlimited */
} ls_count_params;

/* Device timings of the last ls_pileup_run / ls_genotype_run, CUDA events on the ctx stream. */
typedef struct ls_run_stats {
  float ms_total;      /* whole run */
  float ms_segments;   /* segment build (CIGAR walk, read filter) */
  float ms_sort;       /* (tile, cell) radix sort */
  float ms_count;      /* the pileup-count kernel alone */
  float ms_compact;    /* site compaction (ls_pileup_fetch) */
  int64_t n_segments;  /* (read, tile) work items */
  int64_t n_tiles;     /* non-empty tiles */
  int64_t n_aligned;   /* sum of M/=/X lengths over all records of the batch (the bench unit) */
  int64_t n_events;    /* (read, reference position) entries visited by the count kernel */
  int32_t count_launches; /* kernels launched by the last run */
  int32_t reserved;
} ls_run_stats;

/* Compacted result of ls_pileup_count, ordered by (window order, pos). */
typedef struct ls_site_counts {
  int64_t capacity;   /* in: number of sites the arrays can hold */
  int64_t n_sites;    /* out */
  int32_t *tid;       /* [capacity] */
  int32_t *pos;       /* [capacity] 0-based */
  uint8_t *ref;       /* [capacity] upper-cased reference base (BaseCellCounter.py:202-203) */
  uint32_t *counts;   /* [capacity][LS_SITE_WORDS] */
} ls_site_counts;

/* ---- context -------------------------------------------------------------------------- */
int ls_abi_version(void);
int ls_ctx_create(int device, ls_ctx **ctx);
int ls_ctx_destroy(ls_ctx *ctx);
const char *ls_last_error(const ls_ctx *ctx);
/* pinned host staging memory (cudaHostAlloc); optional, pageable buffers also work */
int ls_host_alloc(size_t bytes, void **ptr);
int ls_host_free(void *ptr);

/* ---- K1: per-barcode base pileup -------------------------------------------------------
 * Replaces BaseCellCounter.run_interval (BaseCellCounter.py:182-320) + EasyReadPileup
 * (:152-180) + the htslib pileup engine behind pysam.AlignmentFile.pileup (:190-191).
 *   upload : H2D copy of a batch and its windows (the ctx keeps device copies)
 *   run    : segment build -> (tile,cell) sort -> pileup-count kernel; results stay in HBM
 *   compact: compaction of the passing sites into output order, still in HBM (fetch does it if it has not been done)
 *   fetch  : D2H of the compacted sites into caller arrays
 *   count  : upload + run + fetch in one call (the end-to-end entry point)            */
int ls_pileup_upload(ls_ctx *ctx, const ls_read_batch *batch, const ls_windows *windows);
int ls_pileup_run(ls_ctx *ctx, const ls_count_params *params, int64_t *n_sites, ls_run_stats *stats);
int ls_pileup_compact(ls_ctx *ctx, ls_run_stats *stats); /* device-side half of fetch: passing sites in (window, pos) order */
int ls_pileup_fetch(ls_ctx *ctx, ls_site_counts *out);
int ls_pileup_count(ls_ctx *ctx, const ls_read_batch *batch, const ls_windows *windows,
                    const ls_count_params *params, ls_site_counts *out, ls_run_stats *stats);

/* ---- K1': pileup at candidate sites, per (site, cell) ------------------------------------
 * Replaces SingleCellGenotype.run_interval's pileup loop (SingleCellGenotype.py:114-178) and
 * HCCVSingleCellGenotype.run_interval (:112-176).  Uses the batch of the last
 * ls_pileup_upload (windows may be empty).  Sites sorted by (tid, pos), unique.
 *   alt_class[s]  : class id the site's ALT_expected maps to (LS_CLASS_*), LS_CLASS_NA if the
 *                   string is not one of A,C,T,G,I,D,N (then Alt stays 0)
 *   alt_only      : 0 = --alt_flag All (classes A,C,T,G,I,D,N counted, :149-151)
 *                   1 = --alt_flag Alt (only class == ALT_expected, :153)
 *   cell ids >= n_cells or < 0 are "barcode not in --meta" and skipped (:164-169)
 *   dp, alt       : [n_sites][n_cells] int32, row-major, written in full                     */
typedef struct ls_geno_params {
  int32_t min_bq;
  int32_t min_mq;
  int32_t max_depth;
  int32_t alt_only;
  int32_t bin_size; /* --bin (50000): one pileup() call per CHROM_floor(POS/bin) group of sites
                       (build_dict_variants, SingleCellGenotype.py:253-274); only matters for max_depth */
  int32_t reserved;
} ls_geno_params;
int ls_genotype_count(ls_ctx *ctx, const int32_t *site_tid, const int32_t *site_pos,
                      const uint8_t *alt_class, int64_t n_sites, int32_t n_cells,
                      const ls_geno_params *params, int32_t *dp, int32_t *alt, ls_run_stats *stats);

/* Sparse form of the same computation, for candidate lists whose dense [site][cell] tensors would not fit (2e5 sites
 * x 2e4 cells = 32 GB): only the TOUCHED (site, cell) pairs -- Dp > 0 -- leave the device, sorted by (site, cell), with
 * the beta-binomial tail of SingleCellGenotype.py:204 / HCCVSingleCellGenotype.py:204 already evaluated on the device:
 *   p = betabinom.sf(Alt - eps, Dp, alpha, beta)  for pairs with Alt > 0 at sites with skip_p[site] == 0, NaN otherwise
 * (skip_p marks the sites that take the chrM shortcut, :195-199; may be NULL).  run keeps the tuples in HBM and returns
 * their number, fetch copies them out; the dense rows of the reference are an expansion of these tuples.            */
typedef struct ls_geno_tuples {
  int64_t capacity;  /* in */
  int64_t n_tuples;  /* out */
  int32_t *site;     /* [capacity] index into the site arrays of the run */
  int32_t *cell;     /* [capacity] */
  int32_t *dp;       /* [capacity] */
  int32_t *alt;      /* [capacity] */
  double *p;         /* [capacity] */
} ls_geno_tuples;
int ls_genotype_sparse_run(ls_ctx *ctx, const int32_t *site_tid, const int32_t *site_pos, const uint8_t *alt_class,
                           const uint8_t *skip_p, int64_t n_sites, int32_t n_cells, const ls_geno_params *params,
                           double alpha, double beta, int64_t *n_tuples, ls_run_stats *stats);
int ls_genotype_sparse_fetch(ls_ctx *ctx, ls_geno_tuples *out);

/* ---- K2: beta-binomial tails ---------------------------------------------------------------
 * Replaces scipy.stats.betabinom.sf / 1-cdf as called at BaseCellCalling.step1.py:196,201,
 * 329-330,427-428, SingleCellGenotype.py:204, HCCVSingleCellGenotype.py:204.
 *   p[i] = sf(k[i] - eps, n[i], a, b) = 1 - sum_{j=0}^{k[i]-1} pmf(j)   for 0 < eps < 1
 * with scipy's argument handling (k-eps < 0 -> 1, k-eps >= n -> 0, n < 0 -> NaN). fp64. */
int ls_betabinom_sf(ls_ctx *ctx, const int32_t *k, const int32_t *n, double a, double b,
                    double *p, int64_t m, ls_run_stats *stats);

/* ---- K3: (chrom,pos) membership masks --------------------------------------------------------
 * Replaces step2.build_dict + the EDITING / PON_SR / PON_LR lookups of GetExtraFilters
 * (BaseCellCalling.step2.py:124-221).  keys are (tid<<32 | pos) and need not be sorted
 * or unique; hit[i] = 1 iff query[i] is in keys. */
int ls_site_mask(ls_ctx *ctx, const uint64_t *keys, int64_t n_keys, const uint64_t *query,
                 int64_t m, uint8_t *hit, ls_run_stats *stats);
/* The same in two steps, for a site list that is looked up more than once (step2 holds the
 * editing list and the two panels of normals for the whole run, :197-221): the table is
 * sorted once and stays resident in HBM in slot `table` (0 .. LS_SITE_TABLES-1) until that
 * slot is loaded again.  A lookup in an empty slot is LS_E_STATE. */
#define LS_SITE_TABLES 4
int ls_site_table_load(ls_ctx *ctx, int table, const uint64_t *keys, int64_t n_keys,
                       ls_run_stats *stats);
int ls_site_table_lookup(ls_ctx *ctx, int table, const uint64_t *query, int64_t m, uint8_t *hit,
                         ls_run_stats *stats);

/* ---- genotype matrices ------------------------------------------------------------------------
 * Replaces the pandas pivots of SingleCellGenotype.py:351-379 (pivot_long_dataframe + sort_chr_index): the
 * DpMatrix / AltMatrix / VAFMatrix / BinaryMatrix rows, written as text straight from the touched pairs.
 *   load : the pairs in matrix coordinates (row = output row rank, col = output column rank), sorted on the device
 *          by (row, col) and kept resident until the next load.  A duplicate (row, col) is LS_E_ARG.
 *   text : the rows row_lo .. row_lo + *rows_done - 1 of one matrix kind, as many whole rows as fit in capacity
 *          bytes, each "label <tab> entry <tab> ... entry \n" (no header line).  A row longer than capacity is
 *          LS_E_CAPACITY.
 * Entries, as pandas prints them:
 *   SNV row, touched pair     Dp, Alt as integers; VAF str(round(Alt / Dp, 4)) ('.' when Dp = 0); Binary the
 *                             long table's BinMutationStatus: 3 when Dp = 0, 0 when Alt = 0, chrM shortcut rows
 *                             1 when the rounded VAF >= 0.3, else 1 when p < pvalue, else 0
 *   SNV row, untouched        0, 0, '.', 3; empty in a col_absent column
 *   fusion row, a pair        1, 1, 1, 1
 *   fusion row, no pair       empty
 * With float_mode set (some entry of the matrix is absent) Dp, Alt and Binary print as floats ("2.0").          */
#define LS_GENO_MATRIX_DP 0
#define LS_GENO_MATRIX_ALT 1
#define LS_GENO_MATRIX_VAF 2
#define LS_GENO_MATRIX_BINARY 3
#define LS_GENO_ROW_CHRM 1   /* the chrM shortcut applies to this row (--chrM_contaminant True) */
#define LS_GENO_ROW_FUSION 2 /* a fusion row: every pair prints 1, every other entry is absent */
typedef struct ls_geno_matrix_in {
  int64_t n_rows;
  int64_t n_pairs;
  int32_t n_cols;
  int32_t float_mode;
  const int32_t *row;          /* [n_pairs] */
  const int32_t *col;          /* [n_pairs] */
  const int32_t *dp;           /* [n_pairs] */
  const int32_t *alt;          /* [n_pairs] */
  const double *p;             /* [n_pairs] beta-binomial tail rounded to four places (numpy.round), NaN if none */
  const char *labels;          /* printed row labels back to back, in row order */
  const int64_t *label_off;    /* [n_rows+1] */
  const uint8_t *row_flags;    /* [n_rows] LS_GENO_ROW_* */
  const uint8_t *col_absent;   /* [n_cols] 1: the column is absent from SNV rows (a fusion barcode); may be NULL */
  double pvalue;               /* --pvalue */
} ls_geno_matrix_in;
int ls_geno_matrix_load(ls_ctx *ctx, const ls_geno_matrix_in *in);
int ls_geno_matrix_text(ls_ctx *ctx, int kind, int64_t row_lo, char *out, int64_t capacity, int64_t *rows_done,
                        int64_t *bytes);

/* ---- genotype long table ----------------------------------------------------------------------
 * Replaces the row loops of SingleCellGenotype.py:128-214 / HCCVSingleCellGenotype.py:126-212 (the dense long table,
 * one row per candidate site x metadata barcode), written as text straight from the touched pairs.  The text equals
 * the host writer's (ls_geno_rows).
 *   load : the output sites in the order their rows are written, each with its range of the touched pairs, and the
 *          texts of the rows; kept resident until the next load.  LS_E_ARG for a pair's cell outside [0, n_cells),
 *          cells not strictly increasing inside a site's range, a range outside [0, n_pairs] or with lo > hi, a pair
 *          with alt outside [0, dp], a p neither NaN nor below 4e5 in magnitude, or a null array that is needed.
 *          The alt and p rules go beyond the host writer, which prints such pairs; they keep every number within the
 *          device's 32-bit digit formatting.  K1' counts alt only with dp and K2's tails lie in [0, 1], so the CLIs
 *          never meet them.
 *   text : the rows of the sites site_lo .. site_lo + *sites_done - 1, as many whole sites as fit in capacity bytes
 *          (no header line).  A site longer than capacity is LS_E_CAPACITY; site_lo == n_sites gives (0, 0).
 *   times: device time of the text calls since the load, from events: the write kernels and the device-to-host
 *          copies, with the number of blocks and their bytes.
 * For site s and cell c = 0 .. n_cells-1, one row:
 *   prefix[s] \t cell_text[c] \t Dp \t Alt \t VAF \t BetaBin \t MutationStatus [\t BinMutationStatus \t index[s]] \n
 * (the two bracketed columns only when hccv is 0), with the pair (Dp, Alt, p) of (s, c):
 *   untouched, or Dp = 0         0 \t 0 \t . \t . \t NoCoverage, BinMutationStatus 3
 *   Dp > 0, Alt = 0              VAF 0.0, BetaBin '.', NoAltReads, 0
 *   Alt > 0, LS_GENO_ROW_CHRM    VAF str(round(Alt / Dp, 4)), BetaBin '.', LowVAFChrM when that VAF < 0.3 else PASS
 *   Alt > 0, other sites         VAF as above, BetaBin str(p) ('nan' for NaN), PASS when p < pvalue else
 *                                BetaBin_problem
 *   BinMutationStatus            1 for PASS, 3 for NoCoverage, 0 otherwise                                          */
typedef struct ls_geno_long_in {
  int64_t n_sites;             /* output sites, in the order their rows are written */
  int32_t n_cells;             /* may be 0: every site then has no rows */
  int32_t hccv;                /* 1: 14 columns, no BinMutationStatus / INDEX */
  int64_t n_pairs;
  const int32_t *cell;         /* [n_pairs] touched pairs, sorted by cell inside each site's range */
  const int32_t *dp;           /* [n_pairs] */
  const int32_t *alt;          /* [n_pairs] */
  const double *p;             /* [n_pairs] rounded to four places (numpy.round), NaN where none */
  const int64_t *hit_lo;       /* [n_sites] the site's range of the pair arrays (lo == hi: untouched) */
  const int64_t *hit_hi;       /* [n_sites] */
  const uint8_t *site_flags;   /* [n_sites] LS_GENO_ROW_CHRM */
  const char *prefix;          /* the seven leading columns of each site, tab-joined, back to back */
  const int64_t *prefix_off;   /* [n_sites+1] */
  const char *index;           /* INDEX column of each site; NULL when hccv */
  const int64_t *index_off;    /* [n_sites+1]; NULL when hccv */
  const char *cell_text;       /* "barcode\tcell type" of each cell */
  const int64_t *cell_off;     /* [n_cells+1] */
  double pvalue;               /* --pvalue */
} ls_geno_long_in;
int ls_geno_long_load(ls_ctx *ctx, const ls_geno_long_in *in);
int ls_geno_long_text(ls_ctx *ctx, int64_t site_lo, char *out, int64_t capacity, int64_t *sites_done, int64_t *bytes);
int ls_geno_long_times(ls_ctx *ctx, double *ms_text, double *ms_copy, int64_t *blocks, int64_t *bytes);
/* frees the long table's device buffers (a later text call is LS_E_STATE until the next load) */
int ls_geno_long_release(ls_ctx *ctx);

/* ---- device-resident handles for benchmarking (inputs already in HBM) ----------------------- */
int ls_device_synchronize(ls_ctx *ctx);
/* PCI address ("0000:1b:00.0") of a CUDA device ordinal, for NUMA placement of the host staging buffers; no context */
int ls_device_pci_bus_id(int device, char *buf, int len);
/* flush L2 by writing a scratch buffer larger than the 126 MB L2 */
int ls_flush_l2(ls_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* LONGSOM_B200_H */
