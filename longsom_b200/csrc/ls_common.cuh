// Shared internals of the longsom_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/longsom_b200.h"

#define LS_NUM_SMS_DEFAULT 148

// BAM CIGAR op codes (SAM spec section 4.2): MIDNSHP=X
enum { OP_M = 0, OP_I = 1, OP_D = 2, OP_N = 3, OP_S = 4, OP_H = 5, OP_P = 6, OP_EQ = 7, OP_X = 8 };

// pysam pileup() default flag_filter: UNMAP|SECONDARY|QCFAIL|DUP (SURVEY Appendix A.2)
#define LS_FLAG_FILTER 0x704u
#define LS_FLAG_PAIRED 0x1u
#define LS_FLAG_PROPER 0x2u
#define LS_FLAG_REVERSE 0x10u
#define LS_FLAG_SUPPL 0x800u

// A device buffer that grows on demand and is freed with its owner.
struct DBuf {
  void *p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(const DBuf &) = delete;
  DBuf &operator=(const DBuf &) = delete;
  ~DBuf() { release(); }
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    release();
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      e = cudaMalloc(&p, bytes);
      want = bytes;
    }
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};

// one (read, tile) work item of the pileup-count kernel (16 B, self-contained: the count kernel never touches the
// per-read arrays)
struct __align__(16) Segment {
  uint32_t p0;      // first piece of the segment in pieces[] (consecutive: a read's CIGAR visits a tile once)
  uint32_t np_nu;   // bits 0-15: number of pieces; bits 16-31: number of 32-base units the pieces expand to
  uint32_t boff16;  // base_off[read] / 16: where the read's qualities / bases start
  uint32_t flags;   // bit 0: reverse strand
};

// One CIGAR op clipped to one tile, produced by the segment builder so that the count kernel does not walk
// CIGARs: a match piece covers query bases [ya, ya + n) at tile columns [col, col + n); a deletion piece covers
// n columns that all carry the quality of query base ya (htslib: qpos of a deletion = the next query base).
// `ind` marks a piece whose last column is the op's last column and is followed by an insertion (1) or a
// deletion (2): that column's class becomes I / D.  A ref-skip followed by an indel is a 1-column deletion piece.
// `virt` marks query positions past the stored sequence (malformed record): quality 0, base 'N'.
struct __align__(8) Piece {
  uint32_t ya;
  uint32_t meta;  // col: bits 0-8, n (1..512): bits 9-18, deletion-like: bit 19, ind: bits 20-21, virt: bit 22
};
__host__ __device__ __forceinline__ uint32_t piece_meta(uint32_t col, uint32_t n, uint32_t del, uint32_t ind,
                                                        uint32_t virt) {
  return col | (n << 9) | (del << 19) | (ind << 20) | (virt << 22);
}
// Units of a piece: the piece cut at the 32-column windows of its tile (a unit never crosses a window, so the
// count kernel can keep one window's per-site state in registers and the padded accumulator rows need no carry).
__host__ __device__ __forceinline__ uint32_t piece_units(uint32_t meta) {
  const uint32_t col = meta & 511u, n = (meta >> 9) & 1023u;
  return ((col + n - 1u) >> 5) - (col >> 5) + 1u;
}

// Device copies of qual[] / seq4[] start LS_QPAD bytes into their allocations (and end with as much slack): a unit
// loads the aligned 40-byte / 24-byte blocks around its bases, which may reach a few bytes past either end.
#define LS_QPAD 64

// Device counters of one pileup run (ctx->counters, zeroed at the start of ls_pileup_run).  Kernels get pointers to
// single fields; the 32-bit flags and counters sit in 8-byte slots.
struct RunCounters {
  unsigned long long n_aligned;  // aligned bases (seg_build_kernel)
  unsigned long long n_events;   // pileup entries (pileup_count_kernel)
  uint64_t n_sites;              // passing sites: total of the scan of the per-slot pass counts
  uint64_t n_slots;              // non-empty tiles
  alignas(8) uint32_t n_parts;   // parts of deep tiles (part_build_kernel)
  alignas(8) uint32_t long_run;  // some same-cell run is too long for the packed counters (classify_kernel)
  alignas(8) uint32_t n_light;   // parts of shallow tiles
  alignas(8) uint32_t cap_flag;  // some window fetches more than max_depth records
  // reservation totals of seg_build_kernel, which takes them as one array
  unsigned long long n_segments, n_pieces, n_units;
  uint64_t tot_s, tot_m, tot_u;  // sizes of the S / M / U unit streams
  uint64_t n_groups;             // (cell, window) groups in M
  uint64_t n_members;            // run-member segments
};
static_assert(sizeof(RunCounters) == 128, "RunCounters layout");

// Device counters of one genotype call (the start of ctx->counters, zeroed by ls_genotype_count and
// ls_genotype_sparse_run)
struct GenoCounters {
  unsigned long long n_events;  // real hits (genotype_kernel)
  uint64_t n_slots;             // hit slots: total of the scan of the per-read candidate counts
  uint64_t n_tuples;            // touched (site, cell) pairs: total of the scan of the first-hit flags
  alignas(8) uint32_t n_big;    // pairs K2 leaves to the staged path (p = -1)
};
static_assert(sizeof(GenoCounters) == 32, "GenoCounters layout");

// What K1' keeps between its kernels, and between ls_genotype_sparse_run and ls_genotype_sparse_fetch
struct GenoState {
  DBuf site_key, alt_class, site_bin, skip;  // site table of the last call: keys, ALT classes, bins, skip_p flags
  DBuf slots;           // per read: its candidate sites, scanned in place into its first hit slot
  DBuf hits_a, hits_b;  // hit keys and the radix sort's second buffer
  DBuf flag;            // first hit of a pair: flag, scanned in place into the pair's tuple index
  DBuf tup, p;          // tuples: site, cell, Dp, Alt and the K2 query k, each [n_tuples]; p [n_tuples]
  DBuf dp, alt;         // dense [site][cell] tensors of ls_genotype_count
  int64_t n_tuples = 0;
  bool have_tuples = false;
  double alpha = 0.0, beta = 0.0;
};

// The genotype matrix writer's pairs, kept between ls_geno_matrix_load and the ls_geno_matrix_text calls
struct GenoMatrixState {
  DBuf keys_a, keys_b, vals_a, vals_b;  // (row, col) keys and the radix sort's second buffers
  DBuf in_dp, in_alt, in_p;             // pairs in the caller's order
  DBuf col, dp, alt, p;                 // pairs sorted by (row, col)
  DBuf row_start;                       // [n_rows+1] first pair of each row
  DBuf labels, label_off, row_flags, col_absent;
  DBuf lens, offs, out, result;         // per text call: row lengths, their scan, the block's text, rows / bytes
  int64_t n_rows = 0, n_pairs = 0;
  int32_t n_cols = 0, n_present = 0, float_mode = 0;
  double pvalue = 0.0;
  bool loaded = false;
};

// The genotype long table's layout, kept between ls_geno_long_load and the ls_geno_long_text calls
struct GenoLongState {
  DBuf cell, dp, alt, p;                         // [n_pairs] the touched pairs as given
  DBuf hit_lo, hit_hi, flags;                    // [n_sites] each output site's range of the pairs, LS_GENO_ROW_*
  DBuf tail_base, tail_cum;                      // per site, from tail_base[s]: its pairs' tail lengths, scanned
  DBuf site_len, site_off;                       // [n_sites] text bytes of a site; [n_sites+1] their scan
  DBuf prefix, prefix_off, index, index_off, cell_text, cell_off;  // offsets rebased to 0
  DBuf out, result;                              // per text call: the block's text; load: the input error flags
  std::vector<int64_t> h_site_off;               // [n_sites+1] host copy of site_off: plans the blocks
  int64_t n_sites = 0, n_pairs = 0;
  int32_t n_cells = 0, hccv = 0;
  double pvalue = 0.0;
  double ms_text = 0.0, ms_copy = 0.0;           // device time of the text calls since the load (events)
  int64_t blocks = 0, bytes = 0;                 // blocks and bytes written since the load
  bool loaded = false;
  void release() {
    for (DBuf *b : {&cell, &dp, &alt, &p, &hit_lo, &hit_hi, &flags, &tail_base, &tail_cum, &site_len, &site_off, &prefix,
                    &prefix_off, &index, &index_off, &cell_text, &cell_off, &out, &result})
      b->release();
    std::vector<int64_t>().swap(h_site_off);
    loaded = false;
  }
};

// The counter table's row offsets, kept between ls_pileup_text_load and the ls_pileup_text calls
struct CounterTextState {
  DBuf names, name_off;  // contig names back to back, [n_names+1] offsets rebased to 0
  DBuf lens, off;        // [n_sites] row bytes; [n_sites+1] their 64-bit exclusive scan
  DBuf range, result;    // [2][n_names] each contig's site range; load: input error flags, text: (last site, bytes)
  DBuf out;              // per text call: the block's text
  int64_t n_sites = 0;
  bool loaded = false;   // cleared by ls_pileup_upload and ls_pileup_run
};

// BaseCellCalling.step1 on the device: one byte range of the merged table between ls_step1_load and the
// ls_step1_text calls, and the reference contigs, resident from the first range that names them to ls_step1_release
struct Step1State {
  DBuf data;                      // the range's bytes
  DBuf flag, row_lo;              // [len] line-start flags, scanned; [n_rows+1] line starts, then len
  DBuf rows, calls;               // [n_rows] S1Row; [n_rows][n_ct] S1Call
  DBuf qoff, run;                 // 2 x [n_rows+1] query counts, scanned; contig-run flags and their scan
  DBuf run_lo, run_ctg;           // per contig run: its first row's line start and CHROM length; its contig id
  DBuf q, p;                      // queries k1 n1 k2 n2 (int32) and tails p1 p2 (double)
  DBuf cols, names, name_off;     // the cell-type columns and their header names
  DBuf ctg_ptr, ctg_len;          // per contig id: the resident bases, their number (-1: not resident)
  DBuf lens, off, out, result;    // row lengths, their 64-bit scan, a text call's block, flags and totals
  std::vector<DBuf *> contigs;    // [contig id] resident bases (nullptr: the FASTA does not have it)
  std::vector<int64_t> contig_len;
  std::vector<std::string> contig_names;
  std::vector<int64_t> h_off;     // [n_rows+1] host copy of off: plans the blocks
  int64_t len = 0, n_rows = 0, n_q1 = 0, n_q2 = 0;
  int32_t n_ct = 0, min_cov = 0, min_cells = 0, min_ac_cells = 0, min_ac_reads = 0, min_cell_types = 0,
          max_cell_types = 0;
  double alpha1 = 0.0, beta1 = 0.0, alpha2 = 0.0, beta2 = 0.0;
  bool loaded = false, called = false;
  void release() {
    for (DBuf *b : {&data, &flag, &row_lo, &rows, &calls, &qoff, &run, &run_lo, &run_ctg, &q, &p, &cols, &names,
                    &name_off, &ctg_ptr, &ctg_len, &lens, &off, &out, &result})
      b->release();
    for (DBuf *b : contigs) delete b;
    contigs.clear();
    contig_len.clear();
    contig_names.clear();
    std::vector<int64_t>().swap(h_off);
    loaded = called = false;
  }
  ~Step1State() {
    for (DBuf *b : contigs) delete b;
  }
};

// What a replay of ls_pileup_run takes from the last run on the batch that it can stand for
struct ReplaySnapshot {
  bool valid = false;
  ls_count_params params = {};
  RunCounters mid = {};  // the device counters at the run's middle read-back
  int64_t n_sites = 0;
};

struct ls_ctx {
  int device = 0;
  int num_sms = LS_NUM_SMS_DEFAULT;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[8] = {};
  std::string err;

  // ---- uploaded batch ----
  bool have_batch = false;
  int64_t n_reads = 0, n_cigar = 0, n_bases = 0, n_windows = 0;
  int32_t max_cell = -1;
  DBuf tid, pos, flag, mapq, cell, cigar_off, cigar, base_off, lq, seq4, qual;
  DBuf wtid, wstart, wend, wref_off, ref, wtile_base;
  // seq4 on the device is nibble-swapped at upload (even base in the LOW nibble): base n of the batch then sits at
  // bits 4n .. 4n+3 of the little-endian byte stream, so aligning a unit to its window is one funnel shift
  const uint8_t *qual_d() const { return as_u8(qual) + LS_QPAD; }
  const uint8_t *seq4_d() const { return as_u8(seq4) + LS_QPAD; }
  static const uint8_t *as_u8(const DBuf &b) { return reinterpret_cast<const uint8_t *>(b.p); }
  std::vector<int32_t> h_wtid, h_wstart, h_wend;
  std::vector<int64_t> h_wtile_base;  // [n_windows+1]
  int64_t n_tiles_total = 0;

  // ---- run state ----
  bool have_run = false, compacted = false;
  ReplaySnapshot replay;  // sizes of the last completed run on this batch, for the replay mode of ls_pileup_run
  ls_count_params params = {};
  DBuf segs, pieces, keys_a, keys_b, vals_a, vals_b, rs_hist, scan_tmp, counters;
  DBuf tile_flag, tile_rank, slot_tile, slot_lo, slot_out, slot_mask, slot_npass, slot_off;
  DBuf drop_keys, rend, wcount, part_slot, slot_done, slot_desc, acbuf;  // part_slot: PartDesc records
  DBuf offs_s, offs_m, offs_u, units, goffs, gdir, mrank, mlist;
  int64_t n_drop = 0;
  bool k1_attr_set = false;
  int64_t n_segments = 0, n_pieces = 0, n_slots = 0, n_sites = 0;
  int cell_bits = 0;
  uint64_t *sorted_keys = nullptr;
  uint32_t *sorted_vals = nullptr;
  ls_run_stats stats = {};

  // ---- fetch / misc scratch ----
  DBuf out_tid, out_pos, out_ref, out_counts;
  DBuf l2_scratch;
  DBuf g_a, g_b, g_c, g_d, g_e;  // scratch of K2 and K3: nothing lives in them across an entry-point call
  // K3: resident sorted site tables (slot LS_SITE_TABLES is the scratch table of the one-shot ls_site_mask)
  DBuf site_tab[LS_SITE_TABLES + 1];
  int64_t site_tab_n[LS_SITE_TABLES + 1] = {};
  bool site_tab_ok[LS_SITE_TABLES + 1] = {};
  GenoState geno;  // K1'
  GenoMatrixState gm;  // genotype matrix writer
  GenoLongState gl;    // genotype long-table writer
  CounterTextState ct;  // counter table writer
  Step1State s1;        // BaseCellCalling.step1
};

#define LS_CK(call)                                                                        \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess) {                                                               \
      char _b[512];                                                                        \
      snprintf(_b, sizeof _b, "%s:%d: %s -> %s", __FILE__, __LINE__, #call,                \
               cudaGetErrorString(_e));                                                    \
      ctx->err = _b;                                                                       \
      return LS_E_CUDA;                                                                    \
    }                                                                                      \
  } while (0)

#define LS_FAIL(code, msg) \
  do {                     \
    ctx->err = (msg);      \
    return (code);         \
  } while (0)

static inline int ls_bits_for(uint64_t v) {  // number of bits needed to hold values 0..v
  int b = 0;
  while (v) {
    ++b;
    v >>= 1;
  }
  return b < 1 ? 1 : b;
}

// ---- device helpers ---------------------------------------------------------------------
__device__ __forceinline__ bool op_is_match(uint32_t op) { return op == OP_M || op == OP_EQ || op == OP_X; }
__device__ __forceinline__ bool op_consumes_ref(uint32_t op) {
  return op == OP_M || op == OP_D || op == OP_N || op == OP_EQ || op == OP_X;
}

// read-level filter of the pileup engine (SURVEY Appendix A.2; pysam __advance_samtools)
__device__ __forceinline__ bool read_passes_engine(uint32_t flag, uint32_t mapq, int min_mq) {
  if (flag & LS_FLAG_FILTER) return false;
  if ((int)mapq < min_mq) return false;
  if ((flag & LS_FLAG_PAIRED) && !(flag & LS_FLAG_PROPER)) return false;  // ignore_orphans
  return true;
}

// Sign of htslib's pileup "indel" field at the LAST reference position of op k
// (resolve_cigar2: peek at the following ops).  Returns +1 (insertion follows),
// -1 (deletion follows), 0.
__device__ __forceinline__ int indel_after(const uint32_t *__restrict__ cigar, uint32_t k, uint32_t kend,
                                           uint32_t op) {
  if (k + 1 >= kend) return 0;
  uint32_t op2 = cigar[k + 1] & 15u;
  if (op2 == OP_D && op != OP_D) return -1;
  if (op2 == OP_I) return +1;
  if (op2 == OP_P && k + 2 < kend) {
    uint32_t l3 = 0;
    for (uint32_t kk = k + 2; kk < kend; ++kk) {
      uint32_t c = cigar[kk];
      uint32_t o = c & 15u;
      if (o == OP_I)
        l3 += c >> 4;
      else if (o == OP_D || o == OP_M || o == OP_N || o == OP_EQ || o == OP_X)
        break;
    }
    if (l3 > 0) return +1;
  }
  return 0;
}

// BAM nibble code -> allele class (EasyReadPileup, BaseCellCounter.py:152-180)
__device__ __forceinline__ int class_of_code(uint32_t code) {
  // =ACMGRSVTWYHKDBN : 1=A 2=C 4=G 8=T 15=N
  switch (code) {
    case 1: return LS_CLASS_A;
    case 2: return LS_CLASS_C;
    case 4: return LS_CLASS_G;
    case 8: return LS_CLASS_T;
    case 15: return LS_CLASS_N;
    default: return LS_CLASS_NA;
  }
}

__device__ __forceinline__ uint8_t class_letter(int cls) {
  // "ACTGIDNO" packed little-endian, one byte per class id
  return (uint8_t)((0x4F4E444947544341ull >> (8 * (cls & 7))) & 0xffu);
}

__device__ __forceinline__ uint8_t upper_ascii(uint8_t c) { return (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c; }

int ls_depth_cap_host(ls_ctx *ctx, const std::vector<int32_t> &wtid, const std::vector<int32_t> &wstart,
                      const std::vector<int32_t> &wend, const uint32_t *d_wcount, int min_mq, int max_depth);
int ls_tile_size(void);

// ---- utilities implemented in ls_util.cu --------------------------------------------------
// several independent exclusive scans in one launch (ls_util.cu)
constexpr int LS_SCAN_MAX_JOBS = 6;
struct LsScanJob {
  const uint32_t *in;
  uint32_t *out;
  int64_t n;
  uint64_t *total;  // may be null
  uint64_t *out64 = nullptr;  // ls_scan_exclusive_u32_wide only: the 64-bit prefixes
};
cudaError_t ls_scan_exclusive_u32_multi(const LsScanJob *jobs, int n_jobs, DBuf &tmp, cudaStream_t st);
cudaError_t ls_scan_exclusive_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n, uint64_t *d_total,
                                  DBuf &tmp, cudaStream_t st);
// d_out[0 .. n]: exclusive prefix sums of d_in as 64-bit values, d_out[n] the total; every 2048 consecutive inputs
// must sum below 2^32
cudaError_t ls_scan_exclusive_u32_wide(const uint32_t *d_in, uint64_t *d_out, int64_t n, DBuf &tmp, cudaStream_t st);
cudaError_t ls_radix_sort_pairs(uint64_t *keys_a, uint64_t *keys_b, uint32_t *vals_a, uint32_t *vals_b,
                                int64_t n, int key_bits, DBuf &hist, uint64_t **sorted_keys,
                                uint32_t **sorted_vals, int num_sms, cudaStream_t st, int *launches);
cudaError_t ls_radix_sort_keys32(uint32_t *keys_a, uint32_t *keys_b, int64_t n, int key_bits, DBuf &hist,
                                 uint32_t **sorted_keys, int num_sms, cudaStream_t st, int *launches);
cudaError_t ls_radix_sort_keys(uint64_t *keys_a, uint64_t *keys_b, int64_t n, int key_bits, DBuf &hist,
                               uint64_t **sorted_keys, int num_sms, cudaStream_t st, int *launches);
