// BaseCellCalling.step1 on the device: one line-aligned byte range of the merged table's body in, the output text of
// that range out.  The rules are those of the host passes ls_s1_parse + ls_s1_format (csrc/host/ls_step1.cpp), which
// restate BaseCellCalling.step1.py:78-467 (SURVEY Appendix C); the text is byte for byte theirs.
//
//   load  line starts (newline flags, chained scan), then one thread per row: the columns, the qualifying gate, the
//         candidate alleles and the rest sums, with the strictness of ls_s1_parse (a row it refuses refuses the
//         range, and the lowest such row is reported).  The per-row query counts are scanned, the CHROM runs of the
//         range are mapped to contig ids on the host (a table is grouped by contig: a few runs per range), and the
//         (k, n) queries of both families are written in the host passes' order.
//   call  K2 on the queries (ls_betabinom_device, the long tails through the staged path of ls_betabinom_sf), the
//         tails rounded as np.round(p, 4) does, then one thread per row measures its output row: the label cascade,
//         the contexts from the resident contigs, the twenty INFO columns.  The lengths are scanned to 64-bit offsets.
//   text  as many whole rows as fit the caller's block, one thread per row: a CTA stages its tile of consecutive rows
//         in shared memory and stores it with 16-byte stores (copy_out); a tile longer than the stage is stored row
//         by row.
// Beyond ls_s1_parse, the device refuses a range with a '\r' (the host passes read universal newlines), a candidate
// allele at a depth or cell count of 0 and a VAF / MCF of 4e5 or more (both beyond the 32-bit digit formatting; the
// Python passes fail on the first), so the caller redoes such a range on the host.  ls_s1_format's refusals (a NaN
// among a call's per-allele tails) refuse it at the call.  Compiled with -fmad=false, as K2.
#include <algorithm>
#include <unordered_map>

#include "ls_common.cuh"
#include "ls_text.cuh"

int ls_betabinom_device(ls_ctx *ctx, const int32_t *d_k, const int32_t *d_n, double a, double b, double *d_p, int64_t m,
                        uint32_t *d_nbig);

namespace {

constexpr int S1_THREADS = 128;          // rows per tile of the text kernel
constexpr uint32_t S1_STAGE = 48 << 10;  // bytes of a tile staged in shared memory (typical rows: 250-400 bytes)
constexpr int S1_MAX_CT = 64;            // cell-type columns (ls_s1_format's per-row tables hold 64 calls)
constexpr double S1_RATIO_MAX = 4.0e5;   // VAF / MCF * 1e4 must fit the 32-bit units of put_units4

struct S1Row {
  int64_t lo, pos;
  int64_t sum_bc, sum_cc, sum_dp, sum_nc;  // the rest sums: Sum_alts_bc, Sum_alts_cc, Sum_dp, Sum_nc
  int32_t len, tab4;                       // line length without its end; offset of the 4th tab (-1: none)
  int32_t chrom_len, n_qual, ncall, ctg;   // ctg: contig id (-1 for a verbatim row)
  uint8_t verbatim, nl, rest, pad;         // nl: the line ends in '\n'; rest: the row has the noise test
};

struct S1Call {
  int32_t ct, DP, NC;
  uint32_t has_bc, has_cc;  // bit x: allele x (A, C, T, G) has reads / cells
  int32_t bc[4], cc[4];
};

enum { E_COLS = 1, E_POS, E_FIELDS, E_DPNC, E_LIST, E_BIG, E_NOCELLS, E_ZERO, E_RATIO };
const char *const S1_MSG[] = {"",
                              "fewer columns than the header names",
                              "POS is not a plain integer",
                              "a cell-type column does not have seven '|' fields",
                              "DP / NC is not a plain integer",
                              "CC / BC is not a ':' list of at most eight integers",
                              "count above 2^31",
                              "an allele has reads but no cells",
                              "a candidate allele at a depth or cell count of 0",
                              "a VAF or MCF of 4e5 or more"};
enum { B_CR = 1, B_NAN = 2, B_ROUND = 4 };

// ---- load --------------------------------------------------------------------------------------
__global__ void s1_line_kernel(const char *__restrict__ d, int64_t len, uint32_t *__restrict__ flag,
                               unsigned long long *__restrict__ bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) {
    flag[i] = (i == 0 || d[i - 1] == '\n') ? 1u : 0u;
    if (d[i] == '\r') atomicOr(bad, (unsigned long long)B_CR);
  }
}

__global__ void s1_start_kernel(const char *__restrict__ d, int64_t len, const uint32_t *__restrict__ idx,
                                int64_t *__restrict__ row_lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
    if (i == 0 || d[i - 1] == '\n') row_lo[idx[i]] = i;
}

__device__ __forceinline__ bool parse_uint(const char *p, const char *e, int64_t &v) {
  if (p >= e || e - p > 18) return false;
  int64_t x = 0;
  for (; p < e; ++p) {
    if (*p < '0' || *p > '9') return false;
    x = x * 10 + (*p - '0');
  }
  v = x;
  return true;
}

// "a:b:c..." (at most eight non-negative integers): *sum over the alleles other than REF and 'O'; bit x of *has and
// a[x] for the alleles x < 4 other than REF with a count > 0; *big when one of those is above 2^31 - 1
__device__ __forceinline__ bool parse_list(const char *p, const char *e, int ref_idx, int32_t *a, uint32_t *has,
                                           int64_t *sum, bool *big) {
  for (int x = 0;; ++x) {
    const char *q = p;
    while (q < e && *q != ':') ++q;
    int64_t v;
    if (x >= 8 || !parse_uint(p, q, v)) return false;
    if (x != ref_idx && x != 7) *sum += v;
    if (x < 4 && x != ref_idx && v > 0) {
      if (v > 0x7fffffff) *big = true;
      *has |= 1u << x;
      a[x] = (int32_t)v;
    }
    if (q >= e) return true;
    p = q + 1;
  }
}

struct S1Parse {
  const char *d;
  const int64_t *row_lo;
  int64_t n_rows;
  const int32_t *cols;
  int32_t n_ct, max_col, min_cov, min_cells;
  S1Row *rows;
  S1Call *calls;
  uint32_t *q1c, *q2c, *runf;
  unsigned long long *err;  // lowest (row << 8 | code) of a refused row
};

// one cell-type column [f, fe) of row R; t: the row's next call slot
__device__ int parse_cell(const S1Parse &a, const char *f, const char *fe, int ct, int ref_idx, S1Row &R, S1Call *t,
                          uint32_t &nq1, uint32_t &nq2) {
  if (fe - f >= 2 && f[0] == 'N' && f[1] == 'A') return 0;
  const char *e0 = nullptr, *e1 = nullptr, *e2 = nullptr, *e3 = nullptr;  // ends of DP|NC|CC|BC|BQ|BCf|BCr
  int nb = 0;
  for (const char *c = f; c < fe; ++c)
    if (*c == '|') {
      if (nb >= 6) return E_FIELDS;
      e0 = nb == 0 ? c : e0;
      e1 = nb == 1 ? c : e1;
      e2 = nb == 2 ? c : e2;
      e3 = nb == 3 ? c : e3;
      ++nb;
    }
  if (nb != 6) return E_FIELDS;
  int64_t DP, NC;
  if (!parse_uint(f, e0, DP) || !parse_uint(e0 + 1, e1, NC) || DP > 0x7fffffff || NC > 0x7fffffff) return E_DPNC;
  if (!(DP >= a.min_cov && NC >= a.min_cells)) return 0;
  ++R.n_qual;
  uint32_t has_cc = 0, has_bc = 0;
  int64_t scc = 0, sbc = 0;
  bool big = false;
  if (!parse_list(e1 + 1, e2, ref_idx, t->cc, &has_cc, &scc, &big) ||
      !parse_list(e2 + 1, e3, ref_idx, t->bc, &has_bc, &sbc, &big))
    return E_LIST;
  R.sum_bc += sbc;
  R.sum_cc += scc;
  R.sum_dp += DP;
  R.sum_nc += NC;
  if (big) return E_BIG;
  if (!has_bc) return 0;
  if (has_bc & ~has_cc) return E_NOCELLS;
  if (DP == 0 || NC == 0) return E_ZERO;
  int64_t b0 = 0, c0 = 0;
  for (int x = 0; x < 4; ++x)
    if (has_bc & (1u << x)) {
      if ((double)t->bc[x] >= S1_RATIO_MAX * (double)DP || (double)t->cc[x] >= S1_RATIO_MAX * (double)NC) return E_RATIO;
      b0 += t->bc[x];
      c0 += t->cc[x];
    }
  t->ct = ct;
  t->DP = (int32_t)DP;
  t->NC = (int32_t)NC;
  t->has_bc = has_bc;
  t->has_cc = has_cc;
  R.sum_dp -= b0;
  R.sum_nc -= c0;
  R.sum_bc -= b0;
  R.sum_cc -= c0;
  ++R.ncall;
  nq1 += __popc(has_bc);
  nq2 += __popc(has_cc);
  return 0;
}

__device__ int parse_row(const S1Parse &a, int64_t r, int64_t lo, int64_t hi, S1Row &R, uint32_t &nq1, uint32_t &nq2) {
  const char *d = a.d;
  int ncol = 1;
  for (int64_t i = lo; i < hi; ++i) ncol += d[i] == '\t';
  if (ncol <= a.max_col) return E_COLS;
  const char *const ALLELE = "ACTGIDNO";
  S1Call *slots = a.calls + r * a.n_ct;
  int ref_idx = -1, ci = 0;
  int64_t s = lo;
  for (int64_t j = lo, c = 0;; ++j) {
    if (j < hi && d[j] != '\t') continue;
    if (c == 0) {
      R.chrom_len = (int32_t)(j - lo);
    } else if (c == 1) {
      if (!parse_uint(d + s, d + j, R.pos)) return E_POS;
    } else if (c == 3) {
      if (j - s == 1)
        for (int x = 0; x < 8; ++x)
          if (d[s] == ALLELE[x]) ref_idx = x;
      if (j < hi) R.tab4 = (int32_t)(j - lo);
    } else if (ci < a.n_ct && c == a.cols[ci]) {
      const int e = parse_cell(a, d + s, d + j, ci, ref_idx, R, slots + R.ncall, nq1, nq2);
      if (e) return e;
      ++ci;
    }
    if (j >= hi) break;
    s = j + 1;
    ++c;
  }
  if (R.sum_bc > 0) {  // the noise test
    if (R.sum_bc > 0x7fffffff || R.sum_dp > 0x7fffffff || R.sum_dp < -0x7fffffff || R.sum_cc > 0x7fffffff ||
        R.sum_cc < -0x7fffffff || R.sum_nc > 0x7fffffff || R.sum_nc < -0x7fffffff)
      return E_BIG;
    R.rest = 1;
    ++nq1;
    ++nq2;
  }
  return 0;
}

// a data row starts a contig run unless the row before it is a data row with the same CHROM
__device__ bool run_start(const char *d, const int64_t *row_lo, int64_t r, int64_t lo, int32_t clen) {
  if (r == 0) return true;
  const int64_t p = row_lo[r - 1], pe = lo - 1;  // the row before ends in the '\n' at lo - 1
  if (pe - p >= 2 && d[p] == '#' && d[p + 1] == '#') return true;
  int64_t k = 0;
  while (k < clen && p + k < pe && d[p + k] == d[lo + k]) ++k;
  return !(k == clen && (p + k == pe || d[p + k] == '\t'));
}

__global__ void __launch_bounds__(256) s1_parse_kernel(S1Parse a) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    S1Row R;
    memset(&R, 0, sizeof R);
    const int64_t lo = a.row_lo[r], end = a.row_lo[r + 1];
    const bool nl = end > lo && a.d[end - 1] == '\n';
    const int64_t hi = end - (nl ? 1 : 0);
    R.lo = lo;
    R.len = (int32_t)(hi - lo);
    R.nl = nl ? 1 : 0;
    R.tab4 = -1;
    R.ctg = -1;
    uint32_t nq1 = 0, nq2 = 0, run = 0;
    if (hi - lo >= 2 && a.d[lo] == '#' && a.d[lo + 1] == '#') {
      R.verbatim = 1;
    } else {
      const int e = parse_row(a, r, lo, hi, R, nq1, nq2);
      if (e) atomicMin(a.err, ((unsigned long long)r << 8) | (unsigned long long)e);
      run = run_start(a.d, a.row_lo, r, lo, R.chrom_len) ? 1u : 0u;
    }
    a.rows[r] = R;
    a.q1c[r] = nq1;
    a.q2c[r] = nq2;
    a.runf[r] = run;
  }
}

// each contig run: its first row's line start and CHROM length
__global__ void s1_runs_kernel(const S1Row *__restrict__ rows, const uint32_t *__restrict__ runf,
                               const uint32_t *__restrict__ runx, int64_t n_rows, int64_t *__restrict__ run_lo) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x)
    if (runf[r]) {
      run_lo[2 * runx[r]] = rows[r].lo;
      run_lo[2 * runx[r] + 1] = rows[r].chrom_len;
    }
}

// the contig id of every data row, and its (k, n) queries in the order of the host passes: per call the read counts
// (q1) and the cell counts (q2) of its alleles in A, C, T, G order, then the row's noise test
__global__ void s1_query_kernel(S1Row *__restrict__ rows, const S1Call *__restrict__ calls, int32_t n_ct, int64_t n_rows,
                                const uint32_t *__restrict__ q1off, const uint32_t *__restrict__ q2off,
                                const uint32_t *__restrict__ runf, const uint32_t *__restrict__ runx,
                                const int32_t *__restrict__ run_ctg, int32_t *__restrict__ k1, int32_t *__restrict__ n1,
                                int32_t *__restrict__ k2, int32_t *__restrict__ n2) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    S1Row &R = rows[r];
    if (R.verbatim) continue;
    R.ctg = run_ctg[runx[r] + runf[r] - 1];
    uint32_t o1 = q1off[r], o2 = q2off[r];
    for (int k = 0; k < R.ncall; ++k) {
      const S1Call &t = calls[r * n_ct + k];
#pragma unroll
      for (int x = 0; x < 4; ++x)
        if (t.has_bc & (1u << x)) {
          k1[o1] = t.bc[x];
          n1[o1++] = t.DP;
        }
#pragma unroll
      for (int x = 0; x < 4; ++x)
        if (t.has_cc & (1u << x)) {
          k2[o2] = t.cc[x];
          n2[o2++] = t.NC;
        }
    }
    if (R.rest) {
      k1[o1] = (int32_t)R.sum_bc;
      n1[o1] = (int32_t)R.sum_dp;
      k2[o2] = (int32_t)R.sum_cc;
      n2[o2] = (int32_t)R.sum_nc;
    }
  }
}

// ---- call --------------------------------------------------------------------------------------
// np.round(p, 4) of the tails.  ls_betabinom_device answers k == 0 with NaN ("no query"); the host passes' K2 answers
// it as scipy does (1, NaN for n < 0): the noise test's cell-count query can have k == 0.
__global__ void s1_round_kernel(const int32_t *__restrict__ k, const int32_t *__restrict__ n, double *__restrict__ p,
                                int64_t m) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = k[i] <= 0 ? (n[i] < 0 ? NAN : 1.0) : p[i];  // ls_sf_finish(k, n, 0) of ls_pairwise.h
    p[i] = isnan(v) ? v : rint(v * 10000.0) / 10000.0;
  }
}

// text at o (o null: length only)
struct Out {
  char *o;
  uint32_t n;
  __device__ void ch(char x) {
    if (o) o[n] = x;
    ++n;
  }
  __device__ void str(const char *x) {
    while (*x) ch(*x++);
  }
  __device__ void span(const char *x, int64_t len) {
    if (o)
      for (int64_t i = 0; i < len; ++i) o[n + i] = x[i];
    n += (uint32_t)len;
  }
  __device__ void i64(int64_t v) {
    if (v < 0) ch('-');
    uint64_t u = v < 0 ? (uint64_t)(-(v + 1)) + 1u : (uint64_t)v;
    int nd = 1;
    for (uint64_t q = u; q >= 10u; q /= 10u) ++nd;
    if (o)
      for (int i = nd - 1; i >= 0; --i) {
        o[n + i] = (char)('0' + u % 10u);
        u /= 10u;
      }
    n += nd;
  }
  __device__ void units4(uint32_t k) { n += put_units4(k, o ? o + n : nullptr); }
};

struct S1View {
  const char *d;
  const S1Row *rows;
  const S1Call *calls;
  const uint32_t *q1off, *q2off;
  const double *p1, *p2;
  const char *names;
  const int64_t *name_off;
  const uint64_t *ctg_ptr;
  const int64_t *ctg_len;
  const uint64_t *off;
  int32_t n_ct, n_ctg, min_ac_cells, min_ac_reads, min_cell_types, max_cell_types;
};

// str() of a tail already rounded to four places (put_round4 of ls_step1.cpp; its fast path is exact for these)
__device__ __forceinline__ void put_p(Out &t, double v, uint32_t &bad) {
  if (isnan(v)) {
    t.str("nan");
    return;
  }
  const double sc = v * 1e4, fl = floor(sc), frac = sc - fl;
  if (!(v >= 0.0 && v < S1_RATIO_MAX) || fabs(frac - 0.5) <= 1e-6) {
    bad |= B_ROUND;
    return;
  }
  t.units4((uint32_t)fl + (frac > 0.5 ? 1u : 0u));
}

__device__ __forceinline__ int sorted_allele(int j) { return (0x2310 >> (4 * j)) & 15; }  // A, C, G, T

// the candidate alleles of a call as the reference prints them: "A|C|G|T" at most
template <typename F>
__device__ __forceinline__ void for_alts(uint32_t has_bc, F &&f) {
  bool first = true;
  for (int j = 0; j < 4; ++j) {
    const int x = sorted_allele(j);
    if (!(has_bc & (1u << x))) continue;
    if (!first) f('|');
    first = false;
    f("ACTG"[x]);
  }
}

enum { L_NONSIG, L_LOWSIG, L_MULTI, L_LOWCELLS, L_LOWREADS, L_PASS };
__device__ const char *label_text(int l) {
  switch (l) {
    case L_NONSIG: return "Non-Significant";
    case L_LOWSIG: return "Low-Significance";
    case L_MULTI: return "Multi-allelic";
    case L_LOWCELLS: return "Low_cells";
    case L_LOWREADS: return "Low_reads";
    default: return "PASS";
  }
}

// the type label of one call (step1.py:206-226); b1 / b2: its first read- / cell-count query
__device__ int call_label(const S1View &v, const S1Call &t, uint32_t b1, uint32_t b2, uint32_t &bad) {
  double mb = INFINITY, mc = INFINITY;
  for (int x = 0; x < 4; ++x) {
    if (t.has_bc & (1u << x)) {
      const double p = v.p1[b1 + __popc(t.has_bc & ((1u << x) - 1u))];
      if (isnan(p)) bad |= B_NAN;
      mb = p < mb ? p : mb;
    }
    if (t.has_cc & (1u << x)) {
      const double p = v.p2[b2 + __popc(t.has_cc & ((1u << x) - 1u))];
      if (isnan(p)) bad |= B_NAN;
      mc = p < mc ? p : mc;
    }
  }
  if (mb >= 0.05 || mc >= 0.05) return L_NONSIG;
  if ((0.001 < mb && mb < 0.05) || (0.001 < mc && mc < 0.05)) return L_LOWSIG;
  if (__popc(t.has_bc) > 1) return L_MULTI;
  const int x = __ffs(t.has_bc) - 1;
  if (t.cc[x] < v.min_ac_cells) return L_LOWCELLS;
  if (t.bc[x] < v.min_ac_reads) return L_LOWREADS;
  return L_PASS;
}

struct Run {  // longest run of equal characters (step1.py:478-483)
  int best = 0, cur = 0;
  char prev = 0;
  bool first = true;
  __device__ void operator()(char c) {
    cur = (!first && c == prev) ? cur + 1 : 1;
    first = false;
    prev = c;
    if (cur > best) best = cur;
  }
};

// the row r of the output; bad collects the refusals (only the measuring pass looks at them)
__device__ void put_row(const S1View &v, int64_t r, Out &t, uint32_t &bad) {
  const S1Row R = v.rows[r];
  const char *line = v.d + R.lo;
  if (R.verbatim) {
    t.span(line, R.len);
    if (R.nl) t.ch('\n');
    return;
  }
  t.span(line, R.tab4 >= 0 ? R.tab4 : R.len);
  t.ch('\t');
  // fetch(CHROM, POS - 6, POS + 5).upper(): cl bases (clipped at the contig's end), -1: '.'
  int cl = -1;
  const uint8_t *cb = nullptr;
  if (R.ctg >= 0 && R.ctg < v.n_ctg && v.ctg_len[R.ctg] >= 0 && R.pos >= 6) {
    const int64_t start = R.pos - 6, avail = v.ctg_len[R.ctg] - start;
    cl = avail < 0 ? 0 : (avail > 11 ? 11 : (int)avail);
    cb = reinterpret_cast<const uint8_t *>(v.ctg_ptr[R.ctg]) + start;
  }
  auto base = [&](int k) { return (char)upper_ascii(cb[k]); };
  const int up_n = cl < 0 ? 0 : (cl < 5 ? cl : 5), dn_n = cl > 6 ? cl - 6 : 0;
  const bool up_dot = cl < 0 || (up_n == 1 && base(0) == '.'), dn_dot = cl < 0 || (dn_n == 1 && base(6) == '.');
  auto put_up = [&]() {
    if (cl < 0)
      t.ch('.');
    else
      for (int k = 0; k < up_n; ++k) t.ch(base(k));
  };
  auto put_down = [&]() {
    if (cl < 0)
      t.ch('.');
    else
      for (int k = 0; k < dn_n; ++k) t.ch(base(6 + k));
  };
  const bool has_rest = R.rest;
  const double bc_noise = has_rest ? v.p1[v.q1off[r + 1] - 1] : 1.0, cc_noise = has_rest ? v.p2[v.q2off[r + 1] - 1] : 1.0;
  auto put_rest = [&](int64_t a, int64_t b, double p) {
    t.i64(a);
    t.ch(';');
    t.i64(b);
    t.ch(';');
    if (has_rest)
      put_p(t, p, bad);
    else
      t.ch('1');  // a plain int in the reference (Q7)
  };
  if (R.ncall > 0) {
    const S1Call *tc = v.calls + r * v.n_ct;
    const uint32_t q1 = v.q1off[r], q2 = v.q2off[r];
    // the labels of the calls, recomputed where they are printed
    auto each_label = [&](auto &&f) {
      uint32_t b1 = q1, b2 = q2;
      for (int k = 0; k < R.ncall; ++k) {
        const S1Call &c = tc[k];
        f(k, call_label(v, c, b1, b2, bad));
        b1 += __popc(c.has_bc);
        b2 += __popc(c.has_cc);
      }
    };
    int n_pass = 0, n_nonsig = 0;
    bool any_multi = false;
    uint32_t seen = 0;  // distinct ALT strings: one per candidate set
    each_label([&](int k, int l) {
      n_pass += l == L_PASS;
      n_nonsig += l == L_NONSIG;
      any_multi = any_multi || l == L_MULTI;
      seen |= 1u << tc[k].has_bc;
    });
    const int len_alts = __popc(seen);
    auto homopolymer = [&](bool upstream) {
      if (upstream ? up_dot : dn_dot) return false;
      int m = 0;
      for (int k = 0; k < R.ncall; ++k) {
        Run run;
        if (upstream)
          for (int i = 0; i < up_n; ++i) run(base(i));
        for_alts(tc[k].has_bc, run);
        if (!upstream)
          for (int i = 0; i < dn_n; ++i) run(base(6 + i));
        m = run.best > m ? run.best : m;
      }
      return m >= 4;
    };
    const bool f_mct = n_pass > v.max_cell_types, f_mal = len_alts > 1 || any_multi, f_min = R.n_qual < v.min_cell_types,
               f_noise = R.ncall - n_pass - n_nonsig > 0, f_noisy = bc_noise < 0.05 || cc_noise < 0.05,
               f_lcu = homopolymer(true), f_lcd = homopolymer(false);
    auto join_calls = [&](auto &&f) {
      for (int k = 0; k < R.ncall; ++k) {
        if (k) t.ch(',');
        f(tc[k]);
      }
    };
    auto per_cand = [&](const S1Call &c, auto &&f) {
      bool first = true;
      for (int j = 0; j < 4; ++j) {
        const int x = sorted_allele(j);
        if (!(c.has_bc & (1u << x))) continue;
        if (!first) t.ch('|');
        first = false;
        f(x);
      }
    };
    join_calls([&](const S1Call &c) { for_alts(c.has_bc, [&](char x) { t.ch(x); }); });  // ALT
    t.ch('\t');
    if (f_mct || f_mal || f_min || f_noise || f_noisy || f_lcu || f_lcd) {  // FILTER
      bool first = true;
      auto add = [&](bool on, const char *s) {
        if (!on) return;
        if (!first) t.ch(',');
        first = false;
        t.str(s);
      };
      add(f_mct, "Multiple_cell_types");
      add(f_mal, "Multi-allelic");
      add(f_min, "Min_cell_types");
      add(f_noise, "Cell_type_noise");
      add(f_noisy, "Noisy_site");
      add(f_lcu, "LC_Upstream");
      add(f_lcd, "LC_Downstream");
    } else if (n_pass > 0) {
      t.str("PASS");
    } else {
      each_label([&](int k, int l) {
        if (k) t.ch(',');
        t.str(label_text(l));
      });
    }
    t.ch('\t');
    join_calls([&](const S1Call &c) { t.span(v.names + v.name_off[c.ct], v.name_off[c.ct + 1] - v.name_off[c.ct]); });
    t.ch('\t');
    put_up();
    t.ch('\t');
    put_down();
    t.ch('\t');
    t.i64(len_alts);
    t.ch('\t');
    join_calls([&](const S1Call &c) { t.i64(c.DP); });
    t.ch('\t');
    join_calls([&](const S1Call &c) { t.i64(c.NC); });
    t.ch('\t');
    join_calls([&](const S1Call &c) { per_cand(c, [&](int x) { t.i64(c.bc[x]); }); });
    t.ch('\t');
    join_calls([&](const S1Call &c) { per_cand(c, [&](int x) { t.i64(c.cc[x]); }); });
    t.ch('\t');
    join_calls([&](const S1Call &c) { per_cand(c, [&](int x) { t.units4(vaf_units(c.bc[x], c.DP)); }); });
    t.ch('\t');
    join_calls([&](const S1Call &c) { per_cand(c, [&](int x) { t.units4(vaf_units(c.cc[x], c.NC)); }); });
    t.ch('\t');
    {
      uint32_t b1 = q1;
      join_calls([&](const S1Call &c) {
        per_cand(c, [&](int x) { put_p(t, v.p1[b1 + __popc(c.has_bc & ((1u << x) - 1u))], bad); });
        b1 += __popc(c.has_bc);
      });
    }
    t.ch('\t');
    {
      uint32_t b2 = q2;
      join_calls([&](const S1Call &c) {
        per_cand(c, [&](int x) { put_p(t, v.p2[b2 + __popc(c.has_cc & ((1u << x) - 1u))], bad); });
        b2 += __popc(c.has_cc);
      });
    }
    t.ch('\t');
    t.i64(R.n_qual);
    t.ch('\t');
    t.i64(R.n_qual);  // Cell_types_min_BC printed twice (Q7)
    t.ch('\t');
    put_rest(R.sum_bc, R.sum_dp, bc_noise);
    t.ch('\t');
    put_rest(R.sum_cc, R.sum_nc, cc_noise);
    t.str("\t.\t");  // Fisher_p: '.' when --fisher_cutoff is 1
    each_label([&](int k, int l) {
      if (k) t.ch(',');
      t.str(label_text(l));
    });
  } else {
    t.str(".\t");
    t.str(bc_noise < 0.001 || cc_noise < 0.001 ? "Noisy_site" : ".");
    t.str("\t.\t");
    put_up();
    t.ch('\t');
    put_down();
    t.str("\t.\t.\t.\t.\t.\t.\t.\t.\t.\t");
    t.i64(R.n_qual);
    t.ch('\t');
    t.i64(R.n_qual);
    t.ch('\t');
    put_rest(R.sum_bc, R.sum_dp, bc_noise);
    t.ch('\t');
    put_rest(R.sum_cc, R.sum_nc, cc_noise);
    t.str("\t.\t.");
  }
  if (R.tab4 >= 0) t.span(line + R.tab4, R.len - R.tab4);  // "\t" + the columns from the fifth on
  t.ch('\n');
}

__global__ void __launch_bounds__(256) s1_len_kernel(S1View v, int64_t n_rows, uint32_t *__restrict__ lens,
                                                     unsigned long long *__restrict__ bad) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    Out t{nullptr, 0};
    uint32_t b = 0;
    put_row(v, r, t, b);
    lens[r] = t.n;
    if (b) atomicOr(bad, (unsigned long long)b);
  }
}

// ---- text --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(S1_THREADS) s1_write_kernel(S1View v, int64_t row_lo, int64_t row_hi,
                                                              char *__restrict__ out) {
  __shared__ __align__(16) char stage[S1_STAGE];
  const uint64_t base = v.off[row_lo];
  uint32_t bad = 0;
  for (int64_t t0 = row_lo + (int64_t)blockIdx.x * S1_THREADS; t0 < row_hi; t0 += (int64_t)gridDim.x * S1_THREADS) {
    const int64_t t1 = t0 + S1_THREADS < row_hi ? t0 + S1_THREADS : row_hi, i = t0 + threadIdx.x;
    const uint64_t tb = v.off[t0], tile = v.off[t1] - tb;
    if (tile <= S1_STAGE) {
      if (i < t1) {
        Out t{stage + (v.off[i] - tb), 0};
        put_row(v, i, t, bad);
      }
      __syncthreads();
      copy_out<S1_THREADS>(out + (tb - base), stage, (uint32_t)tile);
      __syncthreads();
    } else if (i < t1) {
      Out t{out + (v.off[i] - base), 0};
      put_row(v, i, t, bad);
    }
  }
}

template <typename T>
cudaError_t upload(DBuf &d, const T *h, int64_t n, cudaStream_t st) {
  cudaError_t e = d.ensure((size_t)n * sizeof(T) + 16);
  if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(d.p, h, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st);
  return e;
}

// the second array of qoff / run starts at this element: the scans take 16-byte aligned arrays
int64_t pair_stride(int64_t n_rows) { return (n_rows + 1 + 3) & ~(int64_t)3; }

unsigned grid_for(const ls_ctx *ctx, int64_t n, int threads) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, (int64_t)ctx->num_sms * 16));
}

// K2 leaves the queries past its in-register range at p = -1: those go through the staged path of ls_betabinom_sf
int long_tails(ls_ctx *ctx, const int32_t *d_k, const int32_t *d_n, double *d_p, int64_t m, double a, double b) {
  cudaStream_t st = ctx->stream;
  std::vector<int32_t> k((size_t)m), n((size_t)m);
  std::vector<double> p((size_t)m);
  LS_CK(cudaMemcpyAsync(k.data(), d_k, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(n.data(), d_n, (size_t)m * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(p.data(), d_p, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  std::vector<int64_t> big;
  for (int64_t i = 0; i < m; ++i)
    if (p[(size_t)i] == -1.0) big.push_back(i);
  std::vector<int32_t> bk(big.size()), bn(big.size());
  std::vector<double> bp(big.size());
  for (size_t j = 0; j < big.size(); ++j) {
    bk[j] = k[(size_t)big[j]];
    bn[j] = n[(size_t)big[j]];
  }
  int rc = ls_betabinom_sf(ctx, bk.data(), bn.data(), a, b, bp.data(), (int64_t)big.size(), nullptr);
  if (rc != LS_OK) return rc;
  for (size_t j = 0; j < big.size(); ++j) p[(size_t)big[j]] = bp[j];
  LS_CK(cudaMemcpyAsync(d_p, p.data(), (size_t)m * 8, cudaMemcpyHostToDevice, st));
  LS_CK(cudaStreamSynchronize(st));
  return LS_OK;
}

unsigned long long *ull(uint64_t *p) { return reinterpret_cast<unsigned long long *>(p); }

S1View make_view(const Step1State &s) {
  S1View v = {};
  v.d = s.data.as<char>();
  v.rows = s.rows.as<S1Row>();
  v.calls = s.calls.as<S1Call>();
  v.q1off = s.qoff.as<uint32_t>();
  v.q2off = v.q1off + pair_stride(s.n_rows);
  v.p1 = s.p.as<double>();
  v.p2 = v.p1 + s.n_q1;
  v.names = s.names.as<char>();
  v.name_off = s.name_off.as<int64_t>();
  v.ctg_ptr = s.ctg_ptr.as<uint64_t>();
  v.ctg_len = s.ctg_len.as<int64_t>();
  v.off = s.off.as<uint64_t>();
  v.n_ct = s.n_ct;
  v.n_ctg = (int32_t)s.contigs.size();
  v.min_ac_cells = s.min_ac_cells;
  v.min_ac_reads = s.min_ac_reads;
  v.min_cell_types = s.min_cell_types;
  v.max_cell_types = s.max_cell_types;
  return v;
}

}  // namespace

extern "C" int ls_step1_load(ls_ctx *ctx, const char *data, int64_t len, const ls_step1_in *in, int64_t *n_rows,
                             int64_t *n_queries, char *new_names, int64_t names_cap, int32_t *first_new,
                             int32_t *n_new) {
  if (!ctx) return LS_E_ARG;
  Step1State &s = ctx->s1;
  s.loaded = s.called = false;
  if (!in || !n_rows || !n_queries || !first_new || !n_new || (len > 0 && !data) || (names_cap > 0 && !new_names))
    LS_FAIL(LS_E_ARG, "ls_step1_load: null argument");
  if (len < 0 || len >= ((int64_t)1 << 31)) LS_FAIL(LS_E_ARG, "ls_step1_load: range length outside [0, 2^31)");
  if (in->n_ct < 0 || in->n_ct > S1_MAX_CT) LS_FAIL(LS_E_ARG, "ls_step1_load: more than 64 cell-type columns");
  if (in->n_ct > 0 && (!in->ct_cols || !in->ct_names || !in->ct_name_off))
    LS_FAIL(LS_E_ARG, "ls_step1_load: null cell-type array");
  for (int i = 0; i < in->n_ct; ++i)
    if (in->ct_cols[i] < 4 || (i > 0 && in->ct_cols[i] <= in->ct_cols[i - 1]))
      LS_FAIL(LS_E_ARG, "ls_step1_load: cell-type columns not ascending from column 4");
  if (!(in->alpha1 > 0.0) || !(in->beta1 > 0.0) || !(in->alpha2 > 0.0) || !(in->beta2 > 0.0))
    LS_FAIL(LS_E_ARG, "ls_step1_load: alpha and beta must be > 0");
  const int32_t n_ct = in->n_ct;
  std::vector<int64_t> name_off((size_t)n_ct + 1, 0);
  for (int i = 0; i < n_ct; ++i) {
    if (in->ct_name_off[i + 1] < in->ct_name_off[i]) LS_FAIL(LS_E_ARG, "ls_step1_load: name offsets not ascending");
    name_off[(size_t)i + 1] = in->ct_name_off[i + 1] - in->ct_name_off[0];
  }
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(s.result.ensure(8 * 8));
  uint64_t *res = s.result.as<uint64_t>();  // 0 rows, 1 error, 2-3 queries, 4 runs, 5 flags, 6-7 long tails
  const uint64_t init[8] = {0, ~0ull, 0, 0, 0, 0, 0, 0};
  LS_CK(cudaMemcpyAsync(res, init, sizeof init, cudaMemcpyHostToDevice, st));
  LS_CK(upload(s.data, data, len, st));
  LS_CK(upload(s.cols, in->ct_cols, n_ct, st));
  LS_CK(upload(s.names, n_ct ? in->ct_names + in->ct_name_off[0] : nullptr, name_off[(size_t)n_ct], st));
  LS_CK(upload(s.name_off, name_off.data(), (int64_t)n_ct + 1, st));
  // rows
  LS_CK(s.flag.ensure((size_t)len * 4 + 16));
  const char *d = s.data.as<char>();
  uint64_t h[8];
  if (len > 0) {
    s1_line_kernel<<<grid_for(ctx, len, 256), 256, 0, st>>>(d, len, s.flag.as<uint32_t>(), ull(res + 5));
    LS_CK(ls_scan_exclusive_u32(s.flag.as<uint32_t>(), s.flag.as<uint32_t>(), len, res, ctx->scan_tmp, st));
  }
  LS_CK(cudaMemcpyAsync(h, res, sizeof h, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (h[5] & B_CR) LS_FAIL(LS_E_ARG, "ls_step1_load: a line ends in '\\r'");
  const int64_t nr = (int64_t)h[0];
  LS_CK(s.row_lo.ensure((size_t)(nr + 1) * 8));
  if (len > 0) s1_start_kernel<<<grid_for(ctx, len, 256), 256, 0, st>>>(d, len, s.flag.as<uint32_t>(), s.row_lo.as<int64_t>());
  LS_CK(cudaMemcpyAsync(s.row_lo.as<int64_t>() + nr, &len, 8, cudaMemcpyHostToDevice, st));
  // parse
  LS_CK(s.rows.ensure((size_t)nr * sizeof(S1Row) + 16));
  LS_CK(s.calls.ensure((size_t)nr * std::max(n_ct, 1) * sizeof(S1Call) + 16));
  const int64_t stride = pair_stride(nr);
  LS_CK(s.qoff.ensure((size_t)stride * 2 * 4));
  LS_CK(s.run.ensure((size_t)stride * 2 * 4));
  uint32_t *q1c = s.qoff.as<uint32_t>(), *q2c = q1c + stride, *runf = s.run.as<uint32_t>(), *runx = runf + stride;
  LS_CK(cudaMemsetAsync(q1c + nr, 0, 4, st));
  LS_CK(cudaMemsetAsync(q2c + nr, 0, 4, st));
  LS_CK(cudaMemsetAsync(runf + nr, 0, 4, st));
  S1Parse a = {};
  a.d = d;
  a.row_lo = s.row_lo.as<int64_t>();
  a.n_rows = nr;
  a.cols = s.cols.as<int32_t>();
  a.n_ct = n_ct;
  a.max_col = n_ct ? std::max(3, in->ct_cols[n_ct - 1]) : 3;
  a.min_cov = in->min_cov;
  a.min_cells = in->min_cells;
  a.rows = s.rows.as<S1Row>();
  a.calls = s.calls.as<S1Call>();
  a.q1c = q1c;
  a.q2c = q2c;
  a.runf = runf;
  a.err = ull(res + 1);
  if (nr > 0) s1_parse_kernel<<<grid_for(ctx, nr, 256), 256, 0, st>>>(a);
  LS_CK(cudaGetLastError());
  const LsScanJob jobs[3] = {{q1c, q1c, nr + 1, res + 2}, {q2c, q2c, nr + 1, res + 3}, {runf, runx, nr + 1, res + 4}};
  LS_CK(ls_scan_exclusive_u32_multi(jobs, 3, ctx->scan_tmp, st));
  LS_CK(cudaMemcpyAsync(h, res, sizeof h, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (h[1] != ~0ull) {
    char b[160];
    snprintf(b, sizeof b, "ls_step1_load: row %lld: %s", (long long)(h[1] >> 8), S1_MSG[h[1] & 255u]);
    LS_FAIL(LS_E_ARG, b);
  }
  // contig runs -> contig ids; the names first met in this range go to the caller
  const int64_t n_runs = (int64_t)h[4];
  LS_CK(s.run_lo.ensure((size_t)n_runs * 16 + 16));
  if (nr > 0) s1_runs_kernel<<<grid_for(ctx, nr, 256), 256, 0, st>>>(a.rows, runf, runx, nr, s.run_lo.as<int64_t>());
  std::vector<int64_t> run_lo((size_t)n_runs * 2);
  if (n_runs) LS_CK(cudaMemcpyAsync(run_lo.data(), s.run_lo.p, (size_t)n_runs * 16, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  std::unordered_map<std::string, int32_t> ids;
  for (size_t i = 0; i < s.contig_names.size(); ++i) ids.emplace(s.contig_names[i], (int32_t)i);
  std::vector<int32_t> run_ctg((size_t)n_runs);
  std::vector<std::string> fresh;
  int64_t need = 0;
  for (int64_t k = 0; k < n_runs; ++k) {
    std::string name(data + run_lo[(size_t)(2 * k)], (size_t)run_lo[(size_t)(2 * k + 1)]);
    auto it = ids.find(name);
    if (it == ids.end()) {
      it = ids.emplace(name, (int32_t)(s.contig_names.size() + fresh.size())).first;
      need += (int64_t)name.size() + 1;
      fresh.push_back(name);
    }
    run_ctg[(size_t)k] = it->second;
  }
  if (need > names_cap) LS_FAIL(LS_E_CAPACITY, "ls_step1_load: the new contig names do not fit names_cap");
  *first_new = (int32_t)s.contig_names.size();
  *n_new = (int32_t)fresh.size();
  char *o = new_names;
  for (const std::string &x : fresh) {
    memcpy(o, x.c_str(), x.size() + 1);
    o += x.size() + 1;
    s.contig_names.push_back(x);
    s.contigs.push_back(nullptr);
    s.contig_len.push_back(-1);
  }
  LS_CK(upload(s.run_ctg, run_ctg.data(), n_runs, st));
  // queries
  s.n_q1 = (int64_t)h[2];
  s.n_q2 = (int64_t)h[3];
  LS_CK(s.q.ensure((size_t)(s.n_q1 + s.n_q2) * 8 + 16));
  int32_t *k1 = s.q.as<int32_t>(), *n1 = k1 + s.n_q1, *k2 = n1 + s.n_q1, *n2 = k2 + s.n_q2;
  if (nr > 0)
    s1_query_kernel<<<grid_for(ctx, nr, 256), 256, 0, st>>>(a.rows, a.calls, n_ct, nr, q1c, q2c, runf, runx,
                                                            s.run_ctg.as<int32_t>(), k1, n1, k2, n2);
  LS_CK(cudaGetLastError());
  LS_CK(cudaStreamSynchronize(st));
  s.len = len;
  s.n_rows = nr;
  s.n_ct = n_ct;
  s.min_cov = in->min_cov;
  s.min_cells = in->min_cells;
  s.min_ac_cells = in->min_ac_cells;
  s.min_ac_reads = in->min_ac_reads;
  s.min_cell_types = in->min_cell_types;
  s.max_cell_types = in->max_cell_types;
  s.alpha1 = in->alpha1;
  s.beta1 = in->beta1;
  s.alpha2 = in->alpha2;
  s.beta2 = in->beta2;
  s.loaded = true;
  *n_rows = nr;
  *n_queries = s.n_q1 + s.n_q2;
  return LS_OK;
}

extern "C" int ls_step1_contig(ls_ctx *ctx, int32_t id, const uint8_t *seq, int64_t len) {
  if (!ctx) return LS_E_ARG;
  Step1State &s = ctx->s1;
  if (id < 0 || id >= (int32_t)s.contigs.size()) LS_FAIL(LS_E_ARG, "ls_step1_contig: no load has named this contig id");
  if (len < 0 || (len > 0 && !seq)) LS_FAIL(LS_E_ARG, "ls_step1_contig: bad sequence");
  LS_CK(cudaSetDevice(ctx->device));
  if (!s.contigs[(size_t)id]) s.contigs[(size_t)id] = new DBuf();
  LS_CK(upload(*s.contigs[(size_t)id], seq, len, ctx->stream));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  s.contig_len[(size_t)id] = len;
  return LS_OK;
}

extern "C" int ls_step1_call(ls_ctx *ctx, int64_t *bytes, int64_t *longest_row) {
  if (!ctx) return LS_E_ARG;
  Step1State &s = ctx->s1;
  if (!s.loaded) LS_FAIL(LS_E_STATE, "ls_step1_call: nothing loaded");
  if (!bytes || !longest_row) LS_FAIL(LS_E_ARG, "ls_step1_call: null argument");
  s.called = false;
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t n1 = s.n_q1, n2 = s.n_q2, nr = s.n_rows;
  int32_t *k1 = s.q.as<int32_t>(), *q1n = k1 + n1, *k2 = q1n + n1, *q2n = k2 + n2;
  LS_CK(s.p.ensure((size_t)(n1 + n2) * 8 + 16));
  double *p1 = s.p.as<double>(), *p2 = p1 + n1;
  uint64_t *res = s.result.as<uint64_t>();
  uint32_t *nbig = reinterpret_cast<uint32_t *>(res + 6);
  LS_CK(cudaMemsetAsync(res + 5, 0, 24, st));
  int rc = ls_betabinom_device(ctx, k1, q1n, s.alpha1, s.beta1, p1, n1, nbig);
  if (rc != LS_OK) return rc;
  rc = ls_betabinom_device(ctx, k2, q2n, s.alpha2, s.beta2, p2, n2, nbig + 2);
  if (rc != LS_OK) return rc;
  uint32_t hb[4];
  LS_CK(cudaMemcpyAsync(hb, nbig, sizeof hb, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (hb[0] && (rc = long_tails(ctx, k1, q1n, p1, n1, s.alpha1, s.beta1)) != LS_OK) return rc;
  if (hb[2] && (rc = long_tails(ctx, k2, q2n, p2, n2, s.alpha2, s.beta2)) != LS_OK) return rc;
  if (n1) s1_round_kernel<<<grid_for(ctx, n1, 256), 256, 0, st>>>(k1, q1n, p1, n1);
  if (n2) s1_round_kernel<<<grid_for(ctx, n2, 256), 256, 0, st>>>(k2, q2n, p2, n2);
  // the resident contigs
  const size_t nc = s.contigs.size();
  std::vector<uint64_t> ptr(nc, 0);
  for (size_t i = 0; i < nc; ++i)
    if (s.contigs[i]) ptr[i] = (uint64_t)(uintptr_t)s.contigs[i]->p;
  LS_CK(upload(s.ctg_ptr, ptr.data(), (int64_t)nc, st));
  LS_CK(upload(s.ctg_len, s.contig_len.data(), (int64_t)nc, st));
  // row lengths and their offsets
  LS_CK(s.lens.ensure((size_t)nr * 4 + 16));
  LS_CK(s.off.ensure((size_t)(nr + 1) * 8 + 16));
  const S1View v = make_view(s);
  if (nr > 0) s1_len_kernel<<<grid_for(ctx, nr, 256), 256, 0, st>>>(v, nr, s.lens.as<uint32_t>(), ull(res + 5));
  LS_CK(cudaGetLastError());
  LS_CK(ls_scan_exclusive_u32_wide(s.lens.as<uint32_t>(), s.off.as<uint64_t>(), nr, ctx->scan_tmp, st));
  s.h_off.assign((size_t)nr + 1, 0);
  uint64_t bad = 0;
  LS_CK(cudaMemcpyAsync(s.h_off.data(), s.off.p, (size_t)(nr + 1) * 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(&bad, res + 5, 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (bad & B_NAN) LS_FAIL(LS_E_ARG, "ls_step1_call: a NaN among a call's per-allele tails");
  if (bad & B_ROUND) LS_FAIL(LS_E_ARG, "ls_step1_call: a tail outside the four-decimal formatting");
  int64_t longest = 0;
  for (int64_t r = 0; r < nr; ++r) longest = std::max(longest, s.h_off[(size_t)r + 1] - s.h_off[(size_t)r]);
  *bytes = s.h_off[(size_t)nr];
  *longest_row = longest;
  s.called = true;
  return LS_OK;
}

extern "C" int ls_step1_text(ls_ctx *ctx, int64_t row_lo, char *out, int64_t capacity, int64_t *rows_done,
                             int64_t *bytes) {
  if (!ctx) return LS_E_ARG;
  Step1State &s = ctx->s1;
  if (!s.called) LS_FAIL(LS_E_STATE, "ls_step1_text: no call since the last load");
  if (!out || !rows_done || !bytes || capacity < 0 || row_lo < 0 || row_lo > s.n_rows)
    LS_FAIL(LS_E_ARG, "ls_step1_text: bad argument");
  *rows_done = 0;
  *bytes = 0;
  if (row_lo == s.n_rows) return LS_OK;
  const std::vector<int64_t> &off = s.h_off;
  int64_t hi = s.n_rows;  // rows row_lo .. hi - 1 fit
  if (off[(size_t)s.n_rows] - off[(size_t)row_lo] > capacity)
    hi = (int64_t)(std::upper_bound(off.begin() + row_lo, off.end(), off[(size_t)row_lo] + capacity) - off.begin()) - 1;
  if (hi == row_lo) LS_FAIL(LS_E_CAPACITY, "ls_step1_text: a row is longer than the capacity");
  const int64_t nb = off[(size_t)hi] - off[(size_t)row_lo];
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(s.out.ensure((size_t)nb + 16));
  s1_write_kernel<<<grid_for(ctx, hi - row_lo, S1_THREADS), S1_THREADS, 0, st>>>(make_view(s), row_lo, hi,
                                                                                 s.out.as<char>());
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(out, s.out.p, (size_t)nb, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  *rows_done = hi - row_lo;
  *bytes = nb;
  return LS_OK;
}

extern "C" int ls_step1_release(ls_ctx *ctx) {
  if (!ctx) return LS_E_ARG;
  LS_CK(cudaSetDevice(ctx->device));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  ctx->s1.release();
  return LS_OK;
}
