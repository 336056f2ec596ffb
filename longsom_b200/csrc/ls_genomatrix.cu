// Genotype matrices (DpMatrix, AltMatrix, VAFMatrix, BinaryMatrix of SingleCellGenotype) written as text on the
// device, straight from the touched (site, cell) pairs: the reference pivots its long table four times in pandas
// (SingleCellGenotype.py:351-379), which holds n_sites x n_cells rows in host memory.
//
// A matrix row is its label, then one "\t entry" per column, then "\n".  Almost every entry is untouched and has a
// fixed text, so a row's length is a fixed part plus one correction per touched pair (length pass); the rows are
// placed by an exclusive scan of those lengths, and as many whole rows as fit the caller's block are written
// (write pass): one CTA per row, column tiles formatted into shared memory at offsets from a block scan, then
// stored to the block with 16-byte stores.
#include "ls_common.cuh"
#include "ls_text.cuh"

namespace {

constexpr int GM_THREADS = 256;
constexpr int GM_COLS_PER_THREAD = 4;
constexpr int GM_TILE = GM_THREADS * GM_COLS_PER_THREAD;
constexpr int GM_ENTRY_MAX = 13;  // tab + "2147483647.0"

__device__ __forceinline__ int put_num(uint32_t v, bool as_float, char *o) {
  int n = put_uint(v, o);
  if (as_float) {
    if (o) o[n] = '.', o[n + 1] = '0';
    n += 2;
  }
  return n;
}

__device__ __forceinline__ int default_len(int kind, int float_mode) {
  return (kind == LS_GENO_MATRIX_VAF || !float_mode) ? 1 : 3;
}

__device__ __forceinline__ int put_default(int kind, int float_mode, char *o) {
  if (o) o[0] = kind == LS_GENO_MATRIX_VAF ? '.' : (kind == LS_GENO_MATRIX_BINARY ? '3' : '0');
  if (kind != LS_GENO_MATRIX_VAF && float_mode) {
    if (o) o[1] = '.', o[2] = '0';
    return 3;
  }
  return 1;
}

// text of a pair's entry (without its tab); o may be null (length only)
__device__ __forceinline__ int put_pair(int kind, int float_mode, uint32_t rflags, int32_t dp, int32_t alt, double p,
                                        double pvalue, char *o) {
  if (rflags & LS_GENO_ROW_FUSION) {
    if (o) o[0] = '1';
    if (kind == LS_GENO_MATRIX_VAF || !float_mode) return 1;
    if (o) o[1] = '.', o[2] = '0';
    return 3;
  }
  switch (kind) {
    case LS_GENO_MATRIX_DP: return put_num((uint32_t)dp, float_mode, o);
    case LS_GENO_MATRIX_ALT: return put_num((uint32_t)alt, float_mode, o);
    case LS_GENO_MATRIX_VAF:
      if (dp == 0) {
        if (o) o[0] = '.';
        return 1;
      }
      return put_units4(vaf_units(alt, dp), o);
    default: {
      uint32_t bin;
      if (dp == 0)
        bin = 3u;
      else if (alt == 0)
        bin = 0u;
      else if (rflags & LS_GENO_ROW_CHRM)
        bin = vaf_units(alt, dp) >= 3000u ? 1u : 0u;  // the double nearest k / 1e4 is >= 0.3 iff k >= 3000
      else
        bin = p < pvalue ? 1u : 0u;
      return put_num(bin, float_mode, o);
    }
  }
}

// ---- load ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gm_keys_kernel(const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                                                      int64_t n, int64_t n_rows, int32_t n_cols, int col_bits,
                                                      uint64_t *__restrict__ keys, uint32_t *__restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t r = row[i], c = col[i];
  if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) {
    atomicOr(bad, 1u);
    return;
  }
  keys[i] = ((uint64_t)r << col_bits) | (uint64_t)c;
}

__global__ void __launch_bounds__(256) gm_gather_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ src,
                                                        int64_t n, int col_bits, const int32_t *__restrict__ in_dp,
                                                        const int32_t *__restrict__ in_alt, const double *__restrict__ in_p,
                                                        int32_t *__restrict__ col, int32_t *__restrict__ dp,
                                                        int32_t *__restrict__ alt, double *__restrict__ p,
                                                        uint32_t *__restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t k = keys[i];
  if (i > 0 && keys[i - 1] == k) atomicOr(bad, 2u);
  const uint32_t s = src[i];
  col[i] = (int32_t)(k & (((uint64_t)1 << col_bits) - 1u));
  dp[i] = in_dp[s];
  alt[i] = in_alt[s];
  p[i] = in_p[s];
}

// row_start[r] = first sorted pair of row r (lower bound of r << col_bits), r = 0 .. n_rows
__global__ void __launch_bounds__(256) gm_row_start_kernel(const uint64_t *__restrict__ keys, int64_t n, int64_t n_rows,
                                                           int col_bits, int64_t *__restrict__ row_start) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  const uint64_t want = (uint64_t)r << col_bits;
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (keys[mid] < want)
      lo = mid + 1;
    else
      hi = mid;
  }
  row_start[r] = lo;
}

// ---- length pass -----------------------------------------------------------------------------
struct GmView {
  const int32_t *col, *dp, *alt;
  const double *p;
  const int64_t *row_start, *label_off;
  const char *labels;
  const uint8_t *row_flags, *col_absent;
  int32_t n_cols, n_present, float_mode;
  double pvalue;
};

// one warp per row: lens[i] = length of row row_lo + i, clamped to 2^32 - 1
__global__ void __launch_bounds__(256) gm_length_kernel(GmView v, int kind, int64_t row_lo, int64_t m,
                                                        uint32_t *__restrict__ lens) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= m) return;
  const int64_t r = row_lo + i;
  const uint32_t fl = v.row_flags[r];
  const bool fusion = fl & LS_GENO_ROW_FUSION;
  const int dl = default_len(kind, v.float_mode);
  int64_t corr = 0;
  for (int64_t j = v.row_start[r] + lane; j < v.row_start[r + 1]; j += 32) {
    const int c = v.col[j];
    const int base = (fusion || (v.col_absent && v.col_absent[c])) ? 0 : dl;
    corr += put_pair(kind, v.float_mode, fl, v.dp[j], v.alt[j], v.p[j], v.pvalue, nullptr) - base;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) corr += __shfl_xor_sync(0xffffffffu, corr, o);
  if (lane == 0) {
    const int64_t fixed = (v.label_off[r + 1] - v.label_off[r]) + 1 + v.n_cols + (fusion ? 0 : (int64_t)v.n_present * dl);
    const int64_t len = fixed + corr;
    lens[i] = len > 0xffffffffll ? 0xffffffffu : (uint32_t)len;
  }
}

// res[0] = rows that fit in cap, res[1] = their bytes.  Offsets past 4 GB wrap, but every row before the first one
// that does not fit starts below cap (< 2^32), so that row's offset and the minimum index are exact.
__global__ void __launch_bounds__(256) gm_fit_kernel(const uint32_t *__restrict__ lens, const uint32_t *__restrict__ offs,
                                                     int64_t m, uint64_t cap, unsigned long long *__restrict__ res) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m && (uint64_t)offs[i] + lens[i] > cap) atomicMin(res, (unsigned long long)i);
}

__global__ void gm_fit_bytes_kernel(const uint32_t *__restrict__ lens, const uint32_t *__restrict__ offs,
                                    unsigned long long *__restrict__ res) {
  const unsigned long long k = res[0];
  res[1] = k == 0 ? 0ull : (unsigned long long)offs[k - 1] + lens[k - 1];
}

// ---- write pass ------------------------------------------------------------------------------
// one CTA per row of the block
__global__ void __launch_bounds__(GM_THREADS) gm_write_kernel(GmView v, int kind, int64_t row_lo,
                                                              const uint32_t *__restrict__ offs, char *__restrict__ out) {
  __shared__ int32_t tile_pair[GM_TILE];
  __shared__ char text[GM_TILE * GM_ENTRY_MAX + 16];
  __shared__ uint32_t sm[GM_THREADS / 32 + 1];
  const int64_t r = row_lo + blockIdx.x;
  char *dst = out + offs[blockIdx.x];
  const uint32_t fl = v.row_flags[r];
  const bool fusion = fl & LS_GENO_ROW_FUSION;
  const int64_t l0 = v.label_off[r];
  const uint32_t ll = (uint32_t)(v.label_off[r + 1] - l0);
  for (uint32_t k = threadIdx.x; k < ll; k += GM_THREADS) dst[k] = v.labels[l0 + k];
  dst += ll;
  int64_t cursor = v.row_start[r];
  const int64_t pend = v.row_start[r + 1];
  for (int32_t c0 = 0; c0 < v.n_cols; c0 += GM_TILE) {
    for (int k = threadIdx.x; k < GM_TILE; k += GM_THREADS) tile_pair[k] = -1;
    __syncthreads();
    // the row's pairs are sorted by column: this tile's pairs are the next ones, at most GM_TILE of them
    int taken = 0;
    for (int k = 0; k < GM_TILE; k += GM_THREADS) {
      const int64_t j = cursor + k + threadIdx.x;
      const bool in = j < pend && v.col[j] < c0 + GM_TILE;
      if (in) tile_pair[v.col[j] - c0] = (int32_t)(j - v.row_start[r]);
      taken += __syncthreads_count(in);
    }
    const int64_t pbase = v.row_start[r];
    cursor += taken;
    uint32_t len = 0;
    const int cb = threadIdx.x * GM_COLS_PER_THREAD;
#pragma unroll
    for (int q = 0; q < GM_COLS_PER_THREAD; ++q) {
      const int32_t c = c0 + cb + q;
      if (c >= v.n_cols) break;
      const int32_t tp = tile_pair[cb + q];
      if (tp >= 0) {
        const int64_t j = pbase + tp;
        len += 1 + put_pair(kind, v.float_mode, fl, v.dp[j], v.alt[j], v.p[j], v.pvalue, nullptr);
      } else {
        len += 1 + ((fusion || (v.col_absent && v.col_absent[c])) ? 0 : default_len(kind, v.float_mode));
      }
    }
    uint32_t total;
    uint32_t o = block_excl_scan<GM_THREADS>(len, &total, sm);
#pragma unroll
    for (int q = 0; q < GM_COLS_PER_THREAD; ++q) {
      const int32_t c = c0 + cb + q;
      if (c >= v.n_cols) break;
      text[o++] = '\t';
      const int32_t tp = tile_pair[cb + q];
      if (tp >= 0) {
        const int64_t j = pbase + tp;
        o += put_pair(kind, v.float_mode, fl, v.dp[j], v.alt[j], v.p[j], v.pvalue, text + o);
      } else if (!(fusion || (v.col_absent && v.col_absent[c]))) {
        o += put_default(kind, v.float_mode, text + o);
      }
    }
    __syncthreads();
    copy_out<GM_THREADS>(dst, text, total);
    dst += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) *dst = '\n';
}

}  // namespace

extern "C" int ls_geno_matrix_load(ls_ctx *ctx, const ls_geno_matrix_in *in) {
  if (!ctx) return LS_E_ARG;
  GenoMatrixState &g = ctx->gm;
  g.loaded = false;
  if (!in) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: input is null");
  const int64_t n = in->n_pairs, nr = in->n_rows;
  const int32_t nc = in->n_cols;
  if (n < 0 || nr < 0 || nc < 0) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: negative size");
  if (n >= (int64_t)0xffffffffll) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: more than 2^32-1 pairs");
  if (nr >= ((int64_t)1 << 31)) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: more than 2^31-1 rows");
  if (n > 0 && (!in->row || !in->col || !in->dp || !in->alt || !in->p))
    LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: null pair array");
  if (!in->label_off || (nr > 0 && !in->row_flags)) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: null row array");
  for (int64_t r = 0; r < nr; ++r)
    if (in->label_off[r + 1] < in->label_off[r]) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: label_off not ascending");
  const int64_t nl = in->label_off[nr] - in->label_off[0];
  if (nl > 0 && !in->labels) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: null labels");
  int32_t present = nc;
  if (in->col_absent)
    for (int32_t c = 0; c < nc; ++c) present -= in->col_absent[c] ? 1 : 0;

  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int col_bits = ls_bits_for(nc > 0 ? (uint64_t)(nc - 1) : 0u);
  const int key_bits = col_bits + ls_bits_for(nr > 0 ? (uint64_t)(nr - 1) : 0u);
  LS_CK(g.keys_a.ensure((size_t)n * 8 + 16));
  LS_CK(g.keys_b.ensure((size_t)n * 8 + 16));
  LS_CK(g.vals_a.ensure((size_t)n * 4 + 16));
  LS_CK(g.vals_b.ensure((size_t)n * 4 + 16));
  LS_CK(g.in_dp.ensure((size_t)n * 4 + 16));
  LS_CK(g.in_alt.ensure((size_t)n * 4 + 16));
  LS_CK(g.in_p.ensure((size_t)n * 8 + 16));
  LS_CK(g.col.ensure((size_t)n * 4 + 16));
  LS_CK(g.dp.ensure((size_t)n * 4 + 16));
  LS_CK(g.alt.ensure((size_t)n * 4 + 16));
  LS_CK(g.p.ensure((size_t)n * 8 + 16));
  LS_CK(g.row_start.ensure((size_t)(nr + 1) * 8));
  LS_CK(g.labels.ensure((size_t)nl + 16));
  LS_CK(g.label_off.ensure((size_t)(nr + 1) * 8));
  LS_CK(g.row_flags.ensure((size_t)nr + 16));
  LS_CK(g.col_absent.ensure((size_t)nc + 16));
  LS_CK(g.result.ensure(16));
  // the caller's row and col go through the sort's second buffers, which the sort overwrites afterwards
  int32_t *d_row = g.vals_b.as<int32_t>(), *d_col = reinterpret_cast<int32_t *>(g.keys_b.as<uint64_t>());
  if (n) {
    LS_CK(cudaMemcpyAsync(d_row, in->row, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(d_col, in->col, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(g.in_dp.p, in->dp, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(g.in_alt.p, in->alt, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(g.in_p.p, in->p, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  }
  if (nl) LS_CK(cudaMemcpyAsync(g.labels.p, in->labels + in->label_off[0], (size_t)nl, cudaMemcpyHostToDevice, st));
  {
    std::vector<int64_t> lo(in->label_off, in->label_off + nr + 1);
    for (auto &x : lo) x -= in->label_off[0];
    LS_CK(cudaMemcpyAsync(g.label_off.p, lo.data(), (size_t)(nr + 1) * 8, cudaMemcpyHostToDevice, st));
    if (nr) LS_CK(cudaMemcpyAsync(g.row_flags.p, in->row_flags, (size_t)nr, cudaMemcpyHostToDevice, st));
    if (nc && in->col_absent) LS_CK(cudaMemcpyAsync(g.col_absent.p, in->col_absent, (size_t)nc, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemsetAsync(g.result.p, 0, 16, st));
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (n) gm_keys_kernel<<<blocks, 256, 0, st>>>(d_row, d_col, n, nr, nc, col_bits, g.keys_a.as<uint64_t>(),
                                                   g.result.as<uint32_t>());
    LS_CK(cudaGetLastError());
    uint64_t *sk = nullptr;
    uint32_t *sv = nullptr;
    LS_CK(ls_radix_sort_pairs(g.keys_a.as<uint64_t>(), g.keys_b.as<uint64_t>(), g.vals_a.as<uint32_t>(),
                              g.vals_b.as<uint32_t>(), n, key_bits, ctx->rs_hist, &sk, &sv, ctx->num_sms, st, nullptr));
    if (n) gm_gather_kernel<<<blocks, 256, 0, st>>>(sk, sv, n, col_bits, g.in_dp.as<int32_t>(), g.in_alt.as<int32_t>(),
                                                     g.in_p.as<double>(), g.col.as<int32_t>(), g.dp.as<int32_t>(),
                                                     g.alt.as<int32_t>(), g.p.as<double>(), g.result.as<uint32_t>());
    gm_row_start_kernel<<<(unsigned)((nr + 1 + 255) / 256), 256, 0, st>>>(sk, n, nr, col_bits, g.row_start.as<int64_t>());
    LS_CK(cudaGetLastError());
    uint32_t bad = 0;
    LS_CK(cudaMemcpyAsync(&bad, g.result.p, 4, cudaMemcpyDeviceToHost, st));
    LS_CK(cudaStreamSynchronize(st));  // also the copy of `lo`
    if (bad & 1u) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: a pair's row or column is out of range");
    if (bad & 2u) LS_FAIL(LS_E_ARG, "ls_geno_matrix_load: duplicate (row, col) pair");
  }
  g.n_rows = nr;
  g.n_pairs = n;
  g.n_cols = nc;
  g.n_present = present;
  g.float_mode = in->float_mode ? 1 : 0;
  g.pvalue = in->pvalue;
  g.loaded = true;
  return LS_OK;
}

extern "C" int ls_geno_matrix_text(ls_ctx *ctx, int kind, int64_t row_lo, char *out, int64_t capacity,
                                   int64_t *rows_done, int64_t *bytes) {
  if (!ctx) return LS_E_ARG;
  GenoMatrixState &g = ctx->gm;
  if (!g.loaded) LS_FAIL(LS_E_STATE, "ls_geno_matrix_text: no pairs loaded");
  if (kind < LS_GENO_MATRIX_DP || kind > LS_GENO_MATRIX_BINARY) LS_FAIL(LS_E_ARG, "ls_geno_matrix_text: bad kind");
  if (!out || !rows_done || !bytes || capacity < 0 || row_lo < 0 || row_lo > g.n_rows)
    LS_FAIL(LS_E_ARG, "ls_geno_matrix_text: bad argument");
  *rows_done = 0;
  *bytes = 0;
  const int64_t m = g.n_rows - row_lo;
  if (m == 0) return LS_OK;
  const uint64_t cap = (uint64_t)(capacity < ((int64_t)1 << 31) ? capacity : ((int64_t)1 << 31));
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(g.lens.ensure((size_t)m * 4 + 16));
  LS_CK(g.offs.ensure((size_t)m * 4 + 16));
  GmView v;
  v.col = g.col.as<int32_t>();
  v.dp = g.dp.as<int32_t>();
  v.alt = g.alt.as<int32_t>();
  v.p = g.p.as<double>();
  v.row_start = g.row_start.as<int64_t>();
  v.label_off = g.label_off.as<int64_t>();
  v.labels = g.labels.as<char>();
  v.row_flags = g.row_flags.as<uint8_t>();
  v.col_absent = g.col_absent.as<uint8_t>();
  v.n_cols = g.n_cols;
  v.n_present = g.n_present;
  v.float_mode = g.float_mode;
  v.pvalue = g.pvalue;
  if (g.n_present == g.n_cols) v.col_absent = nullptr;
  gm_length_kernel<<<(unsigned)((m * 32 + 255) / 256), 256, 0, st>>>(v, kind, row_lo, m, g.lens.as<uint32_t>());
  LS_CK(cudaGetLastError());
  LS_CK(ls_scan_exclusive_u32(g.lens.as<uint32_t>(), g.offs.as<uint32_t>(), m, nullptr, ctx->scan_tmp, st));
  unsigned long long res[2] = {(unsigned long long)m, 0ull};
  LS_CK(cudaMemcpyAsync(g.result.p, res, 8, cudaMemcpyHostToDevice, st));
  gm_fit_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(g.lens.as<uint32_t>(), g.offs.as<uint32_t>(), m, cap,
                                                            g.result.as<unsigned long long>());
  gm_fit_bytes_kernel<<<1, 1, 0, st>>>(g.lens.as<uint32_t>(), g.offs.as<uint32_t>(), g.result.as<unsigned long long>());
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(res, g.result.p, 16, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (res[0] == 0) LS_FAIL(LS_E_CAPACITY, "ls_geno_matrix_text: a row is longer than the capacity");
  const int64_t rows = (int64_t)res[0], nb = (int64_t)res[1];
  LS_CK(g.out.ensure((size_t)nb + 16));
  gm_write_kernel<<<(unsigned)rows, GM_THREADS, 0, st>>>(v, kind, row_lo, g.offs.as<uint32_t>(), g.out.as<char>());
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(out, g.out.p, (size_t)nb, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  *rows_done = rows;
  *bytes = nb;
  return LS_OK;
}
