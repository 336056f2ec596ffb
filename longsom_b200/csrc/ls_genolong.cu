// The dense long table of SingleCellGenotype / HCCVSingleCellGenotype (<prefix>.SingleCellGenotype.tsv, HCCV's
// --outfile) written as text on the device from the touched (site, cell) pairs.  The text is that of the host writer
// ls_geno_rows (csrc/host/ls_genorows.cpp): one row per (output site, metadata cell), almost all "NoCoverage".  The
// load refuses two kinds of pair that ls_geno_rows would print, alt outside [0, dp] and |p| >= 4e5 (inf included), so
// that every number fits the 32-bit digit formatting; the genotype CLIs never produce them.
//
// A row is the site's fixed part (prefix, index and the constant characters), the cell's text, and a tail (Dp .. the
// MutationStatus) that is 18 bytes for an untouched cell.  So the load step scans, per site, the tail lengths of its
// pairs once, and a site's length and a row's offset inside it follow without looking at the other rows:
//   site length  = n_cells * F_s + sum(cell_len) + 18 * (n_cells - m_s) + tail_cum_s[m_s]
//   row offset   = c * F_s + cell_cum[c] + 18 * (c - k) + tail_cum_s[k],  k = the site's pairs with cell < c
// A text call then places as many whole sites as fit the caller's block from the host copy of the site offsets, and
// writes their rows one warp per row, the lanes storing consecutive bytes.
#include <algorithm>

#include "ls_common.cuh"
#include "ls_text.cuh"

namespace {

constexpr int GL_THREADS = 256;
constexpr int GL_WARPS = GL_THREADS / 32;
constexpr int GL_UNTOUCHED_TAIL = 18;  // "0\t0\t.\t.\tNoCoverage"
constexpr int GL_CHUNK = 96;           // '\t' + the longest tail + "\t3\t"
constexpr double GL_P_MAX = 4.0e5;     // |p| * 1e4 must fit the 32-bit units of put_units4

// text at o (o null: length only)
struct TextOut {
  char *o;
  int n;
  __device__ void ch(char x) {
    if (o) o[n] = x;
    ++n;
  }
  __device__ void str(const char *x) {
    while (*x) ch(*x++);
  }
  __device__ void num(uint32_t v) { n += put_uint(v, o ? o + n : nullptr); }
  __device__ void units4(uint32_t k) { n += put_units4(k, o ? o + n : nullptr); }
};

// The columns Dp, ALT, VAF, BetaBin and MutationStatus of one row, tab-joined; returns the BinMutationStatus digit.
// 0 <= alt <= dp (checked at load); p is NaN or rounded to four places with |p| < GL_P_MAX (checked at load).
__device__ __forceinline__ char put_tail(TextOut &t, int32_t dp, int32_t alt, double p, bool chrm, double pvalue) {
  t.num((uint32_t)dp);
  t.ch('\t');
  t.num((uint32_t)alt);
  t.ch('\t');
  if (dp == 0) {
    t.str(".\t.\tNoCoverage");
    return '3';
  }
  const uint32_t k = vaf_units(alt, dp);
  t.units4(k);  // alt = 0 gives "0.0", as both scripts print it
  t.ch('\t');
  if (alt == 0) {
    t.str(".\tNoAltReads");
    return '0';
  }
  bool pass;
  if (chrm) {
    t.ch('.');
    pass = k >= 3000u;  // the double nearest k / 1e4 is >= 0.3 iff k >= 3000
    t.ch('\t');
    t.str(pass ? "PASS" : "LowVAFChrM");
  } else {
    if (isnan(p)) {
      t.str("nan");
    } else {
      if (p < 0.0) t.ch('-');
      t.units4((uint32_t)rint(fabs(p) * 10000.0));
    }
    pass = p < pvalue;
    t.ch('\t');
    t.str(pass ? "PASS" : "BetaBin_problem");
  }
  return pass ? '1' : '0';
}

struct GlView {
  const int32_t *cell, *dp, *alt;
  const double *p;
  const int64_t *hit_lo, *hit_hi, *tail_base, *tail_cum, *site_off;
  const uint8_t *flags;
  const char *prefix, *index, *cell_text;
  const int64_t *prefix_off, *index_off, *cell_off;
  int32_t n_cells, hccv;
  double pvalue;
};

// the bytes of a site's row other than the cell's text and the tail
__device__ __forceinline__ int64_t fixed_len(const GlView &v, int64_t s) {
  const int64_t pl = v.prefix_off[s + 1] - v.prefix_off[s];
  return pl + 3 + (v.hccv ? 0 : 3 + (v.index_off[s + 1] - v.index_off[s]));
}

// ---- load: one CTA per site ---------------------------------------------------------------------
// checks the site's pairs (bad: 1 cell out of range, 2 cells not strictly increasing, 4 alt outside [0, dp], 8 p
// neither NaN nor below GL_P_MAX in magnitude), scans their tail lengths into tail_cum[tail_base[s] ..], m_s + 1
// values, and writes the site's length
__global__ void __launch_bounds__(GL_THREADS) gl_site_kernel(GlView v, int64_t n_sites, int64_t *__restrict__ tail_cum,
                                                             int64_t *__restrict__ site_len, uint32_t *__restrict__ bad) {
  __shared__ uint32_t sm[GL_WARPS + 1];
  for (int64_t s = blockIdx.x; s < n_sites; s += gridDim.x) {
    const int64_t lo = v.hit_lo[s], hi = v.hit_hi[s], base = v.tail_base[s];
    const bool chrm = v.flags[s] & LS_GENO_ROW_CHRM;
    int64_t carry = 0;
    for (int64_t j0 = lo; j0 < hi; j0 += GL_THREADS) {
      const int64_t j = j0 + threadIdx.x;
      uint32_t len = 0;
      if (j < hi) {
        const int32_t c = v.cell[j], dp = v.dp[j], alt = v.alt[j];
        const double p = v.p[j];
        uint32_t b = 0;
        if (c < 0 || c >= v.n_cells) b |= 1u;
        if (j > lo && v.cell[j - 1] >= c) b |= 2u;
        if (alt < 0 || alt > dp) b |= 4u;
        if (!isnan(p) && !(fabs(p) < GL_P_MAX)) b |= 8u;
        if (b) atomicOr(bad, b);
        TextOut t{nullptr, 0};
        if (!(b & 4u)) put_tail(t, dp, alt, p, chrm, v.pvalue);
        len = (uint32_t)t.n;
      }
      uint32_t total;
      const uint32_t ex = block_excl_scan<GL_THREADS>(len, &total, sm);
      if (j < hi) tail_cum[base + (j - lo)] = carry + ex;
      carry += total;
    }
    if (threadIdx.x == 0) {
      const int64_t m = hi - lo, nc = v.n_cells;
      tail_cum[base + m] = carry;
      const int64_t cells = v.cell_off[nc] - v.cell_off[0];
      site_len[s] = nc * fixed_len(v, s) + cells + GL_UNTOUCHED_TAIL * (nc - m) + carry;
    }
  }
}

// ---- text: one warp per row ---------------------------------------------------------------------
__device__ __forceinline__ void warp_copy(char *dst, const char *src, int64_t n, int lane) {
  for (int64_t i = lane; i < n; i += 32) dst[i] = src[i];
}

__global__ void __launch_bounds__(GL_THREADS) gl_write_kernel(GlView v, int64_t site_lo, int64_t n_rows,
                                                              char *__restrict__ out) {
  __shared__ char chunk[GL_WARPS][GL_CHUNK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t base = v.site_off[site_lo];
  for (int64_t r = (int64_t)blockIdx.x * GL_WARPS + w; r < n_rows; r += (int64_t)gridDim.x * GL_WARPS) {
    const int64_t s = site_lo + r / v.n_cells;
    const int32_t c = (int32_t)(r % v.n_cells);
    const int64_t lo = v.hit_lo[s], hi = v.hit_hi[s];
    int64_t a = lo, b = hi;  // the first of the site's pairs with cell >= c
    while (a < b) {
      const int64_t mid = (a + b) >> 1;
      if (v.cell[mid] < c)
        a = mid + 1;
      else
        b = mid;
    }
    const int64_t k = a - lo;
    const bool touched = a < hi && v.cell[a] == c;
    const int64_t fl = fixed_len(v, s);
    const int64_t c0 = v.cell_off[c] - v.cell_off[0], cl = v.cell_off[c + 1] - v.cell_off[c];
    char *dst = out + (v.site_off[s] - base) + c * fl + c0 + GL_UNTOUCHED_TAIL * (c - k) + v.tail_cum[v.tail_base[s] + k];
    __syncwarp();
    int n_chunk = 0;
    if (lane == 0) {
      TextOut t{chunk[w], 0};
      t.ch('\t');
      const char bin = touched ? put_tail(t, v.dp[a], v.alt[a], v.p[a], v.flags[s] & LS_GENO_ROW_CHRM, v.pvalue)
                               : put_tail(t, 0, 0, 0.0, false, v.pvalue);
      if (v.hccv) {
        t.ch('\n');
      } else {
        t.ch('\t');
        t.ch(bin);
        t.ch('\t');
      }
      n_chunk = t.n;
    }
    n_chunk = __shfl_sync(0xffffffffu, n_chunk, 0);
    __syncwarp();
    const int64_t p0 = v.prefix_off[s], pl = v.prefix_off[s + 1] - p0;
    warp_copy(dst, v.prefix + p0, pl, lane);
    dst += pl;
    if (lane == 0) dst[0] = '\t';
    warp_copy(dst + 1, v.cell_text + c0, cl, lane);
    dst += 1 + cl;
    warp_copy(dst, chunk[w], n_chunk, lane);
    dst += n_chunk;
    if (!v.hccv) {
      const int64_t i0 = v.index_off[s], il = v.index_off[s + 1] - i0;
      warp_copy(dst, v.index + i0, il, lane);
      if (lane == 0) dst[il] = '\n';
    }
  }
}

template <typename T>
cudaError_t upload(DBuf &d, const T *h, int64_t n, cudaStream_t st) {
  cudaError_t e = d.ensure((size_t)n * sizeof(T) + 16);
  if (e == cudaSuccess && n > 0) e = cudaMemcpyAsync(d.p, h, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st);
  return e;
}

// off[0 .. n] ascending, rebased to 0 (the text at base + off[0] .. base + off[n] is uploaded with it)
bool rebase(const int64_t *off, int64_t n, std::vector<int64_t> &out) {
  out.resize((size_t)n + 1);
  for (int64_t i = 0; i <= n; ++i) {
    if (i > 0 && off[i] < off[i - 1]) return false;
    out[(size_t)i] = off[i] - off[0];
  }
  return true;
}

}  // namespace

extern "C" int ls_geno_long_load(ls_ctx *ctx, const ls_geno_long_in *in) {
  if (!ctx) return LS_E_ARG;
  GenoLongState &g = ctx->gl;
  g.loaded = false;
  if (!in) LS_FAIL(LS_E_ARG, "ls_geno_long_load: input is null");
  const int64_t ns = in->n_sites, np = in->n_pairs;
  const int32_t nc = in->n_cells;
  const bool hccv = in->hccv != 0;
  if (ns < 0 || np < 0 || nc < 0) LS_FAIL(LS_E_ARG, "ls_geno_long_load: negative size");
  if (ns >= ((int64_t)1 << 31)) LS_FAIL(LS_E_ARG, "ls_geno_long_load: more than 2^31-1 sites");
  if (np > 0 && (!in->cell || !in->dp || !in->alt || !in->p)) LS_FAIL(LS_E_ARG, "ls_geno_long_load: null pair array");
  if (ns > 0 && (!in->hit_lo || !in->hit_hi || !in->site_flags))
    LS_FAIL(LS_E_ARG, "ls_geno_long_load: null site array");
  if (!in->prefix_off || !in->cell_off || (!hccv && !in->index_off))
    LS_FAIL(LS_E_ARG, "ls_geno_long_load: null offset array");
  std::vector<int64_t> prefix_off, index_off, cell_off, tail_base((size_t)ns);
  if (!rebase(in->prefix_off, ns, prefix_off) || !rebase(in->cell_off, nc, cell_off) ||
      (!hccv && !rebase(in->index_off, ns, index_off)))
    LS_FAIL(LS_E_ARG, "ls_geno_long_load: text offsets not ascending");
  if ((prefix_off[(size_t)ns] && !in->prefix) || (cell_off[(size_t)nc] && !in->cell_text) ||
      (!hccv && index_off[(size_t)ns] && !in->index))
    LS_FAIL(LS_E_ARG, "ls_geno_long_load: null text");
  int64_t n_tail = 0;
  for (int64_t s = 0; s < ns; ++s) {
    const int64_t lo = in->hit_lo[s], hi = in->hit_hi[s];
    if (lo < 0 || lo > hi || hi > np) LS_FAIL(LS_E_ARG, "ls_geno_long_load: a site's pair range is outside [0, n_pairs]");
    tail_base[(size_t)s] = n_tail;
    n_tail += hi - lo + 1;
  }

  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(upload(g.cell, in->cell, np, st));
  LS_CK(upload(g.dp, in->dp, np, st));
  LS_CK(upload(g.alt, in->alt, np, st));
  LS_CK(upload(g.p, in->p, np, st));
  LS_CK(upload(g.hit_lo, in->hit_lo, ns, st));
  LS_CK(upload(g.hit_hi, in->hit_hi, ns, st));
  LS_CK(upload(g.flags, in->site_flags, ns, st));
  LS_CK(upload(g.tail_base, tail_base.data(), ns, st));
  LS_CK(upload(g.prefix, in->prefix + in->prefix_off[0], prefix_off[(size_t)ns], st));
  LS_CK(upload(g.prefix_off, prefix_off.data(), ns + 1, st));
  LS_CK(upload(g.cell_text, in->cell_text + in->cell_off[0], cell_off[(size_t)nc], st));
  LS_CK(upload(g.cell_off, cell_off.data(), (int64_t)nc + 1, st));
  if (!hccv) {
    LS_CK(upload(g.index, in->index + in->index_off[0], index_off[(size_t)ns], st));
    LS_CK(upload(g.index_off, index_off.data(), ns + 1, st));
  }
  LS_CK(g.tail_cum.ensure((size_t)n_tail * 8 + 16));
  LS_CK(g.site_len.ensure((size_t)ns * 8 + 16));
  LS_CK(g.site_off.ensure((size_t)(ns + 1) * 8));
  LS_CK(g.result.ensure(16));
  LS_CK(cudaMemsetAsync(g.result.p, 0, 4, st));
  GlView v = {};
  v.cell = g.cell.as<int32_t>();
  v.dp = g.dp.as<int32_t>();
  v.alt = g.alt.as<int32_t>();
  v.p = g.p.as<double>();
  v.hit_lo = g.hit_lo.as<int64_t>();
  v.hit_hi = g.hit_hi.as<int64_t>();
  v.tail_base = g.tail_base.as<int64_t>();
  v.flags = g.flags.as<uint8_t>();
  v.prefix = g.prefix.as<char>();
  v.prefix_off = g.prefix_off.as<int64_t>();
  v.cell_text = g.cell_text.as<char>();
  v.cell_off = g.cell_off.as<int64_t>();
  v.index = hccv ? nullptr : g.index.as<char>();
  v.index_off = hccv ? nullptr : g.index_off.as<int64_t>();
  v.n_cells = nc;
  v.hccv = hccv ? 1 : 0;
  v.pvalue = in->pvalue;
  if (ns) {
    const unsigned grid = (unsigned)std::min<int64_t>(ns, (int64_t)ctx->num_sms * 32);
    gl_site_kernel<<<grid, GL_THREADS, 0, st>>>(v, ns, g.tail_cum.as<int64_t>(), g.site_len.as<int64_t>(),
                                                g.result.as<uint32_t>());
    LS_CK(cudaGetLastError());
  }
  std::vector<int64_t> site_len((size_t)ns);
  uint32_t bad = 0;
  LS_CK(cudaMemcpyAsync(&bad, g.result.p, 4, cudaMemcpyDeviceToHost, st));
  if (ns) LS_CK(cudaMemcpyAsync(site_len.data(), g.site_len.p, (size_t)ns * 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (bad & 1u) LS_FAIL(LS_E_ARG, "ls_geno_long_load: a pair's cell is outside [0, n_cells)");
  if (bad & 2u) LS_FAIL(LS_E_ARG, "ls_geno_long_load: cells not strictly increasing inside a site's range");
  if (bad & 4u) LS_FAIL(LS_E_ARG, "ls_geno_long_load: a pair's alt is outside [0, dp]");
  if (bad & 8u) LS_FAIL(LS_E_ARG, "ls_geno_long_load: a p-value is neither NaN nor below 4e5 in magnitude");
  g.h_site_off.assign((size_t)ns + 1, 0);
  for (int64_t s = 0; s < ns; ++s) g.h_site_off[(size_t)s + 1] = g.h_site_off[(size_t)s] + site_len[(size_t)s];
  LS_CK(cudaMemcpyAsync(g.site_off.p, g.h_site_off.data(), (size_t)(ns + 1) * 8, cudaMemcpyHostToDevice, st));
  LS_CK(cudaStreamSynchronize(st));
  g.n_sites = ns;
  g.n_pairs = np;
  g.n_cells = nc;
  g.hccv = hccv ? 1 : 0;
  g.pvalue = in->pvalue;
  g.ms_text = g.ms_copy = 0.0;
  g.blocks = g.bytes = 0;
  g.loaded = true;
  return LS_OK;
}

extern "C" int ls_geno_long_text(ls_ctx *ctx, int64_t site_lo, char *out, int64_t capacity, int64_t *sites_done,
                                 int64_t *bytes) {
  if (!ctx) return LS_E_ARG;
  GenoLongState &g = ctx->gl;
  if (!g.loaded) LS_FAIL(LS_E_STATE, "ls_geno_long_text: nothing loaded");
  if (!out || !sites_done || !bytes || capacity < 0 || site_lo < 0 || site_lo > g.n_sites)
    LS_FAIL(LS_E_ARG, "ls_geno_long_text: bad argument");
  *sites_done = 0;
  *bytes = 0;
  if (site_lo == g.n_sites) return LS_OK;
  const std::vector<int64_t> &off = g.h_site_off;
  int64_t hi = g.n_sites;  // sites site_lo .. hi - 1 fit
  if (off[(size_t)g.n_sites] - off[(size_t)site_lo] > capacity)
    hi = (int64_t)(std::upper_bound(off.begin() + site_lo, off.end(), off[(size_t)site_lo] + capacity) - off.begin()) - 1;
  if (hi == site_lo) LS_FAIL(LS_E_CAPACITY, "ls_geno_long_text: a site is longer than the capacity");
  const int64_t nb = off[(size_t)hi] - off[(size_t)site_lo], rows = (hi - site_lo) * (int64_t)g.n_cells;
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(g.out.ensure((size_t)nb + 16));
  GlView v = {};
  v.cell = g.cell.as<int32_t>();
  v.dp = g.dp.as<int32_t>();
  v.alt = g.alt.as<int32_t>();
  v.p = g.p.as<double>();
  v.hit_lo = g.hit_lo.as<int64_t>();
  v.hit_hi = g.hit_hi.as<int64_t>();
  v.tail_base = g.tail_base.as<int64_t>();
  v.tail_cum = g.tail_cum.as<int64_t>();
  v.site_off = g.site_off.as<int64_t>();
  v.flags = g.flags.as<uint8_t>();
  v.prefix = g.prefix.as<char>();
  v.prefix_off = g.prefix_off.as<int64_t>();
  v.cell_text = g.cell_text.as<char>();
  v.cell_off = g.cell_off.as<int64_t>();
  v.index = g.hccv ? nullptr : g.index.as<char>();
  v.index_off = g.hccv ? nullptr : g.index_off.as<int64_t>();
  v.n_cells = g.n_cells;
  v.hccv = g.hccv;
  v.pvalue = g.pvalue;
  LS_CK(cudaEventRecord(ctx->ev[0], st));
  if (rows) {
    const unsigned grid = (unsigned)std::min<int64_t>((rows + GL_WARPS - 1) / GL_WARPS, (int64_t)ctx->num_sms * 16);
    gl_write_kernel<<<grid, GL_THREADS, 0, st>>>(v, site_lo, rows, g.out.as<char>());
    LS_CK(cudaGetLastError());
  }
  LS_CK(cudaEventRecord(ctx->ev[1], st));
  if (nb) LS_CK(cudaMemcpyAsync(out, g.out.p, (size_t)nb, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaEventRecord(ctx->ev[2], st));
  LS_CK(cudaStreamSynchronize(st));
  float ms_text = 0.f, ms_copy = 0.f;
  LS_CK(cudaEventElapsedTime(&ms_text, ctx->ev[0], ctx->ev[1]));
  LS_CK(cudaEventElapsedTime(&ms_copy, ctx->ev[1], ctx->ev[2]));
  g.ms_text += ms_text;
  g.ms_copy += ms_copy;
  g.blocks += 1;
  g.bytes += nb;
  *sites_done = hi - site_lo;
  *bytes = nb;
  return LS_OK;
}

extern "C" int ls_geno_long_times(ls_ctx *ctx, double *ms_text, double *ms_copy, int64_t *blocks, int64_t *bytes) {
  if (!ctx || !ms_text || !ms_copy || !blocks || !bytes) return LS_E_ARG;
  const GenoLongState &g = ctx->gl;
  *ms_text = g.ms_text;
  *ms_copy = g.ms_copy;
  *blocks = g.blocks;
  *bytes = g.bytes;
  return LS_OK;
}

extern "C" int ls_geno_long_release(ls_ctx *ctx) {
  if (!ctx) return LS_E_ARG;
  LS_CK(cudaSetDevice(ctx->device));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  ctx->gl.release();
  return LS_OK;
}
