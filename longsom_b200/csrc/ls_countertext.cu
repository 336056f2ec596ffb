// BaseCellCounter's per-site table written as text on the device from the compacted sites of the last pileup run
// (ctx->out_tid / out_pos / out_ref / out_counts, in (window, position) order).  The text is that of the host writer
// ls_write_counter_rows (csrc/host/ls_bamread.cpp): per site
//   chrom \t pos+1 \t REF \t DP|NC|CC|BC|BQ|BCf|BCr \t DP|NC|cc:..:cc|bc:..|bq:..|bcf:..|bcr:..:bcr \n
// with BC = BCf + BCr added in uint32 (wrapping as the host writer does).
//
// The load step measures every row and scans the lengths into 64-bit byte offsets (ls_scan_exclusive_u32_wide), and
// returns each contig's site range; a run's sites are grouped by contig because its windows are sorted by (tid,
// start).  A text call finds on the device how many whole sites from site_lo fit the caller's block, then formats
// them one site per thread: a CTA stages its tile of consecutive rows in shared memory and stores the tile with
// 16-byte stores (copy_out).  A tile longer than the stage (very long contig names) is stored row by row.
#include <algorithm>

#include "ls_common.cuh"
#include "ls_text.cuh"

namespace {

constexpr int CT_THREADS = 128;          // sites per tile
constexpr uint32_t CT_STAGE = 32 << 10;  // bytes of a tile staged in shared memory (typical rows: ~115 bytes)
constexpr int64_t CT_NAME_MAX = 65535;   // longest contig name: 2048 rows of at most 2^16 + 389 bytes scan in 32 bits

struct CtView {
  const int32_t *tid, *pos;
  const uint8_t *ref;
  const uint32_t *counts;  // [n_sites][LS_SITE_WORDS]: DP, NC, CC[6], BCf[6], BCr[6], BQ[6]
  const char *names;
  const int64_t *name_off;
};

// the row of site i at o; W = false: length only
template <bool W>
__device__ __forceinline__ uint32_t put_row(const CtView &v, int64_t i, char *o) {
  const int32_t t = v.tid[i];
  const int64_t n0 = v.name_off[t];
  const uint32_t nl = (uint32_t)(v.name_off[t + 1] - n0);
  uint32_t n = nl;
  if (W)
    for (uint32_t k = 0; k < nl; ++k) o[k] = v.names[n0 + k];
  if (W) o[n] = '\t';
  ++n;
  n += put_uint((uint32_t)v.pos[i] + 1u, W ? o + n : nullptr);
  if (W) {
    o[n] = '\t';
    o[n + 1] = (char)v.ref[i];
    const char *lit = "\tDP|NC|CC|BC|BQ|BCf|BCr\t";
    for (int k = 0; k < 24; ++k) o[n + 2 + k] = lit[k];
  }
  n += 26;
  const uint32_t *r = v.counts + i * LS_SITE_WORDS;
  n += put_uint(r[0], W ? o + n : nullptr);
  if (W) o[n] = '|';
  ++n;
  n += put_uint(r[1], W ? o + n : nullptr);
  if (W) o[n] = '|';
  ++n;
  // CC, BC, BQ, BCf, BCr: six values each, ':'-joined, '|' between the vectors and '\n' at the end
#pragma unroll 1
  for (int f = 0; f < 5; ++f) {
    const uint32_t *a = r + (f == 0 ? 2 : f == 2 ? 20 : f == 4 ? 14 : 8);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      const uint32_t x = f == 1 ? a[k] + r[14 + k] : a[k];
      n += put_uint(x, W ? o + n : nullptr);
      if (W) o[n] = k < 5 ? ':' : (f < 4 ? '|' : '\n');
      ++n;
    }
  }
  return n;
}

// per site: its row length; the first / one-past-last site of each contig; bad: 1 a tid outside [0, n_names), 2 tids
// not ascending
__global__ void __launch_bounds__(256) ct_len_kernel(CtView v, int64_t n, int32_t n_names, uint32_t *__restrict__ lens,
                                                     int64_t *__restrict__ lo, int64_t *__restrict__ hi,
                                                     uint32_t *__restrict__ bad) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t t = v.tid[i];
    uint32_t b = 0;
    if (t < 0 || t >= n_names) b |= 1u;
    if (i > 0 && v.tid[i - 1] > t) b |= 2u;
    if (b) {
      atomicOr(bad, b);
      lens[i] = 0;
      continue;
    }
    if (i == 0 || v.tid[i - 1] != t) lo[t] = i;
    if (i == n - 1 || v.tid[i + 1] != t) hi[t] = i + 1;
    lens[i] = put_row<false>(v, i, nullptr);
  }
}

// the last site h in [site_lo, site_hi] with off[h] - off[site_lo] <= capacity, and those bytes
__global__ void ct_plan_kernel(const uint64_t *__restrict__ off, int64_t site_lo, int64_t site_hi, int64_t capacity,
                               int64_t *__restrict__ res) {
  const uint64_t base = off[site_lo], lim = base + (uint64_t)capacity;
  int64_t a = site_lo, b = site_hi;  // off[a] <= lim
  while (a < b) {
    const int64_t m = (a + b + 1) >> 1;
    if (off[m] <= lim)
      a = m;
    else
      b = m - 1;
  }
  res[0] = a;
  res[1] = (int64_t)(off[a] - base);
}

__global__ void __launch_bounds__(CT_THREADS) ct_write_kernel(CtView v, const uint64_t *__restrict__ off, int64_t site_lo,
                                                              int64_t site_hi, char *__restrict__ out) {
  __shared__ __align__(16) char stage[CT_STAGE];
  const uint64_t base = off[site_lo];
  for (int64_t t0 = site_lo + (int64_t)blockIdx.x * CT_THREADS; t0 < site_hi; t0 += (int64_t)gridDim.x * CT_THREADS) {
    const int64_t t1 = t0 + CT_THREADS < site_hi ? t0 + CT_THREADS : site_hi, i = t0 + threadIdx.x;
    const uint64_t tb = off[t0], tile = off[t1] - tb;
    if (tile <= CT_STAGE) {
      if (i < t1) put_row<true>(v, i, stage + (off[i] - tb));
      __syncthreads();
      copy_out<CT_THREADS>(out + (tb - base), stage, (uint32_t)tile);
      __syncthreads();
    } else if (i < t1) {
      put_row<true>(v, i, out + (off[i] - base));
    }
  }
}

}  // namespace

extern "C" int ls_pileup_sites_upload(ls_ctx *ctx, const ls_site_counts *sites) {
  if (!ctx) return LS_E_ARG;
  if (!sites) LS_FAIL(LS_E_ARG, "ls_pileup_sites_upload: sites is null");
  const int64_t ns = sites->n_sites;
  if (ns < 0 || ns >= ((int64_t)1 << 32)) LS_FAIL(LS_E_ARG, "ls_pileup_sites_upload: n_sites outside [0, 2^32)");
  if (ns > 0 && (!sites->tid || !sites->pos || !sites->ref || !sites->counts))
    LS_FAIL(LS_E_ARG, "ls_pileup_sites_upload: null site array");
  ctx->have_run = false;
  ctx->ct.loaded = false;
  ctx->replay.valid = false;
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  LS_CK(ctx->out_tid.ensure((size_t)ns * 4 + 16));
  LS_CK(ctx->out_pos.ensure((size_t)ns * 4 + 16));
  LS_CK(ctx->out_ref.ensure((size_t)ns + 16));
  LS_CK(ctx->out_counts.ensure((size_t)ns * LS_SITE_WORDS * 4 + 16));
  if (ns) {
    LS_CK(cudaMemcpyAsync(ctx->out_tid.p, sites->tid, (size_t)ns * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->out_pos.p, sites->pos, (size_t)ns * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->out_ref.p, sites->ref, (size_t)ns, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->out_counts.p, sites->counts, (size_t)ns * LS_SITE_WORDS * 4, cudaMemcpyHostToDevice, st));
  }
  LS_CK(cudaStreamSynchronize(st));
  ctx->n_sites = ns;
  ctx->compacted = true;
  ctx->have_run = true;
  return LS_OK;
}

extern "C" int ls_pileup_text_load(ls_ctx *ctx, const char *names, const int64_t *name_off, int32_t n_names,
                                   int64_t *contig_lo, int64_t *contig_hi) {
  if (!ctx) return LS_E_ARG;
  CounterTextState &c = ctx->ct;
  c.loaded = false;
  if (!ctx->have_run) LS_FAIL(LS_E_STATE, "ls_pileup_text_load: ls_pileup_run has not completed");
  if (n_names < 0) LS_FAIL(LS_E_ARG, "ls_pileup_text_load: negative n_names");
  if (!name_off || (n_names > 0 && (!contig_lo || !contig_hi))) LS_FAIL(LS_E_ARG, "ls_pileup_text_load: null array");
  std::vector<int64_t> off0((size_t)n_names + 1);
  for (int32_t t = 0; t <= n_names; ++t) {
    off0[(size_t)t] = name_off[t] - name_off[0];
    if (t > 0 && !(name_off[t] >= name_off[t - 1] && name_off[t] - name_off[t - 1] <= CT_NAME_MAX))
      LS_FAIL(LS_E_ARG, "ls_pileup_text_load: name offsets not ascending, or a name longer than 65535 bytes");
  }
  const int64_t name_bytes = off0[(size_t)n_names];
  if (name_bytes > 0 && !names) LS_FAIL(LS_E_ARG, "ls_pileup_text_load: names is null");
  int rc = ls_pileup_compact(ctx, nullptr);
  if (rc != LS_OK) return rc;
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t ns = ctx->n_sites;
  LS_CK(c.names.ensure((size_t)name_bytes + 16));
  if (name_bytes) LS_CK(cudaMemcpyAsync(c.names.p, names + name_off[0], (size_t)name_bytes, cudaMemcpyHostToDevice, st));
  LS_CK(c.name_off.ensure(((size_t)n_names + 1) * 8));
  LS_CK(cudaMemcpyAsync(c.name_off.p, off0.data(), ((size_t)n_names + 1) * 8, cudaMemcpyHostToDevice, st));
  LS_CK(c.range.ensure((size_t)n_names * 16 + 16));
  LS_CK(cudaMemsetAsync(c.range.p, 0, (size_t)n_names * 16, st));
  LS_CK(c.result.ensure(16));
  LS_CK(cudaMemsetAsync(c.result.p, 0, 4, st));
  LS_CK(c.lens.ensure((size_t)ns * 4 + 16));
  LS_CK(c.off.ensure(((size_t)ns + 1) * 8));
  int64_t *d_lo = c.range.as<int64_t>(), *d_hi = d_lo + n_names;
  CtView v = {ctx->out_tid.as<int32_t>(), ctx->out_pos.as<int32_t>(), ctx->out_ref.as<uint8_t>(),
              ctx->out_counts.as<uint32_t>(), c.names.as<char>(), c.name_off.as<int64_t>()};
  if (ns) {
    const unsigned grid = (unsigned)std::min<int64_t>((ns + 255) / 256, (int64_t)ctx->num_sms * 16);
    ct_len_kernel<<<grid, 256, 0, st>>>(v, ns, n_names, c.lens.as<uint32_t>(), d_lo, d_hi, c.result.as<uint32_t>());
    LS_CK(cudaGetLastError());
  }
  LS_CK(ls_scan_exclusive_u32_wide(c.lens.as<uint32_t>(), c.off.as<uint64_t>(), ns, ctx->scan_tmp, st));
  uint32_t bad = 0;
  LS_CK(cudaMemcpyAsync(&bad, c.result.p, 4, cudaMemcpyDeviceToHost, st));
  if (n_names) {
    LS_CK(cudaMemcpyAsync(contig_lo, d_lo, (size_t)n_names * 8, cudaMemcpyDeviceToHost, st));
    LS_CK(cudaMemcpyAsync(contig_hi, d_hi, (size_t)n_names * 8, cudaMemcpyDeviceToHost, st));
  }
  LS_CK(cudaStreamSynchronize(st));
  if (bad & 1u) LS_FAIL(LS_E_ARG, "ls_pileup_text_load: a site's tid is outside [0, n_names)");
  if (bad & 2u) LS_FAIL(LS_E_ARG, "ls_pileup_text_load: sites not grouped by ascending tid");
  c.n_sites = ns;
  c.loaded = true;
  return LS_OK;
}

extern "C" int ls_pileup_text(ls_ctx *ctx, int64_t site_lo, int64_t site_hi, char *out, int64_t capacity,
                              int64_t *sites_done, int64_t *bytes) {
  if (!ctx) return LS_E_ARG;
  CounterTextState &c = ctx->ct;
  if (!c.loaded) LS_FAIL(LS_E_STATE, "ls_pileup_text: no ls_pileup_text_load since the last run");
  if (!out || !sites_done || !bytes || capacity < 0 || site_lo < 0 || site_lo > site_hi || site_hi > c.n_sites)
    LS_FAIL(LS_E_ARG, "ls_pileup_text: bad argument");
  *sites_done = 0;
  *bytes = 0;
  if (site_lo == site_hi) return LS_OK;
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint64_t *off = c.off.as<uint64_t>();
  int64_t res[2];
  ct_plan_kernel<<<1, 1, 0, st>>>(off, site_lo, site_hi, capacity, c.result.as<int64_t>());
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(res, c.result.p, 16, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  const int64_t hi = res[0], nb = res[1];
  if (hi == site_lo) LS_FAIL(LS_E_CAPACITY, "ls_pileup_text: a row is longer than the capacity");
  LS_CK(c.out.ensure((size_t)nb + 16));
  CtView v = {ctx->out_tid.as<int32_t>(), ctx->out_pos.as<int32_t>(), ctx->out_ref.as<uint8_t>(),
              ctx->out_counts.as<uint32_t>(), c.names.as<char>(), c.name_off.as<int64_t>()};
  const unsigned grid = (unsigned)std::min<int64_t>((hi - site_lo + CT_THREADS - 1) / CT_THREADS, (int64_t)ctx->num_sms * 8);
  ct_write_kernel<<<grid, CT_THREADS, 0, st>>>(v, off, site_lo, hi, c.out.as<char>());
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(out, c.out.p, (size_t)nb, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  *sites_done = hi - site_lo;
  *bytes = nb;
  return LS_OK;
}
