// K2: fp64 beta-binomial upper tails, p = scipy.stats.betabinom.sf(k - eps, n, a, b).
//
// Replaces the scalar scipy calls of BaseCellCalling.step1.py:196,201,329-330,427-428 and
// SingleCellGenotype.py:204 / HCCVSingleCellGenotype.py:204.  scipy evaluates
//   sf = clip(1 - np.sum(exp(logpmf(arange(0, k)))), 0, 1)
// with logpmf built from cephes lbeta (ls_cephes.h) and np.sum's pairwise order
// (ls_pairwise.h); both are restated exactly so that only libm-level (<= 1-2 ulp) differences
// remain.  Compiled with -fmad=false: the reference arithmetic has no fused multiply-adds.
//
// Work decomposition: one thread per pmf TERM (balanced however skewed k is), terms staged
// in an HBM scratch in query-major order, then one thread per query replays numpy's
// pairwise reduction over its slice.
#include <algorithm>

#include "ls_common.cuh"
#include "ls_pairwise.h"

__global__ void bb_const_kernel(double a, double b, double *out) { out[0] = ls_lbeta(a, b); }

__global__ void __launch_bounds__(256) bb_terms_kernel(const int32_t *__restrict__ k, const int32_t *__restrict__ n,
                                                       const uint64_t *__restrict__ off, int64_t m, uint64_t total,
                                                       double a, double b, const double *__restrict__ lab_p,
                                                       double *__restrict__ terms) {
  const double lab = lab_p[0];
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
       t += (uint64_t)gridDim.x * blockDim.x) {
    // query q with off[q] <= t < off[q+1]
    int64_t lo = 0, hi = m;
    while (hi - lo > 1) {
      int64_t mid = (lo + hi) >> 1;
      if (off[mid] <= t)
        lo = mid;
      else
        hi = mid;
    }
    const double nn = (double)n[lo];
    const double i = (double)(t - off[lo]);
    const double lnp1 = log(nn + 1.0);
    terms[t] = exp(ls_betabinom_logpmf(i, nn, a, b, lnp1, lab));
  }
}

__global__ void __launch_bounds__(128) bb_sum_kernel(const int32_t *__restrict__ k, const int32_t *__restrict__ n,
                                                     const uint64_t *__restrict__ off, int64_t m,
                                                     const double *__restrict__ terms, double *__restrict__ p) {
  int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= m) return;
  const uint64_t lo = off[q], hi = off[q + 1];
  double cdf = 0.0;
  if (hi > lo) cdf = ls_pairwise_sum(terms + lo, (long)(hi - lo));
  p[q] = ls_sf_finish(k[q], n[q], cdf);
}

// Queries with k <= BB_SMALL (every beta-binomial call of the genotype path, most of step1's): one thread per
// query, the pmf terms stay in the thread's local array and numpy's pairwise order is replayed on them -- nothing is
// staged in HBM.  k <= 0 (no query / k - eps < 0) and k > n follow ls_sf_finish; a query past BB_SMALL gets p = -1 and
// is counted in *nbig (the staged kernels above take it).  no_query_nan: k == 0 means "no query" -> NaN.
constexpr int BB_SMALL = 128;

__global__ void __launch_bounds__(128) bb_small_kernel(const int32_t *__restrict__ k, const int32_t *__restrict__ n, int64_t m,
                                                       double a, double b, const double *__restrict__ lab_p,
                                                       double *__restrict__ p, uint32_t *__restrict__ nbig, int no_query_nan,
                                                       const double *__restrict__ table, int table_n) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= m) return;
  const int kk = k[q], nn = n[q];
  if (kk == 0 && no_query_nan) {
    p[q] = NAN;
    return;
  }
  if (nn < 0 || kk <= 0 || kk > nn) {
    p[q] = ls_sf_finish(kk, nn, 0.0);
    return;
  }
  if (table && nn <= table_n) {  // the tail is a function of (k, n) only: shallow pairs come from the table
    p[q] = table[nn * (table_n + 1) + kk];
    return;
  }
  if (kk > BB_SMALL) {
    p[q] = -1.0;
    if (nbig) atomicAdd(nbig, 1u);
    return;
  }
  double t[BB_SMALL];
  const double lab = lab_p[0], dn = (double)nn, lnp1 = log(dn + 1.0);
  for (int i = 0; i < kk; ++i) t[i] = exp(ls_betabinom_logpmf((double)i, dn, a, b, lnp1, lab));
  p[q] = ls_sf_finish(kk, nn, ls_pairwise_sum(t, kk));
}

// every (k, n) with 0 <= k, n <= BB_TABLE_N, as queries: entry n * (BB_TABLE_N + 1) + k
constexpr int BB_TABLE_N = 64;
__global__ void bb_table_queries_kernel(int32_t *__restrict__ k, int32_t *__restrict__ n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (BB_TABLE_N + 1) * (BB_TABLE_N + 1)) return;
  k[i] = i % (BB_TABLE_N + 1);
  n[i] = i / (BB_TABLE_N + 1);
}

// device arrays in, device array out (used by the sparse genotype path).  The depth of a (site, cell) pair is a
// handful of reads, so almost every query repeats one of a few hundred (k, n) pairs: those tails are computed once per
// call, by the same kernel (same arithmetic, same summation order), and looked up.
int ls_betabinom_device(ls_ctx *ctx, const int32_t *d_k, const int32_t *d_n, double a, double b, double *d_p, int64_t m,
                        uint32_t *d_nbig) {
  if (m <= 0) return LS_OK;
  cudaStream_t st = ctx->stream;
  constexpr int NT = (BB_TABLE_N + 1) * (BB_TABLE_N + 1);
  LS_CK(ctx->g_c.ensure(64 + (size_t)NT * (4 + 4 + 8)));
  double *d_lab = ctx->g_c.as<double>();
  double *d_tab = d_lab + 8;
  int32_t *d_tk = reinterpret_cast<int32_t *>(d_tab + NT), *d_tn = d_tk + NT;
  bb_const_kernel<<<1, 1, 0, st>>>(a, b, d_lab);
  const double *table = nullptr;
  if (m > 4 * (int64_t)NT) {
    bb_table_queries_kernel<<<(NT + 255) / 256, 256, 0, st>>>(d_tk, d_tn);
    bb_small_kernel<<<(NT + 127) / 128, 128, 0, st>>>(d_tk, d_tn, NT, a, b, d_lab, d_tab, nullptr, 0, nullptr, 0);
    table = d_tab;
  }
  bb_small_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(d_k, d_n, m, a, b, d_lab, d_p, d_nbig, 1, table, BB_TABLE_N);
  LS_CK(cudaGetLastError());
  return LS_OK;
}

extern "C" int ls_betabinom_sf(ls_ctx *ctx, const int32_t *k, const int32_t *n, double a, double b, double *p,
                               int64_t m, ls_run_stats *stats) {
  if (!ctx) return LS_E_ARG;
  if (m < 0 || (m > 0 && (!k || !n || !p))) LS_FAIL(LS_E_ARG, "ls_betabinom_sf: null array");
  if (!(a > 0.0) || !(b > 0.0)) LS_FAIL(LS_E_ARG, "ls_betabinom_sf: a and b must be > 0");
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  ls_run_stats S;
  memset(&S, 0, sizeof S);
  if (m == 0) {
    if (stats) *stats = S;
    return LS_OK;
  }
  const uint64_t CAP = (uint64_t)1 << 26;  // pmf terms staged per chunk (512 MB of doubles)
  LS_CK(ctx->g_e.ensure(64));
  bb_const_kernel<<<1, 1, 0, st>>>(a, b, ctx->g_e.as<double>());
  int launches = 1;
  float ms_total = 0.f;
  // pass 1: every query with k <= BB_SMALL, in registers / local memory
  std::vector<int64_t> big;
  {
    LS_CK(ctx->g_a.ensure((size_t)m * 4));
    LS_CK(ctx->g_b.ensure((size_t)m * 4));
    LS_CK(ctx->g_d.ensure((size_t)m * 8));
    LS_CK(cudaMemcpyAsync(ctx->g_a.p, k, (size_t)m * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->g_b.p, n, (size_t)m * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaEventRecord(ctx->ev[0], st));
    bb_small_kernel<<<(unsigned)((m + 127) / 128), 128, 0, st>>>(ctx->g_a.as<int32_t>(), ctx->g_b.as<int32_t>(), m, a, b,
                                                                 ctx->g_e.as<double>(), ctx->g_d.as<double>(), nullptr, 0, nullptr, 0);
    ++launches;
    LS_CK(cudaGetLastError());
    LS_CK(cudaEventRecord(ctx->ev[1], st));
    LS_CK(cudaMemcpyAsync(p, ctx->g_d.p, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
    LS_CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    LS_CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    ms_total += ms;
    for (int64_t i = 0; i < m; ++i) {
      if (k[i] > BB_SMALL && n[i] >= 0 && k[i] <= n[i]) big.push_back(i);
      if (k[i] > 0 && k[i] <= BB_SMALL && n[i] >= 0 && k[i] <= n[i]) S.n_events += k[i];
    }
  }
  // pass 2: the long tails (k > BB_SMALL), pmf terms staged in HBM, one thread per term
  std::vector<int32_t> bk(big.size()), bn(big.size());
  std::vector<double> bp(big.size());
  for (size_t j = 0; j < big.size(); ++j) {
    bk[j] = k[big[j]];
    bn[j] = n[big[j]];
  }
  double *p_all = p;
  k = bk.data();
  n = bn.data();
  p = bp.data();
  m = (int64_t)big.size();
  std::vector<uint64_t> off;
  int64_t q0 = 0;
  while (q0 < m) {
    off.clear();
    off.push_back(0);
    int64_t q1 = q0;
    uint64_t tot = 0;
    while (q1 < m) {
      uint64_t t = (n[q1] >= 0 && k[q1] > 0 && k[q1] <= n[q1]) ? (uint64_t)k[q1] : 0;
      if (q1 > q0 && tot + t > CAP) break;
      tot += t;
      off.push_back(tot);
      ++q1;
    }
    const int64_t mc = q1 - q0;
    LS_CK(ctx->g_a.ensure((size_t)mc * 4));
    LS_CK(ctx->g_b.ensure((size_t)mc * 4));
    LS_CK(ctx->g_c.ensure((size_t)(mc + 1) * 8));
    LS_CK(ctx->g_d.ensure((size_t)mc * 8));
    LS_CK(ctx->scan_tmp.ensure((size_t)(tot ? tot : 1) * 8));
    LS_CK(cudaMemcpyAsync(ctx->g_a.p, k + q0, (size_t)mc * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->g_b.p, n + q0, (size_t)mc * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(ctx->g_c.p, off.data(), (size_t)(mc + 1) * 8, cudaMemcpyHostToDevice, st));
    LS_CK(cudaEventRecord(ctx->ev[0], st));
    if (tot) {
      uint64_t nb = (tot + 255) / 256;
      unsigned grid = (unsigned)std::min<uint64_t>(nb, (uint64_t)ctx->num_sms * 32);
      bb_terms_kernel<<<grid, 256, 0, st>>>(ctx->g_a.as<int32_t>(), ctx->g_b.as<int32_t>(), ctx->g_c.as<uint64_t>(), mc,
                                            tot, a, b, ctx->g_e.as<double>(), ctx->scan_tmp.as<double>());
      ++launches;
    }
    bb_sum_kernel<<<(unsigned)((mc + 127) / 128), 128, 0, st>>>(ctx->g_a.as<int32_t>(), ctx->g_b.as<int32_t>(),
                                                                ctx->g_c.as<uint64_t>(), mc, ctx->scan_tmp.as<double>(),
                                                                ctx->g_d.as<double>());
    ++launches;
    LS_CK(cudaGetLastError());
    LS_CK(cudaEventRecord(ctx->ev[1], st));
    LS_CK(cudaMemcpyAsync(p + q0, ctx->g_d.p, (size_t)mc * 8, cudaMemcpyDeviceToHost, st));
    LS_CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    LS_CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    ms_total += ms;
    S.n_events += (int64_t)tot;
    q0 = q1;
  }
  for (size_t j = 0; j < big.size(); ++j) p_all[big[j]] = bp[j];
  S.ms_count = ms_total;
  S.ms_total = ms_total;
  S.count_launches = launches;
  if (stats) *stats = S;
  return LS_OK;
}
