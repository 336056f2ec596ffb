// Device-wide exclusive scan and stable LSD radix sort (hand-written; no CUB / Thrust).
// Both are plumbing for the pileup path: the scans turn tile flags / per-tile pass counts into
// offsets, the sort groups (read, tile) segments by (tile, cell).
#include "ls_common.cuh"

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_CHUNK = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

// exclusive scan of one value per thread over the block; returns exclusive prefix, total in *total
template <int THREADS>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total, uint32_t *smem /*THREADS/32+1*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t inc = warp_incl_scan(v, lane);
  if (lane == 31) smem[w] = inc;
  __syncthreads();
  if (w == 0) {
    uint32_t s = (lane < THREADS / 32) ? smem[lane] : 0u;
    uint32_t si = warp_incl_scan(s, lane);
    if (lane < THREADS / 32) smem[lane] = si - s;
    if (lane == THREADS / 32 - 1) smem[THREADS / 32] = si;
  }
  __syncthreads();
  uint32_t r = smem[w] + inc - v;
  *total = smem[THREADS / 32];
  __syncthreads();
  return r;
}

// Single-pass exclusive scan with decoupled look-back: every CTA takes the next chunk in ticket order (so that the
// chunks before it are always running or done), publishes its chunk total, then walks back over its predecessors'
// records until it meets one that already carries an inclusive prefix.  One read and one write of the array.
// state[j]: bits 62-63 = 0 not ready, 1 = chunk total, 2 = inclusive prefix up to and including chunk j; bits 0-61 value.
constexpr uint64_t SCAN_AGG = 1ull << 62, SCAN_PFX = 2ull << 62, SCAN_VAL = (1ull << 62) - 1ull;

struct ScanJobs {
  LsScanJob j[LS_SCAN_MAX_JOBS];
  unsigned long long *state;  // [jobs][nb_max] chunk records
  unsigned int *ticket;       // [jobs]
  int64_t nb_max;
};

// blockIdx.y = the array (several independent scans share one launch).  WIDE: the prefixes go to job.out64 as 64-bit
// values, for sums that may pass 2^32 (a chunk's own sum must still fit 32 bits)
template <bool WIDE>
__global__ void __launch_bounds__(SCAN_THREADS) scan_chained(ScanJobs jobs) {
  __shared__ uint32_t sm[SCAN_THREADS / 32 + 1];
  __shared__ uint32_t bid_s;
  __shared__ unsigned long long pfx_s;
  const LsScanJob job = jobs.j[blockIdx.y];
  const uint32_t *__restrict__ in = job.in;
  uint32_t *__restrict__ out = job.out;
  const int64_t n = job.n;
  uint64_t *__restrict__ total = job.total;
  unsigned long long *__restrict__ state = jobs.state + (size_t)blockIdx.y * jobs.nb_max;
  if (threadIdx.x == 0) bid_s = atomicAdd(jobs.ticket + blockIdx.y, 1u);
  __syncthreads();
  const uint32_t bid = bid_s;
  if ((int64_t)bid * SCAN_CHUNK >= n) return;  // the launch covers the longest array of the batch
  const int64_t base = (int64_t)bid * SCAN_CHUNK + (int64_t)threadIdx.x * SCAN_ITEMS;
  uint32_t v[SCAN_ITEMS];
  uint32_t s = 0;
  if (base + SCAN_ITEMS <= n) {
    const uint4 a = *reinterpret_cast<const uint4 *>(in + base), b = *reinterpret_cast<const uint4 *>(in + base + 4);
    v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w, v[4] = b.x, v[5] = b.y, v[6] = b.z, v[7] = b.w;
  } else {
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) v[i] = base + i < n ? in[base + i] : 0u;
  }
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) s += v[i];
  uint32_t tot;
  uint32_t ex = block_excl_scan<SCAN_THREADS>(s, &tot, sm);
  if (threadIdx.x < 32) {
    // the first warp looks back 32 chunk records at a time
    const int lane = threadIdx.x;
    unsigned long long pfx = 0;
    if (bid > 0) {
      if (lane == 0) atomicExch(state + bid, SCAN_AGG | (unsigned long long)tot);
      for (int64_t j = (int64_t)bid - 1 - lane;; j -= 32) {
        unsigned long long st = SCAN_PFX;  // before the first chunk: an inclusive prefix of zero
        if (j >= 0) {
          do {
            st = *((volatile unsigned long long *)(state + j));
          } while ((st >> 62) == 0ull);
        }
        const uint32_t pm = __ballot_sync(0xffffffffu, (st >> 62) == 2ull);
        const int first = pm ? __ffs(pm) - 1 : 32;  // nearest record that carries a prefix
        unsigned long long val = lane <= first ? (st & SCAN_VAL) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
        pfx += val;
        if (pm) break;
      }
    }
    if (lane == 0) {
      __threadfence();
      atomicExch(state + bid, SCAN_PFX | (pfx + (unsigned long long)tot));
      pfx_s = pfx;
      if (total && (int64_t)(bid + 1) * SCAN_CHUNK >= n) *total = pfx + (unsigned long long)tot;
    }
  }
  __syncthreads();
  if (WIDE) {
    uint64_t e = pfx_s + ex;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
      if (base + i < n) job.out64[base + i] = e;
      e += v[i];
    }
    return;
  }
  ex += (uint32_t)pfx_s;
  if (base + SCAN_ITEMS <= n) {
    uint4 a, b;
    a.x = ex, ex += v[0];
    a.y = ex, ex += v[1];
    a.z = ex, ex += v[2];
    a.w = ex, ex += v[3];
    b.x = ex, ex += v[4];
    b.y = ex, ex += v[5];
    b.z = ex, ex += v[6];
    b.w = ex;
    *reinterpret_cast<uint4 *>(out + base) = a;
    *reinterpret_cast<uint4 *>(out + base + 4) = b;
  } else {
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
      if (base + i < n) out[base + i] = ex;
      ex += v[i];
    }
  }
}

// ---------------- radix sort ------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ROUNDS = 8;                       // items per thread per chunk
constexpr int RS_CHUNK = RS_THREADS * RS_ROUNDS;   // 2048

template <typename K>
__global__ void __launch_bounds__(RS_THREADS) rs_hist(const K *__restrict__ keys, int64_t n, int64_t per_block,
                                                      int shift, uint32_t *__restrict__ hist, int G) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  int64_t lo = (int64_t)blockIdx.x * per_block;
  int64_t hi = lo + per_block < n ? lo + per_block : n;
  for (int64_t i = lo + threadIdx.x; i < hi; i += RS_THREADS) {
    uint32_t d = (uint32_t)(keys[i] >> shift) & 255u;
    atomicAdd(&h[d], 1u);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * G + blockIdx.x] = h[threadIdx.x];
}

// One chunk (RS_CHUNK items) at a time: stable rank of every item inside its digit (match_any inside a warp,
// per-warp digit counters across warps), then the chunk is laid out digit-major in shared memory and written
// from there, so that each digit's items leave the CTA as one contiguous, coalesced run.
template <bool HAS_VALS, typename K>
__global__ void __launch_bounds__(RS_THREADS) rs_scatter(const K *__restrict__ keys_in,
                                                         const uint32_t *__restrict__ vals_in,
                                                         K *__restrict__ keys_out, uint32_t *__restrict__ vals_out,
                                                         int64_t n, int64_t per_block, int shift,
                                                         const uint32_t *__restrict__ hist_scanned, int G, int first_pass) {
  __shared__ uint32_t gbase[256];            // running global offset of each digit for this CTA
  __shared__ uint32_t lbase[256];            // offset of each digit inside the staged chunk
  __shared__ uint32_t wcnt[RS_WARPS][256];   // per-warp digit counts, then per-warp offsets inside the digit
  __shared__ uint32_t scan_sm[RS_THREADS / 32 + 1];
  __shared__ K skey[RS_CHUNK];
  __shared__ uint32_t sval[HAS_VALS ? RS_CHUNK : 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  gbase[threadIdx.x] = hist_scanned[(int64_t)threadIdx.x * G + blockIdx.x] + hist_scanned[(int64_t)256 * G + threadIdx.x];
  int64_t lo = (int64_t)blockIdx.x * per_block;
  int64_t hi = lo + per_block < n ? lo + per_block : n;
  for (int64_t chunk = lo; chunk < hi; chunk += RS_CHUNK) {
    for (int i = threadIdx.x; i < RS_WARPS * 256; i += RS_THREADS) (&wcnt[0][0])[i] = 0;
    __syncthreads();
    K key[RS_ROUNDS];
    uint32_t val[RS_ROUNDS];
    uint32_t rank[RS_ROUNDS];
    // all loads of the chunk first: the ranking below has warp barriers the loads could not be hoisted across
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
      int64_t idx = chunk + (int64_t)w * (32 * RS_ROUNDS) + r * 32 + lane;
      bool valid = idx < hi;
      key[r] = valid ? keys_in[idx] : (K)0;
      if (HAS_VALS) val[r] = valid ? (first_pass ? (uint32_t)idx : vals_in[idx]) : 0u;
    }
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
      int64_t idx = chunk + (int64_t)w * (32 * RS_ROUNDS) + r * 32 + lane;
      bool valid = idx < hi;
      uint32_t d = valid ? ((uint32_t)(key[r] >> shift) & 255u) : 256u;
      uint32_t peers = __match_any_sync(0xffffffffu, d);
      uint32_t before = __popc(peers & lt);
      uint32_t cur = valid ? wcnt[w][d] : 0u;
      rank[r] = cur + before;
      __syncwarp();
      if (valid && before == 0) wcnt[w][d] = cur + __popc(peers);
      __syncwarp();
    }
    __syncthreads();
    uint32_t dtot;
    {  // per digit: exclusive scan across warps; then across digits for the staged layout
      const int d = threadIdx.x;
      uint32_t run = 0;
#pragma unroll
      for (int ww = 0; ww < RS_WARPS; ++ww) {
        uint32_t t = wcnt[ww][d];
        wcnt[ww][d] = run;
        run += t;
      }
      dtot = run;
    }
    {
      uint32_t tot;
      const uint32_t ex = block_excl_scan<RS_THREADS>(dtot, &tot, scan_sm);  // ends with a barrier
      lbase[threadIdx.x] = ex;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ROUNDS; ++r) {
      int64_t idx = chunk + (int64_t)w * (32 * RS_ROUNDS) + r * 32 + lane;
      if (idx < hi) {
        uint32_t d = (uint32_t)(key[r] >> shift) & 255u;
        uint32_t li = lbase[d] + wcnt[w][d] + rank[r];
        skey[li] = key[r];
        if (HAS_VALS) sval[li] = val[r];
      }
    }
    __syncthreads();
    const int cn = (int)((hi - chunk) < (int64_t)RS_CHUNK ? (hi - chunk) : (int64_t)RS_CHUNK);
    for (int i = threadIdx.x; i < cn; i += RS_THREADS) {
      const K k = skey[i];
      const uint32_t d = (uint32_t)(k >> shift) & 255u;
      const uint32_t pos = gbase[d] + ((uint32_t)i - lbase[d]);
      keys_out[pos] = k;
      if (HAS_VALS) vals_out[pos] = sval[i];
    }
    __syncthreads();
    gbase[threadIdx.x] += dtot;
    __syncthreads();
  }
}

// exclusive scan of the (digit-major, block-minor) histogram in two tiny kernels:
// one CTA per digit scans its G entries and records the digit total, one CTA scans the 256 totals.
__global__ void __launch_bounds__(256) rs_scan_digit(uint32_t *__restrict__ hist, int G, uint32_t *__restrict__ totals) {
  __shared__ uint32_t sm[256 / 32 + 1];
  uint32_t *h = hist + (size_t)blockIdx.x * G;
  uint32_t carry = 0;
  for (int base = 0; base < G; base += 256) {
    const int i = base + threadIdx.x;
    const uint32_t v = i < G ? h[i] : 0u;
    uint32_t tot;
    const uint32_t ex = block_excl_scan<256>(v, &tot, sm);
    if (i < G) h[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}

__global__ void __launch_bounds__(256) rs_scan_totals(uint32_t *__restrict__ totals) {
  __shared__ uint32_t sm[256 / 32 + 1];
  uint32_t tot;
  const uint32_t v = totals[threadIdx.x];
  const uint32_t ex = block_excl_scan<256>(v, &tot, sm);
  totals[threadIdx.x] = ex;
}

template <bool HAS_VALS, typename K>
cudaError_t radix_sort_impl(K *keys_a, K *keys_b, uint32_t *vals_a, uint32_t *vals_b, int64_t n,
                            int key_bits, DBuf &hist, K **sorted_keys, uint32_t **sorted_vals, int num_sms,
                            cudaStream_t st, int *launches) {
  *sorted_keys = keys_a;
  if (sorted_vals) *sorted_vals = vals_a;
  if (n <= 0) return cudaSuccess;
  int passes = (key_bits + 7) / 8;
  if (passes < 1) passes = 1;
  int64_t nchunks = (n + RS_CHUNK - 1) / RS_CHUNK;
  int G = (int)(nchunks < (int64_t)num_sms * 4 ? nchunks : (int64_t)num_sms * 4);
  int64_t per_block = ((nchunks + G - 1) / G) * RS_CHUNK;
  cudaError_t e = hist.ensure(((size_t)256 * G + 256) * sizeof(uint32_t));
  if (e != cudaSuccess) return e;
  K *kin = keys_a, *kout = keys_b;
  uint32_t *vin = vals_a, *vout = vals_b;
  for (int p = 0; p < passes; ++p) {
    int shift = p * 8;
    rs_hist<K><<<G, RS_THREADS, 0, st>>>(kin, n, per_block, shift, hist.as<uint32_t>(), G);
    rs_scan_digit<<<256, 256, 0, st>>>(hist.as<uint32_t>(), G, hist.as<uint32_t>() + (size_t)256 * G);
    rs_scan_totals<<<1, 256, 0, st>>>(hist.as<uint32_t>() + (size_t)256 * G);
    rs_scatter<HAS_VALS, K><<<G, RS_THREADS, 0, st>>>(kin, vin, kout, vout, n, per_block, shift, hist.as<uint32_t>(), G,
                                                   p == 0 ? 1 : 0);
    if (launches) *launches += 4;
    K *tk = kin;
    kin = kout;
    kout = tk;
    uint32_t *tv = vin;
    vin = vout;
    vout = tv;
  }
  *sorted_keys = kin;
  if (sorted_vals) *sorted_vals = vin;
  return cudaGetLastError();
}

template <bool WIDE>
cudaError_t scan_multi(const LsScanJob *jobs, int n_jobs, DBuf &tmp, cudaStream_t st) {
  if (n_jobs < 1 || n_jobs > LS_SCAN_MAX_JOBS) return cudaErrorInvalidValue;
  ScanJobs a;
  int64_t nb_max = 0;
  int live = 0;
  for (int k = 0; k < n_jobs; ++k) {
    if (jobs[k].n <= 0) {
      if (jobs[k].total) {
        cudaError_t e = cudaMemsetAsync(jobs[k].total, 0, sizeof(uint64_t), st);
        if (e != cudaSuccess) return e;
      }
      continue;
    }
    if ((reinterpret_cast<uintptr_t>(jobs[k].in) | reinterpret_cast<uintptr_t>(jobs[k].out)) & 15u) return cudaErrorMisalignedAddress;
    if (WIDE != (jobs[k].out64 != nullptr)) return cudaErrorInvalidValue;
    a.j[live++] = jobs[k];
    const int64_t nb = (jobs[k].n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    nb_max = nb > nb_max ? nb : nb_max;
  }
  if (!live) return cudaSuccess;
  // chunk records of every array + the ticket counters behind them, cleared before every launch
  const size_t words = (size_t)live * (size_t)nb_max + LS_SCAN_MAX_JOBS;
  cudaError_t e = tmp.ensure(words * sizeof(uint64_t));
  if (e != cudaSuccess) return e;
  e = cudaMemsetAsync(tmp.p, 0, words * sizeof(uint64_t), st);
  if (e != cudaSuccess) return e;
  a.state = tmp.as<unsigned long long>();
  a.ticket = reinterpret_cast<unsigned int *>(tmp.as<unsigned long long>() + (size_t)live * (size_t)nb_max);
  a.nb_max = nb_max;
  scan_chained<WIDE><<<dim3((unsigned)nb_max, (unsigned)live), SCAN_THREADS, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace

cudaError_t ls_scan_exclusive_u32_multi(const LsScanJob *jobs, int n_jobs, DBuf &tmp, cudaStream_t st) {
  return scan_multi<false>(jobs, n_jobs, tmp, st);
}

cudaError_t ls_scan_exclusive_u32_wide(const uint32_t *d_in, uint64_t *d_out, int64_t n, DBuf &tmp, cudaStream_t st) {
  if (n <= 0) return cudaMemsetAsync(d_out, 0, sizeof(uint64_t), st);
  LsScanJob j;
  j.in = d_in;
  j.out = nullptr;
  j.n = n;
  j.total = d_out + n;
  j.out64 = d_out;
  return scan_multi<true>(&j, 1, tmp, st);
}

cudaError_t ls_scan_exclusive_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n, uint64_t *d_total, DBuf &tmp,
                                  cudaStream_t st) {
  LsScanJob j;
  j.in = d_in;
  j.out = d_out;
  j.n = n;
  j.total = d_total;
  return ls_scan_exclusive_u32_multi(&j, 1, tmp, st);
}

cudaError_t ls_radix_sort_pairs(uint64_t *keys_a, uint64_t *keys_b, uint32_t *vals_a, uint32_t *vals_b, int64_t n,
                                int key_bits, DBuf &hist, uint64_t **sorted_keys, uint32_t **sorted_vals, int num_sms,
                                cudaStream_t st, int *launches) {
  return radix_sort_impl<true, uint64_t>(keys_a, keys_b, vals_a, vals_b, n, key_bits, hist, sorted_keys, sorted_vals, num_sms,
                               st, launches);
}

cudaError_t ls_radix_sort_keys(uint64_t *keys_a, uint64_t *keys_b, int64_t n, int key_bits, DBuf &hist,
                               uint64_t **sorted_keys, int num_sms, cudaStream_t st, int *launches) {
  return radix_sort_impl<false>(keys_a, keys_b, nullptr, nullptr, n, key_bits, hist, sorted_keys, nullptr, num_sms,
                                st, launches);
}

cudaError_t ls_radix_sort_keys32(uint32_t *keys_a, uint32_t *keys_b, int64_t n, int key_bits, DBuf &hist,
                                 uint32_t **sorted_keys, int num_sms, cudaStream_t st, int *launches) {
  return radix_sort_impl<false>(keys_a, keys_b, nullptr, nullptr, n, key_bits, hist, sorted_keys, nullptr, num_sms,
                                st, launches);
}
