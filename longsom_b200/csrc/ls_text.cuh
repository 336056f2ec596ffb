// Device text helpers shared by the genotype writers (ls_genomatrix.cu, ls_genolong.cu): decimal integers, VAF text
// equal to Python's str(round(alt / dp, 4)), a CTA-wide exclusive scan and a store of a shared-memory tile.
#pragma once
#include <stdint.h>

// decimal digits of v at o; o may be null (length only)
__device__ __forceinline__ int put_uint(uint32_t v, char *o) {
  char b[10];
  int n = 0;
  do {
    b[n++] = (char)('0' + v % 10u);
    v /= 10u;
  } while (v);
  if (o)
    for (int i = 0; i < n; ++i) o[i] = b[n - 1 - i];
  return n;
}

// round(alt / dp, 4) as a count of 1e-4 units: Python rounds the exact binary value of the quotient, half to even.
// q = floor(d * 1e4) exactly (the product may round up across an integer), then the sign of 2 * d * 1e4 - (2q + 1),
// computed with one rounding by fma, places d against the tie point.
__device__ __forceinline__ uint32_t vaf_units(int32_t alt, int32_t dp) {
  const double d = (double)alt / (double)dp;
  double q = floor(d * 10000.0);
  if (fma(d, 10000.0, -q) < 0.0) q -= 1.0;
  const double s = fma(d, 20000.0, -(2.0 * q + 1.0));
  const uint32_t k = (uint32_t)q;
  return s > 0.0 ? k + 1u : (s < 0.0 ? k : k + (k & 1u));
}

// str() of the double nearest k / 1e4: "I.FFFF" with trailing zeros stripped, at least one fraction digit
__device__ __forceinline__ int put_units4(uint32_t k, char *o) {
  int n = put_uint(k / 10000u, o);
  const uint32_t f = k % 10000u;
  char d[4] = {(char)('0' + f / 1000u), (char)('0' + f / 100u % 10u), (char)('0' + f / 10u % 10u), (char)('0' + f % 10u)};
  int nf = 4;
  while (nf > 1 && d[nf - 1] == '0') --nf;
  if (o) {
    o[n] = '.';
    for (int i = 0; i < nf; ++i) o[n + 1 + i] = d[i];
  }
  return n + 1 + nf;
}

// exclusive scan of v over a CTA of NT threads; *total = the sum over the CTA
template <int NT>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total, uint32_t *sm /*NT/32+1*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) sm[w] = inc;
  __syncthreads();
  if (w == 0) {
    const uint32_t s = lane < NT / 32 ? sm[lane] : 0u;
    uint32_t si = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) si += t;
    }
    if (lane < NT / 32) sm[lane] = si - s;
    if (lane == NT / 32 - 1) sm[NT / 32] = si;
  }
  __syncthreads();
  const uint32_t r = sm[w] + inc - v;
  *total = sm[NT / 32];
  __syncthreads();
  return r;
}

// n bytes of shared memory to dst by a CTA of NT threads: byte stores up to the first 16-byte boundary of dst and
// after the last one, 16-byte stores between them
template <int NT>
__device__ __forceinline__ void copy_out(char *dst, const char *src, uint32_t n) {
  const uint32_t head = (uint32_t)((16u - ((uintptr_t)dst & 15u)) & 15u);
  const uint32_t h = head < n ? head : n;
  if (threadIdx.x < h) dst[threadIdx.x] = src[threadIdx.x];
  const uint32_t nv = (n - h) / 16u;
  uint4 *d4 = reinterpret_cast<uint4 *>(dst + h);
  for (uint32_t k = threadIdx.x; k < nv; k += NT) {
    const char *s = src + h + 16u * k;
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      w[q] = (uint32_t)(uint8_t)s[4 * q] | ((uint32_t)(uint8_t)s[4 * q + 1] << 8) |
             ((uint32_t)(uint8_t)s[4 * q + 2] << 16) | ((uint32_t)(uint8_t)s[4 * q + 3] << 24);
    d4[k] = make_uint4(w[0], w[1], w[2], w[3]);
  }
  const uint32_t t0 = h + 16u * nv;
  if (t0 + threadIdx.x < n) dst[t0 + threadIdx.x] = src[t0 + threadIdx.x];
}
