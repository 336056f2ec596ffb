// C-ABI plumbing: context, batch upload, pinned memory, depth-cap pre-pass.
#include <algorithm>
#include <queue>

#include "ls_common.cuh"

extern "C" int ls_abi_version(void) { return LS_ABI_VERSION; }

extern "C" int ls_ctx_create(int device, ls_ctx **out) {
  if (!out) return LS_E_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) {
    fprintf(stderr, "longsom_b200: no CUDA device (%s); there is no CPU fallback\n", cudaGetErrorString(e));
    return LS_E_CUDA;
  }
  if (device < 0 || device >= ndev) return LS_E_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return LS_E_CUDA;
  ls_ctx *ctx = new ls_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return LS_E_CUDA;
  }
  for (auto &ev : ctx->ev)
    if (cudaEventCreate(&ev) != cudaSuccess) {
      delete ctx;
      return LS_E_CUDA;
    }
  // device-wide, set once: the beta-binomial kernels keep up to 128 pmf terms / a pairwise-sum recursion on the stack
  cudaDeviceSetLimit(cudaLimitStackSize, 8192);
  *out = ctx;
  return LS_OK;
}

extern "C" int ls_ctx_destroy(ls_ctx *ctx) {
  if (!ctx) return LS_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto &ev : ctx->ev)
    if (ev) cudaEventDestroy(ev);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;  // frees every device buffer
  return LS_OK;
}

extern "C" const char *ls_last_error(const ls_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

extern "C" int ls_host_alloc(size_t bytes, void **ptr) {
  if (!ptr) return LS_E_ARG;
  *ptr = nullptr;
  if (bytes == 0) bytes = 1;
  return cudaHostAlloc(ptr, bytes, cudaHostAllocDefault) == cudaSuccess ? LS_OK : LS_E_CUDA;
}
extern "C" int ls_host_free(void *ptr) {
  if (!ptr) return LS_OK;
  return cudaFreeHost(ptr) == cudaSuccess ? LS_OK : LS_E_CUDA;
}

extern "C" int ls_device_pci_bus_id(int device, char *buf, int len) {
  if (!buf || len < 16) return LS_E_ARG;
  return cudaDeviceGetPCIBusId(buf, len, device) == cudaSuccess ? LS_OK : LS_E_CUDA;
}

extern "C" int ls_device_synchronize(ls_ctx *ctx) {
  if (!ctx) return LS_E_ARG;
  LS_CK(cudaSetDevice(ctx->device));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  return LS_OK;
}

__global__ void l2_flush_kernel(uint4 *p, size_t n, uint32_t v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = make_uint4(v, v, v, v);
}

extern "C" int ls_flush_l2(ls_ctx *ctx) {
  if (!ctx) return LS_E_ARG;
  LS_CK(cudaSetDevice(ctx->device));
  const size_t bytes = (size_t)256 << 20;  // 2x the 126 MB L2
  LS_CK(ctx->l2_scratch.ensure(bytes));
  static uint32_t v = 0;
  l2_flush_kernel<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(ctx->l2_scratch.as<uint4>(), bytes / 16, ++v);
  LS_CK(cudaGetLastError());
  return LS_OK;
}

// BAM packs base 2b in the HIGH nibble of byte b; the kernels want it in the low nibble (see ls_ctx::seq4_d)
__global__ void __launch_bounds__(256) nibble_swap_kernel(uint4 *p, size_t n16) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n16; i += stride) {
    uint4 v = p[i];
    v.x = ((v.x & 0x0f0f0f0fu) << 4) | ((v.x >> 4) & 0x0f0f0f0fu);
    v.y = ((v.y & 0x0f0f0f0fu) << 4) | ((v.y >> 4) & 0x0f0f0f0fu);
    v.z = ((v.z & 0x0f0f0f0fu) << 4) | ((v.z >> 4) & 0x0f0f0f0fu);
    v.w = ((v.w & 0x0f0f0f0fu) << 4) | ((v.w >> 4) & 0x0f0f0f0fu);
    p[i] = v;
  }
}

// Validation of an uploaded batch on the device (it used to be an O(n_reads) host loop inside every upload):
// err bits: 1 = not sorted by (tid, pos), 2 = bad cigar_off, 4 = base_off not aligned, 8 = read bases exceed n_bases
__global__ void __launch_bounds__(256) batch_check_kernel(int64_t n, const int32_t *__restrict__ tid, const int32_t *__restrict__ pos,
                                                          const int32_t *__restrict__ cell, const uint32_t *__restrict__ cigar_off,
                                                          const uint64_t *__restrict__ base_off, const int32_t *__restrict__ lq,
                                                          int64_t n_cigar, int64_t n_bases, uint32_t *__restrict__ err,
                                                          int32_t *__restrict__ max_cell) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t e = 0;
  int32_t c = -1;
  if (i < n) {
    if (i > 0 && (tid[i] < tid[i - 1] || (tid[i] == tid[i - 1] && pos[i] < pos[i - 1]))) e |= 1u;
    if (cigar_off[i + 1] < cigar_off[i] || (int64_t)cigar_off[i + 1] > n_cigar) e |= 2u;
    if (base_off[i] % LS_BASE_ALIGN != 0) e |= 4u;
    if (lq[i] < 0 || base_off[i] + (uint64_t)(lq[i] < 0 ? 0 : lq[i]) > (uint64_t)n_bases) e |= 8u;
    c = cell[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    e |= __shfl_xor_sync(0xffffffffu, e, o);
    const int32_t t = __shfl_xor_sync(0xffffffffu, c, o);
    c = t > c ? t : c;
  }
  if ((threadIdx.x & 31) == 0) {
    if (e) atomicOr(err, e);
    if (c >= 0) atomicMax(max_cell, c);
  }
}

#define UP(buf, src, bytes)                                                                   \
  do {                                                                                        \
    LS_CK(ctx->buf.ensure((bytes) ? (bytes) : 16));                                           \
    if (bytes) LS_CK(cudaMemcpyAsync(ctx->buf.p, (src), (bytes), cudaMemcpyHostToDevice, st)); \
  } while (0)

extern "C" int ls_pileup_upload(ls_ctx *ctx, const ls_read_batch *b, const ls_windows *w) {
  if (!ctx) return LS_E_ARG;
  if (!b) LS_FAIL(LS_E_ARG, "ls_pileup_upload: batch is null");
  ctx->have_batch = false;
  ctx->have_run = false;
  ctx->replay.valid = false;
  const int64_t n = b->n_reads;
  if (n < 0 || b->n_cigar < 0 || b->n_bases < 0) LS_FAIL(LS_E_ARG, "ls_pileup_upload: negative size");
  if (n >= (int64_t)0xffffffffll) LS_FAIL(LS_E_ARG, "ls_pileup_upload: more than 2^32-1 reads per batch");
  if (b->n_bases >= ((int64_t)1 << 36)) LS_FAIL(LS_E_ARG, "ls_pileup_upload: more than 2^36 query bases per batch");
  if (n > 0 && (!b->tid || !b->pos || !b->flag || !b->mapq || !b->cell || !b->cigar_off || !b->base_off || !b->l_qseq))
    LS_FAIL(LS_E_ARG, "ls_pileup_upload: null per-read array");
  if (b->n_cigar > 0 && !b->cigar) LS_FAIL(LS_E_ARG, "ls_pileup_upload: null cigar");
  if (b->n_bases > 0 && (!b->seq4 || !b->qual)) LS_FAIL(LS_E_ARG, "ls_pileup_upload: null seq4/qual");
  const int64_t nw = w ? w->n_windows : 0;
  if (nw < 0) LS_FAIL(LS_E_ARG, "ls_pileup_upload: negative n_windows");
  if (nw > 0 && (!w->tid || !w->start || !w->end || !w->ref_off || !w->ref))
    LS_FAIL(LS_E_ARG, "ls_pileup_upload: null window array");
  const int T = ls_tile_size();
  ctx->h_wtid.assign(nw ? w->tid : nullptr, nw ? w->tid + nw : nullptr);
  ctx->h_wstart.assign(nw ? w->start : nullptr, nw ? w->start + nw : nullptr);
  ctx->h_wend.assign(nw ? w->end : nullptr, nw ? w->end + nw : nullptr);
  ctx->h_wtile_base.assign((size_t)nw + 1, 0);
  for (int64_t i = 0; i < nw; ++i) {
    if (w->end[i] < w->start[i] || w->start[i] < 0) LS_FAIL(LS_E_ARG, "ls_pileup_upload: bad window");
    if (i > 0 && (w->tid[i] < w->tid[i - 1] || (w->tid[i] == w->tid[i - 1] && w->start[i] < w->end[i - 1])))
      LS_FAIL(LS_E_ARG, "ls_pileup_upload: windows must be sorted by (tid, start) and disjoint");
    if (w->ref_off[i + 1] - w->ref_off[i] != (uint64_t)(w->end[i] - w->start[i]))
      LS_FAIL(LS_E_ARG, "ls_pileup_upload: ref_off does not match window length");
    ctx->h_wtile_base[i + 1] = ctx->h_wtile_base[i] + (w->end[i] - w->start[i] + T - 1) / T;
  }
  ctx->n_tiles_total = ctx->h_wtile_base[nw];

  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  UP(tid, b->tid, (size_t)n * 4);
  UP(pos, b->pos, (size_t)n * 4);
  UP(flag, b->flag, (size_t)n * 2);
  UP(mapq, b->mapq, (size_t)n);
  UP(cell, b->cell, (size_t)n * 4);
  UP(cigar_off, b->cigar_off, (size_t)(n + 1) * 4);
  UP(cigar, b->cigar, (size_t)b->n_cigar * 4);
  UP(base_off, b->base_off, (size_t)(n + 1) * 8);
  UP(lq, b->l_qseq, (size_t)n * 4);
  {
    // qual / seq4 sit LS_QPAD bytes into zero-initialised allocations with as much slack behind them
    const size_t nq = (size_t)b->n_bases, ns = (size_t)(b->n_bases + 1) / 2;
    const size_t ns16 = (ns + 15) / 16 * 16;
    LS_CK(ctx->qual.ensure(nq + 2 * LS_QPAD));
    LS_CK(ctx->seq4.ensure(ns16 + 2 * LS_QPAD));
    LS_CK(cudaMemsetAsync(ctx->qual.p, 0, LS_QPAD, st));
    LS_CK(cudaMemsetAsync((uint8_t *)ctx->qual.p + LS_QPAD + nq, 0, LS_QPAD, st));
    LS_CK(cudaMemsetAsync(ctx->seq4.p, 0, LS_QPAD, st));
    LS_CK(cudaMemsetAsync((uint8_t *)ctx->seq4.p + LS_QPAD + ns, 0, ns16 - ns + LS_QPAD, st));
    if (nq) LS_CK(cudaMemcpyAsync((uint8_t *)ctx->qual.p + LS_QPAD, b->qual, nq, cudaMemcpyHostToDevice, st));
    if (ns) {
      LS_CK(cudaMemcpyAsync((uint8_t *)ctx->seq4.p + LS_QPAD, b->seq4, ns, cudaMemcpyHostToDevice, st));
      nibble_swap_kernel<<<ctx->num_sms * 8, 256, 0, st>>>(reinterpret_cast<uint4 *>((uint8_t *)ctx->seq4.p + LS_QPAD), ns16 / 16);
      LS_CK(cudaGetLastError());
    }
  }
  UP(wtid, w ? w->tid : nullptr, (size_t)nw * 4);
  UP(wstart, w ? w->start : nullptr, (size_t)nw * 4);
  UP(wend, w ? w->end : nullptr, (size_t)nw * 4);
  UP(wref_off, w ? w->ref_off : nullptr, (size_t)(nw > 0 ? (nw + 1) * 8 : 0));
  UP(ref, w ? w->ref : nullptr, (size_t)(nw ? w->ref_off[nw] : 0));
  UP(wtile_base, ctx->h_wtile_base.data(), (size_t)(nw + 1) * 8);
  // batch validation + largest cell id, on the device, behind the copies
  LS_CK(ctx->counters.ensure(128));
  int32_t h_chk[2] = {0, -1};
  LS_CK(cudaMemcpyAsync(ctx->counters.p, h_chk, 8, cudaMemcpyHostToDevice, st));
  if (n > 0)
    batch_check_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        n, ctx->tid.as<int32_t>(), ctx->pos.as<int32_t>(), ctx->cell.as<int32_t>(), ctx->cigar_off.as<uint32_t>(),
        ctx->base_off.as<uint64_t>(), ctx->lq.as<int32_t>(), b->n_cigar, b->n_bases, ctx->counters.as<uint32_t>(),
        ctx->counters.as<int32_t>() + 1);
  LS_CK(cudaGetLastError());
  LS_CK(cudaMemcpyAsync(h_chk, ctx->counters.p, 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  if (h_chk[0] & 1) LS_FAIL(LS_E_ARG, "ls_pileup_upload: reads are not sorted by (tid, pos)");
  if (h_chk[0] & 2) LS_FAIL(LS_E_ARG, "ls_pileup_upload: bad cigar_off");
  if (h_chk[0] & 4) LS_FAIL(LS_E_ARG, "ls_pileup_upload: base_off not aligned");
  if (h_chk[0] & 8) LS_FAIL(LS_E_ARG, "ls_pileup_upload: read bases exceed n_bases");
  const int32_t max_cell = h_chk[1];
  if (max_cell >= 0x7ffffffe) LS_FAIL(LS_E_ARG, "ls_pileup_upload: cell id too large");
  ctx->n_reads = n;
  ctx->n_cigar = b->n_cigar;
  ctx->n_bases = b->n_bases;
  ctx->n_windows = nw;
  ctx->max_cell = max_cell;
  ctx->n_drop = 0;
  ctx->have_batch = true;
  return LS_OK;
}

// ---- pileup max_depth -------------------------------------------------------------------------
// htslib bam_plp_push drops a record iff its start equals the engine's current column and more
// than maxcnt records are buffered (SURVEY.md Appendix A.3).  Equivalent, per pileup() call
// (= per window): the first kept record at a start position P is always accepted; a later
// record at P is dropped iff 1 + #{accepted records of this call with end >= P} > maxcnt.
// Only windows that fetch more than max_depth records can ever drop, so the common case
// costs one device-side count of the fetches per window and nothing here.
// The windows (pileup() calls) are host arrays; d_wcount, if not null, holds their fetch counts
// on the device, and windows at or below the cap are skipped.  ctx->rend (reference end of every
// read) must be filled on ctx->stream.  Sets ctx->drop_keys / ctx->n_drop: (window << 32 | read).
int ls_depth_cap_host(ls_ctx *ctx, const std::vector<int32_t> &wtid, const std::vector<int32_t> &wstart,
                      const std::vector<int32_t> &wend, const uint32_t *d_wcount, int min_mq, int max_depth) {
  const int64_t n = ctx->n_reads, nw = (int64_t)wtid.size();
  cudaStream_t st = ctx->stream;
  std::vector<int32_t> tid(n), pos(n), rend(n);
  std::vector<uint16_t> flag(n);
  std::vector<uint8_t> mapq(n);
  std::vector<uint32_t> wcount(d_wcount ? nw : 0);
  LS_CK(cudaMemcpyAsync(tid.data(), ctx->tid.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(pos.data(), ctx->pos.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(rend.data(), ctx->rend.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(flag.data(), ctx->flag.p, (size_t)n * 2, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(mapq.data(), ctx->mapq.p, (size_t)n, cudaMemcpyDeviceToHost, st));
  if (d_wcount) LS_CK(cudaMemcpyAsync(wcount.data(), d_wcount, (size_t)nw * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  std::vector<uint64_t> drops;
  for (int64_t w = 0; w < nw; ++w) {
    if (d_wcount && (int64_t)wcount[w] <= (int64_t)max_depth) continue;
    const int32_t wt = wtid[w], ws = wstart[w], we = wend[w];
    // first read of this contig
    int64_t r0 = std::lower_bound(tid.begin(), tid.end(), wt) - tid.begin();
    std::priority_queue<int32_t, std::vector<int32_t>, std::greater<int32_t>> live;
    int32_t last_p = -1;
    bool any_at_p = false;
    for (int64_t r = r0; r < n && tid[r] == wt && pos[r] < we; ++r) {
      uint32_t f = flag[r];
      if (f & LS_FLAG_FILTER) continue;
      if ((int)mapq[r] < min_mq) continue;
      if ((f & LS_FLAG_PAIRED) && !(f & LS_FLAG_PROPER)) continue;
      int32_t e = rend[r] > pos[r] ? rend[r] : pos[r] + 1;  // fetch overlap uses bam_endpos
      if (e <= ws) continue;
      const int32_t P = pos[r];
      if (P != last_p) {
        last_p = P;
        any_at_p = false;
      }
      while (!live.empty() && live.top() < P) live.pop();
      if (any_at_p && (int64_t)1 + (int64_t)live.size() > (int64_t)max_depth) {
        drops.push_back(((uint64_t)w << 32) | (uint64_t)r);
        continue;
      }
      any_at_p = true;
      live.push(rend[r]);
    }
  }
  std::sort(drops.begin(), drops.end());
  ctx->n_drop = (int64_t)drops.size();
  LS_CK(ctx->drop_keys.ensure(drops.size() * 8 + 16));
  if (!drops.empty()) {
    LS_CK(cudaMemcpyAsync(ctx->drop_keys.p, drops.data(), drops.size() * 8, cudaMemcpyHostToDevice, st));
    LS_CK(cudaStreamSynchronize(st));  // the copy reads `drops`
  }
  return LS_OK;
}
