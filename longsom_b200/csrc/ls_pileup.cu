// K1: per-barcode base pileup for BaseCellCounter.
//
// Reference behaviour restated (not ported) from
//   workflow/scripts/SNVCalling/BaseCellCounter.py:182-320 (run_interval),
//   :152-180 (EasyReadPileup) and the htslib pileup engine behind
//   pysam.AlignmentFile.pileup (SURVEY.md Appendix A).
//
// Design (B200): the reference walks reference columns and, per column, a Python list of reads.  Here the unit of
// work is a TILE of LS_TILE reference positions, and the accumulation of a tile is shared-memory atomics of the CTAs
// that own it.  One run (DESIGN.md §4, K1):
//   1. seg_build_kernel (ls_segments.cuh): one Segment per (read, tile) pair with a pileup entry, plus its Pieces.
//   2. radix sort of the segments by (tile, cell); the sorted segments become the S / M / U unit streams (ls_count.cuh).
//   3. pileup_count_kernel: a CTA per part of a tile, a lane per unit; the site epilogue applies the reference's gates.
//   4. compact_sites_kernel: the passing sites in the reference's output order.
#include <cstddef>
#include <cstdlib>

#include "ls_common.cuh"

#ifndef LS_TILE
#define LS_TILE 512
#endif

#include "ls_segments.cuh"

// tile boundaries in the sorted key array
__global__ void __launch_bounds__(256) slot_fill_kernel(const uint64_t *__restrict__ keys, int64_t n, int cell_bits,
                                                        const uint32_t *__restrict__ flag,
                                                        const uint32_t *__restrict__ rank, int64_t n_slots,
                                                        int64_t *__restrict__ slot_tile, uint32_t *__restrict__ slot_lo) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) slot_lo[n_slots] = (uint32_t)n;
  if (i >= n) return;
  if (flag[i]) {
    uint32_t s = rank[i];
    slot_tile[s] = (int64_t)(keys[i] >> cell_bits);
    slot_lo[s] = (uint32_t)i;
  }
}

#include "ls_count.cuh"

// ---- compaction of passing sites (fetch path) -----------------------------------------------
struct CompactArgs {
  const SlotDesc *slot_desc;
  const uint32_t *slot_off, *slot_lo;
  const uint32_t *out, *mask;
  const uint8_t *ref;
  int32_t *o_tid, *o_pos;
  uint8_t *o_ref;
  uint32_t *o_counts;
};

static_assert(LS_SITE_WORDS % 2 == 0, "records are copied as 8-byte pairs");

__global__ void __launch_bounds__(256) compact_sites_kernel(CompactArgs a) {
  __shared__ uint16_t list[LS_TILE];
  __shared__ uint32_t words[LS_TILE / 32];
  __shared__ uint32_t wpre[LS_TILE / 32 + 1];
  const int64_t slot = blockIdx.x;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x < 32) {  // pass mask of the tile's 16 windows -> exclusive prefix of their counts
    const uint32_t wd = lane < LS_TILE / 32 ? a.mask[(size_t)slot * (LS_TILE / 32) + lane] : 0u;
    uint32_t inc = (uint32_t)__popc(wd);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane < LS_TILE / 32) {
      words[lane] = wd;
      wpre[lane] = inc - (uint32_t)__popc(wd);
    }
    if (lane == LS_TILE / 32 - 1) wpre[LS_TILE / 32] = inc;
  }
  __syncthreads();
  const uint32_t np = wpre[LS_TILE / 32];
  if (np == 0) return;
  const SlotDesc sd = a.slot_desc[slot];
  const uint32_t off = a.slot_off[slot];
  const bool multi = a.slot_lo[slot + 1] - a.slot_lo[slot] > (uint32_t)K1_PART_SEGS;
  for (int s = threadIdx.x; s < LS_TILE; s += blockDim.x) {
    uint32_t wd = words[s >> 5];
    if ((wd >> (s & 31)) & 1u) {
      uint32_t rk = wpre[s >> 5] + __popc(wd & ((1u << (s & 31)) - 1u));
      if (multi) list[rk] = (uint16_t)s;
      a.o_tid[off + rk] = sd.tid;
      a.o_pos[off + rk] = sd.tile_start + s;
      a.o_ref[off + rk] = upper_ascii(a.ref[sd.ref_base + s]);
    }
  }
  const uint32_t *src = a.out + (size_t)slot * LS_SITE_WORDS * LS_TILE;
  uint32_t *dst = a.o_counts + (size_t)off * LS_SITE_WORDS;
  if (multi) {
    // multi-part tile: field-major words of every column
    __syncthreads();
    for (uint32_t e = threadIdx.x; e < np * LS_SITE_WORDS; e += blockDim.x) {
      uint32_t rk = e / LS_SITE_WORDS, f = e - rk * LS_SITE_WORDS;
      dst[e] = src[f * LS_TILE + list[rk]];
    }
  } else {
    // single-part tile: finished records, the passing ones packed at the front of each window's 32-record block
    // -> one contiguous run of words per window, copied by one warp
    for (int g = threadIdx.x >> 5; g < LS_TILE / 32; g += blockDim.x >> 5) {
      // 26 words = 13 eight-byte pairs per record; four loads in flight per lane
      const uint32_t n2 = (wpre[g + 1] - wpre[g]) * (LS_SITE_WORDS / 2);
      const uint2 *sg = reinterpret_cast<const uint2 *>(src + g * (32 * LS_SITE_WORDS));
      uint2 *dg = reinterpret_cast<uint2 *>(dst + wpre[g] * LS_SITE_WORDS);
      for (uint32_t i = lane; i < n2; i += 128u) {
        uint2 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (i + 32u * k < n2) v[k] = __ldcs(sg + i + 32u * k);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (i + 32u * k < n2) dg[i + 32u * k] = v[k];
      }
    }
  }
}

static int enqueue_compact(ls_ctx *ctx, int64_t ns);

// ---- host-side orchestration ------------------------------------------------------------------
static SegArgs make_seg_args(ls_ctx *ctx, const ls_count_params &p, bool emit_uncounted) {
  SegArgs a;
  a.n_reads = ctx->n_reads;
  a.tid = ctx->tid.as<int32_t>();
  a.pos = ctx->pos.as<int32_t>();
  a.cell = ctx->cell.as<int32_t>();
  a.flag = ctx->flag.as<uint16_t>();
  a.mapq = ctx->mapq.as<uint8_t>();
  a.cigar_off = ctx->cigar_off.as<uint32_t>();
  a.cigar = ctx->cigar.as<uint32_t>();
  a.base_off = ctx->base_off.as<uint64_t>();
  a.lq = ctx->lq.as<int32_t>();
  a.n_windows = ctx->n_windows;
  a.wtid = ctx->wtid.as<int32_t>();
  a.wstart = ctx->wstart.as<int32_t>();
  a.wend = ctx->wend.as<int32_t>();
  a.wtile_base = ctx->wtile_base.as<int64_t>();
  a.min_mq = p.min_mq;
  a.cell_bits = ctx->cell_bits;
  a.emit_uncounted = emit_uncounted ? 1 : 0;
  a.uncounted_key = (uint32_t)(ctx->max_cell + 1);
  a.drop_keys = ctx->drop_keys.as<uint64_t>();
  a.n_drop = ctx->n_drop;
  return a;
}

int ls_tile_size(void) { return LS_TILE; }
extern "C" int ls_pileup_tile_size(void) { return LS_TILE; }

static int read_counters(ls_ctx *ctx, const RunCounters *d, RunCounters &h) {
  LS_CK(cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  return LS_OK;
}

// Phase 1: one Segment per (read, tile) pair and its Pieces.  Their numbers are only known after the walk: a cold run
// starts from the previous run's sizes (or an estimate), reads the counters back into h and relaunches with exact
// sizes if the reservations ran past the buffers, or without the (window, read) pairs the depth cap drops.  A replay
// sizes the builder from h (the snapshot) and has no relaunch.
static int build_segments(ls_ctx *ctx, const ls_count_params &p, bool replay, RunCounters *d, RunCounters &h,
                          int &launches) {
  const int64_t n = ctx->n_reads;
  if (n == 0 || ctx->n_windows == 0) return LS_OK;
  cudaStream_t st = ctx->stream;
  ctx->n_drop = 0;
  SegArgs sa = make_seg_args(ctx, p, p.min_ac > 0);
  // the depth cap can only fire in a window that fetches more than max_depth records (replay: known not to fire)
  bool want_wcount = !replay && p.max_depth > 0 && n > (int64_t)p.max_depth;
  if (want_wcount) {
    LS_CK(ctx->rend.ensure((size_t)n * 4));
    LS_CK(ctx->wcount.ensure((size_t)ctx->n_windows * 4));
    LS_CK(cudaMemsetAsync(ctx->wcount.p, 0, (size_t)ctx->n_windows * 4, st));
  }
  uint64_t seg_need = replay ? h.n_segments : (ctx->n_segments > 0 ? (uint64_t)ctx->n_segments : (uint64_t)n * 5 + 1024);
  uint64_t piece_need =
      replay ? h.n_pieces : (ctx->n_pieces > 0 ? (uint64_t)ctx->n_pieces : (uint64_t)ctx->n_cigar + seg_need);
  for (int attempt = 0;; ++attempt) {
    LS_CK(ctx->segs.ensure((size_t)seg_need * sizeof(Segment)));
    LS_CK(ctx->pieces.ensure((size_t)piece_need * sizeof(Piece)));
    LS_CK(ctx->keys_a.ensure((size_t)seg_need * 8));
    LS_CK(ctx->keys_b.ensure((size_t)seg_need * 8));
    LS_CK(ctx->vals_a.ensure((size_t)seg_need * 4));
    LS_CK(ctx->vals_b.ensure((size_t)seg_need * 4));
    seg_build_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        sa, ctx->segs.as<Segment>(), ctx->keys_a.as<uint64_t>(), ctx->pieces.as<Piece>(), seg_need, piece_need,
        &d->n_segments, &d->n_aligned, want_wcount ? ctx->rend.as<int32_t>() : nullptr,
        want_wcount ? ctx->wcount.as<uint32_t>() : nullptr, (uint32_t)p.max_depth, &d->cap_flag);
    ++launches;
    LS_CK(cudaGetLastError());
    if (replay) return LS_OK;
    int rc = read_counters(ctx, d, h);
    if (rc != LS_OK) return rc;
    bool again = false;
    if (want_wcount && h.cap_flag) {  // some window fetches more than max_depth records
      rc = ls_depth_cap_host(ctx, ctx->h_wtid, ctx->h_wstart, ctx->h_wend, ctx->wcount.as<uint32_t>(), p.min_mq,
                             p.max_depth);
      if (rc != LS_OK) return rc;
      if (ctx->n_drop > 0) {  // redo the walk without the dropped (window, read) pairs
        sa = make_seg_args(ctx, p, p.min_ac > 0);
        again = true;
      }
    }
    want_wcount = false;
    if (!again && (h.n_segments > seg_need || h.n_pieces > piece_need)) {
      seg_need = h.n_segments > seg_need ? h.n_segments : seg_need;
      piece_need = h.n_pieces > piece_need ? h.n_pieces : piece_need;
      again = true;
    }
    if (!again) return LS_OK;
    if (attempt >= 3) LS_FAIL(LS_E_STATE, "ls_pileup_run: segment builder did not converge");
    LS_CK(cudaMemsetAsync(&d->n_aligned, 0, sizeof d->n_aligned, st));
    LS_CK(cudaMemsetAsync(&d->n_segments, 0, 3 * sizeof d->n_segments, st));
  }
}

// Phase 2: the segments sorted by (tile, cell), the slot ranks of the non-empty tiles, and the place of every segment
// in the unit streams (S: single segments, M: same-cell runs, U: uncounted reads).  The stream sizes go to the device
// counters; ea comes back set up for the expansion.
static int build_streams(ls_ctx *ctx, const ls_count_params &p, int64_t nseg, RunCounters *d, ExpandArgs &ea,
                         int &launches) {
  cudaStream_t st = ctx->stream;
  const int tile_bits = ls_bits_for((uint64_t)(ctx->n_tiles_total > 0 ? ctx->n_tiles_total - 1 : 0));
  LS_CK(cudaEventRecord(ctx->ev[1], st));
  LS_CK(ls_radix_sort_pairs(ctx->keys_a.as<uint64_t>(), ctx->keys_b.as<uint64_t>(), ctx->vals_a.as<uint32_t>(),
                            ctx->vals_b.as<uint32_t>(), nseg, tile_bits + ctx->cell_bits, ctx->rs_hist,
                            &ctx->sorted_keys, &ctx->sorted_vals, ctx->num_sms, st, &launches));
  LS_CK(ctx->tile_flag.ensure((size_t)nseg * 4));
  LS_CK(ctx->tile_rank.ensure((size_t)nseg * 4));
  const uint64_t cmask = (1ull << ctx->cell_bits) - 1ull;
  const uint64_t unc = (uint64_t)(uint32_t)(ctx->max_cell + 1);
  const bool with_u = p.min_ac > 0;
  LS_CK(ctx->offs_s.ensure((size_t)(nseg + 1) * 4));
  LS_CK(ctx->offs_m.ensure((size_t)(nseg + 1) * 4));
  LS_CK(ctx->goffs.ensure((size_t)(nseg + 1) * 4));
  LS_CK(ctx->mrank.ensure((size_t)(nseg + 1) * 4));
  LS_CK(ctx->mlist.ensure((size_t)(nseg + 1) * 4));
  if (with_u) LS_CK(ctx->offs_u.ensure((size_t)(nseg + 1) * 4));
  uint32_t *os = ctx->offs_s.as<uint32_t>(), *om = ctx->offs_m.as<uint32_t>(), *og = ctx->goffs.as<uint32_t>();
  uint32_t *ou = with_u ? ctx->offs_u.as<uint32_t>() : nullptr, *mr = ctx->mrank.as<uint32_t>();
  classify_kernel<<<(unsigned)((nseg + 1 + 255) / 256), 256, 0, st>>>(
      ctx->sorted_keys, ctx->sorted_vals, ctx->segs.as<Segment>(), nseg, cmask, unc, ctx->cell_bits, os, om, ou, mr,
      ctx->tile_flag.as<uint32_t>(), &d->long_run);
  ++launches;
  // slot ranks, S / M (/ U) stream offsets and run-member ranks: independent scans, one launch
  LsScanJob jobs[5];
  int nj = 0;
  jobs[nj++] = LsScanJob{ctx->tile_flag.as<uint32_t>(), ctx->tile_rank.as<uint32_t>(), nseg, &d->n_slots};
  jobs[nj++] = LsScanJob{os, os, nseg + 1, &d->tot_s};
  jobs[nj++] = LsScanJob{om, om, nseg + 1, &d->tot_m};
  jobs[nj++] = LsScanJob{mr, mr, nseg + 1, &d->n_members};
  if (with_u) jobs[nj++] = LsScanJob{ou, ou, nseg + 1, &d->tot_u};
  LS_CK(ls_scan_exclusive_u32_multi(jobs, nj, ctx->scan_tmp, st));
  ++launches;
  mlist_kernel<<<(unsigned)((nseg + 255) / 256), 256, 0, st>>>(ctx->sorted_keys, nseg, cmask, unc, mr,
                                                               ctx->mlist.as<uint32_t>());
  ++launches;
  ea.keys = ctx->sorted_keys;
  ea.vals = ctx->sorted_vals;
  ea.segs = ctx->segs.as<Segment>();
  ea.pieces = ctx->pieces.as<Piece>();
  ea.n = nseg;
  ea.cmask = cmask;
  ea.unc = unc;
  ea.offs_s = os;
  ea.offs_m = om;
  ea.offs_u = ou;
  ea.tot_s = &d->tot_s;
  ea.tot_m = &d->tot_m;
  ea.tot_g = &d->n_groups;
  ea.tot_ms = &d->n_members;
  ea.mlist = ctx->mlist.as<uint32_t>();
  ea.goffs = og;
  ea.gdir = nullptr;
  ea.units = nullptr;
  // one warp per 32 run members; the grid covers the worst case (every segment a run member)
  LS_CK(cudaMemsetAsync(og, 0, (size_t)(nseg + 1) * 4, st));
  rungroups_kernel<<<(unsigned)((nseg + 255) / 256), 256, 0, st>>>(ea);
  ++launches;
  LS_CK(ls_scan_exclusive_u32(og, og, nseg + 1, &d->n_groups, ctx->scan_tmp, st));
  launches += 1;
  LS_CK(cudaGetLastError());
  return LS_OK;
}

// Phase 3: the units written into their streams, the tiles split into parts, the count kernel, and the scan of the
// per-slot pass counts that places every tile's passing sites in the output (its total goes to n_sites).  Sized by h,
// the counters of the middle read-back.
static int count_tiles(ls_ctx *ctx, const ls_count_params &p, int64_t nseg, const RunCounters &h, RunCounters *d,
                       ExpandArgs ea, int &launches) {
  cudaStream_t st = ctx->stream;
  const int64_t n_slots = (int64_t)h.n_slots;
  const bool with_u = p.min_ac > 0;
  LS_CK(ctx->slot_tile.ensure((size_t)n_slots * 8));
  LS_CK(ctx->slot_lo.ensure((size_t)(n_slots + 1) * 4));
  slot_fill_kernel<<<(unsigned)((nseg + 255) / 256), 256, 0, st>>>(
      ctx->sorted_keys, nseg, ctx->cell_bits, ctx->tile_flag.as<uint32_t>(), ctx->tile_rank.as<uint32_t>(), n_slots,
      ctx->slot_tile.as<int64_t>(), ctx->slot_lo.as<uint32_t>());
  ++launches;
  LS_CK(ctx->units.ensure((size_t)(h.n_units + 1) * 8));
  LS_CK(ctx->gdir.ensure((size_t)(h.n_groups + 1) * 4));
  ea.gdir = ctx->gdir.as<uint32_t>();
  ea.units = ctx->units.as<uint2>();
  expand_single_kernel<<<(unsigned)((nseg + 255) / 256), 256, 0, st>>>(ea);
  if (h.n_members > 0) expand_runs_kernel<<<(unsigned)((h.n_members + 255) / 256), 256, 0, st>>>(ea);
  launches += 2;
  LS_CK(cudaGetLastError());
  LS_CK(cudaEventRecord(ctx->ev[2], st));

  LS_CK(ctx->slot_out.ensure((size_t)n_slots * LS_SITE_WORDS * LS_TILE * 4));
  LS_CK(ctx->slot_mask.ensure((size_t)n_slots * (LS_TILE / 32) * 4));
  LS_CK(ctx->slot_npass.ensure((size_t)n_slots * 4));
  LS_CK(ctx->slot_off.ensure((size_t)n_slots * 4));
  const int64_t max_parts = n_slots + nseg / K1_PART_SEGS + 1;
  LS_CK(ctx->part_slot.ensure((size_t)max_parts * sizeof(PartDesc)));
  LS_CK(ctx->slot_done.ensure((size_t)n_slots * 4));
  LS_CK(ctx->slot_desc.ensure((size_t)n_slots * sizeof(SlotDesc)));
  if (with_u) LS_CK(ctx->acbuf.ensure((size_t)n_slots * LS_TILE * 4));
  LS_CK(cudaMemsetAsync(ctx->part_slot.p, 0xff, (size_t)max_parts * sizeof(PartDesc), st));
  PartBuildArgs pb;
  pb.slot_lo = ctx->slot_lo.as<uint32_t>();
  pb.slot_tile = ctx->slot_tile.as<int64_t>();
  pb.n_slots = n_slots;
  pb.keys = ctx->sorted_keys;
  pb.offs_s = ctx->offs_s.as<uint32_t>();
  pb.offs_u = with_u ? ctx->offs_u.as<uint32_t>() : nullptr;
  pb.goffs = ctx->goffs.as<uint32_t>();
  pb.n_windows = ctx->n_windows;
  pb.wstart = ctx->wstart.as<int32_t>();
  pb.wend = ctx->wend.as<int32_t>();
  pb.wtile_base = ctx->wtile_base.as<int64_t>();
  pb.wref_off = ctx->wref_off.as<uint64_t>();
  pb.parts = ctx->part_slot.as<PartDesc>();
  pb.slot_desc = ctx->slot_desc.as<SlotDesc>();
  pb.wtid = ctx->wtid.as<int32_t>();
  pb.slot_done = ctx->slot_done.as<uint32_t>();
  pb.n_parts = &d->n_parts;
  pb.n_light = &d->n_light;
  pb.max_parts = (uint32_t)max_parts;
  pb.out = ctx->slot_out.as<uint32_t>();
  pb.acbuf = with_u ? ctx->acbuf.as<uint32_t>() : nullptr;
  part_build_kernel<<<(unsigned)n_slots, 128, 0, st>>>(pb);
  ++launches;
  CountArgs ca;
  ca.parts = ctx->part_slot.as<PartDesc>();
  ca.slot_done = ctx->slot_done.as<uint32_t>();
  ca.acbuf = with_u ? ctx->acbuf.as<uint32_t>() : nullptr;
  ca.units = ctx->units.as<uint2>();
  ca.with_u = with_u ? 1 : 0;
  ca.tot_s = &d->tot_s;
  ca.tot_m = &d->tot_m;
  ca.gdir = ctx->gdir.as<uint32_t>();
  ca.seq4 = ctx->seq4_d();
  ca.qual = ctx->qual_d();
  ca.ref = ctx->ref.as<uint8_t>();
  ca.out = ctx->slot_out.as<uint32_t>();
  ca.mask = ctx->slot_mask.as<uint32_t>();
  ca.npass = ctx->slot_npass.as<uint32_t>();
  ca.n_events = &d->n_events;
  ca.cell_bits = ctx->cell_bits;
  ca.uncounted_key = (uint32_t)(ctx->max_cell + 1);
  ca.min_bq = p.min_bq;
  ca.min_dp = p.min_dp;
  ca.min_cc = p.min_cc;
  ca.min_ac = p.min_ac;
  // shared memory per CTA: the acx row sits last and is only allocated with --min_ac > 0
  const size_t sm_p = with_u ? sizeof(TileSmemT<true>) : offsetof(TileSmemT<true>, acx);
  const size_t sm_u = with_u ? sizeof(TileSmemT<false>) : offsetof(TileSmemT<false>, acx);
  if (!ctx->k1_attr_set) {
    LS_CK(cudaFuncSetAttribute(pileup_count_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)sizeof(TileSmemT<true>)));
    LS_CK(cudaFuncSetAttribute(pileup_count_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int)sizeof(TileSmemT<false>)));
    ctx->k1_attr_set = true;
  }
  // 12-bit packed counters unless some cell has > K1_MAX_RUN_PACKED reads in one tile
  const bool packed = h.long_run == 0;
  ca.cnt1 = packed ? (1u << K1_CNT_SHIFT) : 0u;
  if (packed)
    pileup_count_kernel<true><<<(unsigned)max_parts, K1_THREADS, sm_p, st>>>(ca);
  else
    pileup_count_kernel<false><<<(unsigned)max_parts, K1_THREADS, sm_u, st>>>(ca);
  ++launches;
  LS_CK(cudaGetLastError());
  LS_CK(cudaEventRecord(ctx->ev[3], st));
  LS_CK(ls_scan_exclusive_u32(ctx->slot_npass.as<uint32_t>(), ctx->slot_off.as<uint32_t>(), n_slots, &d->n_sites,
                              ctx->scan_tmp, st));
  launches += 1;
  LS_CK(cudaEventRecord(ctx->ev[4], st));
  return LS_OK;
}

// What the device produced in a replayed run against the snapshot its enqueued sizes came from
static bool replay_matches(const ReplaySnapshot &s, const RunCounters &h, bool pre_compacted) {
  const RunCounters &m = s.mid;
  return h.n_aligned == m.n_aligned && h.n_slots == m.n_slots && h.long_run == m.long_run &&
         h.n_segments == m.n_segments && h.n_pieces == m.n_pieces && h.n_units == m.n_units && h.tot_s == m.tot_s &&
         h.tot_m == m.tot_m && h.tot_u == m.tot_u && h.n_groups == m.n_groups && h.n_members == m.n_members &&
         (!pre_compacted || (int64_t)h.n_sites == s.n_sites);
}

extern "C" int ls_pileup_run(ls_ctx *ctx, const ls_count_params *params, int64_t *n_sites, ls_run_stats *stats) {
  if (!ctx) return LS_E_ARG;
  if (!params) LS_FAIL(LS_E_ARG, "ls_pileup_run: params is null");
  if (!ctx->have_batch) LS_FAIL(LS_E_STATE, "ls_pileup_run: no batch uploaded");
  if (params->min_dp < 1) LS_FAIL(LS_E_ARG, "ls_pileup_run: min_dp must be >= 1");
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  ctx->params = *params;
  ctx->have_run = false;
  ctx->compacted = false;
  ctx->ct.loaded = false;
  ls_run_stats S;
  memset(&S, 0, sizeof S);
  int launches = 0;
  // Replay: a run on the SAME uploaded batch with the SAME parameters has the same intermediate sizes as the last one
  // (the pipeline is deterministic), so the two size read-backs in the middle are skipped and everything is enqueued
  // at once; the sizes are verified against the device counters with the final read-back, and the run is repeated
  // with read-backs if they ever differ.
  const bool replay =
      ctx->replay.valid && memcmp(&ctx->replay.params, params, sizeof *params) == 0 && !getenv("LS_NO_REPLAY");
  // A run that is not a replay overwrites the sizes the next run starts from (n_segments, n_pieces), so the snapshot
  // only survives it if the run refreshes it below.
  if (!replay) ctx->replay.valid = false;
  ctx->cell_bits = ls_bits_for((uint64_t)(ctx->max_cell + 1));

  LS_CK(ctx->counters.ensure(sizeof(RunCounters)));
  RunCounters *d = ctx->counters.as<RunCounters>();
  LS_CK(cudaMemsetAsync(d, 0, sizeof *d, st));
  LS_CK(cudaEventRecord(ctx->ev[0], st));
  // host copy of the counters: a cold run reads them back after the builder, in the middle and at the end; a replay
  // takes the middle read-back of the snapshot and reads back only at the end
  RunCounters h = replay ? ctx->replay.mid : RunCounters{};
  int rc = build_segments(ctx, *params, replay, d, h, launches);
  if (rc != LS_OK) return rc;
  const int64_t nseg = (int64_t)h.n_segments;
  if (nseg >= (int64_t)0xffffffffll || h.n_pieces >= 0xffffffffull || h.n_units >= 0xffffffffull)
    LS_FAIL(LS_E_ARG, "ls_pileup_run: more than 2^32 segments, pieces or units in one batch");
  S.n_aligned = (int64_t)h.n_aligned;
  S.n_segments = nseg;
  ctx->n_segments = nseg;
  ctx->n_pieces = (int64_t)h.n_pieces;
  int64_t n_slots = 0;
  if (nseg > 0) {
    ExpandArgs ea;
    rc = build_streams(ctx, *params, nseg, d, ea, launches);
    if (rc != LS_OK) return rc;
    if (!replay) {
      rc = read_counters(ctx, d, h);
      if (rc != LS_OK) return rc;
    }
    const RunCounters mid = h;
    n_slots = (int64_t)mid.n_slots;
    rc = count_tiles(ctx, *params, nseg, mid, d, ea, launches);
    if (rc != LS_OK) return rc;
    // a replayed run knows how many sites will pass: the compaction goes into the same submission, one synchronisation
    // per step instead of two
    const bool pre_compacted = replay && ctx->replay.n_sites > 0;
    if (pre_compacted) {
      ctx->n_slots = n_slots;
      rc = enqueue_compact(ctx, ctx->replay.n_sites);
      if (rc != LS_OK) return rc;
    }
    rc = read_counters(ctx, d, h);
    if (rc != LS_OK) return rc;
    if (replay) {
      if (!replay_matches(ctx->replay, h, pre_compacted)) {
        ctx->replay.valid = false;
        return ls_pileup_run(ctx, params, n_sites, stats);
      }
    } else if (ctx->n_drop == 0 && mid.cap_flag == 0) {  // a replay skips the depth cap: only a run it spared qualifies
      ctx->replay.valid = true;
      ctx->replay.params = *params;
      ctx->replay.mid = mid;
      ctx->replay.n_sites = (int64_t)h.n_sites;
    }
    ctx->n_sites = (int64_t)h.n_sites;
    if (pre_compacted) {
      ctx->compacted = true;
      LS_CK(cudaEventElapsedTime(&S.ms_compact, ctx->ev[5], ctx->ev[6]));  // (the caller counts this launch)
    }
    S.n_events = (int64_t)h.n_events;
    LS_CK(cudaEventElapsedTime(&S.ms_segments, ctx->ev[0], ctx->ev[1]));
    LS_CK(cudaEventElapsedTime(&S.ms_sort, ctx->ev[1], ctx->ev[2]));
    LS_CK(cudaEventElapsedTime(&S.ms_count, ctx->ev[2], ctx->ev[3]));
    LS_CK(cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[4]));
  } else {
    ctx->n_sites = 0;
  }
  ctx->n_slots = n_slots;
  S.n_tiles = n_slots;
  S.count_launches = launches;
  ctx->stats = S;
  ctx->have_run = true;
  if (n_sites) *n_sites = ctx->n_sites;
  if (stats) *stats = S;
  return LS_OK;
}

// Compaction of the passing sites into the reference's output order (window, position): device only.  The site table
// of a run is tile-major with a pass bitmask; this is the step that turns it into the unit the reference emits.
static int enqueue_compact(ls_ctx *ctx, int64_t ns) {
  cudaStream_t st = ctx->stream;
  LS_CK(ctx->out_tid.ensure((size_t)ns * 4));
  LS_CK(ctx->out_pos.ensure((size_t)ns * 4));
  LS_CK(ctx->out_ref.ensure((size_t)ns));
  LS_CK(ctx->out_counts.ensure((size_t)ns * LS_SITE_WORDS * 4));
  CompactArgs a;
  a.slot_desc = ctx->slot_desc.as<SlotDesc>();
  a.slot_off = ctx->slot_off.as<uint32_t>();
  a.slot_lo = ctx->slot_lo.as<uint32_t>();
  a.out = ctx->slot_out.as<uint32_t>();
  a.mask = ctx->slot_mask.as<uint32_t>();
  a.ref = ctx->ref.as<uint8_t>();
  a.o_tid = ctx->out_tid.as<int32_t>();
  a.o_pos = ctx->out_pos.as<int32_t>();
  a.o_ref = ctx->out_ref.as<uint8_t>();
  a.o_counts = ctx->out_counts.as<uint32_t>();
  LS_CK(cudaEventRecord(ctx->ev[5], st));
  compact_sites_kernel<<<(unsigned)ctx->n_slots, 256, 0, st>>>(a);
  LS_CK(cudaGetLastError());
  LS_CK(cudaEventRecord(ctx->ev[6], st));
  return LS_OK;
}

extern "C" int ls_pileup_compact(ls_ctx *ctx, ls_run_stats *stats) {
  if (!ctx) return LS_E_ARG;
  if (!ctx->have_run) LS_FAIL(LS_E_STATE, "ls_pileup_compact: ls_pileup_run has not completed");
  if (!ctx->compacted && ctx->n_sites > 0) {  // (a replayed run has already done it: see ls_pileup_run)
    LS_CK(cudaSetDevice(ctx->device));
    const int rc = enqueue_compact(ctx, ctx->n_sites);
    if (rc != LS_OK) return rc;
    LS_CK(cudaStreamSynchronize(ctx->stream));
    LS_CK(cudaEventElapsedTime(&ctx->stats.ms_compact, ctx->ev[5], ctx->ev[6]));
  }
  ctx->compacted = true;
  if (stats) *stats = ctx->stats;
  return LS_OK;
}

extern "C" int ls_pileup_fetch(ls_ctx *ctx, ls_site_counts *out) {
  if (!ctx) return LS_E_ARG;
  if (!out) LS_FAIL(LS_E_ARG, "ls_pileup_fetch: out is null");
  if (!ctx->have_run) LS_FAIL(LS_E_STATE, "ls_pileup_fetch: ls_pileup_run has not completed");
  out->n_sites = ctx->n_sites;
  if (ctx->n_sites == 0) return LS_OK;
  if (out->capacity < ctx->n_sites) LS_FAIL(LS_E_CAPACITY, "ls_pileup_fetch: capacity < n_sites");
  if (!out->tid || !out->pos || !out->ref || !out->counts) LS_FAIL(LS_E_ARG, "ls_pileup_fetch: null output array");
  int rc = ls_pileup_compact(ctx, nullptr);
  if (rc != LS_OK) return rc;
  cudaStream_t st = ctx->stream;
  const int64_t ns = ctx->n_sites;
  LS_CK(cudaMemcpyAsync(out->tid, ctx->out_tid.p, (size_t)ns * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->pos, ctx->out_pos.p, (size_t)ns * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->ref, ctx->out_ref.p, (size_t)ns, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->counts, ctx->out_counts.p, (size_t)ns * LS_SITE_WORDS * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  return LS_OK;
}

extern "C" int ls_pileup_count(ls_ctx *ctx, const ls_read_batch *batch, const ls_windows *windows,
                               const ls_count_params *params, ls_site_counts *out, ls_run_stats *stats) {
  int rc = ls_pileup_upload(ctx, batch, windows);
  if (rc != LS_OK) return rc;
  int64_t ns = 0;
  rc = ls_pileup_run(ctx, params, &ns, stats);
  if (rc != LS_OK) return rc;
  rc = ls_pileup_fetch(ctx, out);
  if (stats) stats->ms_compact = ctx->stats.ms_compact;
  return rc;
}
