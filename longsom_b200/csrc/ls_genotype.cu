// K1': pileup at candidate sites, per (site, cell) Dp / Alt.
//
// Replaces the pileup loop of SingleCellGenotype.run_interval (SingleCellGenotype.py:114-178)
// and HCCVSingleCellGenotype.run_interval (:112-176): for every candidate site, every read
// entry whose class is in {A,C,T,G,I,D,N} (--alt_flag All) or equals ALT_expected
// (--alt_flag Alt), whose barcode is in --meta, and that is not secondary / duplicate /
// supplementary, adds 1 to Dp[site, cell] and, if its class equals ALT_expected, to Alt.
//
// Design: candidate sites are sparse (<= 2e5) while reads are dense, so the scan is
// read-major: one thread walks one read's CIGAR, binary-searches the sorted site table for
// sites inside each reference-consuming op and either scatters with global atomics into the
// dense [site][cell] tensors (ls_genotype_count; one int32 add per hit, and hits are ~depth x
// sites, tiny next to HBM) or writes one key per hit, which a sort reduces to the touched
// (site, cell) pairs (ls_genotype_sparse_run).
// Bases that cover no candidate site are never loaded.
#include <type_traits>

#include "ls_common.cuh"

struct GenoArgs {
  int64_t n_reads;
  const int32_t *tid, *pos, *cell, *lq;
  const uint16_t *flag;
  const uint8_t *mapq;
  const uint32_t *cigar_off, *cigar;
  const uint64_t *base_off;
  const uint8_t *seq4, *qual;
  const uint64_t *site_key;  // tid<<32 | pos, sorted
  const uint8_t *alt_class;
  const uint32_t *site_bin;  // index of the pileup() call (50 kb bin) of each site
  int64_t n_sites;
  int32_t n_cells;
  int min_bq, min_mq, alt_only;
  const uint64_t *drop_keys;  // (bin<<32 | read) removed by the depth cap
  int64_t n_drop;
  int32_t *dp, *alt;            // dense [site][cell] tensors (genotype_kernel<void>), else null
  const uint32_t *hit_off;      // first hit slot of every read (exclusive scan of its candidate sites)
  void *hits;                   // hit keys: (site * n_cells + cell) << 1 | (class == ALT_expected)
  uint64_t sentinel;            // key of an unused slot (n_sites * n_cells * 2: behind every real key)
  unsigned long long *n_events;
};

// first index i of the sorted keys[0, n) with keys[i] >= key
__device__ __forceinline__ int64_t lower_key(const uint64_t *__restrict__ keys, int64_t n, uint64_t key) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t m = (lo + hi) >> 1;
    if (keys[m] < key)
      lo = m + 1;
    else
      hi = m;
  }
  return lo;
}

__device__ __forceinline__ bool geno_dropped(const GenoArgs &a, uint32_t bin, uint32_t r) {
  if (a.n_drop == 0) return false;
  const uint64_t key = ((uint64_t)bin << 32) | r;
  const int64_t i = lower_key(a.drop_keys, a.n_drop, key);
  return i < a.n_drop && a.drop_keys[i] == key;
}

// K = void: dense atomics into dp / alt.  K = uint32_t / uint64_t: the read's hits as keys of that width at its slots,
// and the sentinel in the slots it does not use.
template <typename K>
__global__ void __launch_bounds__(256) genotype_kernel(GenoArgs a) {
  constexpr bool DENSE = std::is_void<K>::value;
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long nev = 0;
  if (r < a.n_reads) {
    K *hp = nullptr;
    if constexpr (!DENSE) hp = static_cast<K *>(a.hits) + a.hit_off[r];
    const uint32_t flag = a.flag[r];
    const int32_t cell = a.cell[r];
    const int32_t tid = a.tid[r];
    if (tid >= 0 && read_passes_engine(flag, a.mapq[r], a.min_mq) && !(flag & LS_FLAG_SUPPL) && cell >= 0 &&
        cell < a.n_cells) {
      const uint32_t k0 = a.cigar_off[r], kend = a.cigar_off[r + 1];
      int32_t x = a.pos[r];
      uint32_t y = 0;
      const uint64_t boff = a.base_off[r];
      const uint32_t lq = (uint32_t)a.lq[r];
      int64_t s = lower_key(a.site_key, a.n_sites, ((uint64_t)(uint32_t)tid << 32) | (uint32_t)x);
      for (uint32_t k = k0; k < kend && s < a.n_sites; ++k) {
        const uint32_t c = a.cigar[k];
        const uint32_t op = c & 15u;
        const int32_t len = (int32_t)(c >> 4);
        const bool match = op_is_match(op);
        if ((match || op == OP_D || op == OP_N) && len > 0) {
          const uint64_t kend_key = ((uint64_t)(uint32_t)tid << 32) | (uint32_t)(x + len);
          while (s < a.n_sites && a.site_key[s] < kend_key) {
            const int32_t sp = (int32_t)(a.site_key[s] & 0xffffffffu);
            // site_key[s] >= (tid, x) holds because s only moves forward with x
            const int32_t j = sp - x;
            const uint32_t qpos = match ? y + (uint32_t)j : y;
            const uint32_t q = qpos < lq ? a.qual[boff + qpos] : 0u;
            if ((int)q >= a.min_bq && !geno_dropped(a, a.site_bin[s], (uint32_t)r)) {
              int ind = (j == len - 1) ? indel_after(a.cigar, k, kend, op) : 0;
              int cls;
              if (ind < 0)
                cls = LS_CLASS_D;
              else if (ind > 0)
                cls = LS_CLASS_I;
              else if (match) {
                uint32_t code = 15u;
                if (qpos < lq) {
                  uint32_t bb = a.seq4[(boff + qpos) >> 1];
                  code = (qpos & 1u) ? (bb >> 4) : (bb & 15u);  // device copy is nibble-swapped (ls_ctx::seq4_d)
                }
                cls = class_of_code(code);
              } else
                cls = (op == OP_D) ? LS_CLASS_O : LS_CLASS_NA;
              const int ac = a.alt_class[s];
              const bool use = a.alt_only ? (cls == ac && cls != LS_CLASS_NA) : (cls != LS_CLASS_NA && cls != LS_CLASS_O);
              if (use) {
                if constexpr (DENSE) {
                  atomicAdd(&a.dp[(size_t)s * a.n_cells + cell], 1);
                  if (cls == ac) atomicAdd(&a.alt[(size_t)s * a.n_cells + cell], 1);
                } else {
                  *hp++ = (((K)s * (K)a.n_cells + (K)cell) << 1) | (cls == ac ? 1u : 0u);
                }
                ++nev;
              }
            }
            ++s;
          }
        }
        if (match) {
          x += len;
          y += (uint32_t)len;
        } else if (op == OP_D || op == OP_N) {
          x += len;
        } else if (op == OP_I || op == OP_S) {
          y += (uint32_t)len;
        }
      }
    }
    if constexpr (!DENSE)
      for (K *e = static_cast<K *>(a.hits) + a.hit_off[r + 1]; hp < e; ++hp) *hp = (K)a.sentinel;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nev += __shfl_xor_sync(0xffffffffu, nev, o);
  if ((threadIdx.x & 31) == 0 && nev) atomicAdd(a.n_events, nev);
}

// ---- sparse output: sorted hits -> one (site, cell, Dp, Alt) tuple per touched pair ---------------------------
template <typename K>
__global__ void __launch_bounds__(256) hit_flag_kernel(const K *__restrict__ hits, int64_t n, K sentinel, uint32_t *__restrict__ flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  // unused slots carry the sentinel and sort behind every real key
  flag[i] = (i < n && hits[i] != sentinel && (i == 0 || (hits[i] >> 1) != (hits[i - 1] >> 1))) ? 1u : 0u;
}

template <typename K>
__global__ void __launch_bounds__(256) hit_reduce_kernel(const K *__restrict__ hits, int64_t n, K sentinel,
                                                         const uint32_t *__restrict__ rank, int32_t n_cells,
                                                         const uint8_t *__restrict__ skip_p, int32_t *__restrict__ t_site,
                                                         int32_t *__restrict__ t_cell, int32_t *__restrict__ t_dp,
                                                         int32_t *__restrict__ t_alt, int32_t *__restrict__ t_k) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (hits[i] == sentinel) return;  // an unused slot
  const uint64_t key = (uint64_t)(hits[i] >> 1);
  if (i > 0 && (uint64_t)(hits[i - 1] >> 1) == key) return;  // not the first hit of its pair
  int32_t dp = 0, alt = 0;
  for (int64_t j = i; j < n && hits[j] != sentinel && (uint64_t)(hits[j] >> 1) == key; ++j) {  // the hits of a pair are adjacent; the alt ones last
    ++dp;
    alt += (int32_t)(hits[j] & 1u);
  }
  const uint32_t t = rank[i];
  const int32_t site = (int32_t)(key / (uint64_t)n_cells);
  t_site[t] = site;
  t_cell[t] = (int32_t)(key - (uint64_t)site * (uint64_t)n_cells);
  t_dp[t] = dp;
  t_alt[t] = alt;
  // beta-binomial query of the pair: k = Alt (0: none needed -- no alt reads, or the site takes the chrM shortcut)
  t_k[t] = (skip_p && skip_p[site]) ? 0 : alt;
}

// read end (exclusive) per read, for the depth-cap pre-pass
__global__ void __launch_bounds__(256) read_end_kernel(int64_t n, const int32_t *__restrict__ pos,
                                                       const uint32_t *__restrict__ cigar_off,
                                                       const uint32_t *__restrict__ cigar, int32_t *__restrict__ rend) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  int32_t x = pos[r];
  for (uint32_t k = cigar_off[r]; k < cigar_off[r + 1]; ++k) {
    uint32_t op = cigar[k] & 15u;
    if (op_consumes_ref(op)) x += (int32_t)(cigar[k] >> 4);
  }
  rend[r] = x;
}

// Records each pileup() call (bin) would fetch.  Bins are disjoint and sorted by (tid, start).  A read can only be
// dropped in a bin that fetches more than max_depth records (the rule needs max_depth accepted reads alive), so
// the host pre-pass below is skipped unless the add that crosses the cap raises *over.
struct CandArgs {          // sparse path: slots per read = candidate sites inside [pos, reference end)
  const uint64_t *site_key;
  int64_t n_sites;
  const int32_t *cell;
  int32_t n_cells;
  uint32_t *cand_cnt;      // null: bin counts only
};

__global__ void __launch_bounds__(256) bin_fetch_count_kernel(int64_t n, const int32_t *__restrict__ tid,
                                                              const int32_t *__restrict__ pos,
                                                              const uint16_t *__restrict__ flag,
                                                              const uint8_t *__restrict__ mapq,
                                                              const uint32_t *__restrict__ cigar_off,
                                                              const uint32_t *__restrict__ cigar, int64_t n_bins,
                                                              const int32_t *__restrict__ btid,
                                                              const int32_t *__restrict__ bstart,
                                                              const int32_t *__restrict__ bend, int min_mq,
                                                              uint32_t max_depth, uint32_t *__restrict__ bincount,
                                                              uint32_t *__restrict__ over, CandArgs ca) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int32_t t = tid[r];
  uint32_t cand = 0;
  if (t >= 0 && read_passes_engine(flag[r], mapq[r], min_mq)) {
    const int32_t p = pos[r];
    int64_t lo = n_bins;
    if (n_bins > 0) {  // first bin with (btid, bend) > (t, p)
      int64_t hi = n_bins;
      lo = 0;
      while (lo < hi) {
        const int64_t m = (lo + hi) >> 1;
        const int32_t bt = btid[m];
        if (bt < t || (bt == t && bend[m] <= p))
          lo = m + 1;
        else
          hi = m;
      }
      if (lo < n_bins && btid[lo] != t) lo = n_bins;
    }
    const bool want_cand = ca.cand_cnt && !(flag[r] & LS_FLAG_SUPPL) && ca.cell[r] >= 0 && ca.cell[r] < ca.n_cells;
    if (lo < n_bins || want_cand) {
      int32_t x = p;
      for (uint32_t k = cigar_off[r]; k < cigar_off[r + 1]; ++k) {
        const uint32_t c = cigar[k];
        if (op_consumes_ref(c & 15u)) x += (int32_t)(c >> 4);
      }
      const int32_t e = x > p ? x : p + 1;
      for (int64_t b = lo; b < n_bins && btid[b] == t && bstart[b] < e; ++b) {
        const uint32_t old = atomicAdd(&bincount[b], 1u);
        if (old == max_depth) *over = 1u;
      }
      if (want_cand && x > p) {
        const uint64_t kt = (uint64_t)(uint32_t)t << 32;
        cand = (uint32_t)(lower_key(ca.site_key, ca.n_sites, kt | (uint32_t)x) - lower_key(ca.site_key, ca.n_sites, kt | (uint32_t)p));
      }
    }
  }
  if (ca.cand_cnt) ca.cand_cnt[r] = cand;
}

// Depth cap per pileup() call of the genotype scripts: one call per 50 kb bin of candidate sites
// over [min-1, max+1) (SingleCellGenotype.py:110-124); the rule is K1's (ls_depth_cap_host).
static int geno_depth_cap(ls_ctx *ctx, const std::vector<int32_t> &btid, const std::vector<int32_t> &bstart,
                          const std::vector<int32_t> &bend, int min_mq, int max_depth, CandArgs ca = CandArgs{}) {
  const int64_t n = ctx->n_reads;
  ctx->n_drop = 0;
  const bool cap_possible = max_depth > 0 && n > (int64_t)max_depth;
  if (!cap_possible && !ca.cand_cnt) return LS_OK;
  cudaStream_t st = ctx->stream;
  {  // device pre-count: does any bin fetch more than max_depth records at all?  (The same walk over the CIGARs gives
     // the sparse path its per-read slot counts.)
    const size_t nb = cap_possible ? btid.size() : 0;
    LS_CK(ctx->wcount.ensure(nb * 4 * 4 + 16));
    int32_t *d_bt = ctx->wcount.as<int32_t>(), *d_bs = d_bt + nb, *d_be = d_bs + nb;
    uint32_t *d_fetch = reinterpret_cast<uint32_t *>(d_be + nb), *d_over = d_fetch + nb;
    LS_CK(cudaMemcpyAsync(d_bt, btid.data(), nb * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(d_bs, bstart.data(), nb * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemcpyAsync(d_be, bend.data(), nb * 4, cudaMemcpyHostToDevice, st));
    LS_CK(cudaMemsetAsync(d_fetch, 0, nb * 4 + 4, st));
    bin_fetch_count_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        n, ctx->tid.as<int32_t>(), ctx->pos.as<int32_t>(), ctx->flag.as<uint16_t>(), ctx->mapq.as<uint8_t>(),
        ctx->cigar_off.as<uint32_t>(), ctx->cigar.as<uint32_t>(), (int64_t)nb, d_bt, d_bs, d_be, min_mq,
        (uint32_t)max_depth, d_fetch, d_over, ca);
    LS_CK(cudaGetLastError());
    if (!cap_possible) return LS_OK;
    uint32_t over = 0;
    LS_CK(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, st));
    LS_CK(cudaStreamSynchronize(st));
    if (!over) return LS_OK;
  }
  LS_CK(ctx->rend.ensure((size_t)n * 4));
  read_end_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, ctx->pos.as<int32_t>(), ctx->cigar_off.as<uint32_t>(),
                                                               ctx->cigar.as<uint32_t>(), ctx->rend.as<int32_t>());
  LS_CK(cudaGetLastError());
  // every bin is walked: one that fetches at most max_depth records drops nothing
  return ls_depth_cap_host(ctx, btid, bstart, bend, nullptr, min_mq, max_depth);
}

// Site table of a genotype call: sorted keys, the pileup() call (bin) of every site, and the bins.
struct GenoSites {
  std::vector<uint64_t> keys;
  std::vector<uint32_t> sbin;
  std::vector<int32_t> btid, bstart, bend;
};

// The checks both entry points begin with; `who` names the entry point in the errors.
static int geno_check(ls_ctx *ctx, const char *who, const ls_geno_params *params, int64_t n_sites, int32_t n_cells) {
  const std::string w = who;
  if (!params) LS_FAIL(LS_E_ARG, w + ": params is null");
  if (!ctx->have_batch) LS_FAIL(LS_E_STATE, w + ": no batch uploaded");
  if (n_sites < 0 || n_cells < 0) LS_FAIL(LS_E_ARG, w + ": negative size");
  return LS_OK;
}

// Site setup of both entry points: the site table goes to ctx->geno and the counters are zeroed.  g keeps the host
// side, which the uploads read until the stream is next synchronized, and the bins for the depth cap.
static int geno_setup(ls_ctx *ctx, const int32_t *site_tid, const int32_t *site_pos, const uint8_t *alt_class,
                      int64_t n_sites, const ls_geno_params *params, GenoSites &g) {
  const int32_t bin = params->bin_size > 0 ? params->bin_size : 50000;
  g.keys.resize((size_t)n_sites);
  g.sbin.resize((size_t)n_sites);
  for (int64_t i = 0; i < n_sites; ++i) {
    if (site_tid[i] < 0 || site_pos[i] < 0) LS_FAIL(LS_E_ARG, "ls_genotype: negative site coordinate");
    g.keys[i] = ((uint64_t)(uint32_t)site_tid[i] << 32) | (uint32_t)site_pos[i];
    if (i > 0 && g.keys[i] <= g.keys[i - 1]) LS_FAIL(LS_E_ARG, "ls_genotype: sites must be sorted and unique");
    // build_dict_variants: CHROM_floor(POS / bin) with the 1-based POS of the TSV (:253-274)
    const int64_t code = ((int64_t)site_pos[i] + 1) / bin;
    if (i == 0 || site_tid[i] != site_tid[i - 1] || code != ((int64_t)site_pos[i - 1] + 1) / bin) {
      g.btid.push_back(site_tid[i]);
      g.bstart.push_back(site_pos[i] - 1 < 0 ? 0 : site_pos[i] - 1);
      g.bend.push_back(site_pos[i] + 1);
    } else {
      g.bend.back() = site_pos[i] + 1;
    }
    g.sbin[i] = (uint32_t)(g.btid.size() - 1);
  }
  LS_CK(cudaSetDevice(ctx->device));
  GenoState &gs = ctx->geno;
  cudaStream_t st = ctx->stream;
  LS_CK(gs.site_key.ensure((size_t)n_sites * 8));
  LS_CK(gs.alt_class.ensure((size_t)n_sites));
  LS_CK(gs.site_bin.ensure((size_t)n_sites * 4));
  LS_CK(ctx->counters.ensure(sizeof(GenoCounters)));
  LS_CK(cudaMemcpyAsync(gs.site_key.p, g.keys.data(), (size_t)n_sites * 8, cudaMemcpyHostToDevice, st));
  LS_CK(cudaMemcpyAsync(gs.alt_class.p, alt_class, (size_t)n_sites, cudaMemcpyHostToDevice, st));
  LS_CK(cudaMemcpyAsync(gs.site_bin.p, g.sbin.data(), (size_t)n_sites * 4, cudaMemcpyHostToDevice, st));
  LS_CK(cudaMemsetAsync(ctx->counters.p, 0, sizeof(GenoCounters), st));
  return LS_OK;
}

// The kernel arguments of a call: the batch, the site table in ctx->geno and the depth cap's drops; no output yet
static GenoArgs geno_args(ls_ctx *ctx, int64_t n_sites, int32_t n_cells, const ls_geno_params *params) {
  GenoArgs a = {};
  a.n_reads = ctx->n_reads;
  a.tid = ctx->tid.as<int32_t>();
  a.pos = ctx->pos.as<int32_t>();
  a.cell = ctx->cell.as<int32_t>();
  a.lq = ctx->lq.as<int32_t>();
  a.flag = ctx->flag.as<uint16_t>();
  a.mapq = ctx->mapq.as<uint8_t>();
  a.cigar_off = ctx->cigar_off.as<uint32_t>();
  a.cigar = ctx->cigar.as<uint32_t>();
  a.base_off = ctx->base_off.as<uint64_t>();
  a.seq4 = ctx->seq4_d();
  a.qual = ctx->qual_d();
  a.site_key = ctx->geno.site_key.as<uint64_t>();
  a.alt_class = ctx->geno.alt_class.as<uint8_t>();
  a.site_bin = ctx->geno.site_bin.as<uint32_t>();
  a.n_sites = n_sites;
  a.n_cells = n_cells;
  a.min_bq = params->min_bq;
  a.min_mq = params->min_mq;
  a.alt_only = params->alt_only;
  a.drop_keys = ctx->drop_keys.as<uint64_t>();
  a.n_drop = ctx->n_drop;
  a.n_events = &ctx->counters.as<GenoCounters>()->n_events;
  return a;
}

static int read_counters(ls_ctx *ctx, const GenoCounters *d, GenoCounters &h) {
  LS_CK(cudaMemcpyAsync(&h, d, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
  LS_CK(cudaStreamSynchronize(ctx->stream));
  return LS_OK;
}

int ls_betabinom_device(ls_ctx *ctx, const int32_t *d_k, const int32_t *d_n, double a, double b, double *d_p, int64_t m,
                        uint32_t *d_nbig);

// ---- sparse genotyping: only the touched (site, cell) pairs leave the device -------------------------------------
// Phase 1: per read, how many candidate sites lie inside [pos, reference end) -- an upper bound of its hits, which
// sizes its slots -- scanned into its first slot.  The same walk over the CIGARs gives the depth cap its per-bin fetch
// counts, so there is no separate counting pass over the bases.
static int count_slots(ls_ctx *ctx, const GenoSites &g, int64_t n_sites, int32_t n_cells, const ls_geno_params *params,
                       const uint8_t *skip_p, GenoCounters *d, GenoCounters &h) {
  GenoState &gs = ctx->geno;
  cudaStream_t st = ctx->stream;
  const int64_t n = ctx->n_reads;
  LS_CK(gs.skip.ensure((size_t)n_sites));
  LS_CK(gs.slots.ensure((size_t)(n + 1) * 4));
  if (skip_p) LS_CK(cudaMemcpyAsync(gs.skip.p, skip_p, (size_t)n_sites, cudaMemcpyHostToDevice, st));
  LS_CK(cudaMemsetAsync(gs.slots.as<uint32_t>() + n, 0, 4, st));
  LS_CK(cudaEventRecord(ctx->ev[0], st));
  const CandArgs ca = {gs.site_key.as<uint64_t>(), n_sites, ctx->cell.as<int32_t>(), n_cells, gs.slots.as<uint32_t>()};
  int rc = geno_depth_cap(ctx, g.btid, g.bstart, g.bend, params->min_mq, params->max_depth, ca);
  if (rc != LS_OK) return rc;
  LS_CK(ls_scan_exclusive_u32(gs.slots.as<uint32_t>(), gs.slots.as<uint32_t>(), n + 1, &d->n_slots, ctx->scan_tmp, st));
  return read_counters(ctx, d, h);
}

static cudaError_t sort_hits(ls_ctx *ctx, uint32_t *a, uint32_t *b, int64_t n, int bits, uint32_t **sorted, int *launches) {
  return ls_radix_sort_keys32(a, b, n, bits, ctx->rs_hist, sorted, ctx->num_sms, ctx->stream, launches);
}
static cudaError_t sort_hits(ls_ctx *ctx, uint64_t *a, uint64_t *b, int64_t n, int bits, uint64_t **sorted, int *launches) {
  return ls_radix_sort_keys(a, b, n, bits, ctx->rs_hist, sorted, ctx->num_sms, ctx->stream, launches);
}

// Phase 2: the hits of every read as K-wide keys in its nh slots, sorted, and reduced to one (site, cell, Dp, Alt, k)
// tuple per touched pair.  h gets the counters after the tuple count.
template <typename K>
static int hits_to_tuples(ls_ctx *ctx, GenoArgs a, int64_t nh, bool skip, GenoCounters *d, GenoCounters &h,
                          int &launches) {
  GenoState &gs = ctx->geno;
  cudaStream_t st = ctx->stream;
  const K sentinel = (K)a.sentinel;
  LS_CK(gs.hits_a.ensure((size_t)nh * sizeof(K)));
  LS_CK(gs.hits_b.ensure((size_t)nh * sizeof(K)));
  LS_CK(gs.flag.ensure((size_t)(nh + 1) * 4));
  a.hit_off = gs.slots.as<uint32_t>();
  a.hits = gs.hits_a.p;
  genotype_kernel<K><<<(unsigned)((a.n_reads + 255) / 256), 256, 0, st>>>(a);
  K *sorted = nullptr;
  LS_CK(sort_hits(ctx, gs.hits_a.as<K>(), gs.hits_b.as<K>(), nh, ls_bits_for(a.sentinel), &sorted, &launches));
  uint32_t *flag = gs.flag.as<uint32_t>();
  hit_flag_kernel<K><<<(unsigned)((nh + 1 + 255) / 256), 256, 0, st>>>(sorted, nh, sentinel, flag);
  LS_CK(ls_scan_exclusive_u32(flag, flag, nh + 1, &d->n_tuples, ctx->scan_tmp, st));
  int rc = read_counters(ctx, d, h);
  if (rc != LS_OK) return rc;
  const int64_t nt = (int64_t)h.n_tuples;
  LS_CK(gs.tup.ensure((size_t)nt * 5 * 4 + 16));
  LS_CK(gs.p.ensure((size_t)nt * 8 + 16));
  int32_t *t_site = gs.tup.as<int32_t>(), *t_cell = t_site + nt, *t_dp = t_cell + nt, *t_alt = t_dp + nt, *t_k = t_alt + nt;
  hit_reduce_kernel<K><<<(unsigned)((nh + 255) / 256), 256, 0, st>>>(
      sorted, nh, sentinel, flag, a.n_cells, skip ? gs.skip.as<uint8_t>() : nullptr, t_site, t_cell, t_dp, t_alt, t_k);
  launches += 4;
  LS_CK(cudaGetLastError());
  return LS_OK;
}

extern "C" int ls_genotype_sparse_run(ls_ctx *ctx, const int32_t *site_tid, const int32_t *site_pos,
                                      const uint8_t *alt_class, const uint8_t *skip_p, int64_t n_sites, int32_t n_cells,
                                      const ls_geno_params *params, double alpha, double beta, int64_t *n_tuples,
                                      ls_run_stats *stats) {
  if (!ctx) return LS_E_ARG;
  int rc = geno_check(ctx, "ls_genotype_sparse_run", params, n_sites, n_cells);
  if (rc != LS_OK) return rc;
  if (!(alpha > 0.0) || !(beta > 0.0)) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_run: alpha and beta must be > 0");
  GenoState &gs = ctx->geno;
  ls_run_stats S;
  memset(&S, 0, sizeof S);
  gs.n_tuples = 0;
  gs.have_tuples = false;
  gs.alpha = alpha;
  gs.beta = beta;
  if (n_tuples) *n_tuples = 0;
  if (n_sites == 0 || n_cells == 0 || ctx->n_reads == 0) {
    gs.have_tuples = true;
    if (stats) *stats = S;
    return LS_OK;
  }
  if (!site_tid || !site_pos || !alt_class) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_run: null array");
  if ((uint64_t)n_sites * (uint64_t)n_cells >= ((uint64_t)1 << 62)) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_run: too many pairs");
  GenoSites g;
  rc = geno_setup(ctx, site_tid, site_pos, alt_class, n_sites, params, g);
  if (rc != LS_OK) return rc;
  cudaStream_t st = ctx->stream;
  GenoCounters *d = ctx->counters.as<GenoCounters>(), h;
  rc = count_slots(ctx, g, n_sites, n_cells, params, skip_p, d, h);
  if (rc != LS_OK) return rc;
  const int64_t nh = (int64_t)h.n_slots;  // slots (>= hits)
  if (nh >= (int64_t)0xffffffffll) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_run: more than 2^32 hits; split the site list");
  // The stats keep the meaning callers and bench.py read: ms_count from the slot count to the end of the reduction,
  // ms_sort the K2 tails, n_events the real hits, n_segments the tuples.  count_launches counts the slot count and its
  // scan, then, if there are slots, genotype_kernel, the radix sort, hit_flag_kernel, the scan, hit_reduce_kernel and
  // K2's 2 or 4 launches; a capped call's read_end_kernel is not counted.
  int launches = 2;
  if (nh > 0) {
    // keys that fit 32 bits are written, sorted and reduced as 32-bit words (half the traffic of the hit sort)
    const uint64_t key_span = (uint64_t)n_sites * (uint64_t)n_cells * 2u;
    GenoArgs a = geno_args(ctx, n_sites, n_cells, params);
    a.sentinel = key_span;
    if (key_span < (1ull << 32) && !getenv("LS_GENO_KEYS64"))
      rc = hits_to_tuples<uint32_t>(ctx, a, nh, skip_p != nullptr, d, h, launches);
    else
      rc = hits_to_tuples<uint64_t>(ctx, a, nh, skip_p != nullptr, d, h, launches);
    if (rc != LS_OK) return rc;
  }
  const int64_t nt = (int64_t)h.n_tuples;
  LS_CK(cudaEventRecord(ctx->ev[1], st));
  if (nh > 0) {  // Phase 3, K2 on the device: p = betabinom.sf(Alt - eps, Dp, alpha, beta) for the pairs with a query
    const int32_t *t_dp = gs.tup.as<int32_t>() + 2 * nt, *t_k = t_dp + 2 * nt;
    rc = ls_betabinom_device(ctx, t_k, t_dp, alpha, beta, gs.p.as<double>(), nt, &d->n_big);
    if (rc != LS_OK) return rc;
    launches += nt > 4 * 65 * 65 ? 4 : 2;  // constants + tails (+ the (k, n) table and its queries)
  }
  LS_CK(cudaEventRecord(ctx->ev[2], st));
  LS_CK(cudaStreamSynchronize(st));
  LS_CK(cudaEventElapsedTime(&S.ms_count, ctx->ev[0], ctx->ev[1]));
  LS_CK(cudaEventElapsedTime(&S.ms_sort, ctx->ev[1], ctx->ev[2]));
  LS_CK(cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[2]));
  S.n_events = (int64_t)h.n_events;
  S.n_segments = nt;
  S.count_launches = launches;
  gs.n_tuples = nt;
  gs.have_tuples = true;
  ctx->n_drop = 0;
  if (n_tuples) *n_tuples = nt;
  if (stats) *stats = S;
  return LS_OK;
}

extern "C" int ls_genotype_sparse_fetch(ls_ctx *ctx, ls_geno_tuples *out) {
  if (!ctx) return LS_E_ARG;
  if (!out) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_fetch: out is null");
  const GenoState &gs = ctx->geno;
  if (!gs.have_tuples) LS_FAIL(LS_E_STATE, "ls_genotype_sparse_fetch: ls_genotype_sparse_run has not completed");
  const int64_t nt = gs.n_tuples;
  out->n_tuples = nt;
  if (nt == 0) return LS_OK;
  if (out->capacity < nt) LS_FAIL(LS_E_CAPACITY, "ls_genotype_sparse_fetch: capacity < n_tuples");
  if (!out->site || !out->cell || !out->dp || !out->alt || !out->p) LS_FAIL(LS_E_ARG, "ls_genotype_sparse_fetch: null array");
  LS_CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int32_t *t = gs.tup.as<int32_t>();
  LS_CK(cudaMemcpyAsync(out->site, t, (size_t)nt * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->cell, t + nt, (size_t)nt * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->dp, t + 2 * nt, (size_t)nt * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->alt, t + 3 * nt, (size_t)nt * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(out->p, gs.p.p, (size_t)nt * 8, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaStreamSynchronize(st));
  // pairs whose Alt count is past the in-register kernel's range (marked p = -1): the staged path
  std::vector<int64_t> big;
  for (int64_t i = 0; i < nt; ++i)
    if (out->p[i] == -1.0) big.push_back(i);
  if (!big.empty()) {
    std::vector<int32_t> k(big.size()), nn(big.size());
    std::vector<double> pp(big.size());
    for (size_t j = 0; j < big.size(); ++j) {
      k[j] = out->alt[big[j]];
      nn[j] = out->dp[big[j]];
    }
    int rc = ls_betabinom_sf(ctx, k.data(), nn.data(), gs.alpha, gs.beta, pp.data(), (int64_t)big.size(), nullptr);
    if (rc != LS_OK) return rc;
    for (size_t j = 0; j < big.size(); ++j) out->p[big[j]] = pp[j];
  }
  return LS_OK;
}

extern "C" int ls_genotype_count(ls_ctx *ctx, const int32_t *site_tid, const int32_t *site_pos,
                                 const uint8_t *alt_class, int64_t n_sites, int32_t n_cells,
                                 const ls_geno_params *params, int32_t *dp, int32_t *alt, ls_run_stats *stats) {
  if (!ctx) return LS_E_ARG;
  int rc = geno_check(ctx, "ls_genotype_count", params, n_sites, n_cells);
  if (rc != LS_OK) return rc;
  ls_run_stats S;
  memset(&S, 0, sizeof S);
  if (n_sites == 0 || n_cells == 0) {
    if (stats) *stats = S;
    return LS_OK;
  }
  if (!site_tid || !site_pos || !alt_class || !dp || !alt) LS_FAIL(LS_E_ARG, "ls_genotype_count: null array");
  GenoSites g;
  rc = geno_setup(ctx, site_tid, site_pos, alt_class, n_sites, params, g);
  if (rc != LS_OK) return rc;
  rc = geno_depth_cap(ctx, g.btid, g.bstart, g.bend, params->min_mq, params->max_depth);
  if (rc != LS_OK) return rc;
  GenoState &gs = ctx->geno;
  cudaStream_t st = ctx->stream;
  const size_t cells = (size_t)n_sites * (size_t)n_cells;
  LS_CK(gs.dp.ensure(cells * 4));
  LS_CK(gs.alt.ensure(cells * 4));
  LS_CK(cudaEventRecord(ctx->ev[0], st));
  LS_CK(cudaMemsetAsync(gs.dp.p, 0, cells * 4, st));
  LS_CK(cudaMemsetAsync(gs.alt.p, 0, cells * 4, st));
  GenoArgs a = geno_args(ctx, n_sites, n_cells, params);
  a.dp = gs.dp.as<int32_t>();
  a.alt = gs.alt.as<int32_t>();
  LS_CK(cudaEventRecord(ctx->ev[1], st));
  if (ctx->n_reads > 0) genotype_kernel<void><<<(unsigned)((ctx->n_reads + 255) / 256), 256, 0, st>>>(a);
  LS_CK(cudaGetLastError());
  LS_CK(cudaEventRecord(ctx->ev[2], st));
  LS_CK(cudaMemcpyAsync(dp, gs.dp.p, cells * 4, cudaMemcpyDeviceToHost, st));
  LS_CK(cudaMemcpyAsync(alt, gs.alt.p, cells * 4, cudaMemcpyDeviceToHost, st));
  GenoCounters h;
  rc = read_counters(ctx, ctx->counters.as<GenoCounters>(), h);
  if (rc != LS_OK) return rc;
  LS_CK(cudaEventElapsedTime(&S.ms_count, ctx->ev[1], ctx->ev[2]));
  LS_CK(cudaEventElapsedTime(&S.ms_total, ctx->ev[0], ctx->ev[2]));
  S.n_events = (int64_t)h.n_events;
  S.count_launches = 1;
  ctx->n_drop = 0;
  if (stats) *stats = S;
  return LS_OK;
}
