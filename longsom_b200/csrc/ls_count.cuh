// K1 pileup-count kernel (one LANE per 32-column unit) + the unit expansion and part bookkeeping around it.
// Included by ls_pileup.cu.
//
// After the (tile, cell) sort, `classify_kernel` + scans + `expand_single_kernel` / `expand_runs_kernel` turn the sorted
// segments into UNIT STREAMS
// in HBM.  A unit is one piece (CIGAR op clipped to the tile) clipped to one of the tile's sixteen 32-column windows:
// where its query bases start in qual[] / seq4[], the window, the columns [lo, hi) it covers, strand, and whether it
// is a run of deletion columns (which all carry one quality).  Three streams, each in sorted-segment order:
//   S = segments whose (tile, cell) key occurs once,
//   M = same-cell runs (>= 2 segments of one cell in one tile); inside a run the units are ordered WINDOW-MAJOR, so
//       that all entries one cell has at one reference position are consecutive units of the stream,
//   U = visible-but-uncounted reads (only with --min_ac > 0).
//
// Unit of work of a count CTA: a PART = up to K1_PART_SEGS consecutive sorted segments of one tile.  Most tiles are
// one part; deep tiles (chrM, hotspot genes: >1e5 reads per locus) are split so that no CTA owns more than ~4e5
// pileup entries.  Same-cell runs never straddle parts (a run belongs to the part that holds its first segment), so
// NC / CC stay exact and every output word is additive across parts; multi-part tiles add into their HBM slot and
// the last part to finish applies the reference's gates.  `part_build_kernel` writes one 64-byte PartDesc per CTA (tile
// bounds, reference offset, the part's slices of the streams and of the group directory): a CTA starts with one load.
// The same-cell runs (M) are counted first, the single-segment units (S) last, claimed one 32-unit batch at a time: the
// fine-grained stream fills in behind the long groups, so the warps reach the tile's barrier together.  Single-part
// tiles leave the kernel as finished 26-word site records (passing sites packed per 32-column window).
//
// Inside a part (CTA of K1_WARPS warps, tile accumulators in shared memory) every lane owns whole units:
//   * the lane loads the aligned 40-byte block of qualities and 24-byte block of 4-bit bases around its unit and
//     shifts them so that byte / nibble j is the base at column j of the window (seq4 is nibble-swapped at upload so
//     that this is one funnel shift);
//   * 32 fully unrolled columns: byte permute -> packed (count<<20 | quality) word, nibble -> row offset through a
//     16-entry shared-memory table, one `red.shared.add` per column (a zero add for columns that must not count:
//     ptxas never predicates a shared atomic, it branches around it).  Rows are padded by one word per window, so
//     the lanes of a warp -- which work on different windows and strands -- hit different banks;
//   * all 32 lanes work on different reads, so lane occupancy does not depend on piece lengths (the previous
//     generation gave a whole warp to one piece: 2.5 warp-instructions per pileup entry at 21 of 32 lanes).
// Distinct-cell counts: NC/CC = reads minus same-cell duplicates.  In the M stream the units of one (cell, window)
// group are consecutive and handled by ONE lane, which keeps the class bits the cell has shown at each of the 32
// columns in eight registers: a column whose bit / byte is already set is a (cell, class) / (cell) duplicate.  No
// shared-memory state, no atomics and no warp-level serialisation per run.
#pragma once

constexpr int K1_WARPS = 8;              // warps of a count CTA (3 CTAs / SM with packed counters, 1 without)
constexpr int K1_THREADS = K1_WARPS * 32;
constexpr int K1_PART_SEGS = 2048;       // nominal segments per part
constexpr int K1_MAX_RUN_PACKED = 2039;  // packed counters (12-bit) need: part segs + run extension <= 4095
constexpr int K1_CROWS = 18;             // 16 (class, strand) rows + a dump row pair for ignored base codes
constexpr int K1_ROWW = 16 * 33;         // words per row: 16 windows of 32 columns + 1 pad word each
constexpr uint32_t K1_ROW_BYTES = 4u * K1_ROWW;
constexpr uint32_t K1_DUMP_OFF = 16u * K1_ROW_BYTES;
constexpr uint32_t K1_CNT_SHIFT = 20;    // packed word: count << 20 | base-quality sum (<= 4095 * 255 < 2^20)

static_assert(LS_TILE % 32 == 0 && LS_TILE == 512, "tile shape");
static_assert(K1_CROWS + 8 >= LS_SITE_WORDS, "the epilogue transposes through the warp's columns of hist + dup rows");

// unit.x: low 32 bits of q = index in qual[] of the base at column lo (deletion-like: of the one quality byte)
// unit.y: q >> 32: bits 0-3 | window: 4-7 | lo: 8-12 | hi: 13-18 | strand: 19 | deletion-like: 20 | ind: 21-22 |
//         virt: 23 | first unit of its (run, window) group: 24
constexpr uint32_t UM_STRAND = 1u << 19;
constexpr uint32_t UM_DEL = 1u << 20;
constexpr uint32_t UM_VIRT = 1u << 23;
constexpr uint32_t UM_GSTART = 1u << 24;

__host__ __device__ __forceinline__ int k1_col(int s) { return s + (s >> 5); }  // column -> word of a padded row

struct CountArgs {
  const uint8_t *seq4, *qual;                // device copies (padded, seq4 nibble-swapped; see ls_ctx)
  const uint2 *units;                        // S stream, then M, then U
  const uint64_t *tot_s, *tot_m;             // stream sizes (M starts at *tot_s, U at *tot_s + *tot_m)
  const uint32_t *gdir;                      // [n_groups + 1] first unit (in M) of every group, in run / window order
  int with_u;                                // a U stream exists (--min_ac > 0)
  const struct PartDesc *parts;              // [grid] what every CTA of the count kernel works on (part_build_kernel)
  uint32_t *slot_done;
  const uint8_t *ref;
  uint32_t *out;    // [n_slots]: single-part tiles [16 windows][32 records][LS_SITE_WORDS], passing sites packed at the
                    // front of each window block; multi-part tiles [LS_SITE_WORDS][LS_TILE] (their parts merge with atomics)
  uint32_t *acbuf;  // [n_slots][LS_TILE], only when min_ac > 0
  uint32_t *mask;   // [n_slots][LS_TILE/32]
  uint32_t *npass;  // [n_slots]
  unsigned long long *n_events;
  int cell_bits;
  uint32_t uncounted_key;
  int min_bq, min_dp, min_cc, min_ac;
  uint32_t cnt1;  // 1 << K1_CNT_SHIFT for the packed kernel, 0 for the unpacked one (a run-time value on purpose:
                  // as a compile-time constant it takes PRMT's immediate slot and the byte selectors need a MOV each)
};

// Everything a count CTA needs to start, in one 64-byte record: without it the CTA walks a chain of dependent loads
// (part -> slot -> tile -> binary search over the windows -> stream offsets) before its first unit, and that chain was
// an eighth of the kernel's warp time.
struct alignas(16) PartDesc {
  uint32_t slot;     // 0xffffffff: unused grid entry
  uint32_t nparts;   // parts of this slot's tile
  int32_t tile_start, tile_end;
  uint64_t ref_base;  // index in ref[] of the tile's first column
  uint32_t s_lo, s_n;  // the part's units in the S stream
  uint32_t g_lo, g_n;  // its slice of the group directory (runs that START in the part)
  uint32_t u_lo, u_n;  // its units in the U stream (relative to the stream's start)
  uint32_t pad[4];
};
static_assert(sizeof(PartDesc) == 64, "PartDesc layout");

template <bool PACKED>
struct TileSmemT {
  // rows [cls*2+strand] for cls 0..7, rows 16-17 = "dump" (ignored base codes).  PACKED: cnt<<20|bq; else rows
  // [0..17] counts, [18..35] quality sums.  Column s of a row is word k1_col(s).
  uint32_t hist[PACKED ? K1_CROWS : 2 * K1_CROWS][K1_ROWW];
  uint32_t dup[8][K1_ROWW];               // per class: (cell, class) duplicates | (cell) duplicates << 16
  alignas(64) uint32_t lut[16];           // BAM nibble code -> byte offset of the class's row pair (dump rows if ignored)
  uint32_t lut2[2][16];                   // [deletion-like][code] -> 0x80 | class bit (A..D) | byte offset of the class's dup row << 8
  uint8_t ref[LS_TILE];
  uint32_t next1, next2, next3, npass, ticket;
  uint32_t acx[K1_ROWW];                  // alt entries of visible-but-uncounted reads; LAST: only allocated with --min_ac > 0
};

__device__ __forceinline__ int64_t window_of_tile(const int64_t *__restrict__ wtile_base, int64_t n_windows, int64_t tile) {
  int64_t lo = 0, hi = n_windows;  // last w with wtile_base[w] <= tile
  while (hi - lo > 1) {
    int64_t m = (lo + hi) >> 1;
    if (wtile_base[m] <= tile)
      lo = m;
    else
      hi = m;
  }
  return lo;
}

// shared-memory accesses on 32-bit shared-window addresses (no generic->shared conversion per base)
__device__ __forceinline__ void red_shared_add(uint32_t addr, uint32_t v) {
  // no "memory" clobber: nothing reads the accumulators before the CTA barrier, so loads may move across
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v));
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));  // tables are written once, before the first barrier
  return v;
}
template <uint32_t SEL>
__device__ __forceinline__ uint32_t prmt_sel(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "n"(SEL));
  return d;
}
__device__ __forceinline__ uint32_t prmt_var(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ uint2 ldg_v2(const void *p) {
  uint2 v;
  asm volatile("ld.global.nc.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}

struct UData {
  uint32_t qw[8];  // byte j = quality of the base at column j of the window
  uint32_t hw[4];  // nibble j (bits 4j .. 4j+3) = its BAM base code
  uint32_t qlast;  // quality of the base at column hi - 1 (the one that carries a following indel)
};

// What a unit's loads return, untouched: the loads are issued one step ahead of their use, so nothing here may depend
// on the loaded values (the alignment happens in align_unit, at the start of the step that counts the unit).
struct URaw {
  uint32_t w[10];  // 40 bytes of qualities from the 8-byte boundary at or below column 0 (deletion-like: w[0] = the byte)
  uint32_t h[6];   // 24 bytes of base nibbles, likewise
  uint32_t qlast;
};

__device__ __forceinline__ URaw issue_unit(const CountArgs &a, uint2 u) {
  URaw r;
  const uint32_t meta = u.y;
  const uint32_t lo = (meta >> 8) & 31u, hi = (meta >> 13) & 63u;
#pragma unroll
  for (int i = 0; i < 10; ++i) r.w[i] = 0u;
#pragma unroll
  for (int i = 0; i < 6; ++i) r.h[i] = 0u;
  r.qlast = 0u;
  if (hi == 0u || (meta & UM_VIRT)) return r;  // empty lane / positions past the stored sequence: nothing to load
  const int64_t q = (int64_t)(((uint64_t)(meta & 15u) << 32) | u.x);
  if (meta & UM_DEL) {
    r.w[0] = a.qual[q];
  } else {
    const int64_t q0 = q - (int64_t)lo;  // where column 0 of the window would be (possibly before the read)
    const uint8_t *pq = a.qual + (q0 & ~(int64_t)7);
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const uint2 t = ldg_v2(pq + 8 * i);
      r.w[2 * i] = t.x;
      r.w[2 * i + 1] = t.y;
    }
    const uint8_t *ph = a.seq4 + ((q0 >> 1) & ~(int64_t)7);  // arithmetic shift: q0 may be slightly negative
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const uint2 t = ldg_v2(ph + 8 * i);
      r.h[2 * i] = t.x;
      r.h[2 * i + 1] = t.y;
    }
    if ((meta >> 21) & 3u) r.qlast = a.qual[q + (int64_t)(hi - 1u - lo)];
  }
  return r;
}

__device__ __forceinline__ UData align_unit(const URaw &r, uint2 u) {
  UData d;
  const uint32_t meta = u.y;
  const uint32_t lo = (meta >> 8) & 31u;
  d.qlast = r.qlast;
  if (meta & (UM_DEL | UM_VIRT)) {
    // deletion-like units carry one quality on every column and run as 'N' (virtual ones: quality 0)
    const uint32_t q4 = r.w[0] * 0x01010101u;
#pragma unroll
    for (int i = 0; i < 8; ++i) d.qw[i] = q4;
#pragma unroll
    for (int i = 0; i < 4; ++i) d.hw[i] = ~0u;
    d.qlast = r.w[0];
    return d;
  }
  const uint32_t q0 = u.x - lo;  // only its low bits matter here
  {
    const uint32_t sh = q0 & 7u;
    const bool o = (sh & 4u) != 0u;
    uint32_t x[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) x[i] = o ? r.w[i + 1] : r.w[i];
    const uint32_t sel = 0x3210u + 0x1111u * (sh & 3u);
#pragma unroll
    for (int i = 0; i < 8; ++i) d.qw[i] = prmt_var(x[i], x[i + 1], sel);
  }
  {
    const uint32_t shift = 4u * (q0 & 15u);
    const bool o = (shift & 32u) != 0u;
    uint32_t y[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) y[i] = o ? r.h[i + 1] : r.h[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) d.hw[i] = __funnelshift_r(y[i], y[i + 1], shift & 31u);
  }
  return d;
}

struct WarpCtx {
  uint32_t hist_s, lut_s, dup_s;  // shared-window addresses
  uint32_t thr;                   // PACKED: (1 << 20) | min_bq, else min_bq (clamped to [0, 256])
  uint32_t cnt1;                  // PACKED: 1 << 20, else 0
};

// A column that must not count -- outside [lo, hi), below the quality threshold -- adds ZERO to the word it would have
// hit, and an ignored base code adds to a dump row through the nibble table: the 32 unrolled columns are straight-line
// code.  SEEN adds the same-cell bookkeeping on the lane's per-window state `seen` (one byte per column: 0x80 = the
// cell has an entry here, bits 0-5 = classes A..D it has shown): the duplicates go to the class's dup word with one
// more (possibly zero) add.
__device__ __forceinline__ uint32_t lds_u32_pinned(uint32_t addr) {
  uint32_t v;  // volatile: stays where it is written, i.e. ahead of the block's adds (see ColumnBlock)
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}

// Eight columns of a unit.  All table lookups of the block are issued first and only then the adds: a shared-memory
// load cannot be moved above an earlier shared-memory atomic by the compiler (it cannot prove they do not alias), so
// written column by column every column would wait for its own lookup.
template <bool PACKED, bool SEEN, int B>
struct ColumnBlock {
  static __device__ __forceinline__ void run(const WarpCtx &c, const UData &d, uint32_t hs, uint32_t vm, uint32_t ds,
                                             uint32_t lut2p, uint32_t (&seen)[8]) {
    constexpr uint32_t QOFF = (uint32_t)K1_CROWS * K1_ROW_BYTES;
    uint32_t idx[8], off[8], vz[8], okm[8], w2[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      constexpr int dummy = 0;
      (void)dummy;
      const int pos = 4 * t;  // bit position of column (8B + t)'s nibble in word B
      idx[t] = pos >= 2 ? ((d.hw[B] >> (pos >= 2 ? pos - 2 : 0)) & 0x3cu) : ((d.hw[B] << 2) & 0x3cu);
      off[t] = lds_u32_pinned(idx[t] | c.lut_s);  // the table is 64-byte aligned
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int J = 8 * B + t;
      // c.cnt1 = 1 << 20 (0 when !PACKED) lives in a register so that the byte selector can be the immediate
      const uint32_t v = (t & 3) == 0   ? prmt_sel<0x4640u>(d.qw[J >> 2], c.cnt1)
                         : (t & 3) == 1 ? prmt_sel<0x4641u>(d.qw[J >> 2], c.cnt1)
                         : (t & 3) == 2 ? prmt_sel<0x4642u>(d.qw[J >> 2], c.cnt1)
                                        : prmt_sel<0x4643u>(d.qw[J >> 2], c.cnt1);
      // vz = v, okm = 0x3c if column J is inside [lo, hi) and v >= thr; else 0
      asm("{\n .reg .pred p;\n .reg .b32 t;\n and.b32 t, %3, %4;\n setp.ne.u32 p, t, 0;\n setp.ge.and.u32 p, %2, %5, p;\n"
          " selp.u32 %0, %2, 0, p;\n selp.u32 %1, 60, 0, p;\n}"
          : "=r"(vz[t]), "=r"(okm[t])
          : "r"(v), "r"(vm), "r"(1u << J), "r"(c.thr));
      // table 2, looked up at code 0 (an ignored code: word 0) when the column does not count:
      // byte 0 = 0x80 | class bit (classes A..D: bits 0-5), bits 8.. = byte offset of the class's dup row
      if (SEEN) w2[t] = lds_u32_pinned((idx[t] & okm[t]) | lut2p);
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int J = 8 * B + t;
      const uint32_t addr = hs + off[t] + 4u * J;
      if (PACKED) {
        red_shared_add(addr, vz[t]);
      } else {
        red_shared_add(addr, okm[t] >> 5);
        red_shared_add(addr + QOFF, vz[t]);
      }
      if (SEEN) {
        const uint32_t bsh = (t & 3) == 0   ? prmt_sel<0x4440u>(w2[t], 0u)
                             : (t & 3) == 1 ? prmt_sel<0x4404u>(w2[t], 0u)
                             : (t & 3) == 2 ? prmt_sel<0x4044u>(w2[t], 0u)
                                            : prmt_sel<0x0444u>(w2[t], 0u);
        const uint32_t sw = seen[J >> 2];
        // the 0x80 markers meet iff the cell already has an entry at this column; the class bits iff of this class
        const uint32_t dv = (sw & bsh & 0x3f3f3f3fu) ? 0x10001u : ((sw & bsh) ? 0x10000u : 0u);
        seen[J >> 2] = sw | bsh;
        red_shared_add(ds + (w2[t] >> 8) + 4u * J, dv);
      }
    }
  }
};

// One unit per lane: 32 unrolled columns.  The strand selects the row inside the class's row pair through the base
// address; a deletion-like unit runs as 32 'N' bases with the base address one class (row pair) up, which turns N
// into O -- so one 16-entry nibble table serves every lane.
template <bool PACKED, bool SEEN>
__device__ __forceinline__ void count_unit(const WarpCtx &c, uint32_t meta, const UData &d, int lane, uint32_t (&seen)[8]) {
  const uint32_t lo = (meta >> 8) & 31u, hi = (meta >> 13) & 63u;
  const uint32_t ind = (meta >> 21) & 3u;
  // an empty lane (hi == 0) still issues its 32 zero adds: give it a window / strand of its own in the dump rows
  const uint32_t w = hi ? ((meta >> 4) & 15u) : ((uint32_t)lane & 15u);
  const uint32_t strand = hi ? ((meta >> 19) & 1u) : ((uint32_t)lane >> 4);
  const uint32_t del = (meta >> 20) & 1u;
  uint32_t vm = hi ? ((0xffffffffu >> (32u - hi)) & (0xffffffffu << lo)) : 0u;
  if (ind) vm &= ~(1u << (hi - 1u));
  const uint32_t sb = w * 132u;
  const uint32_t hs = c.hist_s + sb + strand * K1_ROW_BYTES + del * (2u * K1_ROW_BYTES);
  const uint32_t ds = c.dup_s + sb;
  const uint32_t lut2p = c.lut_s + 64u + del * 64u;
  ColumnBlock<PACKED, SEEN, 0>::run(c, d, hs, vm, ds, lut2p, seen);
  ColumnBlock<PACKED, SEEN, 1>::run(c, d, hs, vm, ds, lut2p, seen);
  ColumnBlock<PACKED, SEEN, 2>::run(c, d, hs, vm, ds, lut2p, seen);
  ColumnBlock<PACKED, SEEN, 3>::run(c, d, hs, vm, ds, lut2p, seen);
  if (ind) {  // last base of the op, followed by an insertion / deletion: class I / D instead of its letter
    const uint32_t v = PACKED ? ((1u << K1_CNT_SHIFT) | d.qlast) : d.qlast;
    if (v >= c.thr) {
      const uint32_t cls = ind == 2u ? (uint32_t)LS_CLASS_D : (uint32_t)LS_CLASS_I;
      const uint32_t jl = hi - 1u;
      const uint32_t addr = c.hist_s + (cls * 2u + strand) * K1_ROW_BYTES + sb + 4u * jl;
      if (PACKED) {
        red_shared_add(addr, v);
      } else {
        red_shared_add(addr, 1u);
        red_shared_add(addr + (uint32_t)K1_CROWS * K1_ROW_BYTES, v);
      }
      if (SEEN) {
        const uint32_t r = jl >> 2, sh = 8u * (jl & 3u);
        uint32_t sw = 0u;
#pragma unroll
        for (int i = 0; i < 8; ++i) sw = (uint32_t)i == r ? seen[i] : sw;
        const uint32_t bsh = (0x80u | (1u << cls)) << sh;  // cls is I or D here
        const uint32_t dv = (sw & bsh & 0x3f3f3f3fu) ? 0x10001u : ((sw & bsh) ? 0x10000u : 0u);
#pragma unroll
        for (int i = 0; i < 8; ++i) seen[i] = (uint32_t)i == r ? (sw | bsh) : seen[i];
        if (dv) red_shared_add(ds + cls * K1_ROW_BYTES + 4u * jl, dv);
      }
    }
  }
}

// A unit of a visible-but-uncounted read (no CB tag / supplementary): only the AC pre-gate of
// BaseCellCounter.py:165-174,221 sees it.  Rare (--min_ac > 0 only): plain loop, bytes straight from memory.
template <bool PACKED>
__device__ __noinline__ void count_unit_uncounted(const uint8_t *__restrict__ qual, const uint8_t *__restrict__ seq4,
                                                  int min_bq, TileSmemT<PACKED> &sm, uint2 u) {
  const uint32_t meta = u.y;
  const uint32_t w = (meta >> 4) & 15u, lo = (meta >> 8) & 31u, hi = (meta >> 13) & 63u;
  const uint32_t ind = (meta >> 21) & 3u;
  const bool virt = (meta & UM_VIRT) != 0, del = (meta & UM_DEL) != 0;
  const int64_t q = (int64_t)(((uint64_t)(meta & 15u) << 32) | u.x);
  for (uint32_t j = lo; j < hi; ++j) {
    const int64_t qi = del ? q : q + (int64_t)(j - lo);
    const uint32_t qv = virt ? 0u : qual[qi];
    if ((int)qv < min_bq) continue;
    int cls;
    if (ind && j == hi - 1u)
      cls = ind == 2u ? LS_CLASS_D : LS_CLASS_I;
    else if (del)
      cls = LS_CLASS_O;
    else if (virt)
      cls = LS_CLASS_N;
    else
      cls = class_of_code((qi & 1) ? (uint32_t)(seq4[qi >> 1] >> 4) : (seq4[qi >> 1] & 15u));  // nibble-swapped copy
    if (cls == LS_CLASS_NA) continue;
    const int s = (int)(w * 32u + j);
    const bool alt = (cls == LS_CLASS_D || cls == LS_CLASS_I) || (cls != LS_CLASS_O && class_letter(cls) != sm.ref[s]);
    if (alt) atomicAdd(&sm.acx[k1_col(s)], 1u);
  }
}

// ---- sorted segments -> unit streams ---------------------------------------------------------------------------
// Class of sorted segment i: 2 = visible-but-uncounted read, 1 = member of a same-(tile, cell) run, 0 = single.
__device__ __forceinline__ int segment_class(const uint64_t *__restrict__ keys, int64_t i, int64_t n, uint64_t cmask,
                                             uint64_t unc) {
  const uint64_t k = keys[i];
  if ((k & cmask) == unc) return 2;
  if ((i > 0 && keys[i - 1] == k) || (i + 1 < n && keys[i + 1] == k)) return 1;
  return 0;
}

// One pass over the sorted keys: stream class and unit count of every segment (inputs of the S / M / U offset scans and
// of the run-member ranks), the first-segment-of-its-tile flags (input of the slot table scan), and the check for a
// same-cell run too long for the packed counters.
__global__ void __launch_bounds__(256) classify_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                       const Segment *__restrict__ segs, int64_t n, uint64_t cmask,
                                                       uint64_t unc, int cell_bits, uint32_t *__restrict__ nu_s,
                                                       uint32_t *__restrict__ nu_m, uint32_t *__restrict__ nu_u,
                                                       uint32_t *__restrict__ is_m, uint32_t *__restrict__ tile_flag,
                                                       uint32_t *__restrict__ long_run) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) {  // the arrays have n + 1 entries: after the exclusive scans entry n holds the stream size
    nu_s[n] = 0u;
    nu_m[n] = 0u;
    is_m[n] = 0u;
    if (nu_u) nu_u[n] = 0u;
    return;
  }
  const uint64_t k = keys[i];
  const uint64_t kp = i > 0 ? keys[i - 1] : ~k, kn = i + 1 < n ? keys[i + 1] : ~k;
  const int cls = (k & cmask) == unc ? 2 : ((kp == k || kn == k) ? 1 : 0);
  const uint32_t nu = segs[vals[i]].np_nu >> 16;
  nu_s[i] = cls == 0 ? nu : 0u;
  nu_m[i] = cls == 1 ? nu : 0u;
  is_m[i] = cls == 1 ? 1u : 0u;
  if (nu_u) nu_u[i] = cls == 2 ? nu : 0u;
  tile_flag[i] = (i == 0 || (kp >> cell_bits) != (k >> cell_bits)) ? 1u : 0u;
  if (cls == 1 && i >= K1_MAX_RUN_PACKED && keys[i - K1_MAX_RUN_PACKED] == k) *long_run = 1u;
}

// mlist[rank of i among the run members] = i
__global__ void __launch_bounds__(256) mlist_kernel(const uint64_t *__restrict__ keys, int64_t n, uint64_t cmask, uint64_t unc,
                                                    const uint32_t *__restrict__ mrank, uint32_t *__restrict__ mlist) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (segment_class(keys, i, n, cmask, unc) == 1) mlist[mrank[i]] = (uint32_t)i;
}

struct ExpandArgs {
  const uint64_t *keys;
  const uint32_t *vals;
  const Segment *segs;
  const Piece *pieces;
  int64_t n;
  uint64_t cmask, unc;
  const uint32_t *offs_s, *offs_m, *offs_u;
  const uint64_t *tot_s, *tot_m, *tot_g, *tot_ms;  // stream sizes, groups, run-member segments
  const uint32_t *mlist;                           // sorted indices of the run members, in order
  uint32_t *goffs;                                 // rungroups: groups per run at its first segment; then scanned
  uint32_t *gdir;
  uint2 *units;
};

// The units of one segment, piece by piece, window by window.  f(window, unit) places them.
template <typename F>
__device__ __forceinline__ void segment_units(const ExpandArgs &a, int64_t i, F &&f) {
  const uint4 r = *reinterpret_cast<const uint4 *>(a.segs + a.vals[i]);
  const uint32_t p0 = r.x, np = r.y & 0xffffu;
  const uint64_t boff = (uint64_t)r.z << 4;
  const uint32_t strand = r.w & 1u;
  const uint2 *pp = reinterpret_cast<const uint2 *>(a.pieces) + p0;
  uint2 pc = np ? __ldg(pp) : make_uint2(0u, 0u);
  for (uint32_t k = 0; k < np; ++k) {
    const uint2 cur = pc;
    if (k + 1u < np) pc = __ldg(pp + k + 1u);
    const uint32_t meta = cur.y;
    const uint32_t col = meta & 511u, len = (meta >> 9) & 1023u, ind = (meta >> 20) & 3u;
    const uint32_t del = (meta >> 19) & 1u, virt = (meta >> 22) & 1u;
    const uint64_t g0 = boff + cur.x;
    const uint32_t wa = col >> 5, wb = (col + len - 1u) >> 5;
    const uint32_t common = (strand << 19) | (del << 20) | (virt << 23);
    for (uint32_t w = wa; w <= wb; ++w) {
      const uint32_t lo_s = col > 32u * w ? col : 32u * w;
      const uint32_t hi_s = (col + len) < 32u * w + 32u ? (col + len) : 32u * w + 32u;
      const uint64_t q = del ? g0 : g0 + (lo_s - col);
      uint32_t um = common | (uint32_t)(q >> 32) | (w << 4) | ((lo_s - 32u * w) << 8) | ((hi_s - 32u * w) << 13);
      if (w == wb) um |= ind << 21;
      f(w, make_uint2((uint32_t)q, um));
    }
  }
}

// ---- run members, one LANE per segment -----------------------------------------------------------------------
// A warp takes 32 consecutive run members (mlist) and owns the runs that START among them; the last of those may
// continue past the 32, and then the warp follows it to its end in further rounds.  f(i, runlane) is called by every
// lane of every round: i = the lane's sorted segment (-1: nothing this round), runlane = lane (of round 0) that holds
// the first segment of its run.
template <typename F>
__device__ __forceinline__ void warp_runs(const ExpandArgs &a, uint32_t cb, uint32_t nm, int lane, F &&f) {
  const uint32_t m = cb + (uint32_t)lane;
  int64_t i = -1;
  uint64_t key = 0;
  bool start = false;
  if (m < nm) {
    i = a.mlist[m];
    key = a.keys[i];
    start = i == 0 || a.keys[i - 1] != key;
  }
  const uint32_t smask = __ballot_sync(0xffffffffu, start);
  const uint32_t below = smask & (lane == 31 ? 0xffffffffu : ((2u << lane) - 1u));
  const int runlane = below ? 31 - __clz(below) : -1;  // -1: the run started in an earlier warp's range
  f(runlane >= 0 ? i : (int64_t)-1, runlane);
  if (smask == 0u) return;
  const int jlast = 31 - __clz(smask);
  const uint64_t klast = __shfl_sync(0xffffffffu, key, jlast);
  for (uint32_t rb = cb + 32u; rb < nm; rb += 32u) {
    const uint32_t m2 = rb + (uint32_t)lane;
    int64_t i2 = -1;
    bool same = false;
    if (m2 < nm) {
      i2 = a.mlist[m2];
      same = a.keys[i2] == klast;
    }
    const uint32_t same_mask = __ballot_sync(0xffffffffu, same);
    const int cnt = same_mask == 0xffffffffu ? 32 : (__ffs(~same_mask) - 1);
    if (cnt == 0) break;
    f(lane < cnt ? i2 : (int64_t)-1, jlast);
    if (cnt < 32) break;
  }
}

// windows a segment's pieces touch (bit w)
__device__ __forceinline__ uint32_t segment_window_mask(const ExpandArgs &a, int64_t i) {
  const uint4 r = *reinterpret_cast<const uint4 *>(a.segs + a.vals[i]);
  const uint2 *pp = reinterpret_cast<const uint2 *>(a.pieces) + r.x;
  const uint32_t np = r.y & 0xffffu;
  uint32_t mask = 0u;
  for (uint32_t k = 0; k < np; ++k) {
    const uint32_t meta = __ldg(pp + k).y;
    const uint32_t col = meta & 511u, len = (meta >> 9) & 1023u;
    const uint32_t wa = col >> 5, wb = (col + len - 1u) >> 5;
    mask |= (0xffffu >> (15u - wb)) & (0xffffu << wa);
  }
  return mask;
}

// Number of (cell, window) groups of every same-cell run, stored at the run's first segment (the array is zeroed
// first): the windows its pieces touch.  Its exclusive scan places the runs in the group directory.
__global__ void __launch_bounds__(256) rungroups_kernel(ExpandArgs a) {
  __shared__ uint32_t wmask[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t nm = (uint32_t)*a.tot_ms;
  const uint32_t cb = (blockIdx.x * 8u + (uint32_t)warp) * 32u;
  if (cb >= nm) return;
  wmask[warp][lane] = 0u;
  __syncwarp();
  int64_t first = -1;
  bool round0 = true;
  warp_runs(a, cb, nm, lane, [&](int64_t i, int runlane) {
    if (round0 && runlane == lane) first = i;
    round0 = false;
    if (i >= 0) atomicOr(&wmask[warp][runlane], segment_window_mask(a, i));
  });
  __syncwarp();
  if (first >= 0) a.goffs[first] = (uint32_t)__popc(wmask[warp][lane]);
}

// Singles and uncounted reads: one thread per sorted segment, units in piece / window order.
__global__ void __launch_bounds__(256) expand_single_kernel(ExpandArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int cls = segment_class(a.keys, i, a.n, a.cmask, a.unc);
  if (cls == 1 || (cls == 2 && !a.offs_u)) return;
  uint2 *q = a.units + (cls == 2 ? *a.tot_s + *a.tot_m + a.offs_u[i] : (uint64_t)a.offs_s[i]);
  segment_units(a, i, [&](uint32_t, uint2 u) { *q++ = u; });
}

// Run members: the units of a same-cell run are written WINDOW-MAJOR (all units of window 0, then window 1, ...)
// and the first unit of every non-empty window goes into the group directory, so that the count kernel can give a
// whole (cell, window) group to one lane.  Pass 1 counts the run's units per window (shared-memory counters of the
// lane that holds the run's first segment), pass 2 turns the counters into cursors and places the units.
__global__ void __launch_bounds__(256) expand_runs_kernel(ExpandArgs a) {
  __shared__ uint32_t cnt[8][32][17];  // [warp][runlane][window] (+1: no bank conflicts between run lanes)
  __shared__ uint32_t mbase[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t nm = (uint32_t)*a.tot_ms;
  const uint32_t cb = (blockIdx.x * 8u + (uint32_t)warp) * 32u;
  if (blockIdx.x == 0 && threadIdx.x == 0) a.gdir[*a.tot_g] = (uint32_t)*a.tot_m;  // sentinel: end of the last group
  if (cb >= nm) return;
#pragma unroll
  for (int w = 0; w < 16; ++w) cnt[warp][lane][w] = 0u;
  __syncwarp();
  int64_t first = -1;
  bool round0 = true;
  warp_runs(a, cb, nm, lane, [&](int64_t i, int runlane) {
    if (round0 && runlane == lane) first = i;
    round0 = false;
    if (i >= 0) segment_units(a, i, [&](uint32_t w, uint2) { atomicAdd(&cnt[warp][runlane][w], 1u); });
  });
  __syncwarp();
  if (first >= 0) {
    const uint32_t mb = a.offs_m[first];
    mbase[warp][lane] = mb;
    uint32_t *gd = a.gdir + a.goffs[first];
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < 16; ++w) {
      const uint32_t c = cnt[warp][lane][w];
      cnt[warp][lane][w] = run;
      if (c) *gd++ = mb + run;
      run += c;
    }
  }
  __syncwarp();
  uint2 *um = a.units + *a.tot_s;
  warp_runs(a, cb, nm, lane, [&](int64_t i, int runlane) {
    if (i < 0) return;
    const uint32_t mb = mbase[warp][runlane];
    segment_units(a, i, [&](uint32_t w, uint2 u) { um[mb + atomicAdd(&cnt[warp][runlane][w], 1u)] = u; });
  });
}

template <bool PACKED>
__global__ void __launch_bounds__(K1_THREADS, PACKED ? 3 : 1) pileup_count_kernel(CountArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TileSmemT<PACKED> &sm = *reinterpret_cast<TileSmemT<PACKED> *>(smem_raw);
  PartDesc pd;
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(a.parts + blockIdx.x);
    uint4 *dst = reinterpret_cast<uint4 *>(&pd);
    dst[0] = __ldg(src);
    dst[1] = __ldg(src + 1);
    dst[2] = __ldg(src + 2);
  }
  if (pd.slot == 0xffffffffu) return;  // unused entry between the heavy (front) and light (back) parts
  const int lane = threadIdx.x & 31;
  const int64_t slot = pd.slot;
  const uint32_t nparts = pd.nparts;
  const int32_t tile_start = pd.tile_start, tile_end = pd.tile_end;
  const uint64_t ref_base = pd.ref_base;

  {  // zero the accumulators, stage the reference bases, build the nibble tables
    uint4 *z = reinterpret_cast<uint4 *>(&sm);
    constexpr int NZ = ((PACKED ? K1_CROWS : 2 * K1_CROWS) + 8) * K1_ROWW / 4;  // hist + dup
    for (int i = threadIdx.x; i < NZ; i += K1_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
    if (a.min_ac > 0)
      for (int i = threadIdx.x; i < K1_ROWW; i += K1_THREADS) sm.acx[i] = 0u;
    for (int i = threadIdx.x; i < LS_TILE; i += K1_THREADS)
      sm.ref[i] = (tile_start + i < tile_end) ? upper_ascii(a.ref[ref_base + i]) : (uint8_t)'N';
    if (threadIdx.x < 16) {
      const int cls = class_of_code((uint32_t)threadIdx.x);
      sm.lut[threadIdx.x] = cls == LS_CLASS_NA ? K1_DUMP_OFF : (uint32_t)cls * 2u * K1_ROW_BYTES;
      // deletion-like units run as 'N' one class up (N -> O): their table carries O's bit and dup row
      const int c0 = cls == LS_CLASS_NA ? -1 : cls, c1 = cls == LS_CLASS_N ? LS_CLASS_O : -1;
      sm.lut2[0][threadIdx.x] = c0 < 0 ? 0u : (0x80u | (c0 < 6 ? (1u << c0) : 0u) | (((uint32_t)c0 * K1_ROW_BYTES) << 8));
      sm.lut2[1][threadIdx.x] = c1 < 0 ? 0u : (0x80u | (((uint32_t)c1 * K1_ROW_BYTES) << 8));
    }
    if (threadIdx.x == 0) {
      sm.next1 = 0;
      sm.next2 = 0;
      sm.next3 = 0;
      sm.npass = 0;
      sm.ticket = 0;
    }
  }
  __syncthreads();

  WarpCtx c;
  c.hist_s = (uint32_t)__cvta_generic_to_shared(&sm.hist[0][0]);
  c.lut_s = (uint32_t)__cvta_generic_to_shared(&sm.lut[0]);
  c.dup_s = (uint32_t)__cvta_generic_to_shared(&sm.dup[0][0]);
  {
    const int mq = a.min_bq < 0 ? 0 : (a.min_bq > 256 ? 256 : a.min_bq);
    c.thr = PACKED ? ((1u << K1_CNT_SHIFT) + (uint32_t)mq) : (uint32_t)mq;
    c.cnt1 = a.cnt1;
  }
  uint32_t seen[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) seen[i] = 0u;

  // ---- phase 1: the same-cell runs that start in the part.  Every lane works through whole (cell, window) groups,
  // which it claims one ahead from the part's slice of the group directory ---------------------------------------
  {
    const uint32_t g_lo = pd.g_lo, ngr = pd.g_n;
    const uint32_t *gd = a.gdir + g_lo;
    const uint2 *um = a.units + *a.tot_s;
    const uint32_t lt = (1u << lane) - 1u;
    // claim the next group for the lanes that ask; a lane that gets none keeps pn == en
    auto claim = [&](bool want, uint32_t &pn, uint32_t &en) {
      const uint32_t m = __ballot_sync(0xffffffffu, want);
      if (m == 0u) return;
      uint32_t base = 0;
      if (lane == __ffs(m) - 1) base = atomicAdd(&sm.next2, (uint32_t)__popc(m));
      base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
      if (want) {
        const uint32_t gi = base + (uint32_t)__popc(m & lt);
        pn = en = 0u;
        if (gi < ngr) {
          pn = __ldg(gd + gi);
          en = __ldg(gd + gi + 1u);
        }
      }
    };
    // the group in hand [p, e) and the two claimed after it; a lane walks them unit by unit
    uint32_t p = 0, e = 0, p1 = 0, e1 = 0, p2 = 0, e2 = 0;
    claim(true, p, e);
    claim(true, p1, e1);
    claim(true, p2, e2);
    // position of the unit k (1 or 2) steps after the one in hand; ok = there is one
    auto ahead = [&](int k, bool &ok) -> uint32_t {
      uint32_t a0 = p, b0 = e, a1 = p1, b1 = e1, a2 = p2, b2 = e2;
      for (int i = 0; i < k; ++i) {
        if (a0 + 1u < b0) {
          ++a0;
        } else {
          a0 = a1;
          b0 = b1;
          a1 = a2;
          b1 = b2;
          a2 = b2 = 0u;
        }
      }
      ok = a0 < b0;
      return a0;
    };
    bool ok1, ok2;
    uint2 u0 = p < e ? __ldg(um + p) : make_uint2(0u, 0u);
    const uint32_t q1 = ahead(1, ok1);
    uint2 u1 = ok1 ? __ldg(um + q1) : make_uint2(0u, 0u);
    URaw r0 = issue_unit(a, u0);
    bool fresh = true;  // the unit in hand opens its group
    while (__any_sync(0xffffffffu, p < e)) {
      const uint32_t q2 = ahead(2, ok2);
      const uint2 u2 = ok2 ? __ldg(um + q2) : make_uint2(0u, 0u);
      const URaw r1 = issue_unit(a, u1);
      const UData d0 = align_unit(r0, u0);
      if (fresh) {
#pragma unroll
        for (int i = 0; i < 8; ++i) seen[i] = 0u;
      }
      count_unit<PACKED, true>(c, u0.y, d0, lane, seen);
      const bool want = p < e && p + 1u >= e;
      if (p < e) {
        if (want) {
          p = p1;
          e = e1;
          p1 = p2;
          e1 = e2;
        } else {
          ++p;
        }
      }
      fresh = want;
      claim(want, p2, e2);
      u0 = u1;
      u1 = u2;
      r0 = r1;
    }
  }

  // ---- phase 2: the part's single-segment units, one unit per lane and step.  It runs AFTER the same-cell runs:
  // its guided grabs are fine-grained (one 32-unit batch at the end), so the warps that leave phase 1 early absorb
  // the time other warps still spend on their last long groups and the CTA reaches the barrier together ----------
  {
    const uint32_t nun = pd.s_n;
    const uint2 *us = a.units + pd.s_lo;
    // one 32-unit batch per grab; the warp claims its batches two steps ahead, so that the unit descriptors (two
    // ahead) and the units' bases (one ahead) are in flight while it counts -- the pipeline never drains between grabs
    auto grab = [&]() -> uint32_t {
      uint32_t g = 0;
      if (lane == 0) g = atomicAdd(&sm.next1, 32u);
      return __shfl_sync(0xffffffffu, g, 0) + (uint32_t)lane;
    };
    uint32_t k0 = grab(), k1 = grab();
    uint2 u0 = k0 < nun ? __ldg(us + k0) : make_uint2(0u, 0u);
    uint2 u1 = k1 < nun ? __ldg(us + k1) : make_uint2(0u, 0u);
    URaw r0 = issue_unit(a, u0);
    while (k0 - (uint32_t)lane < nun) {
      const uint32_t k2 = grab();
      const uint2 u2 = k2 < nun ? __ldg(us + k2) : make_uint2(0u, 0u);
      const URaw r1 = issue_unit(a, u1);
      const UData d0 = align_unit(r0, u0);
      count_unit<PACKED, false>(c, u0.y, d0, lane, seen);
      u0 = u1;
      u1 = u2;
      r0 = r1;
      k0 = k1;
      k1 = k2;
    }
  }

  // ---- phase 3: visible-but-uncounted reads (only emitted when --min_ac > 0) ---------------------------------
  if (a.with_u) {
    const uint2 *uu = a.units + *a.tot_s + *a.tot_m + pd.u_lo;
    const uint32_t nun = pd.u_n;
    for (;;) {
      uint32_t g = 0;
      if (lane == 0) g = atomicAdd(&sm.next3, 32u);
      g = __shfl_sync(0xffffffffu, g, 0);
      if (g >= nun) break;
      if (g + (uint32_t)lane < nun) count_unit_uncounted<PACKED>(a.qual, a.seq4, a.min_bq, sm, __ldg(uu + g + lane));
    }
  }
  __syncthreads();

  // ---- site epilogue: gates of BaseCellCounter.py:211,220-222,282,294 -------------------
  uint32_t *out = a.out + (size_t)slot * LS_SITE_WORDS * LS_TILE;
  bool last_part = true;
  uint32_t nev = 0;
  for (int pass_no = 0; pass_no < 2; ++pass_no) {
    // pass 0: per-part words (direct store for single-part tiles, atomic merge otherwise)
    // pass 1: only for the last part of a multi-part tile: gates on the merged totals
    if (pass_no == 1) {
      if (nparts == 1) break;
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) sm.ticket = atomicAdd(&a.slot_done[slot], 1u);
      __syncthreads();
      last_part = sm.ticket == nparts - 1;
      if (!last_part) break;
      __threadfence();
    }
    for (int s = threadIdx.x; s < LS_TILE; s += K1_THREADS) {
      const uint8_t rb = sm.ref[s];
      const int sc = k1_col(s);
      uint32_t dp = 0, nc = 0, ac = 0;
      uint32_t f[8], r[8], bq[6], cc[6];
      if (pass_no == 0) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          if (PACKED) {
            const uint32_t hf = sm.hist[k * 2][sc], hr = sm.hist[k * 2 + 1][sc];
            f[k] = hf >> K1_CNT_SHIFT;
            r[k] = hr >> K1_CNT_SHIFT;
            if (k < 6) bq[k] = (hf & ((1u << K1_CNT_SHIFT) - 1u)) + (hr & ((1u << K1_CNT_SHIFT) - 1u));
          } else {
            f[k] = sm.hist[k * 2][sc];
            r[k] = sm.hist[k * 2 + 1][sc];
            if (k < 6) bq[k] = sm.hist[K1_CROWS + k * 2][sc] + sm.hist[K1_CROWS + k * 2 + 1][sc];
          }
          dp += f[k] + r[k];
        }
        nev += dp;
        uint32_t dnc = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint32_t dw = sm.dup[k][sc];
          dnc += dw >> 16;
          if (k < 6) cc[k] = f[k] + r[k] - (dw & 0xffffu);
        }
        nc = dp - dnc;
        if (a.min_ac > 0) {
          ac = sm.acx[sc] + f[LS_CLASS_I] + r[LS_CLASS_I] + f[LS_CLASS_D] + r[LS_CLASS_D];
          const int base_cls[5] = {LS_CLASS_A, LS_CLASS_C, LS_CLASS_T, LS_CLASS_G, LS_CLASS_N};
#pragma unroll
          for (int j = 0; j < 5; ++j)
            if (class_letter(base_cls[j]) != rb) ac += f[base_cls[j]] + r[base_cls[j]];
        }
        if (nparts > 1) {
          if (dp) atomicAdd(&out[LS_SITE_DP * LS_TILE + s], dp);
          if (nc) atomicAdd(&out[LS_SITE_NC * LS_TILE + s], nc);
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            if (cc[k]) atomicAdd(&out[(LS_SITE_CC + k) * LS_TILE + s], cc[k]);
            if (f[k]) atomicAdd(&out[(LS_SITE_BCF + k) * LS_TILE + s], f[k]);
            if (r[k]) atomicAdd(&out[(LS_SITE_BCR + k) * LS_TILE + s], r[k]);
            if (bq[k]) atomicAdd(&out[(LS_SITE_BQ + k) * LS_TILE + s], bq[k]);
          }
          if (a.min_ac > 0 && ac) atomicAdd(&a.acbuf[(size_t)slot * LS_TILE + s], ac);
          continue;  // gates are applied in pass 1 by the last part
        }
      } else {
        dp = __ldcg(&out[LS_SITE_DP * LS_TILE + s]);
        nc = __ldcg(&out[LS_SITE_NC * LS_TILE + s]);
        if (a.min_ac > 0) ac = __ldcg(&a.acbuf[(size_t)slot * LS_TILE + s]);
      }
      bool pass = (tile_start + s < tile_end) && rb != 'N' && dp > 0 && (int)dp >= a.min_dp && (int)nc >= a.min_cc;
      if (pass && a.min_ac > 0) pass = (int)ac >= a.min_ac;
      const uint32_t bal = __ballot_sync(0xffffffffu, pass);
      if (lane == 0) {
        a.mask[(size_t)slot * (LS_TILE / 32) + (s >> 5)] = bal;
        if (bal) atomicAdd(&sm.npass, (uint32_t)__popc(bal));
      }
      if (pass_no == 0) {
        // Single-part tile: the warp's 32 columns leave as finished 26-word site records, the passing ones packed
        // at the front of the window's 32-record block of the slot.  They are transposed through the warp's own
        // columns of the 26 accumulator rows, which nobody reads any more (every lane has its column in registers).
        __syncwarp();
        uint32_t *stg = &sm.hist[0][0] + (s >> 5) * 33;
        if (pass) {
          // record e0/26 occupies words e0 .. e0+25 of the transposed block: at most two 32-word row segments
          const uint32_t e0 = (uint32_t)__popc(bal & ((1u << lane) - 1u)) * LS_SITE_WORDS;
          uint32_t *p0 = stg + (e0 >> 5) * K1_ROWW + (e0 & 31u);
          const int split = 32 - (int)(e0 & 31u);  // fields from `split` on continue in the next row segment
          auto put = [&](int fld, uint32_t v) { p0[fld + (fld >= split ? K1_ROWW - 32 : 0)] = v; };
          put(LS_SITE_DP, dp);
          put(LS_SITE_NC, nc);
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            put(LS_SITE_CC + k, cc[k]);
            put(LS_SITE_BCF + k, f[k]);
            put(LS_SITE_BCR + k, r[k]);
            put(LS_SITE_BQ + k, bq[k]);
          }
        }
        __syncwarp();
        uint32_t *dst = out + (s >> 5) * (32 * LS_SITE_WORDS) + lane;
        const int nw = __popc(bal) * LS_SITE_WORDS;
        const uint32_t *src = stg + lane;
        for (int i = lane; i < nw; i += 32, dst += 32, src += K1_ROWW) __stcs(dst, *src);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nev += __shfl_xor_sync(0xffffffffu, nev, o);
  if (lane == 0 && nev) atomicAdd(a.n_events, (unsigned long long)nev);
  __syncthreads();
  if (last_part && threadIdx.x == 0) a.npass[slot] = sm.npass;
}

// Where a slot's tile lies (compaction reads it instead of searching the window table again)
struct alignas(16) SlotDesc {
  int32_t tile_start, tid;
  uint64_t ref_base;
};

// One CTA per slot: split the slot into parts, write their descriptors (parts[] pre-set to 0xff), zero the HBM slot of
// multi-part tiles (their parts merge with atomics).
struct PartBuildArgs {
  const uint32_t *slot_lo;
  const int64_t *slot_tile;
  int64_t n_slots;
  const uint64_t *keys;
  const uint32_t *offs_s, *offs_u, *goffs;
  int64_t n_windows;
  const int32_t *wstart, *wend;
  const int64_t *wtile_base;
  const uint64_t *wref_off;
  PartDesc *parts;
  struct SlotDesc *slot_desc;
  const int32_t *wtid;
  uint32_t *slot_done;
  uint32_t *n_parts, *n_light;
  uint32_t max_parts;
  uint32_t *out, *acbuf;
};

// first sorted segment at or after i (inside the slot) that starts a same-cell run or a single
__device__ __forceinline__ uint32_t run_start_at_or_after(const uint64_t *__restrict__ keys, uint32_t i, uint32_t slot_lo,
                                                          uint32_t slot_hi) {
  if (i <= slot_lo) return slot_lo;
  while (i < slot_hi && keys[i] == keys[i - 1]) ++i;
  return i < slot_hi ? i : slot_hi;
}

__global__ void __launch_bounds__(128) part_build_kernel(PartBuildArgs a) {
  const int64_t slot = blockIdx.x;
  if (slot >= a.n_slots) return;
  const uint32_t slot_lo = a.slot_lo[slot], slot_hi = a.slot_lo[slot + 1];
  const uint32_t n = slot_hi - slot_lo;
  const uint32_t np = n == 0 ? 1u : (n + K1_PART_SEGS - 1) / K1_PART_SEGS;
  __shared__ uint32_t base;
  __shared__ int32_t sh_start, sh_end;
  __shared__ uint64_t sh_ref;
  if (threadIdx.x == 0) {
    // deep tiles first: their parts sit at the front of the grid, shallow tiles fill in behind (no long tail)
    if (n >= (uint32_t)K1_PART_SEGS / 2)
      base = atomicAdd(a.n_parts, np);
    else
      base = a.max_parts - np - atomicAdd(a.n_light, np);
    a.slot_done[slot] = 0;
    const int64_t tile = a.slot_tile[slot];
    const int64_t w = window_of_tile(a.wtile_base, a.n_windows, tile);
    const int32_t ts = a.wstart[w] + (int32_t)(tile - a.wtile_base[w]) * LS_TILE;
    sh_start = ts;
    sh_end = (ts + LS_TILE) < a.wend[w] ? (ts + LS_TILE) : a.wend[w];
    sh_ref = a.wref_off[w] + (uint64_t)(ts - a.wstart[w]);
    SlotDesc sd;
    sd.tile_start = ts;
    sd.tid = a.wtid[w];
    sd.ref_base = sh_ref;
    a.slot_desc[slot] = sd;
  }
  __syncthreads();
  for (uint32_t k = threadIdx.x; k < np; k += blockDim.x) {
    const uint32_t my_lo = slot_lo + k * K1_PART_SEGS;
    const uint32_t my_hi = (my_lo + K1_PART_SEGS) < slot_hi ? (my_lo + K1_PART_SEGS) : slot_hi;
    // same-cell runs never straddle parts: a run belongs to the part that holds its first segment
    uint32_t r_lo = my_lo, r_hi = my_hi;
    if (np > 1) {
      r_lo = run_start_at_or_after(a.keys, my_lo, slot_lo, slot_hi);
      r_hi = run_start_at_or_after(a.keys, my_hi, slot_lo, slot_hi);
    }
    PartDesc d;
    d.slot = (uint32_t)slot;
    d.nparts = np;
    d.tile_start = sh_start;
    d.tile_end = sh_end;
    d.ref_base = sh_ref;
    d.s_lo = a.offs_s[my_lo];
    d.s_n = a.offs_s[my_hi] - d.s_lo;
    d.g_lo = a.goffs[r_lo];
    d.g_n = a.goffs[r_hi] - d.g_lo;
    d.u_lo = a.offs_u ? a.offs_u[my_lo] : 0u;
    d.u_n = a.offs_u ? a.offs_u[my_hi] - d.u_lo : 0u;
    d.pad[0] = d.pad[1] = d.pad[2] = d.pad[3] = 0u;
    a.parts[base + k] = d;
  }
  if (np > 1) {
    uint32_t *o = a.out + (size_t)slot * LS_SITE_WORDS * LS_TILE;
    for (int i = threadIdx.x; i < LS_SITE_WORDS * LS_TILE; i += blockDim.x) o[i] = 0u;
    if (a.acbuf)
      for (int i = threadIdx.x; i < LS_TILE; i += blockDim.x) a.acbuf[(size_t)slot * LS_TILE + i] = 0u;
  }
}
