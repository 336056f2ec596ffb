// The .bai index format (SAM spec 5.2 / 5.3), header-only: the bin arithmetic, the parser and the region query.
// ls_bamsplit.cpp writes indexes with reg2bin; ls_bamstream.cpp reads them to decode only the BGZF members a run's
// regions need.  No other file knows the binning scheme.
#pragma once

#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

namespace lsbai {

static const uint32_t kMetaBin = 37450;  // samtools' pseudo-bin: per-reference offsets and record counts, not a bin
static const int64_t kMaxPos = (int64_t)1 << 29;
static const int kLinShift = 14;         // linear index windows of 16 kb

// the smallest bin that holds [beg, end)
inline int reg2bin(int64_t beg, int64_t end) {
  --end;
  if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

// every bin that may hold a record overlapping [beg, end)
inline void reg2bins(int64_t beg, int64_t end, std::vector<uint32_t> &out) {
  out.clear();
  if (beg < 0) beg = 0;
  if (end > kMaxPos) end = kMaxPos;
  if (end <= beg) return;
  --end;
  out.push_back(0);
  static const int shift[5] = {26, 23, 20, 17, 14};
  static const uint32_t base[5] = {1, 9, 73, 585, 4681};
  for (int l = 0; l < 5; ++l)
    for (int64_t k = base[l] + (beg >> shift[l]); k <= base[l] + (end >> shift[l]); ++k) out.push_back((uint32_t)k);
}

typedef std::pair<uint64_t, uint64_t> Chunk;  // virtual offsets [beg, end)

struct Ref {
  std::unordered_map<uint32_t, std::vector<Chunk>> bins;
  std::vector<uint64_t> lin;  // smallest virtual offset of a record overlapping each 16 kb window
};

struct Index {
  std::vector<Ref> refs;
};

// Parses a whole .bai; false with a reason in err when a count or a length does not fit the bytes.
inline bool parse(const uint8_t *p, size_t n, Index &idx, std::string &err) {
  size_t o = 0;
  auto need = [&](size_t k) { return n - o >= k; };
  auto u32 = [&]() { uint32_t x; memcpy(&x, p + o, 4); o += 4; return x; };
  auto u64 = [&]() { uint64_t x; memcpy(&x, p + o, 8); o += 8; return x; };
  if (!need(8) || memcmp(p, "BAI\1", 4) != 0) {
    err = "not a BAI file";
    return false;
  }
  o = 4;
  const uint32_t n_ref = u32();
  if (n_ref > (uint32_t)(n / 8)) {
    err = "corrupt index (reference count)";
    return false;
  }
  idx.refs.assign(n_ref, Ref());
  for (uint32_t r = 0; r < n_ref; ++r) {
    Ref &ref = idx.refs[r];
    if (!need(4)) goto truncated;
    const uint32_t n_bin = u32();
    for (uint32_t b = 0; b < n_bin; ++b) {
      if (!need(8)) goto truncated;
      const uint32_t bin = u32(), n_chunk = u32();
      if ((uint64_t)n_chunk * 16 > n - o) goto truncated;
      if (bin == kMetaBin) {
        o += (size_t)n_chunk * 16;
        continue;
      }
      std::vector<Chunk> &ch = ref.bins[bin];
      for (uint32_t c = 0; c < n_chunk; ++c) {
        const uint64_t a = u64(), e = u64();
        ch.emplace_back(a, e);
      }
    }
    if (!need(4)) goto truncated;
    const uint32_t n_intv = u32();
    if ((uint64_t)n_intv * 8 > n - o) goto truncated;
    ref.lin.resize(n_intv);
    for (uint32_t i = 0; i < n_intv; ++i) ref.lin[i] = u64();
  }
  return true;
truncated:
  err = "truncated index";
  return false;
}

// The chunks a query of [beg, end) on ref reads (SAM spec 5.3): those of reg2bins(beg, end) that end past the
// linear index's offset for beg, clipped to start there.  Appended to out, unsorted.
inline void query(const Ref &ref, int64_t beg, int64_t end, std::vector<Chunk> &out) {
  std::vector<uint32_t> bins;
  reg2bins(beg, end, bins);
  if (bins.empty()) return;
  uint64_t min_off = 0;
  if (!ref.lin.empty()) {
    const size_t w = (size_t)(std::max<int64_t>(beg, 0) >> kLinShift);
    min_off = ref.lin[std::min(w, ref.lin.size() - 1)];
  }
  for (uint32_t b : bins) {
    auto it = ref.bins.find(b);
    if (it == ref.bins.end()) continue;
    for (const Chunk &c : it->second)
      if (c.second > min_off) out.emplace_back(std::max(c.first, min_off), c.second);
  }
}

// Sorts the chunks and merges those that overlap or share a BGZF member (the next one starts in the member where the
// current one ends): the result is a sorted list of disjoint spans, no two of which inflate the same member.
inline void merge_spans(std::vector<Chunk> &ch) {
  std::sort(ch.begin(), ch.end());
  size_t k = 0;
  for (size_t i = 0; i < ch.size(); ++i) {
    if (ch[i].second <= ch[i].first) continue;
    if (k && (ch[i].first >> 16) <= (ch[k - 1].second >> 16))
      ch[k - 1].second = std::max(ch[k - 1].second, ch[i].second);
    else
      ch[k++] = ch[i];
  }
  ch.resize(k);
}

}  // namespace lsbai
