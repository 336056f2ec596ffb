// Host-side BAM splitter: the native half of the SplitBamCellTypes drop-in (SURVEY.md 8f-3).
//
// Reference behaviour restated (workflow/scripts/PreProcessing/SplitBamCellTypes.py:39-192; the
// pysam/htslib calls it makes are AlignmentFile.fetch / .write / pysam.index):
//   * every record with a reference id (fetch() without a region visits the placed records only) is
//     counted in Total_reads; no CB:Z tag -> CB_not_found; barcode (text before the first '-') not in
//     the table -> CB_not_matched;
//   * optional filters, evaluated together and reported as a ';'-joined reason: nM > max_nM
//     (nM_not_found when the tag is absent), NH > max_NH (NH_not_found), mapq < min_MQ (only when min_MQ > 0);
//   * optional end trimming: base qualities of the first trim_start and last trim_end query bases are
//     set to 0; a leading / trailing soft clip of length L extends the trim to L + n_trim, except that
//     20 <= L < 30 is treated as 30 (SplitBamCellTypes.py:140-160);
//   * the record is appended, otherwise byte for byte, to the BAM of its cell type; outputs get the
//     input's header, a BGZF EOF marker and a .bai index.
// Streaming: the input is read in ~64 MB compressed chunks whose BGZF members are inflated in parallel;
// each output keeps at most a few MB of pending records and hands full 0xff00-byte members to a background
// stage that deflates them in parallel and appends them to its file while the next input chunk is inflated
// and routed; the .bai is accumulated on uncompressed offsets and translated to virtual offsets at the end.
// Memory is bounded by the chunk sizes, not by the BAM.
// Differences by construction: members are deflated in parallel (so the compressed bytes differ from
// htslib's, the records do not).
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "ls_bai.h"
#include "ls_bgzf.h"

using namespace lsbgzf;

namespace {

// compressed bytes read per round / pending uncompressed bytes per output before a parallel deflate; the
// environment overrides exist for the tests, which force many rounds and mid-stream flushes on small files
static size_t env_size(const char *name, size_t dflt) {
  const char *v = getenv(name);
  if (!v || !*v) return dflt;
  const long long x = atoll(v);
  return x < 4096 ? (size_t)4096 : (size_t)x;
}
static const size_t kReadChunkDefault = 64u << 20, kFlushBytesDefault = 16u << 20;

struct AuxHit {
  bool found = false;
  bool is_int = false, is_float = false, is_text = false;
  int64_t ival = 0;
  double fval = 0;
  const char *text = nullptr;
};

// look one two-letter tag up in the aux block [p, end)
static AuxHit find_aux(const uint8_t *p, const uint8_t *end, char t0, char t1) {
  AuxHit h;
  while (p + 3 <= end) {
    const bool mine = (p[0] == (uint8_t)t0 && p[1] == (uint8_t)t1);
    const uint8_t ty = p[2];
    p += 3;
    switch (ty) {
      case 'A': case 'c': case 'C':
        if (mine) { h.found = h.is_int = true; h.ival = ty == 'c' ? (int8_t)p[0] : p[0]; return h; }
        p += 1; break;
      case 's': case 'S':
        if (mine) { h.found = h.is_int = true; h.ival = ty == 's' ? (int16_t)rd16(p) : rd16(p); return h; }
        p += 2; break;
      case 'i': case 'I':
        if (mine) { h.found = h.is_int = true; h.ival = ty == 'i' ? (int64_t)(int32_t)rd32(p) : (int64_t)rd32(p); return h; }
        p += 4; break;
      case 'f':
        if (mine) { h.found = h.is_float = true; uint32_t u = rd32(p); float f; memcpy(&f, &u, 4); h.fval = f; return h; }
        p += 4; break;
      case 'Z': case 'H': {
        const uint8_t *s = p;
        while (p < end && *p) ++p;
        if (p >= end) return h;
        ++p;
        if (mine) { h.found = h.is_text = true; h.text = reinterpret_cast<const char *>(s); return h; }
        break;
      }
      case 'B': {
        if (p + 5 > end) return h;
        const uint8_t sub = p[0];
        const uint32_t cnt = rd32(p + 1);
        p += 5;
        const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
        if (mine) { h.found = true; return h; }
        p += es * (size_t)cnt;
        break;
      }
      default: return h;
    }
  }
  return h;
}

static void put32(std::vector<uint8_t> &v, uint32_t x) {
  uint8_t b[4];
  wr32(b, x);
  v.insert(v.end(), b, b + 4);
}
static void put64(std::vector<uint8_t> &v, uint64_t x) {
  put32(v, (uint32_t)x);
  put32(v, (uint32_t)(x >> 32));
}

// .bai of a coordinate-sorted record stream (SAM spec 5.2, with the 37450 metadata bin samtools writes),
// accumulated record by record on UNCOMPRESSED stream offsets; finish() maps them to virtual offsets.
struct BaiBuilder {
  struct Ref {
    std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
    std::vector<uint64_t> lin;  // first record start per 16 kb window, UINT64_MAX = none yet
    uint64_t off_beg = 0, off_end = 0, n_map = 0, n_unmap = 0;
    bool any = false;
    int last_bin = -1;
  };
  std::vector<Ref> refs;
  int32_t prev_tid = -1, prev_beg = -1;
  bool sorted = true;

  explicit BaiBuilder(int n_ref) : refs((size_t)n_ref) {}

  void add(int32_t tid, int32_t beg, int32_t end, uint64_t u0, uint64_t u1, bool mapped) {
    if (tid < prev_tid || (tid == prev_tid && beg < prev_beg)) sorted = false;
    prev_tid = tid;
    prev_beg = beg;
    if (tid < 0 || (size_t)tid >= refs.size()) {
      sorted = false;
      return;
    }
    Ref &r = refs[(size_t)tid];
    const int b = lsbai::reg2bin(beg, end);
    auto &ch = r.bins[(uint32_t)b];
    if (b == r.last_bin && !ch.empty() && ch.back().second == u0)
      ch.back().second = u1;  // consecutive records of one bin form one chunk
    else
      ch.emplace_back(u0, u1);
    r.last_bin = b;
    const size_t w0 = (size_t)(beg >> lsbai::kLinShift), w1 = (size_t)((end - 1) >> lsbai::kLinShift);
    if (r.lin.size() <= w1) r.lin.resize(w1 + 1, UINT64_MAX);
    for (size_t w = w0; w <= w1; ++w)
      if (r.lin[w] == UINT64_MAX) r.lin[w] = u0;
    if (!r.any) r.off_beg = u0;
    r.off_end = u1;
    r.any = true;
    (mapped ? r.n_map : r.n_unmap)++;
  }

  template <typename VOFF>
  void finish(VOFF voff, std::vector<uint8_t> &bai) const {
    bai.clear();
    bai.insert(bai.end(), {'B', 'A', 'I', 1});
    put32(bai, (uint32_t)refs.size());
    for (const Ref &r : refs) {
      put32(bai, (uint32_t)(r.bins.size() + (r.any ? 1 : 0)));
      for (const auto &kv : r.bins) {
        put32(bai, kv.first);
        put32(bai, (uint32_t)kv.second.size());
        for (const auto &c : kv.second) {
          put64(bai, voff(c.first));
          put64(bai, voff(c.second));
        }
      }
      if (r.any) {
        put32(bai, lsbai::kMetaBin);
        put32(bai, 2u);
        put64(bai, voff(r.off_beg));
        put64(bai, voff(r.off_end));
        put64(bai, r.n_map);
        put64(bai, r.n_unmap);
      }
      put32(bai, (uint32_t)r.lin.size());
      uint64_t prev = 0;
      for (uint64_t u : r.lin) {  // windows no record starts in inherit the previous offset, as samtools does
        if (u != UINT64_MAX) prev = voff(u);
        put64(bai, prev);
      }
    }
    put64(bai, 0);  // records without coordinates: none are written
  }
};

// One output BAM: pending uncompressed bytes, the file, the compressed offset of every member written so far.
struct OutStream {
  std::string path;
  FILE *f = nullptr;
  std::vector<uint8_t> pending;
  uint64_t flushed = 0;         // uncompressed bytes already deflated (always a multiple of kBlockPayload)
  uint64_t c_total = 0;         // compressed bytes written
  std::vector<uint64_t> coff;   // file offset of member i
  BaiBuilder bai;

  OutStream(const std::string &p, int n_ref) : path(p), bai(n_ref) {}

  uint64_t tell() const { return flushed + pending.size(); }

  // Router side: cut the deflatable prefix off `pending` (everything when final) and account for it; the bytes
  // are handed to the background writer, which is the only thread that touches f / c_total / coff.
  bool take(bool final, std::vector<uint8_t> &chunk) {
    const size_t nbytes = final ? pending.size() : (pending.size() / kBlockPayload) * kBlockPayload;
    chunk.assign(pending.begin(), pending.begin() + (ptrdiff_t)nbytes);
    flushed += nbytes;
    pending.erase(pending.begin(), pending.begin() + (ptrdiff_t)nbytes);
    return nbytes != 0 || final;
  }

  // Writer side.
  bool write_chunk(const std::vector<uint8_t> &chunk, bool final, int threads, int level, std::string &err) {
    if (!chunk.empty()) {
      std::vector<uint8_t> comp;
      std::vector<uint64_t> rel;
      if (!deflate_stream(chunk.data(), chunk.size(), threads, level, comp, rel, err)) return false;
      for (size_t i = 0; i + 1 < rel.size(); ++i) coff.push_back(c_total + rel[i]);
      if (fwrite(comp.data(), 1, comp.size(), f) != comp.size()) {
        err = "short write to " + path;
        return false;
      }
      c_total += comp.size();
    }
    if (final) coff.push_back(c_total);  // virtual offset of the end of the stream = start of the EOF member
    return true;
  }

  uint64_t voff(uint64_t u) const { return (coff[u / kBlockPayload] << 16) | (u % kBlockPayload); }
};

// Background stage: deflates and appends the chunks the router hands over, in order, while the router goes on
// inflating and routing the next input.  Bounded queue (a few chunks) keeps memory bounded.
struct WriterStage {
  struct Job {
    int out;
    bool final;
    std::vector<uint8_t> data;
  };
  std::vector<OutStream> *outs = nullptr;
  int threads = 1, level = 6;
  std::deque<Job> q;
  std::mutex mu;
  std::condition_variable cv_push, cv_pop;
  bool stop = false;
  std::string err;
  std::thread th;
  static constexpr size_t kMaxJobs = 4;

  void start() {
    th = std::thread([this]() {
      for (;;) {
        Job j;
        {
          std::unique_lock<std::mutex> lk(mu);
          cv_pop.wait(lk, [this]() { return stop || !q.empty(); });
          if (q.empty()) return;
          j = std::move(q.front());
          q.pop_front();
        }
        cv_push.notify_one();
        std::string e;
        if (err.empty() && !(*outs)[(size_t)j.out].write_chunk(j.data, j.final, threads, level, e)) {
          std::lock_guard<std::mutex> lk(mu);
          err = e;
        }
      }
    });
  }
  // false when the writer has already failed (message in err)
  bool push(int out, bool final, std::vector<uint8_t> &&data) {
    std::unique_lock<std::mutex> lk(mu);
    cv_push.wait(lk, [this]() { return q.size() < kMaxJobs; });
    if (!err.empty()) return false;
    q.push_back(Job{out, final, std::move(data)});
    lk.unlock();
    cv_pop.notify_one();
    return true;
  }
  void finish() {
    if (!th.joinable()) return;
    {
      std::lock_guard<std::mutex> lk(mu);
      stop = true;
    }
    cv_pop.notify_one();
    th.join();
  }
};

static bool write_whole(const std::string &path, const std::vector<uint8_t> &a, std::string &err) {
  FILE *f = fopen(path.c_str(), "wb");
  if (!f) {
    err = "cannot create " + path;
    return false;
  }
  bool ok = a.empty() || fwrite(a.data(), 1, a.size(), f) == a.size();
  ok = (fclose(f) == 0) && ok;
  if (!ok) err = "short write to " + path;
  return ok;
}

// Sequential reader of a BGZF file: each round() appends the inflated payload of the next ~kReadChunk compressed
// bytes to `out` (members inflated in parallel) and returns false at end of file or on error (err set).
struct BgzfChunkReader {
  FILE *f = nullptr;
  std::vector<uint8_t> cbuf;
  size_t have = 0;
  bool eof = false;
  int threads = 1;
  size_t kReadChunk = kReadChunkDefault;

  bool round(std::vector<uint8_t> &out, std::string &err) {
    if (!eof) {
      cbuf.resize(have + kReadChunk);
      const size_t got = fread(cbuf.data() + have, 1, kReadChunk, f);
      have += got;
      if (got < kReadChunk) eof = true;
    }
    struct M {
      size_t coff, uoff;
      uint32_t csize, usize;
    };
    std::vector<M> ms;
    size_t off = 0, uo = out.size();
    while (off + 18 <= have) {
      const uint8_t *p = cbuf.data() + off;
      if (p[0] != 0x1f || p[1] != 0x8b || !(p[3] & 4)) {
        err = "not a BGZF file (bad gzip member header)";
        return false;
      }
      const uint32_t xlen = rd16(p + 10);
      if (off + 12 + xlen > have) break;
      uint32_t bsize = 0;
      const uint8_t *x = p + 12, *xe = p + 12 + xlen;
      while (x + 4 <= xe) {
        const uint32_t slen = rd16(x + 2);
        if (x[0] == 'B' && x[1] == 'C' && slen == 2) bsize = (uint32_t)rd16(x + 4) + 1;
        x += 4 + slen;
      }
      if (bsize == 0) {
        err = "corrupt BGZF block";
        return false;
      }
      if (off + bsize > have) break;
      M m;
      m.coff = off;
      m.csize = bsize;
      m.usize = rd32(p + bsize - 4);
      m.uoff = uo;
      ms.push_back(m);
      uo += m.usize;
      off += bsize;
    }
    if (ms.empty()) {
      if (eof && have == off) return false;  // clean end
      if (eof) {
        err = "truncated BGZF file";
        return false;
      }
      return true;  // a member larger than what is buffered cannot happen (<= 64 KiB); read more
    }
    out.resize(uo);
    std::atomic<size_t> next(0);
    std::atomic<int> bad(0);
    auto worker = [&]() {
      for (;;) {
        const size_t i = next.fetch_add(16);
        if (i >= ms.size()) break;
        for (size_t j = i; j < i + 16 && j < ms.size(); ++j)
          if (ms[j].usize && !inflate_member(cbuf.data() + ms[j].coff, ms[j].csize, out.data() + ms[j].uoff, ms[j].usize)) bad = 1;
      }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < (threads < 1 ? 1 : threads); ++t) th.emplace_back(worker);
    for (auto &t : th) t.join();
    if (bad) {
      err = "inflate failed";
      return false;
    }
    memmove(cbuf.data(), cbuf.data() + off, have - off);
    have -= off;
    return true;
  }
};

}  // namespace

// Reason bits of a filtered read (reported by the caller as 'nM;NH;MAPQ'-style keys)
enum { LS_SPLIT_NM = 1, LS_SPLIT_NM_MISSING = 2, LS_SPLIT_NH = 4, LS_SPLIT_NH_MISSING = 8, LS_SPLIT_MAPQ = 16 };

extern "C" {

// counters: [0] Total_reads, [1] Pass_reads, [2] CB_not_found, [3] CB_not_matched, [4 + mask] reads filtered
// for reason set `mask` (1..31); first_seen[mask] = ordinal (1-based, among visited reads) of the first read
// filtered for that set, 0 if none -- the reference's report lists reasons in first-occurrence order.
// max_nm / max_nh < 0 switch the filter off.  Returns 0, or -1 with a message in err.
int ls_bam_split(const char *in_path, int n_types, const char *const *out_paths, const char *bc_blob,
                 const uint32_t *bc_off, const int32_t *bc_type, int64_t n_bc, int min_mapq, int max_nm, int max_nh,
                 int n_trim, int threads, int level, int64_t *counters, int64_t *first_seen, char *err, int errlen) {
  std::string e;
  std::vector<OutStream> outs;
  BgzfChunkReader rd;
  WriterStage writer;
  auto fail = [&](const std::string &m) {
    writer.finish();
    snprintf(err, (size_t)errlen, "%s", m.c_str());
    for (auto &o : outs)
      if (o.f) fclose(o.f);
    if (rd.f) fclose(rd.f);
    return -1;
  };
  for (int k = 0; k < 36; ++k) counters[k] = 0;
  for (int k = 0; k < 32; ++k) first_seen[k] = 0;
  rd.f = fopen(in_path, "rb");
  if (!rd.f) return fail(std::string("cannot open ") + in_path);
  rd.threads = threads;
  rd.kReadChunk = env_size("LS_SPLIT_READ_CHUNK", kReadChunkDefault);
  const size_t kFlushBytes = env_size("LS_SPLIT_FLUSH_BYTES", kFlushBytesDefault);

  std::unordered_map<std::string, int32_t> table;
  table.reserve((size_t)n_bc * 2 + 1);
  for (int64_t i = 0; i < n_bc; ++i)
    table[std::string(bc_blob + bc_off[i], bc_off[i + 1] - bc_off[i])] = bc_type[i];  // later rows win, like dict()

  std::vector<uint8_t> ubuf;  // [carry of the previous round | newly inflated bytes]
  bool header_done = false;
  uint32_t n_ref = 0;
  int64_t visited = 0;
  std::string key;
  for (;;) {
    const size_t before = ubuf.size();
    const bool more = rd.round(ubuf, e);
    if (!e.empty()) return fail(e);
    const uint8_t *p = ubuf.data(), *end = ubuf.data() + ubuf.size();
    if (!header_done) {
      // magic, l_text, text, n_ref, then per reference l_name, name, l_ref: wait until all of it is buffered
      bool complete = false;
      size_t hl = 0;
      if (ubuf.size() >= 12) {
        if (memcmp(p, "BAM\1", 4) != 0) return fail("bad BAM magic");
        const uint64_t l_text = rd32(p + 4);
        if (ubuf.size() >= 12 + l_text) {
          n_ref = rd32(p + 8 + l_text);
          size_t q = 12 + (size_t)l_text;
          uint32_t i = 0;
          for (; i < n_ref; ++i) {
            if (q + 4 > ubuf.size()) break;
            const uint64_t l_name = rd32(p + q);
            if (q + 8 + l_name > ubuf.size()) break;
            q += 8 + (size_t)l_name;
          }
          if (i == n_ref) {
            complete = true;
            hl = q;
          }
        }
      }
      if (!complete) {
        if (!more) return fail(ubuf.empty() ? "empty file" : "truncated BAM header");
        continue;
      }
      outs.reserve((size_t)n_types);
      for (int t = 0; t < n_types; ++t) {
        outs.emplace_back(out_paths[t], (int)n_ref);
        outs.back().f = fopen(out_paths[t], "wb");
        if (!outs.back().f) return fail(std::string("cannot create ") + out_paths[t]);
        outs.back().pending.assign(p, p + hl);
      }
      writer.outs = &outs;
      writer.threads = threads;
      writer.level = level;
      writer.start();
      header_done = true;
      p += hl;
    }
    while (p + 4 <= end) {
      const uint32_t bs = rd32(p);
      if (bs < 32) return fail("corrupt BAM record");
      if (p + 4 + (size_t)bs > end) break;  // the rest of this record comes with the next round
      const uint8_t *r = p + 4;
      p = r + bs;
      const int32_t tid = (int32_t)rd32(r);
      if (tid < 0) continue;  // fetch() without a region does not visit reads without a reference
      ++visited;
      ++counters[0];
      const int32_t pos = (int32_t)rd32(r + 4);
      const uint32_t l_name = r[8], mapq = r[9];
      const uint32_t n_cig = rd16(r + 12), flag = rd16(r + 14), l_seq = rd32(r + 16);
      const uint8_t *cig = r + 32 + l_name;
      const uint8_t *seq = cig + 4 * (size_t)n_cig;
      const uint8_t *qual = seq + (l_seq + 1) / 2;
      const uint8_t *aux = qual + l_seq;
      if (aux > r + bs) return fail("corrupt BAM record");
      const AuxHit cb = find_aux(aux, r + bs, 'C', 'B');
      if (!cb.found) {
        ++counters[2];
        continue;
      }
      if (!cb.is_text) return fail("CB tag is not a string (the reference fails on barcode.split here)");
      const char *dash = strchr(cb.text, '-');
      key.assign(cb.text, dash ? (size_t)(dash - cb.text) : strlen(cb.text));
      auto it = table.find(key);
      if (it == table.end()) {
        ++counters[3];
        continue;
      }
      int mask = 0;
      if (max_nm >= 0) {
        const AuxHit h = find_aux(aux, r + bs, 'n', 'M');
        if (!h.found)
          mask |= LS_SPLIT_NM_MISSING;
        else if (!(h.is_int || h.is_float))
          return fail("nM tag is not numeric");
        else if ((h.is_int ? (double)h.ival : h.fval) > (double)max_nm)
          mask |= LS_SPLIT_NM;
      }
      if (max_nh >= 0) {
        const AuxHit h = find_aux(aux, r + bs, 'N', 'H');
        if (!h.found)
          mask |= LS_SPLIT_NH_MISSING;
        else if (!(h.is_int || h.is_float))
          return fail("NH tag is not numeric");
        else if ((h.is_int ? (double)h.ival : h.fval) > (double)max_nh)
          mask |= LS_SPLIT_NH;
      }
      if (min_mapq > 0 && (int)mapq < min_mapq) mask |= LS_SPLIT_MAPQ;
      if (mask) {
        ++counters[4 + mask];
        if (!first_seen[mask]) first_seen[mask] = visited;
        continue;
      }
      ++counters[1];
      OutStream &o = outs[(size_t)it->second];
      const uint64_t u0 = o.tell();
      const size_t at = o.pending.size();
      o.pending.insert(o.pending.end(), r - 4, r + bs);
      if (n_trim > 0) {
        uint32_t trim_start = (uint32_t)n_trim, trim_end = (uint32_t)n_trim;
        if (n_cig > 1) {
          const uint32_t c0 = rd32(cig), c1 = rd32(cig + 4 * (size_t)(n_cig - 1));
          if ((c0 & 15u) == 4u) trim_start = (((c0 >> 4) >= 20 && (c0 >> 4) < 30) ? 30u : (c0 >> 4)) + (uint32_t)n_trim;
          if ((c1 & 15u) == 4u) trim_end = (((c1 >> 4) >= 20 && (c1 >> 4) < 30) ? 30u : (c1 >> 4)) + (uint32_t)n_trim;
        }
        if (l_seq == 0 || qual[0] == 0xff) return fail("read without base qualities cannot be trimmed (TypeError in the reference)");
        if (trim_start > l_seq || trim_end > l_seq)
          return fail("IndexError: read shorter than the trimmed ends (the reference fails here as well)");
        uint8_t *q = o.pending.data() + at + 4 + (size_t)(qual - r);
        memset(q, 0, trim_start);
        memset(q + l_seq - trim_end, 0, trim_end);
      }
      // reference span for the index: M/D/N/=/X lengths (bam_endpos; 1 for records without one)
      int64_t span = 0;
      for (uint32_t k = 0; k < n_cig; ++k) {
        const uint32_t c = rd32(cig + 4 * (size_t)k), op = c & 15u;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += c >> 4;
      }
      const bool mapped = !(flag & 4u);
      o.bai.add(tid, pos, (int32_t)(pos + ((mapped && span > 0) ? span : 1)), u0, o.tell(), mapped);
      if (o.pending.size() >= kFlushBytes) {
        std::vector<uint8_t> chunk;
        if (o.take(false, chunk) && !writer.push(it->second, false, std::move(chunk))) return fail(writer.err);
      }
    }
    // keep the incomplete tail for the next round
    const size_t left = (size_t)(end - p);
    if (left) memmove(ubuf.data(), p, left);
    ubuf.resize(left);
    if (!more) {
      if (left) return fail("truncated BAM record");
      break;
    }
    (void)before;
  }
  if (!header_done) return fail("truncated BAM header");
  fclose(rd.f);
  rd.f = nullptr;

  for (size_t t = 0; t < outs.size(); ++t) {
    std::vector<uint8_t> chunk;
    outs[t].take(true, chunk);
    if (!writer.push((int)t, true, std::move(chunk))) return fail(writer.err);
  }
  writer.finish();
  if (!writer.err.empty()) return fail(writer.err);
  for (auto &o : outs) {
    bool ok = fwrite(kEofBlock, 1, sizeof kEofBlock, o.f) == sizeof kEofBlock;
    ok = (fclose(o.f) == 0) && ok;
    o.f = nullptr;
    if (!ok) return fail("short write to " + o.path);
    if (!o.bai.sorted) return fail("records are not sorted by coordinate: cannot index (" + o.path + ")");
    std::vector<uint8_t> bai;
    o.bai.finish([&](uint64_t u) { return o.voff(u); }, bai);
    if (!write_whole(o.path + ".bai", bai, e)) return fail(e);
  }
  return 0;
}

}  // extern "C"
