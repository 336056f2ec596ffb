// Streaming BAM -> structure-of-arrays decoder (host, no CUDA): the file is consumed a chunk of BGZF members at a
// time, so the memory in flight is bounded by the chunk size whatever the size of the BAM.
//
// Replaces, for the drop-in BaseCellCounter, the per-window `pysam.AlignmentFile.pileup` fetches of
// workflow/scripts/SNVCalling/BaseCellCounter.py:190-191,344-409 (the reference streams windows through a process
// pool; here the reads stream through chunks and the windows are completed on the fly, see pipeline.stream_chunks).
//
//   h = ls_bams_open(path, threads)                    header + contigs
//   ls_bams_set_regions(h, n, tid, beg, end)           optional: read only the BGZF members that the .bai lists for
//                                                      these regions (see read_index for when the index is refused)
//   n = ls_bams_next(h, target_bytes, &n_cigar, &n_bases)   the next chunk: ~target_bytes inflated (members in parallel),
//                                                      complete records indexed; a record cut by the chunk end is
//                                                      carried over.  The chunk AFTER it is inflated and indexed by a
//                                                      background thread while the caller works on this one.
//   ls_bams_fill(h, ...)                               parallel copy of the chunk into CALLER buffers (pinned staging
//                                                      memory of the CUDA library: the decoder writes where the H2D
//                                                      copy reads)
// Barcodes (CB:Z) are interned across chunks: ids are stable for the whole file.
// The compressed input is a list of segments, whole BGZF members each: the whole file, or one per span of virtual
// offsets the index gives for the regions.  A segment's first member is parsed from the span's in-block offset on and
// its last member up to the span's end, so the inflated bytes are exactly the records of the spans, in file order.
// Every length field is checked against the bytes that are actually there: a truncated or corrupt file is an error
// string, never an out-of-bounds read.
#include <zlib.h>

#include "ls_bai.h"
#include "ls_inflate.h"

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace {

inline uint32_t rd32(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline uint16_t rd16(const uint8_t *p) { return (uint16_t)(p[0] | (p[1] << 8)); }
inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Member {
  size_t coff;     // offset in the compressed buffer
  uint32_t csize, usize;
  size_t uoff;     // offset in the inflated buffer (after the carried bytes)
  uint32_t skip, keep_end;  // the member's inflated bytes [skip, keep_end) are kept
};

// Compressed bytes [c0, c1) of the file, whole members.  The first member's inflated bytes start at `skip`; the member
// at last_coff (if any) ends at last_keep.
struct Segment {
  uint64_t c0, c1;
  uint32_t skip;
  uint64_t last_coff;
  uint32_t last_keep;
};

// Byte buffer that grows without zero-filling (a std::vector would clear 256 MB per chunk before inflate overwrites it)
struct ByteBuf {
  uint8_t *p = nullptr;
  size_t n = 0, cap = 0;
  ~ByteBuf() { free(p); }
  bool resize(size_t want) {
    if (want > cap) {
      const size_t c = want + want / 8 + 4096;
      uint8_t *q = (uint8_t *)realloc(p, c);
      if (!q) return false;
      p = q;
      cap = c;
    }
    n = want;
    return true;
  }
};

// One decoded chunk: inflated bytes (the previous chunk's cut record first) and the index of its complete records
struct Chunk {
  ByteBuf raw;
  size_t tail_lo = 0;                 // first byte of raw not covered by a complete record
  std::vector<const uint8_t *> recs;  // records (pointers into raw, past block_size)
  std::vector<const char *> cbp;      // their CB:Z texts (or nullptr)
  std::vector<uint64_t> cbh;          // ... and the hashes of those texts
  std::vector<uint32_t> ncig, lseq;   // n_cigar_op / l_seq of every record (read once, in parallel)
  std::vector<uint32_t> cig_off;
  std::vector<uint64_t> base_off;
  std::vector<int32_t> cb;
  int64_t n = 0;                      // complete records; -1 = error (err)
  int64_t n_cigar = 0, n_bases = 0;
  int64_t comp_bytes = 0, infl_bytes = 0;  // compressed member bytes read and bytes inflated to produce the chunk
  int32_t n_barcodes = 0;             // size of the barcode table when the chunk was indexed
  std::string err;
};

// barcode text -> dense id, ids stable for the whole file; open addressing on a 64-bit FNV-1a hash
struct BarcodeTable {
  std::deque<std::string> names;  // element addresses stay valid while the table grows
  std::vector<int32_t> slot;
  std::vector<uint64_t> hash;
  std::mutex mu;                  // names is read by the caller's thread while the prefetch thread appends
  BarcodeTable() : slot(1 << 12, -1), hash(1 << 12, 0) {}
  static uint64_t fnv(const char *s) {
    uint64_t h = 1469598103934665603ull;
    for (; *s; ++s) h = (h ^ (uint8_t)*s) * 1099511628211ull;
    return h;
  }
  int32_t intern(const char *s, uint64_t h) {
    size_t m = slot.size() - 1, i = (size_t)h & m;
    for (;; i = (i + 1) & m) {
      const int32_t id = slot[i];
      if (id < 0) break;
      if (hash[i] == h && names[(size_t)id] == s) return id;
    }
    std::lock_guard<std::mutex> g(mu);
    const int32_t id = (int32_t)names.size();
    names.emplace_back(s);
    slot[i] = id;
    hash[i] = h;
    if (names.size() * 2 > slot.size()) {  // rehash at load 1/2
      std::vector<int32_t> s2(slot.size() * 2, -1);
      std::vector<uint64_t> h2(slot.size() * 2, 0);
      m = s2.size() - 1;
      for (size_t k = 0; k < slot.size(); ++k) {
        if (slot[k] < 0) continue;
        size_t j = (size_t)hash[k] & m;
        while (s2[j] >= 0) j = (j + 1) & m;
        s2[j] = slot[k];
        h2[j] = hash[k];
      }
      slot.swap(s2);
      hash.swap(h2);
    }
    return id;
  }
};

struct Stream {
  std::string err, path;
  int fd = -1;
  uint64_t file_size = 0;
  int threads = 1;
  double t_read = 0, t_inflate = 0, t_index = 0, t_tags = 0, t_intern = 0, t_fill = 0, t_wait = 0;  // LS_BAM_TIMING
  bool header_done = false, started = false;
  std::vector<std::string> contig_names;
  std::vector<int32_t> contig_lens;
  BarcodeTable bar;
  std::vector<Segment> segs;  // what is read, in file order
  size_t seg = 0;             // the segment being read
  uint64_t rd_off = 0;        // next file offset of segs[seg] to read
  uint64_t comp_file_off = 0; // file offset of comp[comp_lo]
  std::string index_note = "regions not set";  // why the index is not used ("" when it is)
  int64_t comp_bytes = 0, infl_bytes = 0;  // since the last chunk was produced
  int64_t tot_comp = 0, tot_infl = 0;      // of the chunks handed out
  std::vector<uint8_t> comp;  // compressed bytes read but not yet consumed
  size_t comp_lo = 0;         // first unconsumed byte of comp
  Chunk ch[2];
  int cur = 0;                // the chunk the caller sees; the other one is being produced / is the next one
  std::thread pf;
  bool pf_running = false;
};

bool inflate_block(z_stream &zs, const uint8_t *src, uint32_t csize, uint8_t *dst, uint32_t usize) {
  if (csize < 26) return false;
  const uint32_t xlen = rd16(src + 10);
  if (12u + xlen + 8u > csize) return false;
  const uint8_t *def = src + 12 + xlen;
  const uint32_t dlen = csize - 12 - xlen - 8;
  {
    static thread_local lsinf::Tables tabs;  // own decoder first; zlib judges whatever it does not accept
    if (!getenv("LS_ZLIB_INFLATE") && lsinf::inflate_raw(def, dlen, dst, usize, tabs)) return true;
  }
  if (inflateReset(&zs) != Z_OK) return false;
  zs.next_in = const_cast<Bytef *>(def);
  zs.avail_in = dlen;
  zs.next_out = dst;
  zs.avail_out = usize;
  const int rc = inflate(&zs, Z_FINISH);
  return rc == Z_STREAM_END && zs.total_out == usize;
}


// "CB" aux tag of type Z: pointer to its NUL-terminated text, or nullptr
const char *find_cb(const uint8_t *p, const uint8_t *end) {
  while (p + 3 <= end) {
    const uint8_t t0 = p[0], t1 = p[1], ty = p[2];
    p += 3;
    const bool is_cb = (t0 == 'C' && t1 == 'B');
    switch (ty) {
      case 'A': case 'c': case 'C': p += 1; break;
      case 's': case 'S': p += 2; break;
      case 'i': case 'I': case 'f': p += 4; break;
      case 'Z': case 'H': {
        const uint8_t *s = p;
        while (p < end && *p) ++p;
        if (p >= end) return nullptr;
        ++p;
        if (is_cb && ty == 'Z') return reinterpret_cast<const char *>(s);
        break;
      }
      case 'B': {
        if (p + 5 > end) return nullptr;
        const uint8_t sub = p[0];
        const uint32_t cnt = rd32(p + 1);
        p += 5;
        const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
        if ((size_t)(end - p) < es * (size_t)cnt) return nullptr;
        p += es * (size_t)cnt;
        break;
      }
      default: return nullptr;
    }
  }
  return nullptr;
}


bool pread_all(int fd, uint8_t *dst, size_t n, uint64_t off) {
  while (n) {
    const ssize_t k = pread(fd, dst, n, (off_t)off);
    if (k < 0 && errno == EINTR) continue;
    if (k <= 0) return false;
    dst += k;
    n -= (size_t)k;
    off += (uint64_t)k;
  }
  return true;
}

// Make sure at least `want` unconsumed compressed bytes of the current segment are buffered (or the segment is
// exhausted).  Bytes below `pin` (the first member of the call in progress, still to be inflated) are kept; returns
// how far the buffer was shifted.
size_t refill(Stream *s, size_t want, size_t pin) {
  if (s->comp.size() - s->comp_lo >= want || s->seg >= s->segs.size()) return 0;
  const Segment &g = s->segs[s->seg];
  if (s->rd_off >= g.c1) return 0;
  size_t shift = 0;
  if (pin) {
    s->comp.erase(s->comp.begin(), s->comp.begin() + (ptrdiff_t)pin);
    s->comp_lo -= pin;
    shift = pin;
  }
  const size_t have = s->comp.size();
  // the header is read in small steps: with an index, what follows it is not needed
  const size_t step = s->header_done ? (size_t)(8u << 20) : (size_t)(256u << 10);
  const size_t grab = (size_t)std::min<uint64_t>(std::max(want, step), g.c1 - s->rd_off);
  s->comp.resize(have + grab);
  const double t0 = now_s();
  const bool ok = pread_all(s->fd, s->comp.data() + have, grab, s->rd_off);
  s->t_read += now_s() - t0;
  if (!ok) {  // the file is shorter than it was: what is buffered is all there is
    s->comp.resize(have);
    s->rd_off = g.c1;
    return shift;
  }
  s->rd_off += grab;
  return shift;
}

// Inflate members until the inflated size of this call reaches target (at least one member); appended to raw.
bool inflate_some(Stream *s, ByteBuf &raw, size_t target, std::string &err) {
  std::vector<Member> mem;
  size_t usum = 0;
  const size_t raw0 = raw.n;
  size_t pin = s->comp_lo;  // everything from here on is needed until the members below are inflated
  auto need = [&](size_t want) {
    const size_t shift = refill(s, want, pin);
    if (shift) {
      for (auto &m : mem) m.coff -= shift;
      pin = 0;
    }
    return s->comp.size() - s->comp_lo >= want;
  };
  for (;;) {
    if (!need(18)) {
      if (s->comp.size() - s->comp_lo != 0) {
        err = "truncated BGZF member header";
        return false;
      }
      if (s->seg + 1 >= s->segs.size()) break;
      ++s->seg;  // the next segment starts in an empty buffer
      s->rd_off = s->comp_file_off = s->segs[s->seg].c0;
      continue;
    }
    const uint8_t *p = s->comp.data() + s->comp_lo;
    if (p[0] != 0x1f || p[1] != 0x8b || !(p[3] & 4)) {
      err = "not a BGZF file (bad gzip member header)";
      return false;
    }
    const uint32_t xlen = rd16(p + 10);
    if (!need(12 + (size_t)xlen)) {
      err = "truncated BGZF extra field";
      return false;
    }
    p = s->comp.data() + s->comp_lo;
    uint32_t bsize = 0;
    const uint8_t *x = p + 12, *xe = p + 12 + xlen;
    while (x + 4 <= xe) {
      const uint32_t slen = rd16(x + 2);
      if (x[0] == 'B' && x[1] == 'C' && slen == 2 && x + 6 <= xe) bsize = (uint32_t)rd16(x + 4) + 1;
      x += 4 + slen;
    }
    if (bsize < 12 + xlen + 8) {
      err = "corrupt BGZF block (no BC field or bad size)";
      return false;
    }
    if (!need(bsize)) {
      err = "truncated BGZF member";
      return false;
    }
    p = s->comp.data() + s->comp_lo;
    Member m;
    m.coff = s->comp_lo;
    m.csize = bsize;
    m.usize = rd32(p + bsize - 4);
    if (m.usize > 65536u) {
      err = "corrupt BGZF block (ISIZE > 64 KiB)";
      return false;
    }
    const Segment &g = s->segs[s->seg];
    m.skip = s->comp_file_off == g.c0 ? g.skip : 0;
    m.keep_end = s->comp_file_off == g.last_coff ? g.last_keep : m.usize;
    if (m.skip > m.keep_end || m.keep_end > m.usize) {
      err = "index offset past the end of a BGZF member";
      return false;
    }
    m.uoff = raw0 + usum;
    mem.push_back(m);
    usum += m.keep_end - m.skip;
    s->comp_bytes += bsize;
    s->infl_bytes += m.usize;
    s->comp_lo += bsize;
    s->comp_file_off += bsize;
    if (usum >= target) break;
  }
  if (mem.empty()) return true;
  const double t_i0 = now_s();
  if (!raw.resize(raw0 + usum + 8)) {  // + 8: the inflater's word-wide copies may touch bytes past a member's end
    err = "out of memory";
    return false;
  }
  raw.n = raw0 + usum;
  std::atomic<size_t> next(0);
  std::atomic<int> bad(0);
  auto worker = [&]() {
    std::vector<uint8_t> part;  // a member only partly kept is inflated here first
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) {
      bad = 1;
      return;
    }
    for (;;) {
      const size_t i = next.fetch_add(8);
      if (i >= mem.size()) break;
      for (size_t j = i; j < i + 8 && j < mem.size(); ++j) {
        const Member &m = mem[j];
        if (!m.usize) continue;
        if (m.skip == 0 && m.keep_end == m.usize) {
          if (!inflate_block(zs, s->comp.data() + m.coff, m.csize, raw.p + m.uoff, m.usize)) bad = 1;
          continue;
        }
        part.resize((size_t)m.usize + 8);
        if (!inflate_block(zs, s->comp.data() + m.coff, m.csize, part.data(), m.usize)) bad = 1;
        else memcpy(raw.p + m.uoff, part.data() + m.skip, m.keep_end - m.skip);
      }
    }
    inflateEnd(&zs);
  };
  std::vector<std::thread> th;
  for (int t = 0; t < s->threads; ++t) th.emplace_back(worker);
  for (auto &t : th) t.join();
  s->t_inflate += now_s() - t_i0;
  if (bad) {
    err = "inflate failed";
    return false;
  }
  return true;
}

// BAM header + reference table at the start of raw; need_more if more bytes are needed
bool parse_header(Stream *s, const ByteBuf &raw, size_t &consumed, bool &need_more) {
  need_more = false;
  const uint8_t *p = raw.p, *end = p + raw.n;
  if (raw.n < 12) {
    need_more = true;
    return true;
  }
  if (memcmp(p, "BAM\1", 4) != 0) {
    s->err = "bad BAM magic";
    return false;
  }
  const uint64_t l_text = rd32(p + 4);
  if ((uint64_t)(end - p) < 12 + l_text) {
    need_more = true;
    return true;
  }
  const uint8_t *q = p + 8 + l_text;
  const uint32_t n_ref = rd32(q);
  q += 4;
  std::vector<std::string> names;
  std::vector<int32_t> lens;
  for (uint32_t i = 0; i < n_ref; ++i) {
    if (end - q < 4) {
      need_more = true;
      return true;
    }
    const uint64_t l_name = rd32(q);
    if ((uint64_t)(end - q) < 8 + l_name) {
      need_more = true;
      return true;
    }
    names.emplace_back(reinterpret_cast<const char *>(q + 4), l_name ? (size_t)l_name - 1 : 0);
    lens.push_back((int32_t)rd32(q + 4 + l_name));
    q += 8 + l_name;
  }
  s->contig_names.swap(names);
  s->contig_lens.swap(lens);
  consumed = (size_t)(q - p);
  return true;
}

// Produce the chunk that follows `prev` into `dst`: prev's cut record, ~target more inflated bytes, the record index.
// Runs on the caller's thread (first chunk) or on the prefetch thread; touches only dst, the compressed-side state
// of the stream and the barcode table.
void produce(Stream *s, Chunk &dst, const Chunk &prev, size_t target) {
  dst.err.clear();
  dst.recs.clear();
  dst.n = 0;
  dst.n_cigar = dst.n_bases = 0;
  struct Account {  // the bytes read since the previous chunk are this chunk's, whichever way produce() returns
    Stream *s;
    Chunk &c;
    ~Account() {
      c.comp_bytes = s->comp_bytes;
      c.infl_bytes = s->infl_bytes;
      s->comp_bytes = s->infl_bytes = 0;
    }
  } account{s, dst};
  const size_t carry = prev.raw.n - prev.tail_lo;
  if (!dst.raw.resize(carry + 8)) {
    dst.err = "out of memory";
    dst.n = -1;
    return;
  }
  dst.raw.n = carry;
  if (carry) memcpy(dst.raw.p, prev.raw.p + prev.tail_lo, carry);
  dst.tail_lo = 0;
  for (;;) {  // until the chunk holds a complete record (a record may be larger than the chunk) or the file ends
    const size_t before = dst.raw.n;
    if (!inflate_some(s, dst.raw, target > 65536 ? target : 65536, dst.err)) {
      dst.n = -1;
      return;
    }
    const double t_x0 = now_s();
    dst.recs.clear();
    const uint8_t *p = dst.raw.p, *end = p + dst.raw.n;
    while (end - p >= 4) {
      const uint64_t bs = rd32(p);
      if (bs < 32) {
        dst.err = "corrupt BAM record (block_size < 32)";
        dst.n = -1;
        return;
      }
      if ((uint64_t)(end - p) < 4 + bs) break;  // cut by the chunk end: carried over
      dst.recs.push_back(p + 4);
      p += 4 + bs;
    }
    dst.tail_lo = (size_t)(p - dst.raw.p);
    s->t_index += now_s() - t_x0;
    if (!dst.recs.empty()) break;
    if (dst.raw.n == before) {  // nothing more to inflate
      if (dst.raw.n - dst.tail_lo > 0) {
        dst.err = "truncated BAM record at end of file";
        dst.n = -1;
      }
      dst.n_barcodes = (int32_t)s->bar.names.size();
      return;
    }
  }
  const double t_x1 = now_s();
  const int64_t n = (int64_t)dst.recs.size();
  dst.cig_off.resize((size_t)n + 1);
  dst.base_off.resize((size_t)n + 1);
  dst.cb.resize((size_t)n);
  dst.cbp.resize((size_t)n);
  dst.cbh.resize((size_t)n);
  dst.ncig.resize((size_t)n);
  dst.lseq.resize((size_t)n);
  // per record, in parallel: field check and the CB tag's text (each record's aux block is a cache miss)
  std::atomic<int64_t> nx(0);
  std::atomic<int> bad(0);
  auto scan = [&]() {
    for (;;) {
      const int64_t i0 = nx.fetch_add(4096);
      if (i0 >= n) break;
      for (int64_t i = i0; i < i0 + 4096 && i < n; ++i) {
        const uint8_t *r = dst.recs[(size_t)i];
        const uint64_t bs = rd32(r - 4);
        const uint64_t l_name = r[8], n_cig = rd16(r + 12), l_seq = rd32(r + 16);
        const uint64_t fixed = 32 + l_name + 4 * n_cig + (l_seq + 1) / 2 + l_seq;
        dst.ncig[(size_t)i] = (uint32_t)n_cig;
        dst.lseq[(size_t)i] = (uint32_t)l_seq;
        if (fixed > bs) {
          bad = 1;
          dst.cbp[(size_t)i] = nullptr;
          continue;
        }
        const char *cbs = find_cb(r + fixed, r + bs);
        dst.cbp[(size_t)i] = cbs;
        dst.cbh[(size_t)i] = cbs ? BarcodeTable::fnv(cbs) : 0;
      }
    }
  };
  {
    std::vector<std::thread> th;
    for (int t = 0; t < s->threads; ++t) th.emplace_back(scan);
    for (auto &t : th) t.join();
  }
  const double t_x2 = now_s();
  s->t_tags += t_x2 - t_x1;
  if (bad) {
    dst.err = "corrupt BAM record (fields exceed block_size)";
    dst.n = -1;
    return;
  }
  uint64_t co = 0, bo = 0;
  for (int64_t i = 0; i < n; ++i) {
    const uint64_t n_cig = dst.ncig[(size_t)i], l_seq = dst.lseq[(size_t)i];
    dst.cig_off[(size_t)i] = (uint32_t)co;
    dst.base_off[(size_t)i] = bo;
    co += n_cig;
    bo += (l_seq + 15u) & ~(uint64_t)15u;
    const char *cbs = dst.cbp[(size_t)i];
    dst.cb[(size_t)i] = cbs ? s->bar.intern(cbs, dst.cbh[(size_t)i]) : -1;
  }
  if (co >= 0xffffffffull) {
    dst.err = "more than 2^32 CIGAR operations in one chunk";
    dst.n = -1;
    return;
  }
  dst.cig_off[(size_t)n] = (uint32_t)co;
  dst.base_off[(size_t)n] = bo;
  dst.n_cigar = (int64_t)co;
  dst.n_bases = (int64_t)bo;
  dst.n = n;
  dst.n_barcodes = (int32_t)s->bar.names.size();
  s->t_intern += now_s() - t_x2;
}

// The BGZF member at file offset off: its compressed size and ISIZE; false when off is not at a whole member.
bool member_at(const Stream *s, uint64_t off, uint32_t &bsize, uint32_t &isize) {
  uint8_t hd[18], tl[4];
  if (off + 26 > s->file_size || !pread_all(s->fd, hd, 18, off)) return false;
  if (hd[0] != 0x1f || hd[1] != 0x8b || hd[2] != 8 || !(hd[3] & 4) || rd16(hd + 10) != 6 || hd[12] != 'B' ||
      hd[13] != 'C' || rd16(hd + 14) != 2)
    return false;
  bsize = (uint32_t)rd16(hd + 16) + 1;
  if (bsize < 26 || off + bsize > s->file_size || !pread_all(s->fd, tl, 4, off + bsize - 4)) return false;
  isize = rd32(tl);
  return isize <= 65536u;
}

// Reads <bam>.bai (or <bam without .bam>.bai) and turns the regions' queries into segments.  An index that is missing,
// unreadable, older than the BAM, made for another header, or that points anywhere but into whole members of the file
// is not used: false, with the reason in s->index_note.
bool use_index(Stream *s, int64_t n, const int32_t *tid, const int64_t *beg, const int64_t *end,
               std::vector<Segment> &segs) {
  std::string bai = s->path + ".bai";
  struct stat sb, si;
  if (stat(bai.c_str(), &si) != 0 && s->path.size() > 4 && s->path.compare(s->path.size() - 4, 4, ".bam") == 0)
    bai = s->path.substr(0, s->path.size() - 4) + ".bai";
  if (stat(bai.c_str(), &si) != 0) {
    s->index_note = "no .bai index";
    return false;
  }
  if (fstat(s->fd, &sb) != 0 || si.st_mtim.tv_sec < sb.st_mtim.tv_sec ||
      (si.st_mtim.tv_sec == sb.st_mtim.tv_sec && si.st_mtim.tv_nsec < sb.st_mtim.tv_nsec)) {
    s->index_note = bai + " is older than the BAM";
    return false;
  }
  std::vector<uint8_t> buf;
  {
    const int fd = open(bai.c_str(), O_RDONLY | O_CLOEXEC);
    struct stat st;
    bool ok = fd >= 0 && fstat(fd, &st) == 0;
    if (ok) {
      buf.resize((size_t)st.st_size);
      ok = pread_all(fd, buf.data(), buf.size(), 0);
    }
    if (fd >= 0) close(fd);
    if (!ok) {
      s->index_note = "cannot read " + bai;
      return false;
    }
  }
  lsbai::Index idx;
  std::string why;
  if (!lsbai::parse(buf.data(), buf.size(), idx, why)) {
    s->index_note = bai + ": " + why;
    return false;
  }
  if (idx.refs.size() != s->contig_names.size()) {
    s->index_note = bai + " lists " + std::to_string(idx.refs.size()) + " references, the BAM header " +
                    std::to_string(s->contig_names.size());
    return false;
  }
  // regions that overlap or touch are one query
  std::vector<std::pair<int64_t, int64_t>> reg;  // (tid << 32 | beg, end)
  for (int64_t i = 0; i < n; ++i)
    if (tid[i] >= 0 && (size_t)tid[i] < idx.refs.size() && end[i] > beg[i] && end[i] > 0)
      reg.emplace_back(((int64_t)tid[i] << 32) | std::max<int64_t>(beg[i], 0), end[i]);
  std::sort(reg.begin(), reg.end());
  std::vector<lsbai::Chunk> spans;
  for (size_t i = 0; i < reg.size();) {
    const int64_t t = reg[i].first >> 32, b = reg[i].first & 0xffffffffll;
    int64_t e = reg[i].second;
    size_t j = i + 1;
    for (; j < reg.size() && (reg[j].first >> 32) == t && (reg[j].first & 0xffffffffll) <= e; ++j)
      e = std::max(e, reg[j].second);
    lsbai::query(idx.refs[(size_t)t], b, e, spans);
    i = j;
  }
  lsbai::merge_spans(spans);
  segs.clear();
  for (const lsbai::Chunk &c : spans) {
    const uint64_t c0 = c.first >> 16, c1 = c.second >> 16;
    const uint32_t u0 = (uint32_t)(c.first & 0xffff), u1 = (uint32_t)(c.second & 0xffff);
    uint32_t bsize = 0, isize = 0;
    Segment g{c0, c1, u0, c1, u1};
    if (!member_at(s, c0, bsize, isize) || u0 > isize || (!segs.empty() && c0 < segs.back().c1)) {
      s->index_note = bai + ": a chunk starts outside the BAM's BGZF members";
      return false;
    }
    if (u1) {
      if (!member_at(s, c1, bsize, isize) || u1 > isize) {
        s->index_note = bai + ": a chunk ends outside the BAM's BGZF members";
        return false;
      }
      g.c1 = c1 + bsize;
    } else if (c1 > s->file_size || (c1 < s->file_size && !member_at(s, c1, bsize, isize))) {
      s->index_note = bai + ": a chunk ends outside the BAM's BGZF members";
      return false;
    }
    segs.push_back(g);
  }
  return true;
}

}  // namespace

extern "C" {

void *ls_bams_open(const char *path, int threads) {
  Stream *s = new Stream();
  s->threads = threads < 1 ? 1 : threads;
  s->path = path;
  s->fd = open(path, O_RDONLY | O_CLOEXEC);
  struct stat st;
  if (s->fd < 0 || fstat(s->fd, &st) != 0) {
    s->err = std::string("cannot open ") + path;
    return s;
  }
  s->file_size = (uint64_t)st.st_size;
  s->segs.push_back(Segment{0, s->file_size, 0, UINT64_MAX, 0});
  // the header may span several members; what follows it in the inflated bytes is the first chunk's carry
  Chunk &c0 = s->ch[0];
  size_t consumed = 0;
  for (;;) {
    const size_t before = c0.raw.n;
    if (!inflate_some(s, c0.raw, 1u << 20, s->err)) return s;
    bool need_more = false;
    if (!parse_header(s, c0.raw, consumed, need_more)) return s;
    if (!need_more) break;
    if (c0.raw.n == before) {
      s->err = "truncated BAM header";
      return s;
    }
  }
  c0.tail_lo = consumed;
  s->cur = 0;
  s->header_done = true;
  return s;
}

const char *ls_bams_error(void *h) {
  Stream *s = (Stream *)h;
  return s->err.empty() ? nullptr : s->err.c_str();
}
void ls_bams_close(void *h) {
  Stream *s = (Stream *)h;
  if (!s) return;
  if (s->pf_running) s->pf.join();
  if (getenv("LS_BAM_TIMING"))
    fprintf(stderr, "[ls_bamstream] file read %.2f s, inflate %.2f s, record boundaries %.2f s, CB tags %.2f s, barcode ids + offsets "
                    "%.2f s (all on the prefetch thread), fill %.2f s, caller waited %.2f s for prefetched chunks; "
                    "compressed bytes read %lld, inflated bytes %lld, index %s\n",
            s->t_read, s->t_inflate, s->t_index, s->t_tags, s->t_intern, s->t_fill, s->t_wait, (long long)s->tot_comp,
            (long long)s->tot_infl, s->index_note.empty() ? "used" : s->index_note.c_str());
  if (s->fd >= 0) close(s->fd);
  delete s;
}
int32_t ls_bams_n_contigs(void *h) { return (int32_t)((Stream *)h)->contig_names.size(); }
const char *ls_bams_contig_name(void *h, int i) { return ((Stream *)h)->contig_names[i].c_str(); }
int32_t ls_bams_contig_len(void *h, int i) { return ((Stream *)h)->contig_lens[i]; }
// barcodes known when the CURRENT chunk was indexed (the prefetch thread may already have interned later ones)
int32_t ls_bams_n_barcodes(void *h) {
  Stream *s = (Stream *)h;
  return s->ch[s->cur].n_barcodes;
}
const char *ls_bams_barcode(void *h, int i) {
  Stream *s = (Stream *)h;
  std::lock_guard<std::mutex> g(s->bar.mu);
  return s->bar.names[(size_t)i].c_str();
}

int ls_bams_set_regions(void *h, int64_t n, const int32_t *tid, const int64_t *beg, const int64_t *end) {
  Stream *s = (Stream *)h;
  if (!s->err.empty() || !s->header_done || s->started) return -1;
  std::vector<Segment> segs;
  if (!use_index(s, n, tid, beg, end, segs)) return 0;
  // the bytes the header read past itself are not records of the regions
  s->segs.swap(segs);
  s->seg = 0;
  s->rd_off = s->comp_file_off = s->segs.empty() ? 0 : s->segs[0].c0;
  s->comp.clear();
  s->comp_lo = 0;
  s->comp_bytes = s->infl_bytes = 0;
  Chunk &c0 = s->ch[0];
  c0.raw.n = c0.tail_lo;
  s->index_note.clear();
  return 1;
}

const char *ls_bams_index_note(void *h) {
  Stream *s = (Stream *)h;
  return s->index_note.empty() ? nullptr : s->index_note.c_str();
}

void ls_bams_chunk_io(void *h, int64_t *compressed, int64_t *inflated) {
  Stream *s = (Stream *)h;
  *compressed = s->ch[s->cur].comp_bytes;
  *inflated = s->ch[s->cur].infl_bytes;
}

// Next chunk: number of complete records (0 = end of file, -1 = error).  The records stay valid until the next call.
int64_t ls_bams_next(void *h, int64_t target_bytes, int64_t *n_cigar, int64_t *n_bases) {
  Stream *s = (Stream *)h;
  if (!s->err.empty() || !s->header_done) return -1;
  const size_t target = target_bytes > 65536 ? (size_t)target_bytes : 65536;
  Chunk &nxt = s->ch[1 - s->cur];
  if (s->pf_running) {
    const double t0 = now_s();
    s->pf.join();
    s->t_wait += now_s() - t0;
    s->pf_running = false;
  } else {
    produce(s, nxt, s->ch[s->cur], target);
  }
  s->cur = 1 - s->cur;
  Chunk &c = s->ch[s->cur];
  s->started = true;
  s->tot_comp += c.comp_bytes;
  s->tot_infl += c.infl_bytes;
  if (c.n < 0) {
    s->err = c.err.empty() ? "BAM stream: decode failed" : c.err;
    return -1;
  }
  *n_cigar = c.n_cigar;
  *n_bases = c.n_bases;
  if (c.n > 0) {
    // the chunk after this one is produced while the caller copies and processes this one
    Chunk *dst = &s->ch[1 - s->cur];
    const Chunk *prev = &c;
    s->pf = std::thread([s, dst, prev, target]() { produce(s, *dst, *prev, target); });
    s->pf_running = true;
  }
  return c.n;
}

// Copy the current chunk into caller buffers: per-read arrays [n] (cigar_off / base_off: [n + 1]), cigar [n_cigar],
// seq4 [n_bases / 2], qual [n_bases].  Reads start at multiples of 16 bases, the padding is zeroed.
// ref_end (optional): exclusive reference end of every read, pos + its M/D/N/=/X lengths -- what the caller needs to
// decide which windows are complete, computed here while the CIGAR is in cache.
int ls_bams_fill2(void *h, int32_t *tid, int32_t *pos, uint16_t *flag, uint8_t *mapq, int32_t *cb, int32_t *lq,
                  uint32_t *cigar_off, uint64_t *base_off, uint32_t *cigar, uint8_t *seq4, uint8_t *qual, int64_t *ref_end) {
  Stream *s = (Stream *)h;
  if (!s->err.empty()) return -1;
  const Chunk &c = s->ch[s->cur];
  const int64_t n = c.n;
  if (n <= 0) return 0;
  memcpy(cigar_off, c.cig_off.data(), (size_t)(n + 1) * 4);
  memcpy(base_off, c.base_off.data(), (size_t)(n + 1) * 8);
  memcpy(cb, c.cb.data(), (size_t)n * 4);
  std::atomic<int64_t> nx(0);
  auto filler = [&]() {
    for (;;) {
      const int64_t i0 = nx.fetch_add(2048);
      if (i0 >= n) break;
      for (int64_t i = i0; i < i0 + 2048 && i < n; ++i) {
        const uint8_t *r = c.recs[(size_t)i];
        const uint32_t l_name = r[8], n_cig = rd16(r + 12), l_seq = rd32(r + 16);
        tid[i] = (int32_t)rd32(r);
        pos[i] = (int32_t)rd32(r + 4);
        mapq[i] = r[9];
        flag[i] = rd16(r + 14);
        lq[i] = (int32_t)l_seq;
        const uint8_t *cg = r + 32 + l_name;
        memcpy(cigar + c.cig_off[(size_t)i], cg, 4 * (size_t)n_cig);
        if (ref_end) {
          int64_t span = 0;
          for (uint32_t k = 0; k < n_cig; ++k) {
            const uint32_t op = rd32(cg + 4 * k);
            if ((0x18du >> (op & 15u)) & 1u) span += op >> 4;  // M, D, N, =, X consume the reference
          }
          ref_end[i] = (int64_t)(int32_t)rd32(r + 4) + span;
        }
        const uint8_t *sq = cg + 4 * (size_t)n_cig;
        const uint64_t bo = c.base_off[(size_t)i], pad = c.base_off[(size_t)i + 1] - bo;
        const uint32_t sb = (l_seq + 1) / 2;
        memcpy(seq4 + bo / 2, sq, sb);
        memset(seq4 + bo / 2 + sb, 0, (size_t)(pad / 2 - sb));
        memcpy(qual + bo, sq + sb, l_seq);
        memset(qual + bo + l_seq, 0, (size_t)(pad - l_seq));
      }
    }
  };
  const double t_f0 = now_s();
  std::vector<std::thread> th;
  for (int t = 0; t < s->threads; ++t) th.emplace_back(filler);
  for (auto &t : th) t.join();
  s->t_fill += now_s() - t_f0;
  return 0;
}

int ls_bams_fill(void *h, int32_t *tid, int32_t *pos, uint16_t *flag, uint8_t *mapq, int32_t *cb, int32_t *lq,
                 uint32_t *cigar_off, uint64_t *base_off, uint32_t *cigar, uint8_t *seq4, uint8_t *qual) {
  return ls_bams_fill2(h, tid, pos, flag, mapq, cb, lq, cigar_off, base_off, cigar, seq4, qual, nullptr);
}

int ls_inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len) {
  static thread_local lsinf::Tables tabs;
  if (in_len < 0 || out_len < 0) return 0;
  return lsinf::inflate_raw(in, (size_t)in_len, out, (size_t)out_len, tabs) ? 1 : 0;
}

}  // extern "C"
