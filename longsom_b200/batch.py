"""Host-side structure-of-arrays containers handed to the C-ABI (include/longsom_b200.h).

ReadBatch is what the BAM decoder (longsom_b200/bamio.py) produces in place of pysam's
per-column Python objects (reference: BaseCellCounter.py:190-191,214-216,238-249).
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def _chk(a, dtype, name):
    a = np.ascontiguousarray(a, dtype=dtype)
    return a


@dataclass
class ReadBatch:
    tid: np.ndarray        # int32 [n]
    pos: np.ndarray        # int32 [n]
    flag: np.ndarray       # uint16 [n]
    mapq: np.ndarray       # uint8 [n]
    cell: np.ndarray       # int32 [n]  (-1 = no CB tag)
    cigar_off: np.ndarray  # uint32 [n+1]
    cigar: np.ndarray      # uint32 [n_cigar]
    base_off: np.ndarray   # uint64 [n+1], multiples of 16
    l_qseq: np.ndarray     # int32 [n]
    seq4: np.ndarray       # uint8 [n_bases/2]
    qual: np.ndarray       # uint8 [n_bases]

    def __post_init__(self):
        self.tid = _chk(self.tid, np.int32, "tid")
        self.pos = _chk(self.pos, np.int32, "pos")
        self.flag = _chk(self.flag, np.uint16, "flag")
        self.mapq = _chk(self.mapq, np.uint8, "mapq")
        self.cell = _chk(self.cell, np.int32, "cell")
        self.cigar_off = _chk(self.cigar_off, np.uint32, "cigar_off")
        self.cigar = _chk(self.cigar, np.uint32, "cigar")
        self.base_off = _chk(self.base_off, np.uint64, "base_off")
        self.l_qseq = _chk(self.l_qseq, np.int32, "l_qseq")
        self.seq4 = _chk(self.seq4, np.uint8, "seq4")
        self.qual = _chk(self.qual, np.uint8, "qual")

    @property
    def n_reads(self):
        return int(self.pos.shape[0])

    @property
    def n_bases(self):
        return int(self.qual.shape[0])

    def aligned_bases(self):
        """Sum of M/=/X lengths over all records: the unit of the throughput metric (SURVEY 8d)."""
        op = self.cigar & 15
        ln = (self.cigar >> 4).astype(np.int64)
        return int(ln[(op == 0) | (op == 7) | (op == 8)].sum())

    def as_struct(self):
        s = L.LsReadBatch()
        s.n_reads = self.n_reads
        s.n_cigar = int(self.cigar.shape[0])
        s.n_bases = self.n_bases
        for f in ("tid", "pos", "flag", "mapq", "cell", "cigar_off", "cigar", "base_off", "l_qseq", "seq4", "qual"):
            setattr(s, f, _ptr(getattr(self, f)))
        return s

    def nbytes(self):
        return sum(getattr(self, f).nbytes for f in
                   ("tid", "pos", "flag", "mapq", "cell", "cigar_off", "cigar", "base_off", "l_qseq", "seq4", "qual"))

    def slice(self, lo, hi):
        """Sub-batch of the consecutive reads [lo, hi): array slices with rebased offsets (no per-read work)."""
        lo, hi = int(lo), int(hi)
        c0, c1 = int(self.cigar_off[lo]), int(self.cigar_off[hi])
        b0, b1 = int(self.base_off[lo]), int(self.base_off[hi])
        return ReadBatch(self.tid[lo:hi], self.pos[lo:hi], self.flag[lo:hi], self.mapq[lo:hi], self.cell[lo:hi],
                         (self.cigar_off[lo:hi + 1] - np.uint32(c0)).astype(np.uint32), self.cigar[c0:c1],
                         (self.base_off[lo:hi + 1] - np.uint64(b0)).astype(np.uint64), self.l_qseq[lo:hi],
                         self.seq4[b0 // 2:b1 // 2], self.qual[b0:b1])

    def select(self, idx):
        """Sub-batch with the given (sorted) read indices; re-packs cigar / bases.  Every read keeps its base
        padding, and each run of consecutive indices is copied as one slice."""
        idx = np.asarray(idx, dtype=np.int64)
        n = idx.shape[0]
        co, bo = self.cigar_off.astype(np.int64), self.base_off.astype(np.int64)
        cigar_off = np.zeros(n + 1, np.uint32)
        np.cumsum(co[idx + 1] - co[idx], out=cigar_off[1:])
        base_off = np.zeros(n + 1, np.uint64)
        np.cumsum(bo[idx + 1] - bo[idx], out=base_off[1:])
        cut = np.nonzero(np.diff(idx) != 1)[0] + 1
        lo = idx[np.concatenate([[0], cut])] if n else idx
        hi = idx[np.concatenate([cut - 1, [n - 1]])] + 1 if n else idx

        def gather(a, off, div=1):
            parts = [a[off[s] // div:off[e] // div] for s, e in zip(lo.tolist(), hi.tolist())]
            return np.concatenate(parts) if parts else a[:0].copy()
        return ReadBatch(self.tid[idx], self.pos[idx], self.flag[idx], self.mapq[idx], self.cell[idx], cigar_off,
                         gather(self.cigar, co), base_off, self.l_qseq[idx], gather(self.seq4, bo, 2), gather(self.qual, bo))


@dataclass
class Windows:
    tid: np.ndarray      # int32 [w]
    start: np.ndarray    # int32 [w]  0-based, half-open
    end: np.ndarray      # int32 [w]
    ref_off: np.ndarray  # uint64 [w+1]
    ref: np.ndarray      # uint8, reference bases of every window back to back

    def __post_init__(self):
        self.tid = _chk(self.tid, np.int32, "tid")
        self.start = _chk(self.start, np.int32, "start")
        self.end = _chk(self.end, np.int32, "end")
        self.ref_off = _chk(self.ref_off, np.uint64, "ref_off")
        self.ref = _chk(self.ref, np.uint8, "ref")

    @property
    def n_windows(self):
        return int(self.tid.shape[0])

    def as_struct(self):
        s = L.LsWindows()
        s.n_windows = self.n_windows
        for f in ("tid", "start", "end", "ref_off", "ref"):
            setattr(s, f, _ptr(getattr(self, f)))
        return s

    def slice(self, lo, hi):
        """Windows [lo, hi) with their reference bytes."""
        lo, hi = int(lo), int(hi)
        r0, r1 = int(self.ref_off[lo]), int(self.ref_off[hi])
        return Windows(self.tid[lo:hi], self.start[lo:hi], self.end[lo:hi],
                       (self.ref_off[lo:hi + 1] - np.uint64(r0)).astype(np.uint64), self.ref[r0:r1])

    @staticmethod
    def from_intervals(intervals, contig_seqs):
        """intervals: iterable of (tid, start, end) 0-based half-open, sorted, disjoint.
        contig_seqs: mapping tid -> uint8 array (or bytes) of the whole contig."""
        iv = list(intervals)
        tid = np.array([i[0] for i in iv], np.int32)
        start = np.array([i[1] for i in iv], np.int32)
        end = np.array([i[2] for i in iv], np.int32)
        ref_off = np.zeros(len(iv) + 1, np.uint64)
        if len(iv):
            np.cumsum((end - start).astype(np.uint64), out=ref_off[1:])
        ref = np.empty(int(ref_off[-1]), np.uint8)
        for j, (t, s, e) in enumerate(iv):
            seq = contig_seqs[t]
            if not isinstance(seq, np.ndarray):
                seq = np.frombuffer(seq, np.uint8)
            ref[int(ref_off[j]):int(ref_off[j + 1])] = seq[s:e]
        return Windows(tid, start, end, ref_off, ref)


def make_windows(contig_lens, bin_size=50000, chrom=None, first_pos=1):
    """Window grid of the reference's MakeWindows without --bed/--bed_out
    (BaseCellCounter.py:81-113): contigs as (name, 1, len) -> bedtools makewindows -w bin.
    Returns a list of (tid, start, end); note reference position 0 is never covered (:86)."""
    out = []
    for t, ln in enumerate(contig_lens):
        if chrom is not None and t != chrom:
            continue
        s = first_pos
        while s < ln:
            e = min(s + bin_size, ln)
            out.append((t, s, e))
            s = e
    return out


@dataclass
class SiteCounts:
    tid: np.ndarray     # int32 [n]
    pos: np.ndarray     # int32 [n] 0-based
    ref: np.ndarray     # uint8 [n] upper-case reference base
    counts: np.ndarray  # uint32 [n, 26]  (see LS_SITE_* in include/longsom_b200.h)

    @property
    def n_sites(self):
        return int(self.pos.shape[0])

    @staticmethod
    def empty(capacity):
        return SiteCounts(np.zeros(capacity, np.int32), np.zeros(capacity, np.int32), np.zeros(capacity, np.uint8),
                          np.zeros((capacity, L.LS_SITE_WORDS), np.uint32))

    def as_struct(self):
        s = L.LsSiteCounts()
        s.capacity = self.n_sites
        s.n_sites = 0
        s.tid, s.pos, s.ref, s.counts = _ptr(self.tid), _ptr(self.pos), _ptr(self.ref), _ptr(self.counts)
        return s

    def head(self, n):
        return SiteCounts(self.tid[:n], self.pos[:n], self.ref[:n], self.counts[:n])
