"""Host-side file codecs: BAM (BGZF) reader / writer and FASTA(.fai) reader / writer.

The reference reads these formats through pysam/htslib (BaseCellCounter.py:84-86,190-194;
SingleCellGenotype.py:123-127); pysam is not a dependency here.  Reading is done by the native
decoder csrc/host/ls_bamread.cpp (block-parallel inflate, one pass, structure-of-arrays out);
writing (synthetic data, tests) is plain Python + zlib.
"""
import ctypes as C
import os
import struct
import zlib

import numpy as np

from .batch import ReadBatch

_HERE = os.path.dirname(os.path.abspath(__file__))
_HOST_LIB = os.path.join(_HERE, "liblongsom_host.so")
_host = None


def _load_host():
    global _host
    if _host is None:
        if not os.path.exists(_HOST_LIB):
            raise RuntimeError("longsom_b200: %s not built (run __graft_entry__.build())" % _HOST_LIB)
        lib = C.CDLL(_HOST_LIB)
        lib.ls_bam_read.restype = C.c_void_p
        lib.ls_bam_read.argtypes = [C.c_char_p, C.c_int]
        lib.ls_bam_error.restype = C.c_char_p
        lib.ls_bam_error.argtypes = [C.c_void_p]
        lib.ls_bam_free.argtypes = [C.c_void_p]
        for f in ("ls_bam_n_reads", "ls_bam_n_cigar", "ls_bam_n_bases"):
            getattr(lib, f).restype = C.c_int64
            getattr(lib, f).argtypes = [C.c_void_p]
        for f in ("ls_bam_n_contigs", "ls_bam_n_barcodes"):
            getattr(lib, f).restype = C.c_int32
            getattr(lib, f).argtypes = [C.c_void_p]
        lib.ls_bam_contig_name.restype = C.c_char_p
        lib.ls_bam_contig_name.argtypes = [C.c_void_p, C.c_int]
        lib.ls_bam_contig_len.restype = C.c_int32
        lib.ls_bam_contig_len.argtypes = [C.c_void_p, C.c_int]
        lib.ls_bam_barcode.restype = C.c_char_p
        lib.ls_bam_barcode.argtypes = [C.c_void_p, C.c_int]
        lib.ls_bam_array.restype = C.c_void_p
        lib.ls_bam_array.argtypes = [C.c_void_p, C.c_int]
        _host = lib
    return _host


class BamData:
    """Decoded BAM: contigs, a ReadBatch whose `cell` column holds the id of the RAW CB:Z text
    (-1 = no CB tag), and the list of distinct raw barcode strings (id -> text)."""

    def __init__(self, contig_names, contig_lens, batch, barcodes):
        self.contig_names = contig_names
        self.contig_lens = contig_lens
        self.batch = batch
        self.barcodes = barcodes

    def with_cells(self, raw_to_cell):
        """New ReadBatch whose cell ids are raw_to_cell[raw barcode id] (array; -1 keeps 'no CB')."""
        raw_to_cell = np.asarray(raw_to_cell, np.int32)
        b = self.batch
        cell = np.where(b.cell >= 0, raw_to_cell[np.maximum(b.cell, 0)], -1).astype(np.int32)
        return ReadBatch(b.tid, b.pos, b.flag, b.mapq, cell, b.cigar_off, b.cigar, b.base_off, b.l_qseq, b.seq4,
                         b.qual)


class _BamHandle:
    """Owns the native decoder's buffers; the numpy arrays of a decoded batch are views into them and keep
    this object alive through their buffer chain (no 3 GB host copy per million long reads)."""

    def __init__(self, lib, h):
        self.lib, self.h = lib, h

    def __del__(self):
        if self.h:
            self.lib.ls_bam_free(self.h)
            self.h = None


def read_bam(path, threads=None):
    lib = _load_host()
    if threads is None:
        threads = min(32, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    owner = _BamHandle(lib, lib.ls_bam_read(os.fsencode(path), int(threads)))
    h = owner.h
    err = lib.ls_bam_error(h)
    if err:
        raise IOError("read_bam(%s): %s" % (path, err.decode()))
    n, nc, nb = lib.ls_bam_n_reads(h), lib.ls_bam_n_cigar(h), lib.ls_bam_n_bases(h)
    names = [lib.ls_bam_contig_name(h, i).decode() for i in range(lib.ls_bam_n_contigs(h))]
    lens = [lib.ls_bam_contig_len(h, i) for i in range(len(names))]
    barcodes = [lib.ls_bam_barcode(h, i).decode() for i in range(lib.ls_bam_n_barcodes(h))]

    def arr(which, dtype, count):
        if count == 0:
            return np.zeros(0, dtype)
        ct = np.ctypeslib.as_ctypes_type(dtype)
        buf = (ct * count).from_address(lib.ls_bam_array(h, which))
        buf._owner = owner  # array -> memoryview -> buf -> owner: freed with the last array
        return np.frombuffer(buf, dtype=dtype)
    batch = ReadBatch(arr(0, np.int32, n), arr(1, np.int32, n), arr(2, np.uint16, n), arr(3, np.uint8, n),
                      arr(4, np.int32, n), arr(5, np.uint32, n + 1), arr(6, np.uint32, nc),
                      arr(7, np.uint64, n + 1), arr(8, np.int32, n), arr(9, np.uint8, nb // 2),
                      arr(10, np.uint8, nb))
    return BamData(names, lens, batch, barcodes)


# ---- BGZF / BAM writer (synthetic data + tests) -------------------------------------------------
_BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


class BamStream:
    """Chunked decoder over csrc/host/ls_bamstream.cpp: bounded memory, barcodes interned across chunks.

    next_chunk(target_bytes, alloc, head) decodes the next ~target_bytes of inflated BAM and writes the records into
    arrays obtained from alloc(n_reads, n_cigar, n_bases) -- pinned staging memory in the counter CLI -- AFTER the
    `head` reads the caller has already placed at their start (the reads carried over from the previous chunk), and
    returns the ReadBatch of head + chunk with raw barcode ids in .cell (or None at the end of the file)."""

    def __init__(self, path, threads=None):
        self.lib = _load_host()
        lib = self.lib
        if not hasattr(lib, "_bams_ready"):
            lib.ls_bams_open.restype = C.c_void_p
            lib.ls_bams_open.argtypes = [C.c_char_p, C.c_int]
            lib.ls_bams_error.restype = C.c_char_p
            lib.ls_bams_error.argtypes = [C.c_void_p]
            lib.ls_bams_close.argtypes = [C.c_void_p]
            lib.ls_bams_next.restype = C.c_int64
            lib.ls_bams_next.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
            lib.ls_bams_fill.restype = C.c_int
            lib.ls_bams_fill.argtypes = [C.c_void_p] + [C.c_void_p] * 11
            lib.ls_bams_fill2.restype = C.c_int
            lib.ls_bams_fill2.argtypes = [C.c_void_p] + [C.c_void_p] * 12
            for f in ("ls_bams_n_contigs", "ls_bams_n_barcodes"):
                getattr(lib, f).restype = C.c_int32
                getattr(lib, f).argtypes = [C.c_void_p]
            lib.ls_bams_contig_name.restype = C.c_char_p
            lib.ls_bams_contig_name.argtypes = [C.c_void_p, C.c_int]
            lib.ls_bams_contig_len.restype = C.c_int32
            lib.ls_bams_contig_len.argtypes = [C.c_void_p, C.c_int]
            lib.ls_bams_barcode.restype = C.c_char_p
            lib.ls_bams_barcode.argtypes = [C.c_void_p, C.c_int]
            lib.ls_bams_set_regions.restype = C.c_int
            lib.ls_bams_set_regions.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
            lib.ls_bams_index_note.restype = C.c_char_p
            lib.ls_bams_index_note.argtypes = [C.c_void_p]
            lib.ls_bams_chunk_io.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
            lib._bams_ready = True
        threads = threads or min(16, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
        self.h = lib.ls_bams_open(os.fsencode(path), int(threads))
        self._check()
        self.contig_names = [lib.ls_bams_contig_name(self.h, i).decode() for i in range(lib.ls_bams_n_contigs(self.h))]
        self.contig_lens = [lib.ls_bams_contig_len(self.h, i) for i in range(len(self.contig_names))]
        self.barcodes = []
        self.compressed_bytes = self.inflated_bytes = 0  # of the chunks decoded so far

    def set_regions(self, tid, beg, end):
        """Read only the BGZF members the .bai lists for the regions [beg, end) of reference tid (arrays); call before
        the first next_chunk.  Returns None when the index is used, else the one-line reason why the whole file is
        read (see ls_bams_set_regions)."""
        tid = np.ascontiguousarray(tid, np.int32)
        beg = np.ascontiguousarray(beg, np.int64)
        end = np.ascontiguousarray(end, np.int64)
        rc = self.lib.ls_bams_set_regions(self.h, tid.shape[0], tid.ctypes.data, beg.ctypes.data, end.ctypes.data)
        if rc < 0:
            self._check()
            raise ValueError("BamStream.set_regions: call it before the first next_chunk")
        return None if rc == 1 else self.lib.ls_bams_index_note(self.h).decode(errors="replace")

    def _check(self):
        err = self.lib.ls_bams_error(self.h)
        if err:
            raise IOError("BAM stream: " + err.decode())

    def close(self):
        if self.h:
            self.lib.ls_bams_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def next_chunk(self, target_bytes, alloc, head=None, head_ends=None):
        """-> (batch, n_new, ends) or None; ends = exclusive reference end of every read of the batch (head_ends: those of
        the carried reads in `head`)."""
        nc, nb = C.c_int64(0), C.c_int64(0)
        n = self.lib.ls_bams_next(self.h, int(target_bytes), C.byref(nc), C.byref(nb))
        cb, ib = C.c_int64(0), C.c_int64(0)
        self.lib.ls_bams_chunk_io(self.h, C.byref(cb), C.byref(ib))
        self.compressed_bytes += cb.value
        self.inflated_bytes += ib.value
        if n < 0:
            self._check()
            raise IOError("BAM stream: decode failed")
        if n == 0:
            return None
        h_n = head.n_reads if head is not None else 0
        h_c = int(head.cigar.shape[0]) if head is not None else 0
        h_b = head.n_bases if head is not None else 0
        a = alloc(h_n + n, h_c + nc.value, h_b + nb.value)
        if head is not None and h_n:
            for f in ("tid", "pos", "flag", "mapq", "cell", "l_qseq"):
                a[f][:h_n] = getattr(head, f)
            a["cigar_off"][:h_n + 1] = head.cigar_off
            a["base_off"][:h_n + 1] = head.base_off
            a["cigar"][:h_c] = head.cigar
            a["seq4"][:h_b // 2] = head.seq4
            a["qual"][:h_b] = head.qual
        ptr = lambda arr, off: C.c_void_p(arr.ctypes.data + off * arr.itemsize)
        ends = np.empty(h_n + n, np.int64)
        if h_n:
            if head_ends is None:
                raise ValueError("next_chunk: head given without head_ends")
            ends[:h_n] = head_ends
        rc = self.lib.ls_bams_fill2(self.h, ptr(a["tid"], h_n), ptr(a["pos"], h_n), ptr(a["flag"], h_n), ptr(a["mapq"], h_n),
                                   ptr(a["cell"], h_n), ptr(a["l_qseq"], h_n), ptr(a["cigar_off"], h_n),
                                   ptr(a["base_off"], h_n), ptr(a["cigar"], h_c), ptr(a["seq4"], h_b // 2), ptr(a["qual"], h_b),
                                    ptr(ends, h_n))
        if rc != 0:
            self._check()
            raise IOError("BAM stream: fill failed")
        if h_n:  # the chunk's offsets start at 0: rebase them behind the carried reads
            a["cigar_off"][h_n:h_n + n + 1] += np.uint32(h_c)
            a["base_off"][h_n:h_n + n + 1] += np.uint64(h_b)
        nbar = self.lib.ls_bams_n_barcodes(self.h)
        for i in range(len(self.barcodes), nbar):
            self.barcodes.append(self.lib.ls_bams_barcode(self.h, i).decode())
        N, NC, NB = h_n + n, h_c + nc.value, h_b + nb.value
        return ReadBatch(a["tid"][:N], a["pos"][:N], a["flag"][:N], a["mapq"][:N], a["cell"][:N], a["cigar_off"][:N + 1],
                         a["cigar"][:NC], a["base_off"][:N + 1], a["l_qseq"][:N], a["seq4"][:NB // 2], a["qual"][:NB]), n, ends


def _bgzf_block(data, level):
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    bsize = len(comp) + 25
    hdr = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, ord("B"), ord("C"), 2, bsize)
    return hdr + comp + struct.pack("<II", zlib.crc32(data) & 0xffffffff, len(data))


class BgzfWriter:
    def __init__(self, path, level=1):
        self.f = open(path, "wb")
        self.buf = bytearray()
        self.level = level

    def write(self, data):
        self.buf += data
        while len(self.buf) >= 0xff00:
            self.f.write(_bgzf_block(bytes(self.buf[:0xff00]), self.level))
            del self.buf[:0xff00]

    def close(self):
        if self.buf:
            self.f.write(_bgzf_block(bytes(self.buf), self.level))
        self.f.write(_BGZF_EOF)
        self.f.close()


def _reg2bin(beg, end):
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def write_bam(path, contig_names, contig_lens, batch, cb_text, read_names=None, level=1, extra_tags=None):
    """Write a coordinate-sorted BAM.  cb_text: callable read_index -> CB string or None (no tag)."""
    w = BgzfWriter(path, level)
    text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(
        "@SQ\tSN:%s\tLN:%d\n" % (n, l) for n, l in zip(contig_names, contig_lens))
    tb = text.encode()
    hdr = bytearray(b"BAM\1" + struct.pack("<I", len(tb)) + tb + struct.pack("<I", len(contig_names)))
    for n, l in zip(contig_names, contig_lens):
        nb = n.encode() + b"\0"
        hdr += struct.pack("<I", len(nb)) + nb + struct.pack("<I", l)
    w.write(bytes(hdr))
    b = batch
    refop = np.isin(b.cigar & 15, [0, 2, 3, 7, 8])
    for i in range(b.n_reads):
        name = (read_names[i] if read_names is not None else "r%d" % i).encode() + b"\0"
        c0, c1 = int(b.cigar_off[i]), int(b.cigar_off[i + 1])
        cig = b.cigar[c0:c1]
        rlen = int((cig[refop[c0:c1]] >> 4).sum())
        lq = int(b.l_qseq[i])
        bo = int(b.base_off[i])
        seq = b.seq4[bo // 2: bo // 2 + (lq + 1) // 2].tobytes()
        if lq & 1:  # clear the padding nibble
            seq = seq[:-1] + bytes([seq[-1] & 0xf0])
        qual = b.qual[bo: bo + lq].tobytes()
        aux = b""
        cb = cb_text(i)
        if cb is not None:
            aux += b"CBZ" + cb.encode() + b"\0"
        if extra_tags is not None:
            aux += extra_tags(i)
        pos = int(b.pos[i])
        body = struct.pack("<iiBBHHHIiii", int(b.tid[i]), pos, len(name), int(b.mapq[i]),
                           _reg2bin(pos, pos + max(rlen, 1)), c1 - c0, int(b.flag[i]), lq, -1, -1, 0)
        body += name + cig.astype("<u4").tobytes() + seq + qual + aux
        w.write(struct.pack("<I", len(body)) + body)
    w.close()


# ---- FASTA ------------------------------------------------------------------------------------------
def write_fasta(path, names, seqs, width=60):
    """seqs: uint8 arrays / bytes.  Also writes path + '.fai'."""
    with open(path, "wb") as f, open(path + ".fai", "w") as fai:
        off = 0
        for n, s in zip(names, seqs):
            s = bytes(s) if not isinstance(s, np.ndarray) else s.tobytes()
            head = (">%s\n" % n).encode()
            f.write(head)
            off += len(head)
            fai.write("%s\t%d\t%d\t%d\t%d\n" % (n, len(s), off, width, width + 1))
            for i in range(0, len(s), width):
                f.write(s[i:i + width] + b"\n")
            off += len(s) + (len(s) + width - 1) // width


class Fasta:
    """Indexed FASTA reader with the slice of pysam.FastaFile the reference uses
    (.references, .get_reference_length, .fetch; BaseCellCounter.py:84-86,202; step1.py:29,98)."""

    def __init__(self, path):
        self.path = path
        fai = path + ".fai"
        if not os.path.exists(fai):
            raise IOError("FASTA index %s not found" % fai)
        self.references, self._idx = [], {}
        for line in open(fai):
            p = line.rstrip("\n").split("\t")
            if len(p) < 5:
                continue
            self.references.append(p[0])
            self._idx[p[0]] = (int(p[1]), int(p[2]), int(p[3]), int(p[4]))
        self._f = open(path, "rb")
        self._cache = {}

    @property
    def lengths(self):
        return [self._idx[r][0] for r in self.references]

    def get_reference_length(self, name):
        return self._idx[name][0]

    def contig(self, name):
        """Whole contig as a uint8 array (cached)."""
        if name not in self._cache:
            ln, off, lb, lw = self._idx[name]
            nlines = (ln + lb - 1) // lb if lb else 0
            self._f.seek(off)
            raw = self._f.read(ln + nlines * (lw - lb))
            a = np.frombuffer(raw, np.uint8)
            if lw != lb and ln:
                full = (ln // lb) * lw
                body = a[:full].reshape(-1, lw)[:, :lb].reshape(-1) if full else np.zeros(0, np.uint8)
                tail = a[full:full + (ln - (ln // lb) * lb)]
                a = np.concatenate([body, tail])
            self._cache[name] = np.ascontiguousarray(a[:ln])
        return self._cache[name]

    def fetch(self, name, start, end):
        if start < 0:
            raise ValueError("start out of range (%i)" % start)
        seq = self.contig(name)
        return seq[start:min(end, len(seq))].tobytes().decode()

    def close(self):
        self._f.close()
