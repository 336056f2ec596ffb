"""Writes a .bai (SAM spec 5.2) for a coordinate-sorted BAM from its records' virtual offsets, so that a test can give an
index to a BAM written by bamio.write_bam without changing a byte of the BAM.  Independent of the native writer."""
import os
import struct

from bai_query import BgzfReader


def _reg2bin(beg, end):
    end -= 1
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return base + (beg >> shift)
    return 0


def write_bai(bam_path):
    rd = BgzfReader(bam_path)
    head, v = rd.read(0, 8)
    _, v = rd.read(v, struct.unpack_from("<I", head, 4)[0])
    nb, v = rd.read(v, 4)
    n_ref = struct.unpack("<I", nb)[0]
    for _ in range(n_ref):
        ln, v = rd.read(v, 4)
        _, v = rd.read(v, struct.unpack("<I", ln)[0] + 4)
    refs = [({}, {}) for _ in range(n_ref)]
    eof = len(rd.buf) - 28
    while v >> 16 < eof:
        hb, v2 = rd.read(v, 4)
        rec, v3 = rd.read(v2, struct.unpack("<I", hb)[0])
        tid, pos, l_name, _mq, _bin, n_cig, flag, _lseq = struct.unpack_from("<iiBBHHHI", rec, 0)
        if tid >= 0:
            cig = struct.unpack_from("<%dI" % n_cig, rec, 32 + l_name)
            span = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
            end = pos + (span if span > 0 and not flag & 4 else 1)
            bins, lin = refs[tid]
            ch = bins.setdefault(_reg2bin(pos, end), [])
            if ch and ch[-1][1] == v:
                ch[-1][1] = v3
            else:
                ch.append([v, v3])
            for w in range(pos >> 14, ((end - 1) >> 14) + 1):
                lin.setdefault(w, v)
        v = v3
    out = bytearray(b"BAI\1" + struct.pack("<i", n_ref))
    for bins, lin in refs:
        out += struct.pack("<i", len(bins))
        for b in sorted(bins):
            out += struct.pack("<Ii", b, len(bins[b])) + b"".join(struct.pack("<QQ", *c) for c in bins[b])
        n = max(lin) + 1 if lin else 0
        vals, prev = [], 0
        for w in range(n):
            prev = lin.get(w, prev)
            vals.append(prev)
        out += struct.pack("<i", n) + b"".join(struct.pack("<Q", x) for x in vals)
    out += struct.pack("<Q", 0)
    with open(bam_path + ".bai", "wb") as f:
        f.write(bytes(out))
    t = os.stat(bam_path).st_mtime
    os.utime(bam_path + ".bai", (t + 1, t + 1))
