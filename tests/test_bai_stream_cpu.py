"""The streaming reader with a .bai (ls_bams_set_regions): it reads only the BGZF members of the spans the index gives for
a run's regions.  Checked against a brute-force scan of the whole file and against an independent walk of the index's
spans; the compressed bytes it reads are checked exactly; a missing or unusable index reads the whole file as before;
the streamed counter and genotype drivers give the same results with and without the index."""
import ctypes as C
import os
import shutil
import struct
import sys
import zlib

import numpy as np
import pytest

from longsom_b200 import bamio, pipeline, synth
from longsom_b200.batch import ReadBatch
from longsom_b200.engine import CountParams
from longsom_b200.windows import make_windows

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import bai_query  # noqa: E402

LENS = [70_000_000, 300_000, 400_000, 200_000]  # chr1 reaches the 64 Mb bin level; chr2 and chr4 get no reads
BOUNDARIES = [16384 * 3, 131072 * 2, 1 << 20, 8 << 20, 64 << 20, 16384 * 21]


class NumpySlot:
    """pipeline.PinnedSlot without a CUDA context."""

    def __call__(self, n, nc, nb):
        return dict(tid=np.zeros(n, np.int32), pos=np.zeros(n, np.int32), flag=np.zeros(n, np.uint16),
                    mapq=np.zeros(n, np.uint8), cell=np.zeros(n, np.int32), l_qseq=np.zeros(n, np.int32),
                    cigar_off=np.zeros(n + 1, np.uint32), base_off=np.zeros(n + 1, np.uint64), cigar=np.zeros(nc, np.uint32),
                    seq4=np.zeros(nb // 2 + 1, np.uint8), qual=np.zeros(nb, np.uint8))

    def free(self):
        pass


class OracleEngine:
    """pileup_count, upload and genotype_sparse with the CPU oracle's counts (genotype p is not evaluated: NaN)."""

    def __init__(self, device=0):
        self.device, self.last_stats, self.batch = device, {}, None

    def pileup_count(self, batch, windows, params):
        import oracle
        return oracle.pileup_count(batch, windows, params, threads=2)[0]

    def upload(self, batch, windows=None):
        self.batch = batch

    def genotype_sparse(self, st, sp, alt, n_cells, alpha, beta, skip_p=None, bin_size=50000, **kw):
        import oracle
        dp, al = oracle.genotype_count(self.batch, st, sp, alt, n_cells, bin_size=bin_size, **kw)
        site, cell = np.nonzero(dp > 0)
        return (site.astype(np.int32), cell.astype(np.int32), dp[site, cell], al[site, cell],
                np.full(site.shape[0], np.nan))

    def close(self):
        pass


# ---- inputs ---------------------------------------------------------------------------------------------------------
def hand_reads(rng):
    """Large reads across the linear-index and bin boundaries of chr1, and reads whose N intron starts 100-600 kb
    before them; every one with the barcode of cell 0."""
    reads = []  # (tid, pos, cigar [(len, op)])
    for b in BOUNDARIES:
        clip = (12000, 4)  # records of ~36 kB: most of them are cut by a BGZF member boundary
        reads += [(0, b - 120, [clip, (240, 0), clip]), (0, b - 200, [clip, (200, 0), clip]), (0, b, [clip, (150, 0), clip]),
                  (0, b - 1, [clip, (2, 0), clip])]
        for back in (100_000, 300_000, 600_000):
            if b > back:
                reads.append((0, b - back, [clip, (100, 0), (back - 150, 3), (300, 0)]))
    tid = np.array([r[0] for r in reads], np.int32)
    pos = np.array([r[1] for r in reads], np.int32)
    cig = [np.array([(l << 4) | op for l, op in r[2]], np.uint32) for r in reads]
    lq = np.array([sum(l for l, op in r[2] if op in (0, 1, 4)) for r in reads], np.int32)
    cigar_off = np.concatenate([[0], np.cumsum([c.shape[0] for c in cig])]).astype(np.uint32)
    base_off = np.concatenate([[0], np.cumsum((lq + 15) // 16 * 16)]).astype(np.uint64)
    nb = int(base_off[-1])
    return ReadBatch(tid, pos, np.zeros(len(reads), np.uint16), np.full(len(reads), 60, np.uint8),
                     np.zeros(len(reads), np.int32), cigar_off, np.concatenate(cig), base_off, lq,
                     rng.integers(0, 256, nb // 2).astype(np.uint8), rng.integers(2, 41, nb).astype(np.uint8))


def concat(a, b):
    return ReadBatch(np.concatenate([a.tid, b.tid]), np.concatenate([a.pos, b.pos]), np.concatenate([a.flag, b.flag]),
                     np.concatenate([a.mapq, b.mapq]), np.concatenate([a.cell, b.cell]),
                     np.concatenate([a.cigar_off[:-1], b.cigar_off + np.uint32(a.cigar.shape[0])]),
                     np.concatenate([a.cigar, b.cigar]),
                     np.concatenate([a.base_off[:-1], b.base_off + np.uint64(a.n_bases)]),
                     np.concatenate([a.l_qseq, b.l_qseq]), np.concatenate([a.seq4, b.seq4]), np.concatenate([a.qual, b.qual]))


def split_one_type(src, dst, barcodes):
    """ls_bam_split with every barcode routed to one type and its filters off: dst (+ .bai) holds the placed records of
    src that carry a barcode."""
    host = bamio._load_host()
    host.ls_bam_split.restype = C.c_int
    keys = [b.encode() for b in barcodes]
    off = (C.c_uint32 * (len(keys) + 1))(*np.concatenate([[0], np.cumsum([len(k) for k in keys])]).tolist())
    counters, first_seen, err = (C.c_int64 * 36)(), (C.c_int64 * 32)(), C.create_string_buffer(512)
    rc = host.ls_bam_split(os.fsencode(src), 1, (C.c_char_p * 1)(os.fsencode(dst)), b"".join(keys), off,
                           (C.c_int32 * len(keys))(*([0] * len(keys))), C.c_int64(len(keys)), 0, -1, -1, 0, 4, 6,
                           counters, first_seen, err, 512)
    assert rc == 0, err.value


def append_unplaced(path, n):
    """Appends n unplaced records (tid -1) in BGZF members of their own before the EOF marker; the index stays valid."""
    data = open(path, "rb").read()
    assert data[-28:] == bamio._BGZF_EOF
    recs = b""
    for i in range(n):
        name = b"u%d\0" % i
        body = struct.pack("<iiBBHHHIiii", -1, -1, len(name), 0, 4680, 0, 4, 4, -1, -1, 0) + name + b"\x11\x11" + \
            bytes([30] * 4) + b"CBZ" + synth.barcode_of(0).encode() + b"\0"
        recs += struct.pack("<I", len(body)) + body
    with open(path, "wb") as f:
        f.write(data[:-28] + bamio._bgzf_block(recs, 1) + bamio._BGZF_EOF)


@pytest.fixture(scope="module")
def case(tmp_path_factory, built):
    """chr1 (70 Mb) and chr3 with reads, chr2 and chr4 without; unplaced reads at the end; indexed by ls_bam_split."""
    # the genes are generated on the first 2 Mb of chr1, so that chr3 gets its share; chr1's far bins get hand_reads
    d = synth.generate(seed=91, contig_lens=[2_000_000] + LENS[1:], n_genes=24, n_reads=6000, n_cells=40)
    b = d.batch
    keep = np.nonzero((b.tid == 0) | (b.tid == 2))[0]
    allr = concat(b.select(keep), hand_reads(np.random.default_rng(92)))
    order = np.lexsort((allr.pos, allr.tid))
    allr = allr.select(order)
    tmp = tmp_path_factory.mktemp("bai_stream")
    raw, bam = str(tmp / "raw.bam"), str(tmp / "x.bam")
    bamio.write_bam(raw, d.contig_names, LENS, allr,
                    lambda i: None if allr.cell[i] < 0 else synth.barcode_of(int(allr.cell[i])) + "-1")
    split_one_type(raw, bam, [synth.barcode_of(c) for c in range(d.n_cells + d.n_extra_cells)])
    append_unplaced(bam, 50)
    t = os.stat(bam).st_mtime
    os.utime(bam + ".bai", (t + 1, t + 1))
    plain = str(tmp / "plain" / "x.bam")  # the same BAM without an index
    os.makedirs(os.path.dirname(plain))
    shutil.copy(bam, plain)
    fa = str(tmp / "ref.fa")
    pad = np.frombuffer(b"ACGT", np.uint8)[np.random.default_rng(93).integers(0, 4, LENS[0] - 2_000_000)]
    bamio.write_fasta(fa, d.contig_names, [np.concatenate([d.contig_seq(0), pad])] +
                      [d.contig_seq(i) for i in range(1, len(LENS))])
    return d, bam, plain, fa, tmp


# ---- the independent side: records of the file and of the index's spans ------------------------------------------------
def walk(bam):
    """Every record of the file in order: (virtual offset, next virtual offset, name, fields)."""
    rd = bai_query.BgzfReader(bam)
    head, v = rd.read(0, 12)
    l_text = struct.unpack_from("<I", head, 4)[0]
    _, v = rd.read(v, l_text - 4)
    n_ref_b, v = rd.read(v, 4)
    for _ in range(struct.unpack("<I", n_ref_b)[0]):
        ln, v = rd.read(v, 4)
        _, v = rd.read(v, struct.unpack("<I", ln)[0] + 4)
    out = []
    while True:
        try:
            hb, v2 = rd.read(v, 4)
        except EOFError:
            break
        if not hb:
            break
        rec, v3 = rd.read(v2, struct.unpack("<I", hb)[0])
        tid, pos, l_name, mapq, _bin, n_cig, flag, l_seq = struct.unpack_from("<iiBBHHHI", rec, 0)
        cig = struct.unpack_from("<%dI" % n_cig, rec, 32 + l_name)
        q0 = 32 + l_name + 4 * n_cig + (l_seq + 1) // 2
        out.append((v, v3, rec[32:32 + l_name - 1].decode(),
                    (tid, pos, flag, mapq, l_seq, cig, zlib.crc32(rec[q0:q0 + l_seq]))))
        v = v3
        if v >> 16 >= len(rd.buf) - 28:
            break
    return out


def index_spans(bam, regions):
    """SAM spec 5.3 over the merged regions, chunks merged where they share a BGZF member: [(start, end)] voffsets."""
    refs, _ = bai_query.read_bai(bam + ".bai")
    merged = []
    for t, s, e in sorted(regions):
        if merged and merged[-1][0] == t and s <= merged[-1][2]:
            merged[-1][2] = max(merged[-1][2], e)
        else:
            merged.append([t, s, e])
    chunks = []
    for t, s, e in merged:
        bins, lin = refs[t]
        min_off = lin[min(s >> 14, len(lin) - 1)] if lin else 0
        chunks += [(max(c0, min_off), c1) for b in bai_query.reg2bins(s, e) if b in bins and b != 37450
                   for c0, c1 in bins[b] if c1 > min_off]
    spans = []
    for c0, c1 in sorted(chunks):
        if spans and c0 >> 16 <= spans[-1][1] >> 16:
            spans[-1][1] = max(spans[-1][1], c1)
        else:
            spans.append([c0, c1])
    return spans


def member_bytes(bam, spans):
    """Compressed bytes of the BGZF members the spans touch."""
    rd = bai_query.BgzfReader(bam)
    total = 0
    for s, e in spans:
        c, last = s >> 16, (e >> 16) if e & 0xffff else (e >> 16) - 1
        while c <= last:
            bsize = rd.block(c)[1]
            total += bsize
            c += bsize
    return total


def overlaps(fields, regions):
    tid, pos, flag, _mq, _lq, cig, _q = fields
    span = sum(c >> 4 for c in cig if (c & 15) in (0, 2, 3, 7, 8))
    end = max(pos + span, pos + 1)
    return any(t == tid and s < end and pos < e for t, s, e in regions)


# ---- the reader under test ---------------------------------------------------------------------------------------------
def stream_records(bam, regions, chunk_bytes=64 << 10):
    """(records as field tuples, index note, compressed bytes, inflated bytes) of BamStream, regions set or not."""
    bs = bamio.BamStream(bam, threads=3)
    note = "not set"
    if regions is not None:
        r = np.array(regions, np.int64).reshape(-1, 3)
        note = bs.set_regions(r[:, 0], r[:, 1], r[:, 2])
    out, slot = [], NumpySlot()
    while True:
        got = bs.next_chunk(chunk_bytes, slot)
        if got is None:
            break
        b, _n, _ends = got
        for i in range(b.n_reads):
            c0, c1, b0 = int(b.cigar_off[i]), int(b.cigar_off[i + 1]), int(b.base_off[i])
            lq = int(b.l_qseq[i])
            out.append((int(b.tid[i]), int(b.pos[i]), int(b.flag[i]), int(b.mapq[i]), lq,
                        tuple(int(x) for x in b.cigar[c0:c1]), zlib.crc32(b.qual[b0:b0 + lq].tobytes())))
    io = (bs.compressed_bytes, bs.inflated_bytes)
    bs.close()
    return out, note, io[0], io[1]


def random_regions(rng, n, width):
    tids = rng.choice([0, 0, 0, 1, 2, 2, 3], n)
    out = []
    for t in tids.tolist():
        s = int(rng.integers(0, LENS[t] - width))
        out.append((t, s, s + int(rng.integers(1, width))))
    return out


def boundary_regions():
    out = []
    for b in BOUNDARIES:
        out += [(0, b - 1, b), (0, b, b + 1), (0, b - 30, b + 30)]
    return out + [(1, 1000, 60000), (3, 0, 200_000), (3, 150_000, 150_010)]


REGION_SETS = {
    "boundaries": lambda rng: boundary_regions(),
    "sparse sites": lambda rng: random_regions(rng, 60, 3),
    "windows": lambda rng: random_regions(rng, 25, 50_000),
    "touching windows": lambda rng: [(0, s, s + 50_000) for s in range((8 << 20) - 200_000, (8 << 20) + 200_000, 50_000)],
    "whole contigs": lambda rng: [(t, 0, l) for t, l in enumerate(LENS)],
}


@pytest.mark.parametrize("name", sorted(REGION_SETS))
def test_span_reader_returns_the_index_spans_records(case, name):
    d, bam, plain, fa, tmp = case
    regions = REGION_SETS[name](np.random.default_rng(sorted(REGION_SETS).index(name)))
    recs = walk(bam)
    spans = index_spans(bam, regions)
    want = [f for v0, _v1, _nm, f in recs if any(s <= v0 < e for s, e in spans)]
    got, note, comp, _infl = stream_records(bam, regions)
    assert note is None
    assert got == want  # exactly the records of the spans, in file order
    # after the overlap filter: the brute-force scan of the whole file, and the independent index query
    brute = [f for _v0, _v1, _nm, f in recs if overlaps(f, regions)]
    assert [f for f in got if overlaps(f, regions)] == brute
    names = {nm for _v0, _v1, nm, f in recs if overlaps(f, regions)}
    assert names == {nm for t, s, e in regions for nm, _p in bai_query.query(bam, t, s, e)}
    assert comp == member_bytes(bam, spans)  # the saving is exact
    if name == "boundaries":
        assert brute and any(f[5] and any((c & 15) == 3 and (c >> 4) >= 99_850 for c in f[5]) for f in brute)
    if name == "whole contigs":
        assert got == [r[3] for r in recs if r[3][0] >= 0]  # every placed record, none of the unplaced ones


def test_region_sets_cut_records_at_span_edges(case):
    """The region sets above include spans whose first record and spans whose last record are cut by a BGZF member
    boundary, so the reader is checked on both."""
    d, bam, plain, fa, tmp = case
    recs = walk(bam)
    cut = [(v0, v1) for v0, v1, _nm, _f in recs if v0 >> 16 != v1 >> 16 and v1 & 0xffff]
    starts, ends = set(), set()
    for name in sorted(REGION_SETS):
        spans = index_spans(bam, REGION_SETS[name](np.random.default_rng(sorted(REGION_SETS).index(name))))
        starts |= {s for s, _e in spans}
        ends |= {e for _s, e in spans}
    assert any(v0 in starts for v0, _v1 in cut) and any(v1 in ends for _v0, v1 in cut)


def test_sparse_sites_read_a_small_part_of_the_file(case):
    d, bam, plain, fa, tmp = case
    regions = random_regions(np.random.default_rng(7), 20, 2)
    got, note, comp, infl = stream_records(bam, regions)
    assert note is None
    assert comp == member_bytes(bam, index_spans(bam, regions))
    assert comp < os.path.getsize(bam) // 4
    whole, note0, comp0, infl0 = stream_records(plain, regions)
    assert note0 == "no .bai index" and infl < infl0 // 4
    assert comp0 == os.path.getsize(plain)  # every member, the header's and the EOF marker included


def write_bai(path, refs, n_no_coor, extra_refs=0):
    out = bytearray(b"BAI\1" + struct.pack("<i", len(refs) + extra_refs))
    for bins, lin in refs:
        out += struct.pack("<i", len(bins))
        for b, ch in bins.items():
            out += struct.pack("<Ii", b, len(ch)) + b"".join(struct.pack("<QQ", *c) for c in ch)
        out += struct.pack("<i", len(lin)) + b"".join(struct.pack("<Q", x) for x in lin)
    out += struct.pack("<ii", 0, 0) * extra_refs
    if n_no_coor is not None:
        out += struct.pack("<Q", n_no_coor)
    open(path, "wb").write(bytes(out))


def shifted(refs, delta):
    return [({b: [(c0 + delta, c1 + delta) for c0, c1 in ch] for b, ch in bins.items()}, lin) for bins, lin in refs]


@pytest.mark.parametrize("damage", ["missing", "truncated", "stale", "n_ref", "past EOF", "not at a member"])
def test_unusable_index_reads_the_whole_file(case, tmp_path, damage):
    d, bam, plain, fa, tmp = case
    x = str(tmp_path / "x.bam")
    shutil.copy(bam, x)
    blob = open(bam + ".bai", "rb").read()
    refs, n_no_coor = bai_query.read_bai(bam + ".bai")
    size = os.path.getsize(bam)
    if damage == "truncated":
        open(x + ".bai", "wb").write(blob[:len(blob) // 2])
    elif damage == "n_ref":
        write_bai(x + ".bai", refs, n_no_coor, extra_refs=1)
    elif damage == "past EOF":
        write_bai(x + ".bai", shifted(refs, size << 16), n_no_coor)
    elif damage == "not at a member":
        write_bai(x + ".bai", shifted(refs, 1 << 16), n_no_coor)
    elif damage == "stale":
        open(x + ".bai", "wb").write(blob)
    t = os.stat(x).st_mtime
    if damage == "stale":
        os.utime(x + ".bai", (t - 10, t - 10))
    elif damage != "missing":
        os.utime(x + ".bai", (t + 1, t + 1))
    regions = random_regions(np.random.default_rng(3), 30, 5000)
    got, note, comp, _ = stream_records(x, regions)
    whole, _n, _c, _i = stream_records(x, None)
    assert isinstance(note, str) and note and "\n" not in note, note
    assert {"missing": "no .bai", "truncated": "truncated", "stale": "older", "n_ref": "references",
            "past EOF": "outside", "not at a member": "outside"}[damage] in note
    assert got == whole and len(whole) == len(walk(bam))


def test_index_named_without_the_bam_suffix(case, tmp_path):
    d, bam, plain, fa, tmp = case
    x = str(tmp_path / "x.bam")
    shutil.copy(bam, x)
    shutil.copy(bam + ".bai", str(tmp_path / "x.bai"))
    t = os.stat(x).st_mtime
    os.utime(str(tmp_path / "x.bai"), (t + 1, t + 1))
    regions = boundary_regions()
    assert stream_records(x, regions)[:2] == stream_records(bam, regions)[:2]
    assert stream_records(x, regions)[1] is None


# ---- the streamed drivers with and without the index ---------------------------------------------------------------------
def table_body(path):
    with open(path) as f:
        return [l for l in f if not l.startswith("##fileDate")]


@pytest.mark.parametrize("chrom", ["all", "chr3", "bed"])
def test_stream_count_same_with_and_without_index(case, monkeypatch, chrom):
    d, bam, plain, fa_path, tmp = case
    fa = bamio.Fasta(fa_path)
    bed = None
    if chrom == "bed":
        bed = str(tmp / "focus.bed")
        with open(bed, "w") as f:
            for t, s, e in random_regions(np.random.default_rng(11), 40, 20_000) + boundary_regions():
                f.write("%s\t%d\t%d\n" % (d.contig_names[t], s, e))
    named = make_windows(fa.references, fa.lengths, "all" if chrom == "bed" else chrom, 50000,
                         **({"bed": bed} if bed else {}))
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", OracleEngine)
    prm = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=30)
    out = {}
    for label, path in (("indexed", bam), ("plain", plain)):
        stats = []
        pipeline.stream_count(path, named, fa, prm, str(tmp / ("count_%s_%s.tsv" % (chrom, label))), "x", [0, 0],
                              chunk_bytes=64 << 10, stats_out=stats)
        out[label] = (table_body(str(tmp / ("count_%s_%s.tsv" % (chrom, label)))), stats)
    assert out["indexed"][0] == out["plain"][0] and len(out["indexed"][0]) > 100
    si, sp = out["indexed"][1], out["plain"][1]
    assert all(s["indexed"] for s in si) and not any(s["indexed"] for s in sp)
    assert sum(s["compressed_bytes"] for s in si) <= sum(s["compressed_bytes"] for s in sp)
    if chrom == "chr3":
        assert sum(s["inflated_bytes"] for s in si) < sum(s["inflated_bytes"] for s in sp) // 2


@pytest.mark.parametrize("chunk_kb,bins", [(64, 5000), (1024, 50000)])
def test_stream_genotype_same_with_and_without_index(case, monkeypatch, chunk_kb, bins):
    d, bam, plain, fa, tmp = case
    recs = [r[3] for r in walk(bam) if r[3][0] >= 0]
    rng = np.random.default_rng(chunk_kb)
    pick = rng.choice(len(recs), 300, replace=False)
    keys = sorted({(recs[i][0], recs[i][1] + int(rng.integers(0, 300))) for i in pick} |
                  {(0, b) for b in BOUNDARIES} | {(1, 5000), (3, 100)})
    st = np.array([k[0] for k in keys], np.int32)
    sp = np.array([k[1] for k in keys], np.int32)
    alt = rng.integers(0, 4, st.shape[0]).astype(np.uint8)
    col = {synth.barcode_of(c): c for c in range(30)}
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", OracleEngine)
    kw = dict(min_bq=30, min_mq=60, max_depth=20, alt_only=False)
    res = {}
    for label, path in (("indexed", bam), ("plain", plain)):
        stats = []
        res[label] = pipeline.stream_genotype(path, (st, sp, alt), bins, 30, lambda t: col.get(t.split("-")[0], -1), kw,
                                              0.2, 100.0, None, [0, 0, 0], chunk_bytes=chunk_kb << 10, stats_out=stats)
        res[label + " stats"] = stats
    for x, y in zip(res["indexed"][:4], res["plain"][:4]):
        assert x.dtype == y.dtype and np.array_equal(x, y)
    assert res["indexed"][0].shape[0] > 100
    si, sp_ = res["indexed stats"], res["plain stats"]
    assert all(s["indexed"] for s in si)
    assert sum(s["compressed_bytes"] for s in si) < sum(s["compressed_bytes"] for s in sp_)
