"""The host side of the counter table written on the device, with a stand-in engine that formats rows in Python: the
contig ranges and whole-row blocks of blocks.counter_text, and the streamed counter's part files fed with per-contig
text instead of counts (pipeline.stream_count), against the host writer's table."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from longsom_b200 import bamio, blocks, pipeline, synth
from longsom_b200.batch import SiteCounts
from longsom_b200.engine import CountParams
from longsom_b200.windows import make_windows

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_stream_driver_cpu import NumpySlot, OracleEngine  # noqa: E402


class HostBlock:
    """Stand-in for blocks.PinnedBlock: pageable memory."""

    def __init__(self, nbytes):
        self.nbytes, self._buf = nbytes, C.create_string_buffer(nbytes)
        self.addr = C.addressof(self._buf)
        self.view = memoryview((C.c_char * nbytes).from_address(self.addr)).cast('B')

    def free(self):
        self.view.release()


class TextEngine:
    """pileup_text_load / pileup_text over a SiteCounts, rows formatted by pipeline.format_counter_lines; records every
    text call."""

    def __init__(self, sites):
        self.sites, self.calls, self.rows = sites, [], None

    def pileup_text_load(self, names):
        s = self.sites
        self.rows = [r.encode() for t in np.unique(s.tid).tolist() for r in pipeline.format_counter_lines(
            names[t].decode(), s.pos[s.tid == t], s.ref[s.tid == t], s.counts[s.tid == t])]
        lo, hi = np.zeros(len(names), np.int64), np.zeros(len(names), np.int64)
        for t in np.unique(s.tid).tolist():
            lo[t], hi[t] = np.searchsorted(s.tid, t, "left"), np.searchsorted(s.tid, t, "right")
        return lo, hi

    def pileup_text(self, site_lo, site_hi, addr, cap):
        n, nb = 0, 0
        while site_lo + n < site_hi and nb + len(self.rows[site_lo + n]) <= cap:
            nb += len(self.rows[site_lo + n])
            n += 1
        if n == 0:
            raise RuntimeError("a row is longer than the capacity")
        C.memmove(addr, b"".join(self.rows[site_lo:site_lo + n]), nb)
        self.calls.append((site_lo, site_hi, n, nb, cap))
        return n, nb


def random_sites(seed, n, n_contigs):
    rng = np.random.default_rng(seed)
    tid = np.sort(rng.choice(n_contigs, n)).astype(np.int32)
    counts = rng.integers(0, 2**32, (n, 26), dtype=np.uint64).astype(np.uint32) >> rng.integers(0, 32, (n, 26)).astype(np.uint32)
    return SiteCounts(tid, rng.integers(0, 2**31 - 1, n).astype(np.int32), rng.choice(np.frombuffer(b"ACGTN", np.uint8), n),
                      counts)


@pytest.mark.parametrize("cap", [None, 0, 1, 7, 1000])
def test_counter_text_blocks_hold_whole_rows(cap):
    names = [b"c0", b"chrUn_KI270742v1", b"x" * 200, b"unused", b"chrM"]
    sites = random_sites(5, 3000, 5)
    sites = SiteCounts(*(a[sites.tid != 3] for a in (sites.tid, sites.pos, sites.ref, sites.counts)))
    eng = TextEngine(sites)
    longest = len(names[2]) + blocks.COUNTER_ROW_MAX
    nbytes = blocks.counter_block_bytes(names) if cap is None else longest + cap
    assert nbytes >= longest
    bufs = [HostBlock(nbytes) for _ in range(2)]
    got = blocks.counter_text(eng, names, bufs)
    for b in bufs:
        b.free()
    assert sorted(got) == [0, 1, 2, 4]  # contigs with sites, each once
    for t, text in got.items():
        sel = sites.tid == t
        want = "".join(pipeline.format_counter_lines(names[t].decode(), sites.pos[sel], sites.ref[sel], sites.counts[sel]))
        assert text == want.encode()
    # the calls walk each contig's range in order, every block as full as whole rows allow
    for (lo, hi, n, nb, c), nxt in zip(eng.calls, eng.calls[1:] + [None]):
        assert c == nbytes and nb <= c
        if lo + n < hi:
            assert nb + len(eng.rows[lo + n]) > c and nxt[0] == lo + n
    if cap is not None and cap < 100:
        assert len(eng.calls) > 100


def test_counter_row_max_bounds_every_row():
    names = [b"n" * 200]
    c = np.full((1, 26), 2**32 - 1, np.uint32)
    row = pipeline.format_counter_lines(names[0].decode(), np.array([2**31 - 2], np.int32), np.array([ord("A")], np.uint8), c)[0]
    assert len(row.encode()) == len(names[0]) + blocks.COUNTER_ROW_MAX


class OracleTextEngine(OracleEngine):
    """The oracle's counts, given back as pileup_count_text does: {tid: text} through counter_text and small blocks."""

    def pileup_count_text(self, batch, windows, params, names):
        eng = TextEngine(self.pileup_count(batch, windows, params))
        bufs = [HostBlock(len(max(names, key=len)) + blocks.COUNTER_ROW_MAX + 300) for _ in range(2)]
        text = blocks.counter_text(eng, names, bufs)
        self.last_stats = dict(n_sites=eng.sites.n_sites, text_s=0.0)
        return text


@pytest.fixture(scope="module")
def bam_case(tmp_path_factory, built):
    d = synth.generate(seed=44, contig_lens=[120000, 60000, 16600], chrm=True, n_genes=8, n_reads=4000, n_cells=40)
    b = d.batch
    tmp = tmp_path_factory.mktemp("countertext")
    bam, ref = str(tmp / "x.bam"), str(tmp / "ref.fa")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    bamio.write_fasta(ref, d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    return bam, ref, tmp


def test_streamed_counter_with_text_engine_equals_host_writer(bam_case, monkeypatch):
    bam, ref, tmp = bam_case
    fa = bamio.Fasta(ref)
    named = make_windows(fa.references, fa.lengths, "all", 5000)
    prm = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=40)
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", OracleTextEngine)
    out = {}
    for mode in ("host", "device"):
        monkeypatch.setenv("LONGSOM_COUNTER_TEXT", mode)
        stats = []
        path = str(tmp / (mode + ".tsv"))
        n = pipeline.stream_count(bam, named, fa, prm, path, "x", [0, 0, 0], chunk_bytes=64 << 10, stats_out=stats)
        assert ("text_s" in stats[0]) == (mode == "device") and len(stats) >= 8
        with open(path) as f:
            out[mode] = (n, [l for l in f if not l.startswith("##fileDate")])
        assert not [f for f in os.listdir(str(tmp)) if ".part." in f]
    assert out["device"] == out["host"] and out["host"][0] > 1000
