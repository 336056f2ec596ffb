"""The streamed BAM driver (pipeline.stream_chunks) under the counter and the genotype scripts, with the CPU oracle or
stand-ins in place of the engine: an engine error surfaces as an exception instead of a hang, the streamed counter's
table equals the whole-file table with the depth cap firing and with gaps between the windows, and results come back in
chunk order whatever order the workers finish in."""
import os
import threading
import time

import numpy as np
import pytest

from longsom_b200 import bamio, pipeline, synth
from longsom_b200.engine import CountParams
from longsom_b200.windows import make_windows


class NumpySlot:
    """Stand-in for pipeline.PinnedSlot without a GPU (pinned memory needs a CUDA context); counts the frees."""
    freed = 0

    def __call__(self, n, nc, nb):
        return dict(tid=np.zeros(n, np.int32), pos=np.zeros(n, np.int32), flag=np.zeros(n, np.uint16),
                    mapq=np.zeros(n, np.uint8), cell=np.zeros(n, np.int32), l_qseq=np.zeros(n, np.int32),
                    cigar_off=np.zeros(n + 1, np.uint32), base_off=np.zeros(n + 1, np.uint64), cigar=np.zeros(nc, np.uint32),
                    seq4=np.zeros(nb // 2 + 1, np.uint8), qual=np.zeros(nb, np.uint8))

    def free(self):
        NumpySlot.freed += 1


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


class FailingEngine(OracleEngine):
    """Raises on its second device call."""
    calls = 0

    def _count(self):
        self.calls += 1
        if self.calls == 2:
            raise RuntimeError("device error")

    def pileup_count(self, batch, windows, params):
        self._count()
        return super().pileup_count(batch, windows, params)

    def upload(self, batch, windows=None):
        self._count()
        super().upload(batch, windows)


def failing_take_engine(dev):
    raise RuntimeError("no engine")


@pytest.fixture(scope="module")
def inputs(tmp_path_factory, built):
    """A synthetic BAM with a hot gene (half the reads) on the first of two contigs, its FASTA and a --bed with gaps."""
    d = synth.generate(seed=41, contig_lens=[120000, 16600], chrm=True, n_genes=5, n_reads=4000, n_cells=40,
                       n_hot_genes=1, hot_fraction=0.5)
    b = d.batch
    tmp = tmp_path_factory.mktemp("stream")
    bam, ref, bed = str(tmp / "x.bam"), str(tmp / "ref.fa"), str(tmp / "focus.bed")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    bamio.write_fasta(ref, d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    with open(bed, "w") as f:
        for c, l in zip(d.contig_names, d.contig_lens):
            for s in range(0, int(l), 9000):
                f.write("%s\t%d\t%d\n" % (c, s, min(s + 6000, int(l))))
    return d, bam, ref, bed, tmp


def whole_file_table(bam, fa, named, prm, ID, out):
    """The LONGSOM_STREAM=0 counter with the oracle as the engine."""
    import oracle
    from longsom_b200.batch import Windows
    bd, batch, _ = pipeline.load_bam_for_counting(bam)
    iv = pipeline.prune_and_sort_windows(named, bd.contig_names, batch, pipeline.read_ends(batch))
    win = Windows.from_intervals(iv, {t: fa.contig(bd.contig_names[t]) for t in {w[0] for w in iv}})
    pipeline.write_counter_tsv(out, ID, oracle.pileup_count(batch, win, prm, threads=4)[0], bd.contig_names)


def table_body(path):
    with open(path) as f:
        return [l for l in f if not l.startswith("##fileDate")]


def test_streamed_counter_equals_whole_file_with_cap_and_gaps(inputs, monkeypatch):
    d, bam, ref, bed, tmp = inputs
    fa = bamio.Fasta(ref)
    named = make_windows(fa.references, fa.lengths, "all", 5000, bed=bed)
    assert any(a[2] < b[1] for a, b in zip(named, named[1:]) if a[0] == b[0])  # gaps between windows
    capped, free = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=40), \
        CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=0)
    whole_file_table(bam, fa, named, capped, "x", str(tmp / "whole.tsv"))
    whole_file_table(bam, fa, named, free, "x", str(tmp / "free.tsv"))
    assert table_body(str(tmp / "whole.tsv")) != table_body(str(tmp / "free.tsv"))  # the cap fires
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", OracleEngine)
    stats = []
    n = pipeline.stream_count(bam, named, fa, capped, str(tmp / "stream.tsv"), "x", [0, 0, 0], chunk_bytes=64 << 10,
                              stats_out=stats)
    assert n > 0 and len(stats) >= 8
    assert max(s["n_carried"] for s in stats) > capped.max_depth  # capped windows were cut by chunk boundaries
    assert table_body(str(tmp / "stream.tsv")) == table_body(str(tmp / "whole.tsv"))


def run_with_timeout(fn, timeout=120):
    box = {}

    def target():
        try:
            box["value"] = fn()
        except BaseException as e:
            box["error"] = e
    t = threading.Thread(target=target, daemon=True)
    t.start()
    t.join(timeout)
    assert not t.is_alive(), "the streamed run did not finish within %d s" % timeout
    return box


@pytest.mark.parametrize("failure", ["second call", "take_engine"])
def test_counter_engine_error_raises_and_leaves_no_files(inputs, monkeypatch, failure):
    d, bam, ref, bed, tmp = inputs
    out_dir = tmp / ("fail_" + failure.replace(" ", "_"))
    out_dir.mkdir()
    fa = bamio.Fasta(ref)
    named = make_windows(fa.references, fa.lengths, "all", 5000)
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", FailingEngine if failure == "second call" else failing_take_engine)
    out = str(out_dir / "x.tsv")
    box = run_with_timeout(lambda: pipeline.stream_count(bam, named, fa, CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1),
                                                         out, "x", [0, 0, 0], chunk_bytes=64 << 10))
    assert isinstance(box.get("error"), RuntimeError), box
    assert str(box["error"]) == ("device error" if failure == "second call" else "no engine")
    assert os.listdir(str(out_dir)) == []  # neither the table nor a .part. file


@pytest.mark.parametrize("failure", ["second call", "take_engine"])
def test_genotype_engine_error_raises(inputs, monkeypatch, failure):
    d, bam, ref, bed, tmp = inputs
    b = d.batch
    keys = sorted({(int(b.tid[i]), int(b.pos[i]) + 10) for i in range(0, b.n_reads, 20)})
    st, sp = np.array([k[0] for k in keys], np.int32), np.array([k[1] for k in keys], np.int32)
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    monkeypatch.setattr(pipeline, "take_engine", FailingEngine if failure == "second call" else failing_take_engine)
    box = run_with_timeout(lambda: pipeline.stream_genotype(bam, (st, sp, np.zeros(st.shape[0], np.uint8)), 5000, 40,
                                                            lambda t: 0, dict(min_bq=30, min_mq=60), 0.2, 100.0, None,
                                                            [0, 0, 0], chunk_bytes=64 << 10))
    assert isinstance(box.get("error"), RuntimeError), box
    assert str(box["error"]) == ("device error" if failure == "second call" else "no engine")


def test_results_come_back_in_chunk_order(inputs, monkeypatch):
    """Earlier chunks take longer, so the workers finish out of order; the driver still yields in chunk order, and
    closing it early stops the stream and frees every slot."""
    d, bam, ref, bed, tmp = inputs
    fa = bamio.Fasta(ref)
    names = fa.references
    win = [(names.index(c), s, e) for c, s, e in make_windows(fa.references, fa.lengths, "all", 5000)]
    start = np.array([(t << 32) | s for t, s, e in win], np.int64)
    end = np.array([(t << 32) | e for t, s, e in win], np.int64)
    monkeypatch.setattr(pipeline, "PinnedSlot", NumpySlot)
    finished, lock = [], threading.Lock()

    def run(eng, batch, ends, lo, done):
        time.sleep(0.3 if lo == 0 else 0.1 if len(finished) < 6 else 0.0)
        with lock:
            finished.append(lo)
        return lo, done, batch.n_reads

    got = list(pipeline.stream_chunks(bam, start, end, [0, 0, 0], lambda t: 0, run, 64 << 10, OracleEngine))
    assert [g[1] for g in got] == sorted(finished) and finished != sorted(finished)
    assert got[0][1] == 0 and got[-1][2] == len(win)
    assert all(a[2] == b[1] for a, b in zip(got, got[1:]))  # chunk i + 1 starts at the region chunk i completed
    assert all(r == (lo, done, st["n_reads"]) for r, lo, done, st in got)
    NumpySlot.freed, n_threads = 0, threading.active_count()
    chunks = pipeline.stream_chunks(bam, start, end, [0, 0, 0], lambda t: 0, run, 64 << 10, OracleEngine)
    assert next(chunks)[1] == 0
    chunks.close()
    assert NumpySlot.freed == 4 and threading.active_count() == n_threads
