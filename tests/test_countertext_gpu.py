"""GPU suite for the counter table written on the device (ls_countertext.cu): the text equals the host writer
ls_write_counter_rows on real runs, on random site tables and at the edges of the number formats; the block, state and
argument rules of the two entry points; BaseCellCounter against the goldens with the device writer; and device-text
against host-text streamed runs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from longsom_b200 import _lib as L
from longsom_b200 import bamio, pipeline, synth
from longsom_b200.batch import SiteCounts, Windows, make_windows
from longsom_b200.blocks import COUNTER_ROW_MAX, PinnedBlock, counter_text
from longsom_b200.engine import CountParams

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "support"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_cli_gpu import CASES, assert_same, file_lines, gold_lines, has_gold  # noqa: E402

SCRIPTS = os.path.join(ROOT, "workflow", "scripts")
U32 = 0xffffffff


def host_text(sites, names, tmp_path):
    """{tid: bytes} of ls_write_counter_rows for every contig of `sites`."""
    out = {}
    for t in np.unique(sites.tid).tolist():
        path = str(tmp_path / ("host_%d.txt" % t))
        if os.path.exists(path):
            os.remove(path)
        pipeline.write_counter_rows(path, names[t].decode("latin-1"), sites, t)
        with open(path, "rb") as f:
            out[t] = f.read()
    return out


def device_text(eng, names, cap=None):
    """counter_text of the last run's sites through two pinned blocks of `cap` bytes."""
    blocks = [PinnedBlock(eng, cap or 64 << 20) for _ in range(2)]
    try:
        return {t: bytes(v) for t, v in counter_text(eng, names, blocks).items()}
    finally:
        for b in blocks:
            b.free()


def random_sites(rng, n, n_contigs):
    """A site table ordered as a run orders it (grouped by ascending tid) with counts over the whole uint32 range."""
    tid = np.sort(rng.integers(0, n_contigs, n)).astype(np.int32)
    pos = rng.integers(0, 2**31 - 1, n).astype(np.int32)
    ref = rng.choice(np.frombuffer(b"ACGTN", np.uint8), n)
    digits = rng.integers(0, 10, (n, 26))  # every number of decimal digits, 1 .. 10
    counts = np.minimum(rng.integers(0, 10, (n, 26)) * 10 ** digits.astype(np.float64) + rng.integers(0, 10, (n, 26)),
                        U32).astype(np.uint32)
    return SiteCounts(tid, pos, ref, counts)


@pytest.fixture(scope="module")
def run_case(built):
    d = synth.generate(seed=23, contig_lens=[150000, 90000, 16600], chrm=True, n_genes=12, n_reads=8000, n_cells=120)
    w = Windows.from_intervals(make_windows(d.contig_lens, 50000), d.contig_seqs())
    return d, w


def test_real_run_text_matches_host(engine, run_case, tmp_path):
    d, w = run_case
    names = [n.encode() for n in d.contig_names]
    prm = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1)
    sites = engine.pileup_count(d.batch, w, prm)
    assert sites.n_sites > 10000 and len(np.unique(sites.tid)) == 3
    want = host_text(sites, names, tmp_path)
    got = engine.pileup_count_text(d.batch, w, prm, names)
    assert engine.last_stats["n_sites"] == sites.n_sites
    assert got == want
    # the load of a run that was not compacted yet compacts it; small blocks split every contig
    engine.upload(d.batch, w)
    engine.run(prm)
    assert device_text(engine, names, cap=4096) == want


@pytest.mark.parametrize("n", [0, 1, 5000, 300000])
def test_random_sites_match_host(engine, tmp_path, n):
    rng = np.random.default_rng(n)
    names = [b"c", b"chr1", b"x" * 200, b"HLA-DRB1*15:01:01:01", b"chrUn_KI270742v1"]
    sites = random_sites(rng, n, len(names))
    engine.pileup_sites_upload(sites)
    lo, hi = engine.pileup_text_load(names)
    for t in range(len(names)):
        sel = np.nonzero(sites.tid == t)[0]
        assert (lo[t], hi[t]) == ((sel[0], sel[-1] + 1) if sel.size else (0, 0))
    want = host_text(sites, names, tmp_path)
    assert device_text(engine, names) == want
    if n:
        assert device_text(engine, names, cap=COUNTER_ROW_MAX + 200) == want  # at most a few rows per block


def edge_sites():
    """Counts and BQ sums at 2^32-1, BCf + BCr wrapping, pos at 2^31-2 and at 0, on a 1-byte and a 200-byte name."""
    rows = []
    c = np.full(26, U32, np.uint32)
    rows.append((0, 2**31 - 2, ord("A"), c))
    c = np.zeros(26, np.uint32)
    c[8:14], c[14:20] = U32, [1, 2, 3, U32, 2**31, 0]  # BC wraps to 0, 1, 2, 2^32-2, 2^31-1, 2^32-1
    rows.append((0, 0, ord("N"), c))
    c = np.arange(26, dtype=np.uint32) * 1000003
    rows.append((1, 2**31 - 2, ord("T"), c))
    rows.append((1, 9, ord("G"), np.zeros(26, np.uint32)))
    tid, pos, ref, counts = zip(*rows)
    return SiteCounts(np.array(tid, np.int32), np.array(pos, np.int32), np.array(ref, np.uint8), np.stack(counts))


def test_edges_match_host(engine, tmp_path):
    names = [b"Z", b"n" * 200]
    sites = edge_sites()
    engine.pileup_sites_upload(sites)
    want = host_text(sites, names, tmp_path)
    got = device_text(engine, names)
    assert got == want
    assert b"\t2147483647\tA\t" in got[0] and b"|0:1:2:4294967294:2147483647:4294967295|" in got[0]
    for i in range(sites.n_sites):  # one site at a time
        one = SiteCounts(sites.tid[i:i + 1], sites.pos[i:i + 1], sites.ref[i:i + 1], sites.counts[i:i + 1])
        engine.pileup_sites_upload(one)
        assert device_text(engine, names) == host_text(one, names, tmp_path)


def test_block_capacity_and_state(engine, run_case, tmp_path):
    names = [b"Z", b"n" * 200]
    sites = edge_sites()
    engine.pileup_sites_upload(sites)
    want = host_text(sites, names, tmp_path)
    rows = want[0].splitlines(keepends=True)
    lo, hi = engine.pileup_text_load(names)
    assert (lo.tolist(), hi.tolist()) == ([0, 2], [2, 4])
    blk = PinnedBlock(engine, 1024)
    try:
        n0 = len(rows[0])
        assert engine.pileup_text(0, 2, blk.addr, n0) == (1, n0)  # exactly one row
        assert bytes(blk.view[:n0]) == rows[0]
        assert engine.pileup_text(0, 2, blk.addr, n0 + len(rows[1]) - 1) == (1, n0)
        assert engine.pileup_text(1, 2, blk.addr, 1024) == (1, len(rows[1]))
        assert bytes(blk.view[:len(rows[1])]) == rows[1]
        assert engine.pileup_text(2, 2, blk.addr, 0) == (0, 0)
        with pytest.raises(L.LongSomError) as e:  # one byte short of the first row
            engine.pileup_text(0, 2, blk.addr, n0 - 1)
        assert e.value.code == L.LS_E_CAPACITY
        with pytest.raises(L.LongSomError) as e:
            engine.pileup_text(0, 5, blk.addr, 1024)
        assert e.value.code == L.LS_E_ARG
        # no sites: empty ranges, and every text call is (0, 0)
        engine.pileup_sites_upload(SiteCounts.empty(0))
        lo, hi = engine.pileup_text_load(names)
        assert not lo.any() and not hi.any() and engine.pileup_text(0, 0, blk.addr, 1024) == (0, 0)
        assert device_text(engine, names) == {}
        # a new run discards the load; an engine without a run refuses the load
        d, w = run_case
        engine.upload(d.batch, w)
        engine.run(CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1))
        with pytest.raises(L.LongSomError) as e:
            engine.pileup_text(0, 0, blk.addr, 1024)
        assert e.value.code == L.LS_E_STATE
        from longsom_b200.engine import Engine
        with Engine(0) as fresh:
            for call in (lambda: fresh.pileup_text_load(names), lambda: fresh.pileup_text(0, 0, blk.addr, 1024)):
                with pytest.raises(L.LongSomError) as e:
                    call()
                assert e.value.code == L.LS_E_STATE
    finally:
        blk.free()


def test_load_refuses_bad_tids(engine):
    sites = edge_sites()
    engine.pileup_sites_upload(sites)
    with pytest.raises(L.LongSomError) as e:  # tid 1 has no name
        engine.pileup_text_load([b"only"])
    assert e.value.code == L.LS_E_ARG
    bad = SiteCounts(sites.tid[::-1].copy(), sites.pos, sites.ref, sites.counts)
    engine.pileup_sites_upload(bad)
    with pytest.raises(L.LongSomError) as e:
        engine.pileup_text_load([b"a", b"b"])
    assert e.value.code == L.LS_E_ARG


# ---- BaseCellCounter end to end -------------------------------------------------------------------------------------
def run_counter(args, gpus, text=None):
    env = dict(os.environ, LS_STREAM_TIMING="1")
    env.pop("LONGSOM_GPUS", None)
    env.pop("LONGSOM_COUNTER_TEXT", None)
    if gpus:
        env["LONGSOM_GPUS"] = gpus
    if text:
        env["LONGSOM_COUNTER_TEXT"] = text
    cmd = [sys.executable, os.path.join(SCRIPTS, "SNVCalling", "BaseCellCounter.py")] + [str(a) for a in args]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, "%s failed:\n%s" % (" ".join(cmd), r.stdout[-3000:])
    busy = [l for l in r.stdout.splitlines() if l.startswith("[stream_count] busy seconds:")]
    assert len(busy) == 1, r.stdout[-3000:]
    return float(busy[0].split("text ")[1].split(",")[0])


@pytest.mark.parametrize("bai", [False, True])
@pytest.mark.parametrize("gpus", [None, "0,0,0"])
@pytest.mark.parametrize("case", CASES)
def test_counter_cli_matches_goldens(tmp_path, built, case, gpus, bai):
    import bai_write
    import pipeline_inputs as pi
    d = str(tmp_path)
    p, data = pi.write_inputs(case, d)
    if bai:
        for k in ("cancer", "normal", "full"):
            if k in p:
                bai_write.write_bai(p[k])
    for name, bam in (("Cancer", p["cancer"]), ("Non-Cancer", p["normal"])):
        text_s = run_counter(["--bam", bam, "--ref", p["ref"], "--chrom", "all", "--out_folder", d, "--id", "s." + name,
                              "--min_bq", 20, "--min_mq", 60, "--tmp_dir", os.path.join(d, "tmp")], gpus)
        assert text_s > 0  # the rows were formatted on the device
        assert_same(file_lines(os.path.join(d, "s.%s.tsv" % name)), gold_lines(case, "counts.%s.tsv" % name),
                    "BaseCellCounter " + name)
    if has_gold(case, "counts.full_bed.tsv"):
        bed, bed_out = pi.write_beds(case, d, data)
        for name, extra in (("bed", ["--bed", bed, "--chrom", "all"]),
                            ("bed_out", ["--bed", bed, "--bed_out", bed_out, "--chrom", data.contig_names[0]]),
                            ("bedout_only", ["--bed_out", bed_out, "--bin", 20000, "--chrom", "all"])):
            run_counter(["--bam", p["full"], "--ref", p["ref"], "--out_folder", d, "--id", "full." + name, "--min_bq", 20,
                         "--min_mq", 60, "--min_dp", 3, "--min_cc", 2, "--tmp_dir", os.path.join(d, "tmp")] + extra, gpus)
            assert_same(file_lines(os.path.join(d, "full.%s.tsv" % name)), gold_lines(case, "counts.full_%s.tsv" % name),
                        "BaseCellCounter --" + name)
    assert not [f for f in os.listdir(d) if ".part." in f]


@pytest.mark.parametrize("devices", [[0], [0, 0, 0]])
def test_streamed_device_text_equals_host_text(tmp_path, built, monkeypatch, devices):
    """Small chunks, so that contigs are split across chunks and engines."""
    d = synth.generate(seed=61, contig_lens=[400000, 300000, 200000, 16600], chrm=True, n_genes=30, n_reads=30000,
                       n_cells=60, n_hot_genes=1, hot_fraction=0.2)
    b = d.batch
    bam, fa_path = str(tmp_path / "x.bam"), str(tmp_path / "ref.fa")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b,
                    lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    bamio.write_fasta(fa_path, d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    fa = bamio.Fasta(fa_path)
    from longsom_b200.windows import make_windows as named_windows
    named = named_windows(fa.references, fa.lengths, "all", 50000)
    prm = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=300)
    out = {}
    for mode in ("host", "device"):
        monkeypatch.setenv("LONGSOM_COUNTER_TEXT", mode)
        stats = []
        n = pipeline.stream_count(bam, named, fa, prm, str(tmp_path / (mode + ".tsv")), "x", devices, chunk_bytes=1 << 20,
                                  stats_out=stats)
        assert len(stats) >= 4
        assert ("text_s" in stats[0]) == (mode == "device")
        out[mode] = (n, file_lines(str(tmp_path / (mode + ".tsv"))))
    assert out["device"] == out["host"] and out["host"][0] > 10000
