"""The streamed genotype scripts on the GPU: the CLIs with many small chunks against the whole-file path and the
reference goldens, on one engine and on three, and pipeline.stream_genotype against one Engine.genotype_sparse call over
the whole batch, bit for bit, with the depth cap firing in bins that chunk boundaries cut."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from longsom_b200 import bamio, pipeline, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "support"))
GOLD = os.path.join(ROOT, "tests", "golden")
SCRIPTS = os.path.join(ROOT, "workflow", "scripts")
CASES = [c for c in ("g1", "g2", "g3") if os.path.isdir(os.path.join(GOLD, c))]
AB = (0.2474528917555431, 162.03696139428595)
SCG = ("SingleCellGenotype", "DpMatrix", "AltMatrix", "VAFMatrix", "BinaryMatrix")


@pytest.fixture(scope="module", params=CASES)
def inputs(request, tmp_path_factory, built):
    import pipeline_inputs as pi
    case = request.param
    d = str(tmp_path_factory.mktemp("gstream_" + case))
    p, _ = pi.write_inputs(case, d)
    p["cand"] = os.path.join(d, "candidates.tsv")
    with gzip.open(os.path.join(GOLD, case, "candidates.tsv.gz"), "rb") as f, open(p["cand"], "wb") as o:
        o.write(f.read())
    return case, d, p


def run(script, args, **env):
    e = dict(os.environ, **env)
    cmd = [sys.executable, os.path.join(SCRIPTS, script)] + [str(a) for a in args]
    r = subprocess.run(cmd, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, "%s failed:\n%s" % (" ".join(cmd), r.stdout[-3000:])
    return r.stdout


def gold_text(case, name):
    """The golden's text, or (lines, sha256) for one too large to commit."""
    path = os.path.join(GOLD, case, name)
    if os.path.exists(path + ".gz"):
        with gzip.open(path + ".gz", "rb") as f:
            return f.read()
    if os.path.exists(path + ".sha256.json"):
        import json
        meta = json.load(open(path + ".sha256.json"))
        return meta["lines"], meta["sha256"]
    return None


def same_as_gold(got, want, what):
    if isinstance(want, tuple):
        import hashlib
        assert (got.count(b"\n"), hashlib.sha256(got).hexdigest()) == want, what + ": differs from the golden's SHA-256"
    else:
        assert got == want, what + ": differs from the golden"


@pytest.mark.parametrize("hccv", [False, True], ids=["SingleCellGenotype", "HCCVSingleCellGenotype"])
@pytest.mark.parametrize("flag", ["All", "Alt"])
def test_streamed_cli_bytes(inputs, flag, hccv):
    """Chunks of 0.2 MB of inflated BAM (tens of chunks per file): every output equals the whole-file run's and the
    golden's, byte for byte, on one engine and with three engines sharing one device."""
    import pipeline_inputs as pi
    case, d, p = inputs
    outs = {}
    for mode, env in (("whole", dict(LONGSOM_STREAM="0")), ("stream", dict(LONGSOM_STREAM="1", LONGSOM_CHUNK_MB="0.2")),
                      ("stream3", dict(LONGSOM_STREAM="1", LONGSOM_CHUNK_MB="0.2", LONGSOM_GPUS="0,0,0"))):
        out = os.path.join(d, "%s_%s_%s" % ("hccv" if hccv else "geno", flag, mode))
        common = ["--bam", p["full"], "--infile", p["cand"], "--ref", p["ref"], "--meta", p["meta"], "--alt_flag", flag,
                  "--nprocs", 4, "--min_mq", 60, "--pvalue", 0.01, "--chrM_contaminant", "True", "--tmp_dir", out + ".tmp"]
        if hccv:
            run("CellTypeReannotation/HCCVSingleCellGenotype.py", common + ["--outfile", out + ".tsv"], **env)
            outs[mode] = {"hccv.tsv": open(out + ".tsv", "rb").read()}
        else:
            run("CellClustering/SingleCellGenotype.py", common + ["--fusions", "--outfile", out, "--alpha2", pi.ALPHA2,
                                                                   "--beta2", pi.BETA2], **env)
            outs[mode] = {"geno_%s.%s.tsv" % (flag, s): open("%s.%s.tsv" % (out, s), "rb").read() for s in SCG}
    for name, whole in outs["whole"].items():
        assert len(whole) > 1000, name
        for mode in ("stream", "stream3"):
            assert outs[mode][name] == whole, "%s: %s differs from the whole-file run" % (name, mode)
        # the HCCV golden was written with --alt_flag All
        want = gold_text(case, name) if not (hccv and flag == "Alt") else None
        if want is not None:
            same_as_gold(outs["stream"][name], want, name)


def _hot_chrM_case(tmp_path):
    """A seeded batch with a chrM and a hot gene, its BAM, 1500 candidate sites and the raw-tag -> column map."""
    d = synth.generate(seed=61, contig_lens=[150000, 16600], chrm=True, n_genes=8, n_reads=12000, n_cells=80,
                       n_hot_genes=1, hot_fraction=0.4, chrm_fraction=0.1)
    b = d.batch
    bam = str(tmp_path / "x.bam")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    rng = np.random.default_rng(62)
    pick = rng.choice(b.n_reads, 1500, replace=False)
    keys = sorted({(int(b.tid[i]), int(b.pos[i]) + int(rng.integers(0, 600))) for i in pick})
    st = np.array([k[0] for k in keys], np.int32)
    sp = np.array([k[1] for k in keys], np.int32)
    alt = rng.integers(0, 9, st.shape[0]).astype(np.uint8)
    n_cells = 70  # the barcodes of cells 70.. are not in the table
    col = {synth.barcode_of(c): c for c in range(n_cells)}
    whole = bamio.read_bam(bam)
    raw = np.array([col.get(t.split("-")[0], -1) for t in whole.barcodes], np.int32)
    return d, bam, (st, sp, alt), n_cells, (lambda t: col.get(t.split("-")[0], -1)), whole.with_cells(raw)


@pytest.mark.parametrize("alt_only", [False, True])
def test_stream_genotype_tuples_bit_exact(engine, tmp_path, alt_only):
    """stream_genotype over ~17 chunks and three engines == one genotype_sparse over the whole batch: cell, dp and alt
    equal, p bit-identical with its NaNs, for both skip_p settings; max_depth 40 fires in bins cut by chunk boundaries."""
    d, bam, sites, n_cells, cell_of, batch = _hot_chrM_case(tmp_path)
    st = sites[0]
    kw = dict(min_bq=30, min_mq=60, max_depth=40, alt_only=alt_only)
    engine.upload(batch)
    capped = engine.genotype_sparse(*sites, n_cells, *AB, bin_size=5000, **kw)
    free = engine.genotype_sparse(*sites, n_cells, *AB, bin_size=5000, **dict(kw, max_depth=0))
    assert free[2].sum() > capped[2].sum()  # the cap fires
    chrM = (st == d.contig_names.index("chrM")).astype(np.uint8)
    assert chrM.any() and not chrM.all()
    for skip in (None, chrM):
        want = engine.genotype_sparse(*sites, n_cells, *AB, skip_p=skip, bin_size=5000, **kw)
        stats = []
        got = pipeline.stream_genotype(bam, sites, 5000, n_cells, cell_of, kw, *AB, skip, [0, 0, 0],
                                       chunk_bytes=150_000, stats_out=stats)
        for name, x, y in zip(("site", "cell", "dp", "alt"), got[:4], want[:4]):
            assert x.dtype == y.dtype and np.array_equal(x, y), name
        assert np.array_equal(got[4].view(np.uint64), want[4].view(np.uint64))  # bit for bit, NaNs included
        assert (~np.isnan(want[4])).any()
        if skip is not None or not alt_only:  # pairs without a tail: ALT = 0, or a skipped chrM site
            assert np.isnan(want[4]).any()
        assert len(stats) >= 10
        assert max(s["n_carried"] for s in stats) > kw["max_depth"]  # capped bins spanned chunk boundaries


def test_stream_genotype_really_streams(tmp_path):
    """The largest batch a device receives is a small part of the file."""
    d = synth.generate(seed=71, contig_lens=[400000, 300000], n_genes=40, n_reads=20000, n_cells=50)
    b = d.batch
    bam = str(tmp_path / "s.bam")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b, lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])))
    sel = np.arange(0, b.n_reads, 7)
    keys = sorted({(int(b.tid[i]), int(b.pos[i]) + 20) for i in sel})
    st = np.array([k[0] for k in keys], np.int32)
    sp = np.array([k[1] for k in keys], np.int32)
    col = {synth.barcode_of(c): c for c in range(d.n_cells)}
    stats = []
    tup = pipeline.stream_genotype(bam, (st, sp, np.zeros(st.shape[0], np.uint8)), 50000, d.n_cells,
                                   lambda t: col.get(t, -1), dict(min_bq=30, min_mq=60), *AB, None, [0],
                                   chunk_bytes=1 << 19, stats_out=stats)
    assert tup[0].shape[0] > 1000
    assert len(stats) >= 10
    assert max(s["n_reads"] for s in stats) < b.n_reads // 5, [s["n_reads"] for s in stats]
