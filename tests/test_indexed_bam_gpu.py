"""GPU suite for the indexed BAM reader: with a .bai next to the BAM, BaseCellCounter, SingleCellGenotype and
HCCVSingleCellGenotype read only the BGZF members their regions need, and their tables stay byte-identical to the
goldens and to a run without the index, on one engine and on several, with the depth cap firing."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from longsom_b200 import bamio, pipeline, synth
from longsom_b200.engine import CountParams
from longsom_b200.windows import make_windows

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "support"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_cli_gpu import assert_same, file_lines, gold_lines, has_gold  # noqa: E402

SCRIPTS = os.path.join(ROOT, "workflow", "scripts")
AB = (0.2, 100.0)


def run_script(rel, args, gpus=None):
    env = dict(os.environ, LS_BAM_TIMING="1")
    if gpus:
        env["LONGSOM_GPUS"] = gpus
    cmd = [sys.executable, os.path.join(SCRIPTS, rel)] + [str(a) for a in args]
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, "%s failed:\n%s" % (" ".join(cmd), r.stdout[-3000:])
    return r.stdout


@pytest.mark.parametrize("case", ["g1", "g2"])
@pytest.mark.parametrize("gpus", [None, "0,0,0"])
def test_clis_with_index_match_goldens(tmp_path, built, case, gpus):
    import bai_write
    import pipeline_inputs as pi
    d = str(tmp_path)
    p, data = pi.write_inputs(case, d)
    for k in ("full", "cancer"):
        bai_write.write_bai(p[k])
    log = run_script("SNVCalling/BaseCellCounter.py", ["--bam", p["cancer"], "--ref", p["ref"], "--chrom", "all",
                     "--out_folder", d, "--min_bq", 20, "--min_mq", 60, "--tmp_dir", os.path.join(d, "tmp_c")], gpus)
    assert "index used" in log
    assert_same(file_lines(os.path.join(d, "s.Cancer.tsv")), gold_lines(case, "counts.Cancer.tsv"), "BaseCellCounter")
    if has_gold(case, "counts.full_ac.tsv"):
        run_script("SNVCalling/BaseCellCounter.py", ["--bam", p["full"], "--ref", p["ref"], "--chrom", data.contig_names[0],
                   "--out_folder", d, "--id", "full.ac", "--min_bq", 30, "--min_mq", 0, "--min_ac", 2, "--min_dp", 3,
                   "--min_cc", 2, "--bin", 30000, "--tmp_dir", os.path.join(d, "tmp_ac")], gpus)
        assert_same(file_lines(os.path.join(d, "full.ac.tsv")), gold_lines(case, "counts.full_ac.tsv"),
                    "BaseCellCounter --chrom " + data.contig_names[0])
    cand = os.path.join(d, "candidates.tsv")
    import gzip
    with gzip.open(os.path.join(ROOT, "tests", "golden", case, "candidates.tsv.gz"), "rb") as f, open(cand, "wb") as o:
        o.write(f.read())
    log = run_script("CellClustering/SingleCellGenotype.py", ["--bam", p["full"], "--infile", cand, "--ref", p["ref"], "--meta",
                     p["meta"], "--fusions", "--outfile", os.path.join(d, "geno_All"), "--alt_flag", "All", "--nprocs", 4,
                     "--min_mq", 60, "--pvalue", 0.01, "--alpha2", pi.ALPHA2, "--beta2", pi.BETA2, "--chrM_contaminant",
                     "True", "--tmp_dir", os.path.join(d, "tmp_g")], gpus)
    assert "index used" in log
    for suf in ("SingleCellGenotype", "DpMatrix", "AltMatrix", "VAFMatrix", "BinaryMatrix"):
        assert_same(file_lines(os.path.join(d, "geno_All.%s.tsv" % suf)), gold_lines(case, "geno_All.%s.tsv" % suf),
                    "SingleCellGenotype " + suf)
    run_script("CellTypeReannotation/HCCVSingleCellGenotype.py", ["--bam", p["full"], "--infile", cand, "--ref", p["ref"],
               "--meta", p["meta"], "--outfile", os.path.join(d, "hccv.tsv"), "--alt_flag", "All", "--nprocs", 4, "--min_mq",
               60, "--pvalue", 0.01, "--chrM_contaminant", "True", "--tmp_dir", os.path.join(d, "tmp_h")], gpus)
    assert_same(file_lines(os.path.join(d, "hccv.tsv")), gold_lines(case, "hccv.tsv"), "HCCVSingleCellGenotype")


@pytest.fixture(scope="module")
def sparse_case(tmp_path_factory, built):
    """A larger BAM over six contigs with a hot gene and a chrM, indexed, its copy without the index, its FASTA, and a
    sparse site list with a hot locus where max_depth fires."""
    import bai_write
    d = synth.generate(seed=81, contig_lens=[600000, 500000, 400000, 300000, 300000, 16600], chrm=True, n_genes=40,
                       n_reads=40000, n_cells=80, n_hot_genes=1, hot_fraction=0.3, chrm_fraction=0.05)
    b = d.batch
    tmp = tmp_path_factory.mktemp("indexed_gpu")
    bam = str(tmp / "x.bam")
    bamio.write_bam(bam, d.contig_names, d.contig_lens, b,
                    lambda i: None if b.cell[i] < 0 else synth.barcode_of(int(b.cell[i])) + "-1")
    bai_write.write_bai(bam)
    plain = str(tmp / "plain.bam")
    shutil.copy(bam, plain)
    fa = str(tmp / "ref.fa")
    bamio.write_fasta(fa, d.contig_names, [d.contig_seq(i) for i in range(len(d.contig_lens))])
    rng = np.random.default_rng(82)
    pick = rng.choice(b.n_reads, 200, replace=False)
    # the hot gene's reads are ~30 % of the file: its sites are the hot locus
    keys = sorted({(int(b.tid[i]), int(b.pos[i]) + int(rng.integers(0, 600))) for i in pick})
    st = np.array([k[0] for k in keys], np.int32)
    sp = np.array([k[1] for k in keys], np.int32)
    alt = rng.integers(0, 9, st.shape[0]).astype(np.uint8)
    col = {synth.barcode_of(c): c for c in range(70)}
    return d, bam, plain, fa, (st, sp, alt), (lambda t: col.get(t.split("-")[0], -1))


@pytest.mark.parametrize("devices", [[0], [0, 0, 0]])
def test_stream_genotype_indexed_equals_plain(sparse_case, devices):
    d, bam, plain, fa, sites, cell_of = sparse_case
    kw = dict(min_bq=30, min_mq=60, max_depth=40, alt_only=False)
    res, stats = {}, {}
    for label, path in (("indexed", bam), ("plain", plain)):
        stats[label] = []
        res[label] = pipeline.stream_genotype(path, sites, 5000, 70, cell_of, kw, *AB, None, devices,
                                              chunk_bytes=1 << 20, stats_out=stats[label])
    for x, y in zip(res["indexed"], res["plain"]):
        assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8))
    assert res["indexed"][0].shape[0] > 100
    free = pipeline.stream_genotype(bam, sites, 5000, 70, cell_of, dict(kw, max_depth=0), *AB, None, devices,
                                    chunk_bytes=1 << 20)
    assert free[2].sum() > res["indexed"][2].sum()  # the depth cap fires
    assert all(s["indexed"] for s in stats["indexed"]) and not any(s["indexed"] for s in stats["plain"])
    assert sum(s["compressed_bytes"] for s in stats["indexed"]) < sum(s["compressed_bytes"] for s in stats["plain"])


@pytest.mark.parametrize("chrom", ["chr2", "all"])
def test_stream_count_indexed_equals_plain(sparse_case, tmp_path, chrom):
    d, bam, plain, fa_path, sites, cell_of = sparse_case
    fa = bamio.Fasta(fa_path)
    named = make_windows(fa.references, fa.lengths, chrom, 50000)
    prm = CountParams(min_bq=20, min_mq=60, min_dp=1, min_cc=1, max_depth=200)
    out, stats = {}, {}
    for label, path in (("indexed", bam), ("plain", plain)):
        stats[label] = []
        pipeline.stream_count(path, named, fa, prm, str(tmp_path / (label + ".tsv")), "x", [0, 0], chunk_bytes=1 << 20,
                              stats_out=stats[label])
        out[label] = file_lines(str(tmp_path / (label + ".tsv")))
    assert out["indexed"] == out["plain"] and len(out["indexed"]) > 1000
    ci = sum(s["compressed_bytes"] for s in stats["indexed"])
    cp = sum(s["compressed_bytes"] for s in stats["plain"])
    assert ci < cp if chrom == "chr2" else ci <= cp
