"""The device writer of the genotype long table (ls_genolong.cu via Engine.geno_long_* and cli.genotype.write_long_table)
against the host writer ls_geno_rows, byte for byte: seeded rows of both scripts, every 0 <= a <= d <= 2048 on chrM
sites, blocks of whole sites, the capacity and load errors, the make_case inputs and one of about 10^7 entries, and
main() of both scripts on a golden case with the host writer disabled."""
import argparse
import ctypes as C
import gzip
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "support"))
import genomatrix_cases as gc  # noqa: E402
from longsom_b200 import _lib as L  # noqa: E402
from longsom_b200 import bamio  # noqa: E402
from longsom_b200.cli import genotype as G  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
P_CUT = [0.0, 1e-4, 0.0099, 0.01, 0.0101, 1.0, np.nan]


class Sites:
    """Inputs of both writers: per site prefix, index, chrM flag and pair range; per cell its text; the pairs."""

    def __init__(self, prefix, index, chrm, lo, hi, cell, dp, alt, p, cells):
        self.prefix, self.index, self.chrm, self.lo, self.hi = prefix, index, np.asarray(chrm, np.uint8), lo, hi
        self.cell, self.dp, self.alt, self.p, self.cells = cell, dp, alt, p, cells


def host_rows(x, hccv, pvalue=0.01):
    host = bamio._load_host()
    host.ls_geno_rows.restype = C.c_int64
    host.ls_geno_rows.argtypes = [C.c_int32] + [C.c_void_p] * 9 + [C.c_int32, C.c_void_p, C.c_int32, C.c_double, C.c_void_p]
    host.ls_geno_rows_free.argtypes = [C.c_void_p]
    ns, nc = len(x.prefix), len(x.cells)
    a = lambda v, dt: np.ascontiguousarray(np.asarray(v, dt))
    tc, td, ta, tp = a(x.cell, np.int32), a(x.dp, np.int32), a(x.alt, np.int32), a(x.p, np.float64)
    lo, hi, chrm = a(x.lo, np.int64), a(x.hi, np.int64), a(x.chrm, np.uint8)
    pre = (C.c_char_p * max(1, ns))(*x.prefix)
    idx = None if hccv else (C.c_char_p * max(1, ns))(*x.index)
    cells = (C.c_char_p * max(1, nc))(*x.cells)
    text = C.c_void_p()
    n = host.ls_geno_rows(ns, pre, idx, chrm.ctypes.data, lo.ctypes.data, hi.ctypes.data, tc.ctypes.data, td.ctypes.data,
                          ta.ctypes.data, tp.ctypes.data, nc, cells, 1 if hccv else 0, pvalue, C.byref(text))
    assert n >= 0
    got = C.string_at(text.value, n) if n else b""
    if text.value:
        host.ls_geno_rows_free(text)
    return got


def load(engine, x, hccv, pvalue=0.01):
    engine.geno_long_load(x.cell, x.dp, x.alt, x.p, x.lo, x.hi, x.chrm, x.prefix, None if hccv else x.index, x.cells,
                          hccv, pvalue)


def device_rows(engine, n_sites, cap):
    """Every site of the loaded table through blocks of at most cap bytes: (text, sites per block)."""
    buf = np.zeros(max(cap, 1), np.uint8)
    out, per, s = [], [], 0
    while s < n_sites:
        k, nb = engine.geno_long_text(s, buf.ctypes.data, cap)
        out.append(buf[:nb].tobytes())
        per.append(k)
        s += k
    return b"".join(out), per


def seeded_sites(seed, n_sites, n_cells, untouched=(), full=()):
    """Random sites and pairs: chrM-flagged and plain sites, p on both sides of the cutoff and NaN, cell texts of 1 to
    about 80 bytes with non-ASCII cell types; the sites in `untouched` have no pair, those in `full` every cell."""
    rng = np.random.default_rng(seed)
    types = ["Cancer", "T cell", "Non-Cancer", "Épithélium", "細胞", "x" * 60]
    cells = []
    for c in range(n_cells):
        bc = "".join(rng.choice(list("ACGT"), int(rng.integers(0, 18))))
        cells.append((bc + "\t" + str(rng.choice(types))).encode()[:int(rng.integers(1, 81))] if c % 5 == 0
                     else (bc + "\t" + str(rng.choice(types))).encode())
    prefix, index, chrm, lo, hi = [], [], [], [], []
    cell, dp, alt, p = [], [], [], []
    for s in range(n_sites):
        chrom = str(rng.choice(["chr1", "chrM", "chr10", "MT"]))
        pos = int(rng.integers(1, 10 ** 9))
        prefix.append(("\t".join([chrom, str(pos), str(pos), "A", "G,T", "Cancer", str(int(rng.integers(1, 50)))])).encode())
        index.append(("%s:%d:G" % (chrom, pos)).encode())
        chrm.append(1 if chrom == "chrM" and rng.random() < 0.8 else 0)
        if s in untouched:
            cs = np.zeros(0, np.int64)
        elif s in full:
            cs = np.arange(n_cells)
        else:
            cs = np.sort(rng.choice(n_cells, int(rng.integers(0, min(n_cells, 60) + 1)), replace=False))
        lo.append(len(cell))
        for c in cs:
            d = int(rng.choice([0, 1, 2, 3, 7, 10, 33, 100, 1000, 65535, 2 ** 31 - 1]))
            a = min(d, int(rng.choice([0, 0, 1, d // 3, (3 * d + 9) // 10, d])))
            cell.append(int(c)); dp.append(d); alt.append(a)
            p.append(float(np.round(rng.choice(P_CUT + [rng.random()]), 4)))
        hi.append(len(cell))
    return Sites(prefix, index, chrm, np.array(lo, np.int64), np.array(hi, np.int64), np.array(cell, np.int32),
                 np.array(dp, np.int32), np.array(alt, np.int32), np.array(p, np.float64), cells)


@pytest.mark.parametrize("hccv", [False, True])
@pytest.mark.parametrize("n_cells", [0, 1, 37, 5000])
def test_device_rows_equal_host_writer(engine, built, hccv, n_cells):
    n_sites = 30 if n_cells < 5000 else 12
    x = seeded_sites(100 * n_cells + hccv, n_sites, n_cells, untouched={1, 7}, full={3} if n_cells else set())
    want = host_rows(x, hccv)
    load(engine, x, hccv)
    got, per = device_rows(engine, n_sites, 64 << 20)
    assert got == want
    assert per == [n_sites]
    if n_cells >= 37:
        for label in (b"NoCoverage", b"NoAltReads", b"PASS", b"BetaBin_problem", b"LowVAFChrM", b"\tnan\t"):
            assert label in got, label


def test_every_vaf_on_chrm_sites(engine, built):
    """Site d (1 .. 2048, chrM shortcut) has the pairs (d, a) for a = 0 .. d at cells 0 .. d: the VAF text and the 0.3
    boundary of LowVAFChrM for every 0 <= a <= d <= 2048, and the untouched cells past d."""
    d = np.repeat(np.arange(1, 2049), np.arange(2, 2050)).astype(np.int32)
    a = np.concatenate([np.arange(k + 1) for k in range(1, 2049)]).astype(np.int32)
    hi = np.cumsum(np.arange(2, 2050)).astype(np.int64)
    lo = np.concatenate([[0], hi[:-1]]).astype(np.int64)
    x = Sites([b"chrM\t%d" % k for k in range(1, 2049)], [b"chrM:%d:A" % k for k in range(1, 2049)], np.ones(2048),
              lo, hi, a.copy(), d, a, np.full(len(d), np.nan), [b"c%d\tT" % c for c in range(2049)])
    want = host_rows(x, False)
    load(engine, x, False)
    got, _ = device_rows(engine, 2048, 64 << 20)
    assert got == want
    # the statements themselves on one row: d = 10, a = 3
    line = got.split(b"\n", 2049 * 9 + 4)[2049 * 9 + 3].split(b"\t")
    assert line[4:9] == [b"10", b"3", b"0.3", b".", b"PASS"]


def test_blocks_capacity_and_state(engine, built):
    x = seeded_sites(5, 40, 50, untouched={0, 5})
    load(engine, x, False)
    whole, per = device_rows(engine, 40, 64 << 20)
    rows = whole.split(b"\n")[:-1]
    site_text = [b"".join(r + b"\n" for r in rows[s * 50:(s + 1) * 50]) for s in range(40)]
    assert b"".join(site_text) == whole == host_rows(x, False)
    for cap in (max(len(t) for t in site_text), 10_000, 100_000, len(whole) - 1):
        got, per = device_rows(engine, 40, cap)
        assert got == whole and sum(per) == 40 and len(per) > 1, cap
    buf = np.zeros(1 << 20, np.uint8)
    for s in (0, 17, 39):
        n = len(site_text[s])
        assert engine.geno_long_text(s, buf.ctypes.data, n) == (1, n)
        assert buf[:n].tobytes() == site_text[s]
        with pytest.raises(L.LongSomError) as e:
            engine.geno_long_text(s, buf.ctypes.data, n - 1)
        assert e.value.code == L.LS_E_CAPACITY
    assert engine.geno_long_text(40, buf.ctypes.data, 16) == (0, 0)
    from longsom_b200.engine import Engine
    with Engine(0) as fresh:
        with pytest.raises(L.LongSomError) as e:
            fresh.geno_long_text(0, buf.ctypes.data, 16)
        assert e.value.code == L.LS_E_STATE
    # a released table is gone until the next load
    engine.geno_long_release()
    with pytest.raises(L.LongSomError) as e:
        engine.geno_long_text(0, buf.ctypes.data, 16)
    assert e.value.code == L.LS_E_STATE
    load(engine, x, False)
    assert device_rows(engine, 40, 64 << 20)[0] == whole


def test_load_errors(engine, built):
    def case(**kw):
        x = Sites([b"chr1\t1", b"chr1\t2"], [b"i1", b"i2"], [0, 1], np.array([0, 2], np.int64), np.array([2, 3], np.int64),
                  np.array([0, 2, 1], np.int32), np.array([3, 3, 3], np.int32), np.array([1, 0, 2], np.int32),
                  np.array([0.5, np.nan, np.nan]), [b"a\tT", b"b\tT", b"c\tT"])
        for k, v in kw.items():
            setattr(x, k, np.asarray(v, getattr(x, k).dtype))
        return x

    load(engine, case(), False)
    for kw in (dict(cell=[0, 3, 1]), dict(cell=[-1, 2, 1]), dict(cell=[2, 0, 1]), dict(cell=[1, 1, 1]),
               dict(hi=[2, 4]), dict(lo=[-1, 2]), dict(lo=[0, 3], hi=[2, 2]), dict(alt=[4, 0, 2]), dict(dp=[-1, 3, 3])):
        with pytest.raises(L.LongSomError) as e:
            load(engine, case(**kw), False)
        assert e.value.code == L.LS_E_ARG, kw
    # a null array that is needed
    x = case()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    off = np.array([0, 6, 12], np.int64)
    coff = np.array([0, 3, 6, 9], np.int64)
    base = dict(n_sites=2, n_cells=3, hccv=0, n_pairs=3, cell=vp(x.cell), dp=vp(x.dp), alt=vp(x.alt), p=vp(x.p),
                hit_lo=vp(x.lo), hit_hi=vp(x.hi), site_flags=vp(x.chrm), prefix=C.cast(C.c_char_p(b"chr1\t1chr1\t2"), C.c_void_p),
                prefix_off=vp(off), index=C.cast(C.c_char_p(b"i1i2"), C.c_void_p), index_off=vp(np.array([0, 2, 4], np.int64)),
                cell_text=C.cast(C.c_char_p(b"a\tTb\tTc\tT"), C.c_void_p), cell_off=vp(coff), pvalue=0.01)
    lib = L.load()
    assert lib.ls_geno_long_load(engine._ctx, C.byref(L.LsGenoLongIn(**base))) == L.LS_OK
    for k in ("cell", "p", "hit_lo", "site_flags", "prefix", "prefix_off", "index", "index_off", "cell_text", "cell_off"):
        assert lib.ls_geno_long_load(engine._ctx, C.byref(L.LsGenoLongIn(**dict(base, **{k: None})))) == L.LS_E_ARG, k


def _tables(tmp_path, hccv, args, src, engine, tag):
    a = argparse.Namespace(**dict(vars(args), outfile=str(tmp_path / tag)))
    G.write_long_table(a, hccv, src.blocks, src.keys, src.contig_names, src.tuples, src.barcodes, src.meta_dict,
                       engine)
    path = a.outfile if hccv else a.outfile + ".SingleCellGenotype.tsv"
    with open(path, "rb") as f:
        return f.read()


CASES = [
    dict(seed=1),
    dict(seed=2, alt_flag="Alt"),
    dict(seed=3, chrM_contaminant="False"),
    dict(seed=6, missing_contig=True, untouched_sites=8),
    dict(seed=7, n_cells=1, cover=0.5),
    dict(seed=8, n_sites=300, n_cells=700, cover=0.3),
]


@pytest.mark.parametrize("hccv", [False, True])
@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_write_long_table_device_equals_host(engine, built, tmp_path, case, hccv):
    args, src, _ = gc.make_case(str(tmp_path), **case)
    host = _tables(tmp_path, hccv, args, src, None, "host")
    dev = _tables(tmp_path, hccv, args, src, engine, "dev")
    assert dev == host and len(host.splitlines()) == 1 + len(src.barcodes) * sum(len(t) for _, t in src.blocks)


def big_case(d, n_sites, n_cells, cover, seed=9):
    """About n_sites x n_cells entries: candidates on three contigs (chrM among them), pairs drawn with numpy."""
    rng = np.random.default_rng(seed)
    contigs = ["chr1", "chr2", "chrM"]
    pos = rng.choice(10 ** 7, n_sites, replace=False) + 1
    chrom = rng.integers(0, 3, n_sites)
    with open(os.path.join(d, "cand.tsv"), "w") as f:
        f.write("#CHROM\tStart\tEnd\tREF\tALT\n")
        for c, q in sorted(zip(chrom.tolist(), pos.tolist())):
            f.write("\t".join([contigs[c], str(q), str(q), "A", "ACGT"[q % 4], ".", "Cancer", ".", ".", ".", ".", ".", ".",
                               "3"]) + "\n")
    barcodes = ["BC%07d" % i for i in range(n_cells)]
    with open(os.path.join(d, "meta.tsv"), "w") as f:
        f.write("Index\tCell_type\n")
        for i, b in enumerate(barcodes):
            f.write("%s-1\t%s\n" % (b, "Cancer" if i % 3 else "Non Cancer"))
    meta = G.meta_to_dict(os.path.join(d, "meta.tsv"), None)
    bins = G.build_dict_variants(os.path.join(d, "cand.tsv"), 50000)
    bin_info, keys, site_tid, _, _ = G.candidate_sites(bins, contigs)
    t_site, t_cell = np.nonzero(rng.random((len(keys), n_cells)) < cover)
    n = len(t_site)
    t_dp = rng.choice(np.array([1, 2, 3, 7, 10, 30, 333, 2048], np.int32), n)
    t_alt = np.where(rng.random(n) < 0.7, (rng.random(n) * (t_dp + 1)).astype(np.int32), 0).astype(np.int32)
    t_p = rng.choice(np.array([0.01, 0.00999, 0.010049, 0.5, 1e-9, 0.01005]), n)
    t_p[(t_alt == 0) | (site_tid[t_site] == 2)] = np.nan
    args = argparse.Namespace(outfile=os.path.join(d, "out"), chrM_contaminant="True", pvalue=0.01, alt_flag="All")
    src = G.MatrixSource(None, bin_info, keys, contigs, (t_site.astype(np.int32), t_cell.astype(np.int32), t_dp, t_alt, t_p),
                         list(meta.keys()), meta)
    return args, src


def test_write_long_table_ten_million_entries(engine, built, tmp_path):
    args, src = big_case(str(tmp_path), 2000, 5000, 0.05)
    for hccv in (False, True):
        host = _tables(tmp_path, hccv, args, src, None, "host")
        dev = _tables(tmp_path, hccv, args, src, engine, "dev")
        assert len(dev) == len(host) and hashlib.sha256(dev).digest() == hashlib.sha256(host).digest(), hccv
        assert len(host.splitlines()) == 1 + 2000 * 5000
        del host, dev


def _gold(case, name):
    gz = os.path.join(GOLD, case, name + ".gz")
    if os.path.exists(gz):
        with gzip.open(gz, "rb") as f:
            return hashlib.sha256(f.read()).hexdigest()
    return json.load(open(os.path.join(GOLD, case, name + ".sha256.json")))["sha256"]


def test_main_takes_the_device_writer(built, tmp_path, monkeypatch):
    """Both scripts on golden case g1 with the host writer made to raise: the long tables are the golden bytes."""
    import pipeline_inputs as pi
    d = str(tmp_path)
    p, _ = pi.write_inputs("g1", d)
    cand = os.path.join(d, "candidates.tsv")
    with gzip.open(os.path.join(GOLD, "g1", "candidates.tsv.gz"), "rb") as f, open(cand, "wb") as o:
        o.write(f.read())

    def refuse(*a, **k):
        raise AssertionError("the host writer ran")
    host = bamio._load_host()
    monkeypatch.setattr(host, "ls_geno_rows", refuse)
    pre = os.path.join(d, "geno_All")
    G.main(["--bam", p["full"], "--infile", cand, "--ref", p["ref"], "--meta", p["meta"], "--fusions", "--outfile", pre,
            "--alt_flag", "All", "--min_mq", "60", "--pvalue", "0.01", "--alpha2", str(pi.ALPHA2), "--beta2",
            str(pi.BETA2), "--chrM_contaminant", "True", "--tmp_dir", os.path.join(d, "tg")])
    for suf in ("SingleCellGenotype", "DpMatrix", "AltMatrix", "VAFMatrix", "BinaryMatrix"):
        with open("%s.%s.tsv" % (pre, suf), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == _gold("g1", "geno_All.%s.tsv" % suf), suf
    out = os.path.join(d, "hccv.tsv")
    G.main(["--bam", p["full"], "--infile", cand, "--ref", p["ref"], "--meta", p["meta"], "--outfile", out, "--alt_flag",
            "All", "--min_mq", "60", "--pvalue", "0.01", "--chrM_contaminant", "True", "--tmp_dir", os.path.join(d, "th")],
           hccv=True)
    with open(out, "rb") as f:
        assert hashlib.sha256(f.read()).hexdigest() == _gold("g1", "hccv.tsv")
