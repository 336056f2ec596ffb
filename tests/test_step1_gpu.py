"""BaseCellCalling.step1 called on the device (ls_step1.cu through Engine.step1_*): the goldens byte for byte, and the
same bytes as the host passes of ls_step1.cpp (given the same K2 tails) on randomised tables, on hand-made edge rows,
on ranges the device refuses and at a million rows; the block API's capacities and call order."""
import gzip
import os
import sys

import numpy as np
import pytest

from longsom_b200 import bamio
from longsom_b200._lib import LS_E_CAPACITY, LS_E_STATE, LongSomError
from longsom_b200.cli import step1

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "support"))
sys.path.insert(0, HERE)
from test_step1_native_cpu import _random_table  # noqa: E402

GOLD = os.path.join(HERE, "golden")
A1, B1, A2, B2 = 0.21356677091082193, 104.95163748636298, 0.2474528917555431, 162.03696139428595
LABELS = ("PASS", "Non-Significant", "Low-Significance", "Multi-allelic", "Low_cells", "Low_reads", "Multiple_cell_types",
          "Min_cell_types", "Cell_type_noise", "Noisy_site", "LC_Upstream", "LC_Downstream")

pytestmark = pytest.mark.gpu


class K2Only:
    """The CUDA engine's K2 without its step1 entry points: the host passes run, with bitwise the same tails."""

    def __init__(self, eng):
        self.eng = eng

    def betabinom_sf(self, k, n, a, b):
        return self.eng.betabinom_sf(k, n, a, b)


def _run(infile, outfile, fasta, eng, native=True, **kw):
    args = dict(min_ac_cells=2, min_ac_reads=3, min_cells=5, min_reads=5, min_cell_types=2, max_cell_types=1,
                fisher_cutoff=1)
    args.update(kw)
    old = os.environ.get("LONGSOM_STEP1_NATIVE")
    os.environ["LONGSOM_STEP1_NATIVE"] = "1" if native else "0"
    try:
        return step1.variant_calling_step1(infile, outfile, fasta, A1, B1, A2, B2, args["min_ac_cells"],
                                           args["min_ac_reads"], args["min_cells"], args["min_reads"],
                                           args["min_cell_types"], args["max_cell_types"], args["fisher_cutoff"], eng,
                                           procs=1)
    finally:
        if old is None:
            del os.environ["LONGSOM_STEP1_NATIVE"]
        else:
            os.environ["LONGSOM_STEP1_NATIVE"] = old


def _host_passes_fail(m):
    """Make both host paths raise, so that a silent fall-back cannot pass for the device path."""
    def boom(*a, **k):
        raise AssertionError("a host pass ran")
    m.setattr(step1, "_parse_rows", boom)
    m.setattr(step1, "_NativeRange", boom)


def _both_arms(engine, infile, fasta, tmp_path, monkeypatch, strict=True, **kw):
    """(device text, host-passes text) of one table."""
    dev, host = str(tmp_path / "dev.tsv"), str(tmp_path / "host.tsv")
    _run(infile, host, fasta, K2Only(engine), **kw)
    with monkeypatch.context() as m:
        if strict:
            _host_passes_fail(m)
        _run(infile, dev, fasta, engine, **kw)
    return open(dev, "rb").read(), open(host, "rb").read()


@pytest.mark.parametrize("case", ["g1", "g2", "g3"])
def test_goldens(case, engine, tmp_path, monkeypatch):
    import pipeline_inputs as pi
    p, _ = pi.write_inputs(case, str(tmp_path))
    merged = str(tmp_path / "merged.tsv")
    with gzip.open(os.path.join(GOLD, case, "merged.tsv.gz"), "rb") as f, open(merged, "wb") as o:
        o.write(f.read())
    out = str(tmp_path / "s.tsv")
    with monkeypatch.context() as m:
        _host_passes_fail(m)
        _run(merged, out, p["ref"], engine)
    with gzip.open(os.path.join(GOLD, case, "step1.tsv.gz"), "rb") as f:
        want = [l for l in f.read().splitlines(True) if not l.startswith(b"##fileDate")]
    got = [l for l in open(out, "rb").read().splitlines(True) if not l.startswith(b"##fileDate")]
    assert got == want
    assert step1.last_times["host_rows"] == 0


def _retype(src, dst, n_types, crlf):
    """The generator's table with n_types cell-type columns (its three, repeated under new names), CRLF optional."""
    with open(src) as f:
        lines = f.read().split("\n")
    out = []
    for l in lines:
        if not l or l.startswith("##"):
            out.append(l)
            continue
        c = l.split("\t")
        extra = ["T%d" % i for i in range(n_types)] if l.startswith("#CHROM") else [c[5 + i % 3] for i in range(n_types)]
        out.append("\t".join(c[:5] + extra))
    with open(dst, "w", newline="") as f:
        f.write(("\r\n" if crlf else "\n").join(out))


@pytest.mark.parametrize("seed,n_types,crlf", [(1, 1, False), (2, 2, True), (3, 3, False), (4, 4, False), (5, 5, True),
                                               (6, 3, False)])
def test_random_tables(seed, n_types, crlf, engine, tmp_path, monkeypatch):
    raw, merged = str(tmp_path / "raw.tsv"), str(tmp_path / "rand.tsv")
    _random_table(raw, 6000, seed)
    _retype(raw, merged, n_types, crlf)
    rng = np.random.default_rng(seed)
    fa = str(tmp_path / "ref.fa")
    bamio.write_fasta(fa, ["chr1", "chr2"], ["".join(rng.choice(list("ACGTacgt"), 200000, p=[.5, .1, .1, .1, .05, .05, .05, .05])).encode()
                                             for _ in range(2)])
    outs = []
    for kw in (dict(), dict(min_ac_cells=1, min_ac_reads=1, min_cell_types=1, max_cell_types=2, min_reads=3, min_cells=1),
               dict(min_ac_cells=100000), dict(min_ac_cells=1, min_ac_reads=100000)):
        dev, host = _both_arms(engine, merged, fa, tmp_path, monkeypatch, strict=not crlf, **kw)
        assert dev == host
        outs.append(dev)
        if crlf:   # the device refuses a range with '\r': the host passes redo it, with the same bytes
            assert step1.last_times["host_rows"] == step1.last_times["rows"] > 0
    if n_types >= 3:
        text = b"".join(outs).decode()
        for label in LABELS:
            assert label in text, label


def _cell(dp, nc, cc, bc):
    cc, bc = list(cc) + [0] * (6 - len(cc)), list(bc) + [0] * (6 - len(bc))
    return "|".join([str(dp), str(nc), ":".join(map(str, cc)), ":".join(map(str, bc)), ":".join(["30"] * 6),
                     ":".join(map(str, bc)), ":".join(["0"] * 6)])


def _exact_tail(engine, target, a, b):
    """(k, n) whose tail rounds to exactly `target`."""
    n = np.repeat(np.arange(5, 400, dtype=np.int32), 40)
    k = np.tile(np.arange(1, 41, dtype=np.int32), n.shape[0] // 40)
    keep = k <= n
    k, n = k[keep], n[keep]
    p = np.round(engine.betabinom_sf(k, n, a, b), 4)
    i = np.nonzero(p == target)[0]
    assert i.shape[0], target
    return int(k[i[0]]), int(n[i[0]])


def test_edge_rows(engine, tmp_path, monkeypatch):
    fa = str(tmp_path / "ref.fa")
    bamio.write_fasta(fa, ["chrE", "chrF"], [b"acgtAAAAAcccccGGGGGtttttACGTac", b"AAAAAAAAAATTTTTTTTTTggggg" * 40])
    k05, n05 = _exact_tail(engine, 0.05, A1, B1)
    k001, n001 = _exact_tail(engine, 0.001, A1, B1)
    std = _cell(40, 20, [20], [40])
    rows = [
        ("chrE", 3, "A", [_cell(40, 20, [10, 5], [30, 10]), std]),           # POS < 6: '.' contexts
        ("chrE", 28, "G", [_cell(40, 20, [10, 0, 0, 5], [30, 0, 0, 10]), std]),  # context cut at the contig's end
        ("chrZ", 100, "A", [_cell(40, 20, [10, 5], [30, 10]), std]),         # a contig the FASTA does not have
        ("chrE", 12, "C", [_cell(40, 20, [5, 10], [10, 30]), std]),          # lowercase reference bases
        ("chrF", 50, "A", [_cell(n05, n05, [n05 - k05, k05], [n05 - k05, k05]), std]),       # a tail of exactly 0.05
        ("chrF", 60, "A", [_cell(n001, n001, [n001 - k001, k001], [n001 - k001, k001]), std]),  # exactly 0.001
        ("chrF", 70, "A", [_cell(5, 5, [0, 3, 0, 0, 2], [0, 10, 0, 0, 3]), "NA"]),   # rest depth < 0: nan (Q6)
        ("chrF", 80, "A", [_cell(32, 32, [31, 1], [31, 1]), std]),            # 1/32: a VAF / MCF tie; Sum_alts_bc 0 (Q7)
        ("chrF", 90, "A", [_cell(400000, 5000, [4000, 300, 0, 0, 90], [399000, 800, 0, 0, 200]), std]),  # rest k > 128
        ("chrF", 95, "A", ["NA", std]),
        ("chrF", 97, "A", [_cell(40, 20, [10, 0, 5, 5], [20, 0, 10, 10]), _cell(40, 20, [10, 5, 0, 5], [20, 10, 0, 10])]),
        ("chrF", 99, "N", [_cell(40, 20, [5, 5, 5, 5], [10, 10, 10, 10]), std]),
    ]
    hdr = "##fileDate=x\n#CHROM\tStart\tEnd\tREF\tINFO\tCancer\tNon-Cancer\n"
    body = []
    for i, (c, pos, ref, cols) in enumerate(rows):
        body.append("\t".join([c, str(pos), str(pos), ref, "DP|NC|CC|BC|BQ|BCf|BCr"] + cols) + "\n")
        if i == 4:
            body.append("##a comment in the body\n")
    merged = str(tmp_path / "edge.tsv")
    open(merged, "w").write(hdr + "".join(body))
    for kw in (dict(), dict(min_cell_types=1, min_ac_cells=1, min_ac_reads=1)):
        dev, host = _both_arms(engine, merged, fa, tmp_path, monkeypatch, **kw)
        assert dev == host
        py = str(tmp_path / "py.tsv")
        _run(merged, py, fa, K2Only(engine), native=False, **kw)
        assert dev == open(py, "rb").read()
    lines = dev.decode().split("\n")
    info = {int(l.split("\t")[1]): l.split("\t")[4:24] for l in lines if l.startswith("chr")}
    assert info[3][3:5] == [".", "."]
    assert info[28][3:5] == ["TTACG", "AC"]
    assert info[100][3:5] == [".", "."]
    assert info[12][3:5] == ["AAACC", "CCGGG"]
    assert info[50][12] == "0.05" and info[60][12] == "0.001"
    assert info[70][16].endswith(";nan")
    assert info[80][10] == "0.0312" and info[80][11] == "0.0312" and info[80][16] == "0;71;1"
    assert "##a comment in the body\n" in dev.decode()
    # '##' lines after the #CHROM line and no data row: the script reads them as header (the range API is tested with
    # such a body in test_block_api)
    only = str(tmp_path / "only.tsv")
    open(only, "w").write(hdr + "##one\n##two\n")
    dev, host = _both_arms(engine, only, fa, tmp_path, monkeypatch, strict=False)
    assert dev == host and dev.endswith(b"##one\n##two\n")


def test_refusals(engine, tmp_path, monkeypatch):
    good = str(tmp_path / "good.tsv")
    _random_table(good, 300, 9)
    lines = open(good).read().split("\n")
    body0 = next(i for i, l in enumerate(lines) if l and not l.startswith("#"))
    # rows the reference fails on: the same exception as the Python passes
    for mutate in (lambda l: "\t".join(l.split("\t")[:-1]),
                   lambda l: "\t".join([l.split("\t")[0], "12x"] + l.split("\t")[2:]),
                   lambda l: "\t".join(l.split("\t")[:5] + ["9|9|1:1:1:1:0:0|9:0:0:0:0:0|1:1|1:1"] + l.split("\t")[6:])):
        bad = str(tmp_path / "bad.tsv")
        ls = list(lines)
        ls[body0 + 50] = mutate(ls[body0 + 50])
        open(bad, "w").write("\n".join(ls))
        errs = []
        for eng, native in ((K2Only(engine), False), (engine, True)):
            with pytest.raises(Exception) as e:
                _run(bad, str(tmp_path / "o.tsv"), None, eng, native=native)
            errs.append(type(e.value))
        assert errs[0] == errs[1]
    # a row the device refuses and the host passes print (a VAF of 4e5): the range is redone on the host
    ls = list(lines)
    c = ls[body0 + 20].split("\t")
    ls[body0 + 20] = "\t".join(c[:3] + ["A", c[4], _cell(1, 1, [0, 1], [0, 400000])] + c[6:])
    odd = str(tmp_path / "odd.tsv")
    open(odd, "w").write("\n".join(ls))
    dev, host = _both_arms(engine, odd, None, tmp_path, monkeypatch, strict=False, min_reads=1, min_cells=1)
    assert dev == host and b"400000.0" in dev
    assert step1.last_times["host_rows"] > 0


def test_block_api(engine, tmp_path):
    engine.step1_release()
    for f in (engine.step1_call, lambda: engine.step1_text(0, 0, 0)):
        with pytest.raises(LongSomError) as e:
            f()
        assert e.value.code == LS_E_STATE
    merged = str(tmp_path / "t.tsv")
    _random_table(merged, 3000, 17)
    data = open(merged, "rb").read()
    body = data[data.index(b"\n#CHROM"):]
    body = body[body.index(b"\n", 1) + 1:]
    rng = np.random.default_rng(17)
    seqs = {c: rng.choice(np.frombuffer(b"ACGTa", np.uint8), 200000) for c in ("chr1", "chr2")}
    cols, names = [5, 6, 7], [b"Cancer", b"Non-Cancer", b"T_cell"]
    prm = (5, 5, 2, 3, 2, 1, A1, B1, A2, B2)
    import ctypes as C
    buf = C.create_string_buffer(len(body) * 3 + 4096)

    def text_of(piece, caps):
        rows, nq, new = engine.step1_load(piece, cols, names, *prm)
        for cid, name in new:
            if name in seqs:
                engine.step1_contig(cid, seqs[name])
        nbytes, longest = engine.step1_call()
        out = []
        for cap in caps:
            got, lo = b"", 0
            while lo < rows:
                c = cap(lo)
                done, nb = engine.step1_text(lo, C.addressof(buf), c)
                assert 0 < done and nb <= c
                got += buf.raw[:nb]
                lo += done
            assert len(got) == nbytes
            out.append(got)
        return out, new, longest

    full, new, longest = text_of(body, [lambda lo: 1 << 30])
    lens = [len(x) for x in full[0].splitlines(True)]
    assert max(lens) == longest and sorted(n for _, n in new) == ["chr1", "chr2", "chr3"]
    outs, _, _ = text_of(body, [lambda lo: longest, lambda lo: 4096, lambda lo: lens[lo]])   # the last: one-row blocks
    assert all(o == full[0] for o in outs)
    with pytest.raises(LongSomError) as e:
        engine.step1_text(int(np.argmax(lens)), C.addressof(buf), longest - 1)
    assert e.value.code == LS_E_CAPACITY
    # a second range of the same contigs: nothing new, the contigs are still resident
    cut = body.index(b"\n", len(body) // 2) + 1
    a, new_a, _ = text_of(body[:cut], [lambda lo: 1 << 30])
    b, new_b, _ = text_of(body[cut:], [lambda lo: 1 << 30])
    assert new_a == [] and new_b == []
    assert a[0] + b[0] == full[0]
    # a range of '##' lines only: zero data rows, copied through
    (only,), new, _ = text_of(b"##one\n##two", [lambda lo: 1 << 30])
    assert only == b"##one\n##two" and new == []
    engine.step1_release()
    with pytest.raises(LongSomError) as e:
        engine.step1_text(0, C.addressof(buf), 10)
    assert e.value.code == LS_E_STATE


def test_million_rows(engine, tmp_path, monkeypatch):
    raw = str(tmp_path / "raw.tsv")
    _random_table(raw, 50000, 31)
    data = open(raw, "rb").read()
    head = data[:data.index(b"\n", data.index(b"#CHROM")) + 1]
    body = data[len(head):]
    merged = str(tmp_path / "big.tsv")
    with open(merged, "wb") as f:
        f.write(head)
        for _ in range(20):
            f.write(body)
    rng = np.random.default_rng(31)
    fa = str(tmp_path / "ref.fa")
    bamio.write_fasta(fa, ["chr1", "chr2", "chr3"], ["".join(rng.choice(list("ACGT"), 2000000)).encode() for _ in range(3)])
    dev, host = _both_arms(engine, merged, fa, tmp_path, monkeypatch)
    assert dev == host
    assert step1.last_times["rows"] >= 10 ** 6
