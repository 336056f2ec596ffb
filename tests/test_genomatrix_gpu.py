"""The device writer of SingleCellGenotype's four matrices (ls_genomatrix.cu via cli.genotype.write_matrices) against
pivot_long_dataframe run on the same long table, byte for byte; its VAF text against Python's str(round(a / d, 4)) for
every 0 <= a <= d <= 2048; its blocks of whole rows; and the inputs it leaves to pandas."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import genomatrix_cases as gc  # noqa: E402
from longsom_b200 import _lib as L  # noqa: E402
from longsom_b200.cli import genotype as G  # noqa: E402

pytestmark = pytest.mark.gpu
KINDS = [k for k, _ in G.MATRIX_KINDS]


def text(eng, kind, n_rows, cap):
    """Every row of a loaded matrix through blocks of at most cap bytes: (text, rows per block)."""
    buf = np.zeros(max(cap, 1), np.uint8)
    out, per, row = [], [], 0
    while row < n_rows:
        rows, nb = eng.geno_matrix_text(kind, row, buf.ctypes.data, cap)
        out.append(buf[:nb].tobytes())
        per.append(rows)
        row += rows
    return b"".join(out).decode(), per


def test_vaf_text_is_python_round(engine):
    d = np.repeat(np.arange(1, 2049), np.arange(2, 2050))
    a = np.concatenate([np.arange(x + 1) for x in range(1, 2049)])
    n_rows = 2048
    row_flags = np.full(n_rows, L.LS_GENO_ROW_CHRM, np.uint8)
    engine.geno_matrix_load(d - 1, a, d, a, np.full(len(d), np.nan), [str(x).encode() for x in range(1, 2049)],
                            row_flags, 2049, pvalue=0.01)
    vaf, _ = text(engine, L.LS_GENO_MATRIX_VAF, n_rows, 64 << 20)
    binary, _ = text(engine, L.LS_GENO_MATRIX_BINARY, n_rows, 64 << 20)
    for line_v, line_b, dp in zip(vaf.splitlines(), binary.splitlines(), range(1, 2049)):
        v, b = line_v.split("\t"), line_b.split("\t")
        assert v[0] == str(dp)
        want = [str(round(x / dp, 4)) for x in range(dp + 1)]
        assert v[1:dp + 2] == want, dp
        assert all(x == "." for x in v[dp + 2:])
        # chrM shortcut rows: 1 iff the rounded VAF is >= 0.3 (Alt = 0 prints 0)
        assert b[1:dp + 2] == [("1" if (x > 0 and round(x / dp, 4) >= 0.3) else "0") for x in range(dp + 1)], dp


CASES = [
    dict(seed=1),
    dict(seed=2, alt_flag="Alt"),
    dict(seed=3, chrM_contaminant="False"),
    dict(seed=4, fusions=[("F1--F2", None), ("F1--F2", 0), ("F1--F2", 0), ("G--H", 3), ("G--H", None), ("K--L", 7)]),
    dict(seed=5, fusions=[("F1--F2", i) for i in range(6)] + [("A--B", i) for i in range(6)], n_cells=6),
    dict(seed=6, missing_contig=True, untouched_sites=8),
    dict(seed=7, n_cells=1, cover=0.5),
    dict(seed=8, n_sites=1000, n_cells=2000, cover=0.5, fusions=[("F1--F2", None), ("F1--F2", 5)]),
]


@pytest.mark.parametrize("case", CASES, ids=[str(i) for i in range(len(CASES))])
def test_matrices_match_pandas(built, tmp_path, case):
    args, src, ff = gc.make_case(str(tmp_path), **case)
    assert G.write_matrices(args, src, gc.fusions_of(ff))
    got = {k: open(args.outfile + "." + k + ".tsv", "rb").read() for k in KINDS}
    G.pivot_long_dataframe(args.outfile, gc.fusions_of(ff))
    for k in KINDS:
        want = open(args.outfile + "." + k + ".tsv", "rb").read()
        assert got[k] == want, k


def test_blocks_of_one_row_and_capacity(engine, built, tmp_path):
    args, src, ff = gc.make_case(str(tmp_path), seed=21, n_sites=30, n_cells=50,
                                 fusions=[("F1--F2", None), ("F1--F2", 2)])
    lay = G.matrix_layout(src, gc.fusions_of(ff), args.chrM_contaminant)
    engine.geno_matrix_load(lay.row, lay.col, lay.dp, lay.alt, lay.p, [x.encode() for x in lay.labels], lay.row_flags,
                            len(lay.columns), lay.col_absent, lay.float_mode, args.pvalue)
    for name, kind in G.MATRIX_KINDS:
        rows = gc.format_rows(lay, name, args.pvalue)
        want = "".join(rows.values())
        whole, per = text(engine, kind, len(rows), 64 << 20)
        assert whole == want and per == [len(rows)]
        # a block of exactly one row's length holds that row and nothing more
        buf = np.zeros(1 << 20, np.uint8)
        for r in range(len(rows)):
            n = len(rows[r].encode())
            got = engine.geno_matrix_text(kind, r, buf.ctypes.data, n)
            assert got == (1, n) and buf[:n].tobytes().decode() == rows[r]
        shortest = min(len(x.encode()) for x in rows.values())
        r0 = min(r for r in rows if len(rows[r].encode()) > shortest)
        with pytest.raises(L.LongSomError) as e:
            engine.geno_matrix_text(kind, r0, buf.ctypes.data, len(rows[r0].encode()) - 1)
        assert e.value.code == L.LS_E_CAPACITY
        assert engine.geno_matrix_text(kind, len(rows), buf.ctypes.data, 16) == (0, 0)


def test_duplicate_pair_is_an_argument_error(engine):
    with pytest.raises(L.LongSomError) as e:
        engine.geno_matrix_load([0, 1, 0], [2, 0, 2], [1, 1, 1], [0, 0, 0], [np.nan] * 3, [b"a", b"b"],
                                np.zeros(2, np.uint8), 3)
    assert e.value.code == L.LS_E_ARG


@pytest.mark.parametrize("refusal", ["na_barcode", "digit_barcodes", "no_dot", "no_table"])
def test_refused_inputs_go_to_pandas(built, tmp_path, refusal):
    """A refused input writes no matrix; main() then runs pivot_long_dataframe, whose files or error are the
    reference's."""
    kw = dict(seed=31, n_cells=4)
    if refusal == "na_barcode":
        kw["barcodes"] = ["AAAA", "NA", "CCCC", "GGGG"]
    elif refusal == "digit_barcodes":
        kw["barcodes"] = ["1", "2", "3", "4"]
    elif refusal == "no_dot":
        kw.update(cover=1.0, n_sites=3)
    args, src, ff = gc.make_case(str(tmp_path), **kw)
    if refusal == "no_table":
        os.remove(src.long_path)
        src.long_path = None
    assert not G.write_matrices(args, src, gc.fusions_of(ff))
    assert not any(os.path.exists(args.outfile + "." + k + ".tsv") for k in KINDS)
    if refusal == "no_table":
        with pytest.raises(FileNotFoundError):
            G.pivot_long_dataframe(args.outfile, gc.fusions_of(ff))
    else:
        G.pivot_long_dataframe(args.outfile, gc.fusions_of(ff))
        assert all(os.path.exists(args.outfile + "." + k + ".tsv") for k in KINDS)
