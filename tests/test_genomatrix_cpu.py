"""The layout of SingleCellGenotype's four matrices (cli.genotype.matrix_layout): row order and printed labels, columns,
the float-mode decision and the inputs left to pandas.  The layout, printed by a plain Python formatter, must give the
files pivot_long_dataframe writes from the same long table; the device writer prints the same layout
(test_genomatrix_gpu.py)."""
import os
import sys

import pandas as pd
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import genomatrix_cases as gc  # noqa: E402
from longsom_b200.cli import genotype as G  # noqa: E402

KINDS = [k for k, _ in G.MATRIX_KINDS]


def pandas_files(args, fusion_file):
    G.pivot_long_dataframe(args.outfile, gc.fusions_of(fusion_file))
    return {k: open(args.outfile + "." + k + ".tsv").read() for k in KINDS}


def layout_files(args, src, fusion_file):
    lay = G.matrix_layout(src, gc.fusions_of(fusion_file), args.chrM_contaminant)
    assert lay is not None
    head = "\t" + "\t".join(lay.columns) + "\n"
    return lay, {k: head + "".join(gc.format_rows(lay, k, args.pvalue).values()) for k in KINDS}


def test_chr_index_order_labels():
    labels = sorted(["chrM:5:A", "chr10:7:C", "chr2:9:G", "chrX:1:T", "zzz:F1--F2", "1:5:A", "10:3:A", "MT:4:C",
                     "chr01:8:A", "chr1:8:A", "chrZ:2:A", "zzz:A--B"])
    keyed, order, printed = G.chr_index_order(labels)
    assert printed == ["1:5:A", "10:3:A", "MT:4:C", "chr01:8:A", "chr1:8:A", "chr2:9:G", "chr10:7:C", "chrX:1:T",
                       "chrM:2:A", "chrM:5:A", "A--B", "F1--F2"]
    assert [keyed[i] for i in order][:3] == ["1:5:A", "10:3:A", "MT:4:C"]
    # the leading-zero contig ties chr1 in the natural key: the lexicographic order before the stable sort decides
    assert printed.index("chr01:8:A") < printed.index("chr1:8:A")


def test_sort_chr_index_uses_the_same_order():
    df = pd.DataFrame({"x": range(4)}, index=["zzz:F", "chrM:1:A", "chr10:1:A", "chr2:1:A"])
    out = G.sort_chr_index(df)
    assert list(out.index) == ["chr2:1:A", "chr10:1:A", "chrM:1:A", "F"]
    assert list(out["x"]) == [3, 2, 1, 0]


@pytest.mark.parametrize("case", [
    dict(seed=1),
    dict(seed=2, chrM_contaminant="False"),
    dict(seed=3, fusions=[("F1--F2", None), ("F1--F2", 0), ("F1--F2", 0), ("G--H", 3), ("G--H", None)]),
    dict(seed=4, fusions=[("F1--F2", i) for i in range(5)], n_cells=5),
    dict(seed=5, missing_contig=True, untouched_sites=6),
    dict(seed=6, n_cells=1, cover=0.5),
])
def test_layout_prints_the_pandas_files(built, tmp_path, case):
    args, src, ff = gc.make_case(str(tmp_path), **case)
    want = pandas_files(args, ff)
    lay, got = layout_files(args, src, ff)
    for k in KINDS:
        assert got[k] == want[k], k
    if case.get("fusions") and case["seed"] == 4:
        assert not lay.float_mode  # the fusion covers every barcode: nothing absent, integers
    elif case.get("fusions"):
        assert lay.float_mode
        assert "\t1.0" in want["DpMatrix"] and "\t3.0" in want["BinaryMatrix"]
    else:
        assert not lay.float_mode


def test_float_mode_decision(built, tmp_path):
    args, src, ff = gc.make_case(str(tmp_path), seed=7, n_cells=4, fusions=[("F--G", 0), ("F--G", 1)])
    lay = G.matrix_layout(src, gc.fusions_of(ff), args.chrM_contaminant)
    assert lay.float_mode and not lay.col_absent.any()  # absent only in the fusion row
    args, src, ff = gc.make_case(str(tmp_path), seed=7, n_cells=4, fusions=[("F--G", i) for i in range(4)])
    assert not G.matrix_layout(src, gc.fusions_of(ff), args.chrM_contaminant).float_mode


@pytest.mark.parametrize("value,ok", [
    ("AAACGT", True), ("AAAC GT", True), ("NA", False), ("nan", False), ("null", False), ("None", False),
    ("", False), ("123", False), ("1e5", False), ("True", False), ("a\tb", False), ('a"b', False), ("a\rb", False),
])
def test_prints_as_itself(value, ok):
    assert G.prints_as_itself(value) is ok


@pytest.mark.parametrize("refusal", ["na_barcode", "digit_barcodes", "quote_barcode", "no_dot", "no_table", "tab_fusion"])
def test_refusals(built, tmp_path, refusal):
    d = str(tmp_path)
    kw = dict(seed=11, n_cells=4)
    if refusal == "na_barcode":
        kw["barcodes"] = ["AAAA", "NA", "CCCC", "GGGG"]
    elif refusal == "digit_barcodes":
        kw["barcodes"] = ["1", "2", "3", "4"]
    elif refusal == "quote_barcode":
        kw["barcodes"] = ["AAAA", 'C"C', "GGGG", "TTTT"]
    elif refusal == "no_dot":
        kw.update(cover=1.0, n_sites=3)
    elif refusal == "tab_fusion":
        kw["fusions"] = [("F--G", 0)]
    args, src, ff = gc.make_case(d, **kw)
    fus = gc.fusions_of(ff)
    if refusal == "no_table":
        src.long_path = None
    if refusal == "tab_fusion":
        fus.iloc[0, 7] = "A\tB"
    assert G.matrix_layout(src, fus, args.chrM_contaminant) is None


def test_refuses_zero_columns_and_duplicate_labels(built, tmp_path):
    args, src, ff = gc.make_case(str(tmp_path), seed=12, n_cells=3)
    src.barcodes = []
    assert G.matrix_layout(src, gc.fusions_of(ff), args.chrM_contaminant) is None
    args, src, ff = gc.make_case(str(tmp_path), seed=12, n_cells=3)
    chrom, target = src.blocks[0]
    pos = next(iter(target))
    # a fusion whose label is an SNV row's label
    fus = pd.DataFrame([[".", ".", ".", ".", ".", ".", ".", src.barcodes[0], ".", 1, 1, 1, ".", ".", 1,
                         "%s:%d:%s" % (chrom, pos + 1, target[pos][1])]])
    assert G.matrix_layout(src, fus, args.chrM_contaminant) is None
