"""Seeded inputs of SingleCellGenotype's matrix stage, and a plain Python formatter of the matrices.

make_case writes a candidate list and (optionally) a fusion file, draws touched (site, cell) pairs as K1' + K2 return
them, and writes the long table through cli.genotype.write_long_table, so that pivot_long_dataframe and the device
writer read the same input.  format_rows prints the rows of a MatrixLayout entry by entry, the way pandas does."""
import argparse
import os

import numpy as np

from longsom_b200.cli import genotype as G

CONTIGS = ["chr1", "chr2", "chr10", "chrX", "chrM", "1", "10", "MT", "chr01", "chrZ"]


def barcode(rng, used):
    while True:
        b = "".join(rng.choice(list("ACGT"), 8))
        if b not in used:
            used.add(b)
            return b


def make_case(d, seed, n_sites=40, n_cells=12, cover=0.3, alt_flag="All", chrM_contaminant="True", fusions=None,
              missing_contig=False, untouched_sites=0, pvalue=0.01, barcodes=None):
    """fusions: None (no file), or a list of (#FusionName, BC) rows; BC None is a random metadata barcode + '-1', an
    int i the cleaned metadata barcode i.
    Returns (args, src, fusion_file or None)."""
    rng = np.random.default_rng(seed)
    used = set()
    if barcodes is None:
        barcodes = [barcode(rng, used) for _ in range(n_cells)]
    with open(os.path.join(d, "meta.tsv"), "w") as f:
        f.write("Index\tCell_type\n")
        for i, b in enumerate(barcodes):
            f.write("%s-1\t%s\n" % (b, "Cancer" if i % 3 else "Non Cancer"))
    in_bam = CONTIGS if not missing_contig else CONTIGS[:-2]
    sites = set()
    while len(sites) < n_sites:
        sites.add((CONTIGS[int(rng.integers(len(CONTIGS)))], int(rng.integers(1, 300000))))
    with open(os.path.join(d, "cand.tsv"), "w") as f:
        f.write("#CHROM\tStart\tEnd\tREF\tALT\n")
        for c, p in sorted(sites):
            alt = "ACGT"[p % 4] + ("" if p % 5 else ",T")
            f.write("\t".join([c, str(p), str(p), "A", alt, ".", "Cancer", ".", ".", ".", ".", ".", ".", "3"]) + "\n")
    meta = G.meta_to_dict(os.path.join(d, "meta.tsv"), None)
    bc = list(meta.keys())
    bins = G.build_dict_variants(os.path.join(d, "cand.tsv"), 50000)
    bin_info, keys, site_tid, site_pos, alt_cls = G.candidate_sites(bins, in_bam)
    # touched pairs sorted by (site, cell); a few sites stay untouched
    t = []
    quiet = set(rng.choice(len(keys), min(untouched_sites, len(keys)), replace=False).tolist()) if len(keys) else set()
    for r, (tid, _) in enumerate(keys):
        if r in quiet:
            continue
        for c in range(len(bc)):
            if rng.random() < cover:
                dp = int(rng.choice([1, 2, 3, 7, 10, 30, 333, 2048]))
                alt = int(rng.integers(0, dp + 1)) if rng.random() < 0.7 else 0
                skip = chrM_contaminant == "True" and in_bam[tid] == "chrM"
                p = np.nan if (alt == 0 or skip) else float(rng.choice([pvalue, 0.00999, 0.010049, 0.5, 1e-9, 0.01005]))
                t.append((r, c, dp, alt, p))
    t_site = np.array([x[0] for x in t], np.int32)
    t_cell = np.array([x[1] for x in t], np.int32)
    t_dp = np.array([x[2] for x in t], np.int32)
    t_alt = np.array([x[3] for x in t], np.int32)
    t_p = np.array([x[4] for x in t], np.float64)
    fusion_file = None
    if fusions is not None:
        fusion_file = os.path.join(d, "fusions.tsv")
        with open(fusion_file, "w") as f:
            f.write("#FusionName\tBC\tJunctionReads\n")
            for name, b in fusions:
                if b is None:  # a raw barcode: fusion BCs are not cleaned, so this is a column of its own
                    b = bc[int(rng.integers(len(bc)))] + "-1"
                elif isinstance(b, int):  # the metadata barcode's column
                    b = bc[b]
                f.write("%s\t%s\t1\n" % (name, b))
    args = argparse.Namespace(outfile=os.path.join(d, "out"), chrM_contaminant=chrM_contaminant, pvalue=pvalue,
                              alt_flag=alt_flag)
    src = G.write_long_table(args, False, bin_info, keys, in_bam, (t_site, t_cell, t_dp, t_alt, t_p), bc, meta)
    return args, src, fusion_file


def fusions_of(fusion_file):
    import pandas as pd
    return G.collect_cells_with_fusions(fusion_file) if fusion_file else pd.DataFrame()


def entry(lay, flags, col, pair, kind, pvalue):
    fl = lay.float_mode and kind != "VAFMatrix"
    if flags & G.LS_GENO_ROW_FUSION:
        return "" if pair is None else ("1.0" if fl else "1")
    if pair is None:
        if lay.col_absent[col]:
            return ""
        v = {"DpMatrix": 0, "AltMatrix": 0, "VAFMatrix": ".", "BinaryMatrix": 3}[kind]
    else:
        dp, alt, p = pair
        if kind == "DpMatrix":
            v = dp
        elif kind == "AltMatrix":
            v = alt
        elif kind == "VAFMatrix":
            v = "." if dp == 0 else round(alt / dp, 4)
        elif dp == 0:
            v = 3
        elif alt == 0:
            v = 0
        elif flags & G.LS_GENO_ROW_CHRM:
            v = 1 if round(alt / dp, 4) >= 0.3 else 0
        else:
            v = 1 if p < pvalue else 0
    return str(float(v)) if fl and kind != "VAFMatrix" else str(v)


def format_rows(lay, kind, pvalue, rows=None):
    """{row rank: text of the row} for the given rows (all by default), without the header."""
    rows = range(len(lay.labels)) if rows is None else rows
    order = np.lexsort((lay.col, lay.row))
    r_sorted = lay.row[order]
    out = {}
    for r in rows:
        lo, hi = np.searchsorted(r_sorted, [r, r + 1])
        pairs = {int(lay.col[j]): (int(lay.dp[j]), int(lay.alt[j]), float(lay.p[j])) for j in order[lo:hi]}
        flags = int(lay.row_flags[r])
        out[r] = lay.labels[r] + "".join("\t" + entry(lay, flags, c, pairs.get(c), kind, pvalue)
                                         for c in range(len(lay.columns))) + "\n"
    return out
