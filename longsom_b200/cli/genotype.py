"""Drop-in SingleCellGenotype / HCCVSingleCellGenotype (reference:
workflow/scripts/CellClustering/SingleCellGenotype.py and
workflow/scripts/CellTypeReannotation/HCCVSingleCellGenotype.py).

GPU part: K1' (ls_genotype_sparse_run / _fetch) counts Dp / Alt of every touched (site, cell)
pair of the run in one pass over the reads, and K2 evaluates on the device the beta-binomial
tails of the pairs with ALT > 0; only the touched pairs come back, and the dense rows of the
long table are expanded from them on the device (ls_geno_long_*, write_long_table).  The reference
does this with one pysam pileup per 50 kb bin, a Python dict per (site, barcode) and one scipy
call per pair (:114-218).

The BAM streams by default (pipeline.stream_genotype): chunks of LONGSOM_CHUNK_MB of inflated BAM go
through pinned staging buffers to one engine per LONGSOM_GPUS device, each chunk with the bins no
later read can reach, so host memory stays bounded whatever the size of the tumour BAM.
LONGSOM_STREAM=0 decodes the whole file and runs one call on the first device; both give the same
pairs.  The long table's rows are written in blocks of whole sites, two pinned blocks in flight, so its
text is never held whole either; the host writer (ls_geno_rows) takes the place of the device
writer when the genotyping engine is a stand-in without one.

Host part kept byte-compatible: barcode cleaning, bin codes and temp-file order,
Python set iteration order of the sites inside a bin (:112,130) and row formatting.  The four matrices
(:342-379) are formatted on the device from the same touched pairs (write_matrices); the reference's
pandas pivots stay for the inputs the device writer refuses."""
import argparse
import ctypes as C
import math
import os
import re
import sys
import threading
import timeit
from contextlib import nullcontext

import numpy as np
import pandas as pd
from pandas._libs.parsers import STR_NA_VALUES

from .. import bamio
from .._lib import (CLASS_ID, LS_CLASS_NA, LS_GENO_MATRIX_ALT, LS_GENO_MATRIX_BINARY, LS_GENO_MATRIX_DP,
                    LS_GENO_MATRIX_VAF, LS_GENO_ROW_CHRM, LS_GENO_ROW_FUSION, LS_E_ARG, LongSomError)
from ..blocks import PinnedBlock, write_blocks
from ..engine import Engine
from ..pipeline import devices_from_env, stream_genotype

_NUM = re.compile(r"(\d+)")


def natural_key(s):
    """natsort's default key: digit runs compare as integers, the rest as text."""
    parts = _NUM.split(str(s))
    return tuple(int(p) if i % 2 else p for i, p in enumerate(parts))


def meta_to_dict(meta_file, tissue):
    # SingleCellGenotype.py:230-250
    metadata = pd.read_csv(meta_file, delimiter="\t")
    metadata['Index_clean'] = metadata['Index'].str.replace('-.*$', '', regex=True)
    metadata['Cell_type_clean'] = metadata['Cell_type'].str.replace(' ', '_', regex=True)
    if tissue is not None:
        tissue = tissue.replace(" ", "_")
        metadata['Cell_type_clean'] = str(tissue) + '__' + metadata['Cell_type_clean'].astype(str)
    return metadata.set_index('Index_clean')['Cell_type_clean'].to_dict()


def build_dict_variants(variant_file, window):
    # SingleCellGenotype.py:253-274: bins keyed CHROM_floor(POS/window), insertion ordered
    d = {}
    with open(variant_file) as f:
        for line in f:
            if not line.startswith('#') and not line.startswith('Chr'):
                line = line.rstrip('\n')
                e = line.split('\t')
                code = e[0] + '_' + str(math.floor(int(e[1]) / float(window)))
                d.setdefault(code, []).append(line)
    return d


def candidate_sites(bins, contig_names):
    """Site and bin setup: (bin_info, keys, site_tid, site_pos, alt_cls).  bin_info lists every bin of the variant file
    as (chrom, Target_sites dict in file order); keys are the sorted (tid, pos0) of the sites on contigs of the BAM."""
    tid_of = {n: i for i, n in enumerate(contig_names)}
    bin_info = []  # (chrom, Target_sites dict in file order)
    site_keys = {}
    for code, lines in bins.items():
        target = {}
        chrom = lines[0].split('\t')[0]
        for g in lines:
            g = g.split('\t')
            target[int(g[1]) - 1] = [g[3], g[4].split(',')[0], g[6], g[13]]
        bin_info.append((chrom, target))
        if chrom in tid_of:  # the reference would raise inside pysam for an unknown contig
            for pos0, v in target.items():
                site_keys[(tid_of[chrom], pos0)] = CLASS_ID.get(v[1], LS_CLASS_NA)
    keys = sorted(site_keys)
    site_tid = np.array([k[0] for k in keys], np.int32)
    site_pos = np.array([k[1] for k in keys], np.int32)
    alt_cls = np.array([site_keys[k] for k in keys], np.uint8)
    return bin_info, keys, site_tid, site_pos, alt_cls


def genotype(args, hccv):
    """The long table of one run: (MatrixSource, the engine that wrote it or None); the caller closes the engine."""
    if args.tmp_dir != '.':
        try:
            os.mkdir(args.tmp_dir)
            print("Directory ", args.tmp_dir, " created\n")
        except FileExistsError:
            print("Directory ", args.tmp_dir, " already exists\n")
    else:
        print("Not temp directory specified, using working directory as temp")
    meta_dict = meta_to_dict(args.meta, args.tissue)
    barcodes = list(meta_dict.keys())
    bc_index = {b: i for i, b in enumerate(barcodes)}
    bins = build_dict_variants(args.infile, args.bin)
    devices = devices_from_env()
    stream = os.environ.get("LONGSOM_STREAM", "1") != "0"
    if stream:
        bs = bamio.BamStream(args.bam)  # the header only: the reads are decoded chunk by chunk below
        contig_names = bs.contig_names
        bs.close()
    else:
        # the CUDA context comes up in the background while the BAM is decoded (the native decoder releases the GIL)
        warm = {}

        def _make_engine():
            try:
                warm["engine"] = Engine(devices[0])
            except Exception as e:
                warm["error"] = e
        warm_thread = threading.Thread(target=_make_engine, daemon=True)
        warm_thread.start()
        bam = bamio.read_bam(args.bam)
        contig_names = bam.contig_names
    bin_info, keys, site_tid, site_pos, alt_cls = candidate_sites(bins, contig_names)

    # ---- touched (site, cell) pairs ------------------------------------------------------------------
    # only the touched pairs come back, each with its beta-binomial tail already evaluated on the device (ALT > 0, not
    # the chrM shortcut); the dense rows of the reference are expanded from them below
    if hccv:
        # HCCVSingleCellGenotype.py:163-169 looks the RAW tag up in the cleaned metadata keys
        cell_of = lambda b: bc_index.get(b, -1)
    else:
        cell_of = lambda b: bc_index.get(b.split("-")[0], -1)
    n_cells = len(barcodes)
    chrM_rows = np.array([contig_names[t] == 'chrM' for t in site_tid], bool) if len(keys) else np.zeros(0, bool)
    skip = chrM_rows.astype(np.uint8) if args.chrM_contaminant == 'True' else None
    params = dict(min_bq=args.min_bq, min_mq=args.min_mq, max_depth=200000, alt_only=(args.alt_flag != 'All'))
    if stream:
        # default: chunks of the BAM through pinned staging buffers, over every LONGSOM_GPUS device (bounded host
        # memory); the workers' CUDA contexts come up while the first chunk is decoded.  LONGSOM_STREAM=0 decodes the
        # whole file and runs one call on the first device
        tuples = stream_genotype(args.bam, (site_tid, site_pos, alt_cls), args.bin, n_cells, cell_of, params, args.alpha2,
                                 args.beta2, skip, devices, make_engine=Engine)
    else:
        raw_to_cell = np.array([cell_of(b) for b in bam.barcodes], np.int32)
        batch = bam.with_cells(raw_to_cell) if len(bam.barcodes) else bam.batch
        warm_thread.join()
        if "error" in warm:
            raise warm["error"]
        with warm["engine"] as eng:
            eng.upload(batch, None)
            tuples = eng.genotype_sparse(site_tid, site_pos, alt_cls, n_cells, args.alpha2, args.beta2, skip_p=skip,
                                         bin_size=args.bin, **params)
        del bam, batch
    # the long table is formatted on the first device by the library's writer; a stand-in genotyping engine (the CPU
    # oracle's) has none, and the host writer formats it
    eng = Engine(devices[0]) if hasattr(Engine, 'geno_long_load') else None
    try:
        return write_long_table(args, hccv, bin_info, keys, contig_names, tuples, barcodes, meta_dict, eng), eng
    except BaseException:
        if eng is not None:
            eng.close()
        raise


class MatrixSource:
    """What the matrix writer takes from the long table: its path, its bins (after the CHROM_min_max overwrite rule),
    the touched pairs (p rounded as printed) and the barcodes of its CB column.  long_stats: the device writer's times
    (long_rows_device), None when the host wrote the table."""

    def __init__(self, long_path, blocks, keys, contig_names, tuples, barcodes, meta_dict, long_stats=None):
        self.long_path, self.blocks, self.keys, self.contig_names = long_path, blocks, keys, contig_names
        self.tuples, self.barcodes, self.meta_dict, self.long_stats = tuples, barcodes, meta_dict, long_stats


LONG_BLOCK_BYTES = 64 << 20
LONG_TAIL_MAX = 57  # Dp .. MutationStatus of a row at most: two 10-digit counts, "0.xxxx", "-xxxxxx.xxxx", BetaBin_problem


class LongLayout:
    """The long table's sites in output order: per site its prefix (the seven leading columns), index (the INDEX
    column), chrM flag (the chrM shortcut applies; LS_GENO_ROW_CHRM) and range hit_lo .. hit_hi of the touched pairs.
    The sites of bin b are bin_start[b] .. bin_start[b + 1] - 1."""

    def __init__(self, prefix, index, chrm, hit_lo, hit_hi, bin_start):
        self.prefix, self.index, self.chrm, self.hit_lo, self.hit_hi = prefix, index, chrm, hit_lo, hit_hi
        self.bin_start = bin_start


def long_layout(args, blocks, tid_of, row_of, bounds):
    """The LongLayout of the bins `blocks` (in their (chrom name, lo) order) over the touched pairs split by site at
    `bounds`.  Inside a bin the sites come in the reference's Python set order (:112,130)."""
    prefix, index, chrm, hlo, hhi, bin_start = [], [], [], [], [], []
    for key in sorted(blocks):
        chrom, target = blocks[key]
        bin_start.append(len(prefix))
        for POS in set(target.keys()):  # CELLS dict comprehension iterates the set (:130)
            Ref_exp, Alt_exp, Cell_type_exp, Num_cells_exp = target[POS]
            prefix.append('\t'.join([str(chrom), str(POS + 1), str(POS + 1), Ref_exp, Alt_exp, str(Cell_type_exp),
                                     str(Num_cells_exp)]).encode())
            index.append((str(chrom) + ':' + str(POS + 1) + ':' + Alt_exp.split(',')[0]).encode())
            chrm.append(LS_GENO_ROW_CHRM if (args.chrM_contaminant == 'True' and str(chrom) == 'chrM') else 0)
            r = row_of.get((tid_of.get(chrom, -1), POS))
            hlo.append(bounds[r] if r is not None else 0)
            hhi.append(bounds[r + 1] if r is not None else 0)
    bin_start.append(len(prefix))
    return LongLayout(prefix, index, np.array(chrm, np.uint8), np.array(hlo, np.int64), np.array(hhi, np.int64),
                      bin_start)


def write_long_table(args, hccv, bin_info, keys, contig_names, tuples, barcodes, meta_dict, engine=None):
    """Row assembly: the dense rows of every bin, expanded from the touched pairs, written straight into the long table
    in the reference's (chrom name, lo) bin order.  With an engine the rows are formatted on its device in blocks of
    whole sites (long_rows_device); without one the host writer formats them bin after bin (long_rows_host).  Either
    way no more than two blocks or one bin of text are held at a time."""
    tid_of = {n: i for i, n in enumerate(contig_names)}
    row_of = {k: i for i, k in enumerate(keys)}
    t_site, t_cell, t_dp, t_alt, t_p = tuples
    t_p = np.round(t_p, 4)
    tuples = (t_site, t_cell, t_dp, t_alt, t_p)
    bounds = np.searchsorted(t_site, np.arange(len(keys) + 1))
    native = os.environ.get("LONGSOM_GENO_NATIVE", "1") != "0"
    touched = [None] * len(keys)
    if not native:
        # per site: {cell: (Dp, Alt, BetaBin)}
        tc, td, ta, tp = t_cell.tolist(), t_dp.tolist(), t_alt.tolist(), t_p.tolist()
        for r in range(len(keys)):
            lo_, hi_ = int(bounds[r]), int(bounds[r + 1])
            if hi_ > lo_:
                touched[r] = {tc[i]: (td[i], ta[i], tp[i]) for i in range(lo_, hi_)}

    def bin_rows(chrom, target):
        sites = set(target.keys())  # same construction as the reference => same iteration order
        rows = []
        for POS in sites:  # CELLS dict comprehension iterates the set (:130)
            Ref_exp, Alt_exp, Cell_type_exp, Num_cells_exp = target[POS]
            r = row_of.get((tid_of.get(chrom, -1), POS))
            hits = (touched[r] if r is not None else None) or {}
            for c, bc in enumerate(barcodes):
                CTYPE = meta_dict[bc]
                DP, ALT, PV = hits.get(c, (0, 0, None))
                VAF, BETABIN, MUTATED = '.', '.', 'NoCoverage'
                if DP > 0:
                    if not hccv:
                        VAF = round(ALT / DP, 4)
                    if ALT > 0:
                        if hccv:
                            VAF = round(ALT / DP, 4)
                        if args.chrM_contaminant == 'True' and str(chrom) == 'chrM':
                            MUTATED = 'LowVAFChrM' if VAF < 0.3 else 'PASS'
                        else:
                            BETABIN = np.float64(PV)
                            MUTATED = 'PASS' if BETABIN < args.pvalue else 'BetaBin_problem'
                    else:
                        if hccv:
                            VAF = float(0)
                        MUTATED = 'NoAltReads'
                group = [str(chrom), str(POS + 1), str(POS + 1), Ref_exp, Alt_exp, str(Cell_type_exp), str(Num_cells_exp),
                         bc, CTYPE, str(DP), str(ALT), str(VAF), str(BETABIN), str(MUTATED)]
                if not hccv:
                    BIN = 1 if MUTATED == "PASS" else (3 if MUTATED == "NoCoverage" else 0)
                    group += [str(BIN), str(chrom) + ':' + str(POS + 1) + ':' + Alt_exp.split(',')[0]]
                rows.append(('\t'.join(group) + '\n').encode())
        return rows

    # temp file CHROM_min_max; a later bin with the same name overwrites an earlier one (:117-120)
    blocks = {}
    for chrom, target in bin_info:
        blocks[(str(chrom), min(target))] = (chrom, target)
    header = ['#CHROM', 'Start', 'End', 'REF', 'ALT_expected', 'Cell_type_expected', 'Num_cells_expected', 'CB',
              'Cell_type_observed', 'Dp', 'ALT', 'VAF', 'BetaBin', 'MutationStatus']
    if not hccv:
        header += ['BinMutationStatus', 'INDEX']
    long_path = args.outfile if hccv else args.outfile + '.SingleCellGenotype.tsv'
    stats = None
    if blocks:
        with open(long_path, 'wb') as out:
            out.write(('\t'.join(header) + '\n').encode())
            if not native:
                for key in sorted(blocks):
                    out.writelines(bin_rows(*blocks[key]))
            else:
                lay = long_layout(args, blocks, tid_of, row_of, bounds)
                cell_text = [(bc + '\t' + meta_dict[bc]).encode() for bc in barcodes]
                if engine is not None:
                    stats = long_rows_device(engine, out, lay, tuples, cell_text, hccv, args.pvalue)
                else:
                    long_rows_host(out, lay, tuples, cell_text, hccv, args.pvalue)
    else:
        print('No temporary files found')
    return MatrixSource(long_path if blocks else None, [blocks[k] for k in sorted(blocks)], keys, contig_names, tuples,
                        barcodes, meta_dict, stats)


def long_rows_host(out, lay, tuples, cell_text, hccv, pvalue):
    """The rows of `lay` to file `out` through the host writer (csrc/host/ls_genorows.cpp), one bin's text at a time."""
    host = bamio._load_host()
    host.ls_geno_rows.restype = C.c_int64
    host.ls_geno_rows.argtypes = [C.c_int32] + [C.c_void_p] * 9 + [C.c_int32, C.c_void_p, C.c_int32, C.c_double, C.c_void_p]
    host.ls_geno_rows_free.argtypes = [C.c_void_p]
    _, t_cell, t_dp, t_alt, t_p = tuples
    t_cell = np.ascontiguousarray(t_cell, np.int32)
    t_dp = np.ascontiguousarray(t_dp, np.int32)
    t_alt = np.ascontiguousarray(t_alt, np.int32)
    t_p = np.ascontiguousarray(t_p, np.float64)
    n_cells = len(cell_text)
    cells = (C.c_char_p * max(1, n_cells))(*cell_text)
    for s0, s1 in zip(lay.bin_start[:-1], lay.bin_start[1:]):
        ns = s1 - s0
        pre_a = (C.c_char_p * ns)(*lay.prefix[s0:s1])
        idx_a = None if hccv else (C.c_char_p * ns)(*lay.index[s0:s1])
        text = C.c_void_p()
        n = host.ls_geno_rows(ns, pre_a, idx_a, lay.chrm[s0:].ctypes.data, lay.hit_lo[s0:].ctypes.data,
                              lay.hit_hi[s0:].ctypes.data, t_cell.ctypes.data, t_dp.ctypes.data, t_alt.ctypes.data,
                              t_p.ctypes.data, n_cells, cells, 1 if hccv else 0, float(pvalue), C.byref(text))
        if n < 0:
            raise RuntimeError("ls_geno_rows failed (%d)" % n)
        try:
            if n:
                out.write(C.string_at(text.value, n))
        finally:
            if text.value:
                host.ls_geno_rows_free(text)


def long_rows_device(eng, out, lay, tuples, cell_text, hccv, pvalue):
    """The rows of `lay` to file `out`, formatted on the engine's device (ls_genolong.cu) in blocks of whole sites
    through two pinned buffers.  Returns the device times of the text calls (Engine.geno_long_times) and the seconds
    the file writes took (write_s)."""
    _, t_cell, t_dp, t_alt, t_p = tuples
    eng.geno_long_load(t_cell, t_dp, t_alt, t_p, lay.hit_lo, lay.hit_hi, lay.chrm, lay.prefix,
                       None if hccv else lay.index, cell_text, hccv, pvalue)
    # whole sites per block: the longest possible site fits any block
    n_cells = len(cell_text)
    fixed = np.fromiter((len(x) for x in lay.prefix), np.int64, len(lay.prefix)) + 3 + 18
    if not hccv:
        fixed += 3 + np.fromiter((len(x) for x in lay.index), np.int64, len(lay.index))
    longest = fixed * n_cells + sum(len(x) for x in cell_text) + (LONG_TAIL_MAX - 18) * (lay.hit_hi - lay.hit_lo)
    cap = max(LONG_BLOCK_BYTES, int(longest.max()) if len(longest) else 0)
    bufs = [PinnedBlock(eng, cap) for _ in range(2)]
    try:
        write_s = write_blocks(out, eng.geno_long_text, len(lay.prefix), bufs, cap)
        times = eng.geno_long_times()
    finally:
        for b in bufs:
            b.free()
        eng.geno_long_release()  # the matrix stage that follows on the same engine does not hold the table's buffers
    return dict(times, write_s=write_s)


def collect_cells_with_fusions(fusion_file):
    # SingleCellGenotype.py:325-340
    fusions = pd.read_csv(fusion_file, sep='\t')
    fusions['INDEX'] = fusions['#FusionName'] + ':' + fusions['BC']
    fusions = fusions.drop_duplicates(subset='INDEX', keep="last")
    lines = []
    for _, row in fusions.iterrows():
        lines.append(['.', '.', '.', '.', '.', '.', '.', row['BC'], '.', 1, 1, 1, '.', '.', 1, 'zzz:' + row['#FusionName']])
    return pd.DataFrame(lines)


def chr_index_order(labels):
    """Row order of the matrices (:342-348): chrM sorts last (renamed to chrZ for a stable natural sort), fusions
    ('zzz:') after everything.  Returns the renamed labels, the order of the rows and the labels printed in that order
    (chrZ, literal or not, prints as chrM; the 'zzz:' prefix is dropped)."""
    keyed = [i.replace('chrM', 'chrZ') for i in labels]
    order = sorted(range(len(keyed)), key=lambda i: natural_key(keyed[i]))
    return keyed, order, [keyed[i].replace('chrZ', 'chrM').replace('zzz:', '') for i in order]


def sort_chr_index(df):
    keyed, order, printed = chr_index_order(df.index)
    df.index = keyed
    df = df.reindex([keyed[i] for i in order])
    df.index = printed
    return df


def pivot_long_dataframe(out_prefix, fusions):
    long_df = pd.read_csv(out_prefix + '.SingleCellGenotype.tsv', sep='\t')
    if not fusions.empty:
        fusions.columns = long_df.columns
        long_df = pd.concat([long_df, fusions]).fillna(3)
    for values, name in (('Dp', 'DpMatrix'), ('ALT', 'AltMatrix'), ('VAF', 'VAFMatrix'), ('BinMutationStatus', 'BinaryMatrix')):
        m = long_df.pivot(index='INDEX', columns='CB', values=values)
        m = sort_chr_index(m)
        m.to_csv(out_prefix + '.' + name + '.tsv', sep='\t', index=True)


# ---- the four matrices, written on the device --------------------------------------------------------------------
_CSV_SPECIAL = ('\t', '\n', '\r', '"')
_BOOL_TOKENS = {'True', 'TRUE', 'true', 'False', 'FALSE', 'false'}
MATRIX_KINDS = (('DpMatrix', LS_GENO_MATRIX_DP), ('AltMatrix', LS_GENO_MATRIX_ALT), ('VAFMatrix', LS_GENO_MATRIX_VAF),
                ('BinaryMatrix', LS_GENO_MATRIX_BINARY))
MATRIX_BLOCK_BYTES = 64 << 20


def prints_as_itself(s):
    """True when a value pandas reads from the long table comes back as the same string whatever the other values of
    its column (read_csv infers types chunk by chunk, so one numeric, boolean or NA-like value can change its own type)
    and to_csv prints it unquoted."""
    if not isinstance(s, str) or s in STR_NA_VALUES or s in _BOOL_TOKENS or any(c in s for c in _CSV_SPECIAL):
        return False
    try:
        float(s)
    except ValueError:
        return True
    return False


class MatrixLayout:
    """Rows, columns and pairs of the four matrices in output coordinates, as pivot_long_dataframe lays them out."""

    def __init__(self, labels, columns, col_absent, float_mode, row_flags, row, col, dp, alt, p):
        self.labels, self.columns, self.col_absent, self.float_mode = labels, columns, col_absent, float_mode
        self.row_flags, self.row, self.col, self.dp, self.alt, self.p = row_flags, row, col, dp, alt, p


def matrix_layout(src, fusions, chrM_contaminant):
    """The layout of the matrices pivot_long_dataframe writes from the long table of `src` and the fusion rows of
    collect_cells_with_fusions, or None for an input whose matrices only pandas can say (the reason is printed)."""
    def refuse(why):
        print('Matrices written by pandas: ' + why)
        return None
    if src.long_path is None:
        return refuse('no long table')
    barcodes = src.barcodes
    if not barcodes:
        return refuse('no barcodes')
    if not all(prints_as_itself(b) for b in barcodes):
        return refuse('a barcode pandas would not read back as itself')
    fusion_labels, fusion_bcs = [], []  # 'zzz:' + #FusionName, BC
    if not fusions.empty:
        fusion_labels, fusion_bcs = list(fusions[15]), list(fusions[7])
        if not all(isinstance(x, str) and not any(c in x for c in _CSV_SPECIAL) for x in fusion_labels + fusion_bcs):
            return refuse('a fusion name or barcode that is not plain text')
    # the long table's other text fields: a quote or carriage return there changes how read_csv splits the table
    if any(('"' in x or '\r' in x) for x in src.meta_dict.values()):
        return refuse('a cell type with a quote or carriage return')
    tid_of = {n: i for i, n in enumerate(src.contig_names)}
    row_of = {k: i for i, k in enumerate(src.keys)}
    site_label = np.full(len(src.keys), -1, np.int64)
    labels, chrm = [], []
    for chrom, target in src.blocks:
        for POS, fields in target.items():
            if any(('"' in x or '\r' in x) for x in [str(chrom)] + [str(v) for v in fields]):
                return refuse('a site field with a quote or carriage return')
            r = row_of.get((tid_of.get(chrom, -1), POS))
            if r is not None:
                site_label[r] = len(labels)
            labels.append(str(chrom) + ':' + str(POS + 1) + ':' + fields[1].split(',')[0])
            chrm.append(chrM_contaminant == 'True' and str(chrom) == 'chrM')
    n_snv = len(labels)
    names = sorted(set(fusion_labels))
    labels += names
    if len(set(labels)) < len(labels):
        return refuse('two rows with the same label')
    lex = sorted(range(len(labels)), key=lambda i: labels[i])  # pivot's index order, then the stable natural sort
    keyed, order, printed = chr_index_order([labels[i] for i in lex])
    if len(set(keyed)) < len(keyed):
        return refuse('two rows with the same label once chrM is renamed')
    rank = np.empty(len(labels), np.int32)
    rank[np.asarray(lex, np.int64)[np.asarray(order, np.int64)]] = np.arange(len(labels), dtype=np.int32)
    columns = sorted(set(barcodes) | set(fusion_bcs))
    col_of = {b: i for i, b in enumerate(columns)}
    meta_cols = set(barcodes)
    col_absent = np.array([b not in meta_cols for b in columns], np.uint8)

    t_site, t_cell, t_dp, t_alt, t_p = src.tuples
    srow = site_label[np.asarray(t_site, np.int64)] if len(t_site) else np.zeros(0, np.int64)
    keep = srow >= 0
    cell_col = np.array([col_of[b] for b in barcodes], np.int32)
    row = [rank[srow[keep]]]
    col = [cell_col[np.asarray(t_cell, np.int64)[keep]]]
    dp, alt = [np.asarray(t_dp, np.int32)[keep]], [np.asarray(t_alt, np.int32)[keep]]
    p = [np.asarray(t_p, np.float64)[keep]]
    # the VAF column is read as text only when it holds a '.' (an SNV entry with Dp = 0)
    if int(np.count_nonzero(dp[0] > 0)) >= n_snv * len(barcodes):
        return refuse('every SNV entry is covered, so pandas reads VAF as numbers')
    name_row = {n: n_snv + i for i, n in enumerate(names)}
    fpairs = sorted({(name_row[n], col_of[b]) for n, b in zip(fusion_labels, fusion_bcs)})
    if fpairs:
        fr, fc = np.array(fpairs, np.int64).T
        row.append(rank[fr])
        col.append(fc.astype(np.int32))
        dp.append(np.ones(len(fpairs), np.int32))
        alt.append(np.ones(len(fpairs), np.int32))
        p.append(np.full(len(fpairs), np.nan))
    float_mode = bool(col_absent.any()) or len(fpairs) < len(names) * len(columns)
    row_flags = np.zeros(len(labels), np.uint8)
    row_flags[rank[:n_snv]] = np.where(np.array(chrm, bool), LS_GENO_ROW_CHRM, 0)
    row_flags[rank[n_snv:]] = LS_GENO_ROW_FUSION
    return MatrixLayout(printed, columns, col_absent, float_mode, row_flags, np.concatenate(row), np.concatenate(col),
                        np.concatenate(dp), np.concatenate(alt), np.concatenate(p))


def write_matrices(args, src, fusions, engine=None):
    """DpMatrix, AltMatrix, VAFMatrix and BinaryMatrix as pivot_long_dataframe writes them, formatted on the first
    LONGSOM_GPUS device from the touched pairs in blocks of whole rows, so host memory does not grow with
    n_sites x n_cells.  Runs after the long table is written.  Returns False, writing nothing, for an input it refuses
    (matrix_layout); pivot_long_dataframe then writes the matrices, or raises as the reference does."""
    if not hasattr(Engine, 'geno_matrix_load'):
        return False  # a stand-in genotyping engine (the CPU oracle's) has no matrix writer: pandas writes them
    lay = matrix_layout(src, fusions, args.chrM_contaminant)
    if lay is None:
        return False
    # the caller's engine when it passes one (main: the long table's), else one of our own
    with nullcontext(engine) if engine is not None else Engine(devices_from_env()[0]) as eng:
        try:
            eng.geno_matrix_load(lay.row, lay.col, lay.dp, lay.alt, lay.p, [x.encode() for x in lay.labels],
                                 lay.row_flags, len(lay.columns), lay.col_absent, lay.float_mode, args.pvalue)
        except LongSomError as e:
            if e.code != LS_E_ARG:  # a duplicate (row, col): pandas raises on it as the reference does
                raise
            print('Matrices written by pandas: ' + str(e))
            return False
        # whole rows per block: the longest possible row fits any block
        longest = max(len(x.encode()) for x in lay.labels) + 1 + 13 * len(lay.columns) + 16
        cap = max(MATRIX_BLOCK_BYTES, longest)
        bufs = [PinnedBlock(eng, cap) for _ in range(2)]
        header = ('\t' + '\t'.join(lay.columns) + '\n').encode()
        try:
            for name, kind in MATRIX_KINDS:
                with open(args.outfile + '.' + name + '.tsv', 'wb') as f:
                    f.write(header)
                    write_blocks(f, lambda row, addr, n, kind=kind: eng.geno_matrix_text(kind, row, addr, n),
                                 len(lay.labels), bufs, cap)
        finally:
            for b in bufs:
                b.free()
    return True


def initialize_parser(hccv):
    if hccv:
        p = argparse.ArgumentParser(description='Script to get the alleles observed in each unique cell for the variant sites')
    else:
        p = argparse.ArgumentParser(description='Script to get the SNV/fusions observed in each unique cell')
    p.add_argument('--bam', type=str, default=1, help='Tumor bam file to be analysed', required=True)
    p.add_argument('--infile', type=str, default=1, help='Base calling file (obtained by BaseCellCalling.step2.py), ideally only the PASS variants', required=True)
    p.add_argument('--ref', type=str, default=1, help='Reference genome. *fai must be available in the same folder as reference', required=True)
    p.add_argument('--meta', type=str, default=1, help='Metadata with cell barcodes per cell type', required=True)
    if not hccv:
        p.add_argument('--fusions', type=str, help='Fusions file from CTAT_fusion', nargs='?', const='', required=True)
    p.add_argument('--outfile', default='Matrix.tsv', help='Out file', required=False)
    p.add_argument('--alt_flag', default='All', choices=['Alt', 'All'], help='Flag to search for cells carrying the expected alt variant (Alt) or all cells independent of the alt allele observed (All)', required=False)
    p.add_argument('--nprocs', default=1, help='Number of processes [Default = 1] (accepted for compatibility)', required=False, type=int)
    p.add_argument('--bin', type=int, default=50000, help='Bin size for running the analysis [Default 50000]', required=False)
    p.add_argument('--min_bq', type=int, default=30, help='Minimum base quality permited for the base counts. Default = 30', required=False)
    p.add_argument('--min_mq', type=int, default=255, help='Minimum mapping quality required to analyse read. Default = 255', required=False)
    p.add_argument('--tissue', type=str, default=None, help='Tissue of the sample', required=False)
    p.add_argument('--tmp_dir', type=str, default='tmpDir', help='Temporary folder for tmp files', required=False)
    # the two scripts ship different defaults (SingleCellGenotype.py:396-397, HCCVSingleCellGenotype.py:332-333)
    p.add_argument('--alpha2', type=float, default=0.260288007167716 if hccv else 0.2474528917555431, help='Alpha parameter for Beta-binomial distribution of read counts.', required=False)
    p.add_argument('--beta2', type=float, default=173.94711910763732 if hccv else 162.03696139428595, help='Beta parameter for Beta-binomial distribution of read counts.', required=False)
    p.add_argument('--pvalue', type=float, default=0.01, help='P-value for the beta-binomial test to be significant', required=False)
    p.add_argument('--chrM_contaminant', type=str, default='True', help='Use this option if chrM contaminants are observed in non-cancer cells', required=False)
    return p


def main(argv=None, hccv=False):
    args = initialize_parser(hccv).parse_args(argv)
    start = timeit.default_timer()
    print("Outfile: " if hccv else "Outfile prefix: ", args.outfile, "\n")
    src, eng = genotype(args, hccv)
    try:
        if not hccv:
            fusions = collect_cells_with_fusions(args.fusions) if args.fusions else pd.DataFrame()
            if not write_matrices(args, src, fusions, engine=eng):
                pivot_long_dataframe(args.outfile, fusions)
    finally:
        if eng is not None:
            eng.close()
    print("Computation time: " + str(round(timeit.default_timer() - start)) + ' seconds')


if __name__ == '__main__':
    main(sys.argv[1:])
