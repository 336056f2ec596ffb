"""Drop-in BaseCellCalling.step1 (reference: workflow/scripts/SNVCalling/BaseCellCalling.step1.py).

The reference streams the merged table and, per site and cell type, calls scipy's scalar
betabinom.sf 2-12 times (~100 us each, :196,201,329-330).  Here the table is parsed once, every
(k, n) query of the run is gathered into two arrays (read counts with alpha1/beta1, cell counts
with alpha2/beta2), the tails are computed in two GPU launches (K2, ls_betabinom_sf), and the
label cascade (SURVEY.md Appendix C) is applied on the rounded p-values exactly as the
reference does.  Output bytes are identical, including its quirks (Q5-Q8).  With the CUDA engine the whole row loop
runs on the device (ls_step1.cu), one byte range of the table at a time; the host passes of ls_step1.cpp serve
stand-in engines and the ranges the device refuses.  The Python passes stay as the statement of the reference; when
they run on a table above 8 MB, it is cut into byte ranges handled by forked worker processes (LONGSOM_PROCS, default
min(16, cores)); the GPU calls stay in the parent."""
import argparse
import os
import sys
import timeit

import numpy as np

from .. import bamio
from ..engine import Engine
from ..pipeline import devices_from_env

ALLELES = ["A", "C", "T", "G", "I", "D", "N", "O"]  # step1.py:20 (the count vectors only carry the first six)

INFO_HEADER = [  # step1.py:48-70
    ('ALT', "##INFO=ALT,Description=Alternative alleles found"),
    ('FILTER', "##INFO=FILTER,Description=Filter status of the variant site"),
    ('Cell_types', "##INFO=Cell_types,Description=Cell type/s with the variant"),
    ('Up_context', "##INFO=Up_context,Description=Up-stream bases in reference (4 bases)"),
    ('Down_context', "##INFO=Down_context,Description=Down-stream bases in reference (4 bases)"),
    ('N_ALT', "##INFO=N_ALT,Description=Cell type/s with the variant"),
    ('Dp', "##INFO=Dp,Description=Depth of coverage (reads) in the cell type supporting the variant"),
    ('Nc', "##INFO=Nc,Description=Number of distinct cells found in the cell type with the mutation"),
    ('Bc', "##INFO=Bc,Description=Number of reads (base count) supporting the variants in the cell type with the mutation"),
    ('Cc', "##INFO=Cc,Description=Number of distinct cells supporting the variant in the cell type with the mutation"),
    ('VAF', "##INFO=VAF,Description=Variant allele frequency of variant in the cell type with the mutation"),
    ('MCF', "##INFO=MCF,Description=Cancer cell fraction (fraction of ditinct cells) supporting the alternative allele in the cell type with the mutation"),
    ('BCp', "##INFO=BCp,Description=Beta-binomial p-value for the variant allele (considering read counts)"),
    ('CCp', "##INFO=CCp,Description=Beta-binomial p-value for the variant allele (considering cell counts)"),
    ('Cell_types_min_BC', "##INFO=Cell_types_min_BC,Description=Number of cell types with a minimum number of reads covering a site"),
    ('Cell_types_min_CC', "##INFO=Cell_types_min_CC,Description=Number of cell types with a minimum number of distinct cells found in a specific site"),
    ('Rest_BC', "##INFO=Rest_BC,Description=Base counts (reads) supporting other alternative alleles in this site. BC;DP;P-value (betabin)"),
    ('Rest_CC', "##INFO=Rest_CC,Description=Cell counts supporting other alternative alleles in this site. CC;NC;P-value (betabin)"),
    ('Fisher_p', "##INFO=Fisher_p,Description=Strand bias test. Fisher exact test p-value between forward and reverse reads in variant and reference allele"),
    ('Cell_type_Filter', "##INFO=Cell_type_Filter,Description=Filter status of the variant site in each cell type"),
]


def longest_run(s):
    """Length of the longest run of equal characters (step1.py:478-483)."""
    best, cur = 0, 0
    prev = None
    for ch in s:
        cur = cur + 1 if ch == prev else 1
        prev = ch
        best = max(best, cur)
    return best


def homopolymer(context, alts, upstream):
    """step1.py:511-529 (the second definition wins): longest run of context+alt >= 4."""
    if context == '.':
        return 0
    m = max(longest_run(context + x) if upstream else longest_run(x + context) for x in alts)
    return 1 if m >= 4 else 0


class _TypeCall:
    __slots__ = ("cell_type", "DP", "NC", "cand", "bc", "cc", "q_bc", "q_cc", "bcf", "REF")


def _fisher_p(cand, bcf, REF):
    # step1.py:228-231: forward and "reverse" vectors are both built from BCf, so the table is degenerate
    import scipy.stats as stats
    Fw = {ALLELES[x]: int(bcf[x]) for x in range(len(bcf))}
    return "|".join(str(round(stats.fisher_exact([[Fw[x], Fw[x]], [Fw[REF], Fw[REF]]])[1], 4)) for x in cand)


class _Params:
    """The thresholds both passes need (picklable: the worker processes receive one)."""

    def __init__(self, min_ac_cells, min_ac_reads, min_cells, min_reads, min_cell_types, max_cell_types, fisher_cutoff):
        self.min_ac_cells, self.min_ac_reads, self.min_cells, self.min_reads = min_ac_cells, min_ac_reads, min_cells, min_reads
        self.min_cell_types, self.max_cell_types, self.fisher_cutoff = min_cell_types, max_cell_types, fisher_cutoff


def _text_lines(data):
    """bytes -> lines the way the reference's text-mode `for line in f` sees them (:32-33): universal newlines
    ('\\r\\n' and a lone '\\r' both end a line and read as '\\n'), nothing else splits a line."""
    text = data.decode()
    if '\r' in text:
        text = text.replace('\r\n', '\n').replace('\r', '\n')
    parts = text.split('\n')
    lines = [x + '\n' for x in parts[:-1]]
    if parts[-1]:
        lines.append(parts[-1])
    return lines


def _header_lines(path):
    """(byte offset, line) for the leading lines of the file, line ends normalised to '\\n'; (offset of EOF, None) at
    the end.  The caller stops at the first line that is not header, whose offset is where the body starts."""
    import re
    size = os.path.getsize(path)
    want = 1 << 16
    while True:
        with open(path, 'rb') as f:
            data = f.read(want)
        complete = len(data) >= size
        out, pos = [], 0
        for m in re.finditer(rb'([^\r\n]*)(\r\n|\n|\r)', data):
            if not complete and m.end() == len(data):
                break   # a '\r' at the end of the chunk may be half of a '\r\n'
            out.append((m.start(), m.group(1).decode() + '\n'))
            pos = m.end()
        if complete and pos < len(data):
            out.append((pos, data[pos:].decode()))
            pos = len(data)
        # enough if the chunk holds a line that is not header (the caller stops there) or the whole file
        if complete or any(not ln.startswith('#') for _, ln in out):
            for item in out:
                yield item
            yield (pos, None)
            return
        want *= 4


def _available_cpus():
    """CPUs this process may run on (the cgroup / affinity of a `threads: 1` Snakemake rule), not the machine's."""
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def _parse_rows(lines, cell_types_idx, fa, P):
    """Pass 1 over data lines: per row the parsed pieces, plus the beta-binomial queries of the rows
    (q1: read counts with alpha1/beta1, q2: cell counts with alpha2/beta2); row indices into the query arrays are
    relative to this call."""
    min_reads, min_cells = P.min_reads, P.min_cells
    rows = []
    q1k, q1n, q2k, q2n = [], [], [], []
    for line in lines:
            if line.startswith('##'):   # a '##' line anywhere in the file is copied through where it stands (:34-35)
                rows.append({"verbatim": line})
                continue
            elements = line.rstrip('\n').split('\t')
            CHROM, POS, REF = str(elements[0]), int(elements[1]), elements[3]
            up_context = down_context = '.'
            if fa is not None:
                try:  # any failure (unknown contig, negative start) -> '.', like the bare except at :97-104
                    context = fa.fetch(CHROM, POS - 6, POS + 5).upper()
                    up_context, down_context = context[0:5], context[6:11]
                except Exception:
                    up_context = down_context = '.'
            calls = []
            n_qual = 0
            Sum_alts_bc = Sum_alts_cc = Sum_dp = Sum_nc = 0
            for ci in cell_types_idx:
                INFO_i = elements[ci]
                if INFO_i.startswith('NA'):
                    continue
                DP, NC, CC, BC, BQ, BCf, BCr = INFO_i.split('|')
                DP, NC = int(DP), int(NC)
                if not (DP >= min_reads and NC >= min_cells):
                    continue
                n_qual += 1
                cc = [int(x) for x in CC.split(":")]
                bc = [int(x) for x in BC.split(":")]
                Sum_alts_bc += sum(bc[x] for x in range(len(bc)) if ALLELES[x] not in (REF, "O"))
                Sum_alts_cc += sum(cc[x] for x in range(len(cc)) if ALLELES[x] not in (REF, "O"))
                Sum_dp += DP
                Sum_nc += NC
                alt_bc = {ALLELES[x]: bc[x] for x in range(len(bc)) if ALLELES[x] not in (REF, "I", "D", "N", "O") and bc[x] > 0}
                alt_cc = {ALLELES[x]: cc[x] for x in range(len(cc)) if ALLELES[x] not in (REF, "I", "D", "N", "O") and cc[x] > 0}
                cand = sorted(alt_bc)
                if not cand:
                    continue
                t = _TypeCall()
                t.cell_type, t.DP, t.NC, t.cand, t.bc, t.cc, t.REF = cell_types_idx[ci], DP, NC, cand, alt_bc, alt_cc, REF
                t.bcf = BCf.split(":")
                t.q_bc = {a: len(q1k) + i for i, a in enumerate(alt_bc)}
                for a in alt_bc:
                    q1k.append(alt_bc[a])
                    q1n.append(DP)
                t.q_cc = {a: len(q2k) + i for i, a in enumerate(alt_cc)}
                for a in alt_cc:
                    q2k.append(alt_cc[a])
                    q2n.append(NC)
                b0 = sum(alt_bc[x] for x in cand)
                c0 = sum(alt_cc[x] for x in cand)  # KeyError here == the reference's own failure mode (bc>0 but cc==0 cannot happen)
                Sum_dp -= b0
                Sum_nc -= c0
                Sum_alts_bc -= b0
                Sum_alts_cc -= c0
                calls.append(t)
            row = dict(elements=elements, up=up_context, down=down_context, calls=calls, n_qual=n_qual,
                       sums=(Sum_alts_bc, Sum_alts_cc, Sum_dp, Sum_nc), rest=None)
            if Sum_alts_bc > 0:  # noise test queries (:328-330 / :426-428)
                row["rest"] = (len(q1k), len(q2k))
                q1k.append(Sum_alts_bc)
                q1n.append(Sum_dp)
                q2k.append(Sum_alts_cc)
                q2n.append(Sum_nc)
            rows.append(row)
    return rows, (np.array(q1k, np.int32), np.array(q1n, np.int32), np.array(q2k, np.int32), np.array(q2n, np.int32))


def _format_rows(rows, r1, r2, P):
    """Pass 2: the label cascade on the rounded p-values (r1 / r2 hold the tails of THESE rows' queries) and the
    output lines."""
    min_ac_cells, min_ac_reads, min_cell_types = P.min_ac_cells, P.min_ac_reads, P.min_cell_types
    max_cell_types, fisher_cutoff = P.max_cell_types, P.fisher_cutoff
    lines = []
    for row in rows:
        if "verbatim" in row:
            lines.append(row["verbatim"])
            continue
        elements, calls = row["elements"], row["calls"]
        Sum_alts_bc, Sum_alts_cc, Sum_dp, Sum_nc = row["sums"]
        if row["rest"] is not None:
            BC_noise_p, CC_noise_p = r1[row["rest"][0]], r2[row["rest"][1]]
        else:
            BC_noise_p, CC_noise_p = 1, 1  # plain ints, printed as '1' (:334-335)
        rest_BC = ";".join([str(Sum_alts_bc), str(Sum_dp), str(BC_noise_p)])
        rest_CC = ";".join([str(Sum_alts_cc), str(Sum_nc), str(CC_noise_p)])
        n_qual = str(row["n_qual"])
        if calls:
            Alts, Cell_types, DPs, NCs, BCs, CCs, BCp, CCp, VAF, MCF, Filter, Fisher_p = ([] for _ in range(12))
            for t in calls:
                cand = t.cand
                Alts.append("|".join(cand))
                Cell_types.append(t.cell_type)
                DPs.append(str(t.DP))
                NCs.append(str(t.NC))
                P_BC = [r1[i] for i in t.q_bc.values()]
                P_CC = [r2[i] for i in t.q_cc.values()]
                fisher_p = None
                if fisher_cutoff != 1:
                    fisher_p = _fisher_p(cand, t.bcf, t.REF)
                    Fisher_p.append(fisher_p)
                b = "|".join(str(t.bc[x]) for x in cand)
                c = "|".join(str(t.cc[x]) for x in cand)
                BCs.append(b)
                CCs.append(c)
                BCp.append("|".join(str(r1[t.q_bc[x]]) for x in cand))
                CCp.append("|".join(str(r2[t.q_cc[x]]) for x in cand))
                VAF.append("|".join(str(round(t.bc[x] / float(t.DP), 4)) for x in cand))
                MCF.append("|".join(str(round(t.cc[x] / float(t.NC), 4)) for x in cand))
                mb, mc = min(P_BC), min(P_CC)
                if mb >= 0.05 or mc >= 0.05:
                    Filter.append('Non-Significant')
                elif 0.001 < mb < 0.05 or 0.001 < mc < 0.05:
                    Filter.append('Low-Significance')
                elif len(cand) > 1:
                    Filter.append('Multi-allelic')
                elif int(c) < min_ac_cells:
                    Filter.append('Low_cells')
                elif int(b) < min_ac_reads:
                    Filter.append('Low_reads')
                elif fisher_cutoff != 1:
                    if float(fisher_p) < fisher_cutoff:  # may append nothing (Q8)
                        Filter.append('Fisher')
                else:
                    Filter.append('PASS')
            FILTER = []
            n_pass = sum(1 for x in Filter if x == 'PASS')
            n_nonsig = sum(1 for x in Filter if x == 'Non-Significant')
            if n_pass > max_cell_types:
                FILTER.append('Multiple_cell_types')
            LEN_Alts = len(set(Alts))
            if LEN_Alts > 1 or 'Multi-allelic' in Filter:
                FILTER.append('Multi-allelic')
            if row["n_qual"] < min_cell_types:
                FILTER.append('Min_cell_types')
            if len(Filter) - n_pass - n_nonsig > 0:
                FILTER.append('Cell_type_noise')
            if BC_noise_p < 0.05 or CC_noise_p < 0.05:
                FILTER.append('Noisy_site')
            if homopolymer(row["up"], Alts, True) == 1:
                FILTER.append("LC_Upstream")
            if homopolymer(row["down"], Alts, False) == 1:
                FILTER.append("LC_Downstream")
            if len(FILTER) == 0:
                FILTER = 'PASS' if 'PASS' in Filter else ",".join(Filter)
            else:
                FILTER = ",".join(FILTER)
            INFO = [",".join(Alts), FILTER, ",".join(Cell_types), row["up"], row["down"], str(LEN_Alts), ",".join(DPs),
                    ",".join(NCs), ",".join(BCs), ",".join(CCs), ",".join(VAF), ",".join(MCF), ",".join(BCp),
                    ",".join(CCp), n_qual, n_qual, rest_BC, rest_CC,
                    ",".join(Fisher_p) if fisher_cutoff != 1 else '.', ",".join(Filter)]
        else:
            FILTER = 'Noisy_site' if (BC_noise_p < 0.001 or CC_noise_p < 0.001) else '.'
            INFO = [".", FILTER, ".", row["up"], row["down"], ".", ".", ".", ".", ".", ".", ".", ".", ".", n_qual, n_qual,
                    rest_BC, rest_CC, '.', '.']
        elements.insert(4, "\t".join(INFO))
        lines.append('\t'.join(elements) + '\n')
    return lines


# ---- native row passes (liblongsom_host.so, csrc/host/ls_step1.cpp) -------------------------------------------
# The two per-row passes above restated in C++: a byte range of the table in, queries out; rounded tails in, output
# text out.  Anything the strict native parser refuses (a row the reference itself would fail on) and the strand-bias
# column (--fisher_cutoff != 1) go through the Python passes above, which stay the statement of the reference's
# behaviour; LONGSOM_STEP1_NATIVE=0 switches the native path off.
def _s1_lib():
    import ctypes as C
    lib = bamio._load_host()
    if not getattr(lib, "_s1_ready", False):
        lib.ls_s1_parse.restype = C.c_void_p
        lib.ls_s1_parse.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_int32]
        lib.ls_s1_free.argtypes = [C.c_void_p]
        for f in ("ls_s1_n_rows", "ls_s1_n_data_rows", "ls_s1_n_q1", "ls_s1_n_q2"):
            getattr(lib, f).restype = C.c_int64
            getattr(lib, f).argtypes = [C.c_void_p]
        lib.ls_s1_queries.argtypes = [C.c_void_p] * 5
        lib.ls_s1_n_chroms.restype = C.c_int32
        lib.ls_s1_n_chroms.argtypes = [C.c_void_p]
        lib.ls_s1_chrom.restype = C.c_char_p
        lib.ls_s1_chrom.argtypes = [C.c_void_p, C.c_int32]
        lib.ls_s1_sites.argtypes = [C.c_void_p] * 3
        lib.ls_s1_format.restype = C.c_int64
        lib.ls_s1_format.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        lib._s1_ready = True
    return lib


class _NativeRange:
    """One byte range of the table held by the native parser."""

    def __init__(self, data, cell_types_idx, P):
        import ctypes as C
        self.C, self.lib = C, _s1_lib()
        self.data = data                      # keeps the bytes alive: the handle points into them
        self.cols = np.array(sorted(cell_types_idx), np.int32)
        self.names = [cell_types_idx[int(c)].encode() for c in self.cols]
        err = C.create_string_buffer(256)
        self.h = self.lib.ls_s1_parse(C.c_char_p(data), len(data), self.cols.ctypes.data, len(self.cols), int(P.min_reads),
                                      int(P.min_cells), err, 256)
        if not self.h:
            raise ValueError(err.value.decode())
        n1, n2 = self.lib.ls_s1_n_q1(self.h), self.lib.ls_s1_n_q2(self.h)
        self.q = tuple(np.zeros(n, np.int32) for n in (n1, n1, n2, n2))
        self.lib.ls_s1_queries(self.h, *[a.ctypes.data for a in self.q])
        self.n_rows = self.lib.ls_s1_n_rows(self.h)
        self.n_data = self.lib.ls_s1_n_data_rows(self.h)

    def contexts(self, fa):
        """ctx[row][11], ctx_len[row] = fa.fetch(CHROM, POS - 6, POS + 5).upper() of every row; -1 where the reference
        prints '.' (no FASTA, unknown contig, POS < 6: the bare except at step1.py:97-104)."""
        n = self.n_rows
        ctx, clen = np.zeros((n, 11), np.uint8), np.full(n, -1, np.int8)
        if fa is None or n == 0:
            return ctx, clen
        chrom, pos = np.zeros(n, np.int32), np.zeros(n, np.int64)
        self.lib.ls_s1_sites(self.h, chrom.ctypes.data, pos.ctypes.data)
        offs = np.arange(11, dtype=np.int64)
        for ci in range(self.lib.ls_s1_n_chroms(self.h)):
            name = self.lib.ls_s1_chrom(self.h, ci).decode()
            try:
                seq = fa.contig(name)
            except Exception:
                continue
            rows = np.nonzero((chrom == ci) & (pos >= 6))[0]
            if rows.shape[0] == 0:
                continue
            start = pos[rows] - 6
            L = np.clip(seq.shape[0] - start, 0, 11)
            idx = np.minimum(start[:, None] + offs[None, :], max(seq.shape[0] - 1, 0))
            block = seq[idx] if seq.shape[0] else np.zeros((rows.shape[0], 11), np.uint8)
            lower = (block >= 97) & (block <= 122)
            block = np.where(lower, block - 32, block).astype(np.uint8)
            block[offs[None, :] >= L[:, None]] = 0
            ctx[rows] = block
            clen[rows] = L.astype(np.int8)
        return ctx, clen

    def format(self, r1, r2, fa, P):
        """Output text of the range as a buffer that lives in the native handle (valid until close())."""
        C = self.C
        ctx_p = clen_p = None
        if fa is not None:
            ctx, clen = self.contexts(fa)
            ctx_p, clen_p = ctx.ctypes.data, clen.ctypes.data
        r1 = np.ascontiguousarray(r1, np.float64)
        r2 = np.ascontiguousarray(r2, np.float64)
        names = (C.c_char_p * max(1, len(self.names)))(*self.names)
        text = C.c_void_p()
        n = self.lib.ls_s1_format(self.h, r1.ctypes.data, r2.ctypes.data, ctx_p, clen_p, names,
                                  int(P.min_ac_cells), int(P.min_ac_reads), int(P.min_cell_types), int(P.max_cell_types),
                                  C.byref(text))
        if n < 0:   # a NaN among the per-allele tails (min() over NaNs is order dependent), or > 64 calls in a row
            raise ValueError("ls_s1_format: left to the Python passes")
        return (C.c_char * n).from_address(text.value) if n else b""

    def close(self):
        if self.h:
            self.lib.ls_s1_free(self.h)
            self.h = None


STEP1_BLOCK_BYTES = 16 << 20   # text block of the device path (two pinned blocks, one filled while the other is written)
last_times = {}                # busy seconds of the stages of the last device-called table (tools/cli_step1_timing.py)


def _device_ranges(eng, out, ranges, read, cell_types_idx, fa, P, alphas, tails):
    """The byte ranges of the table called on the device, one at a time, their text written to `out` in blocks of whole
    rows: the parse, the tails, the labels, the contexts (from contigs kept resident on the device) and the rows are
    computed in HBM.  The next range is read from the file while the device works on the current one.  A range the
    device refuses is redone by the host passes (_NativeRange, with the same K2 tails), which give the same bytes; a
    range they refuse raises ValueError.  Returns (rows, beta-binomial tails)."""
    from concurrent.futures import ThreadPoolExecutor
    import time
    from .._lib import LS_E_ARG, LongSomError
    from ..blocks import PinnedBlock, write_blocks
    cols = sorted(cell_types_idx)
    names = [cell_types_idx[c].encode() for c in cols]
    n_rows = n_queries = n_host = 0
    bufs, cap = [], 0
    T = dict(read_s=0.0, call_s=0.0, text_s=0.0, write_s=0.0)  # text_s: the block loop, its file writes overlapped

    def timed_read(rng):
        t = time.perf_counter()
        data = read(rng)
        T["read_s"] += time.perf_counter() - t
        return data

    def host_range(data):
        r = _NativeRange(data, cell_types_idx, P)
        try:
            r1, r2 = tails(r.q)
            out.write(r.format(r1, r2, fa, P))
            return r.n_rows, len(r1) + len(r2)
        finally:
            r.close()
    try:
        with ThreadPoolExecutor(1) as reader:
            nxt = reader.submit(timed_read, ranges[0]) if ranges else None
            for i in range(len(ranges)):
                data = nxt.result()
                nxt = reader.submit(timed_read, ranges[i + 1]) if i + 1 < len(ranges) else None
                t0 = time.perf_counter()
                try:
                    rows, nq, new = eng.step1_load(data, cols, names, P.min_reads, P.min_cells, P.min_ac_cells,
                                                   P.min_ac_reads, P.min_cell_types, P.max_cell_types, *alphas)
                    for cid, name in new:   # a contig is made resident the first time a range names it
                        if fa is None:
                            continue
                        try:
                            seq = fa.contig(name)
                        except Exception:
                            continue        # not in the FASTA: its rows print '.' contexts
                        eng.step1_contig(cid, seq)
                    nbytes, longest = eng.step1_call()
                except LongSomError as e:
                    if getattr(e, "code", None) != LS_E_ARG:
                        raise
                    r, q = host_range(data)
                    n_rows, n_queries, n_host = n_rows + r, n_queries + q, n_host + r
                    T["call_s"] += time.perf_counter() - t0
                    continue
                t1 = time.perf_counter()
                T["call_s"] += t1 - t0
                if max(STEP1_BLOCK_BYTES, longest) > cap:
                    for b in bufs:
                        b.free()
                    bufs = []
                    cap = max(STEP1_BLOCK_BYTES, longest)
                    bufs = [PinnedBlock(eng, cap) for _ in range(2)]
                T["write_s"] += write_blocks(out, eng.step1_text, rows, bufs, cap)
                T["text_s"] += time.perf_counter() - t1
                n_rows += rows
                n_queries += nq
    finally:
        for b in bufs:
            b.free()
        eng.step1_release()
    T.update(rows=n_rows, host_rows=n_host)
    last_times.clear()
    last_times.update(T)
    return n_rows, n_queries


def _native_ok(P):
    return P.fisher_cutoff == 1 and os.environ.get("LONGSOM_STEP1_NATIVE", "1") != "0"


# ---- worker processes: the per-row Python of both passes is the cost of this step (tens of microseconds per row, the
# GPU tails are milliseconds), so large tables are cut into byte ranges handled by forked workers; each parses its
# range, sends its queries, receives its tails, formats its lines.  The order of the output is the order of the ranges.
def _worker(conn, infile, lo, hi, cell_types_idx, fasta, P):
    try:
        fa = bamio.Fasta(fasta) if fasta is not None else None
        with open(infile, 'rb') as f:
            f.seek(lo)
            lines = _text_lines(f.read(hi - lo))
        rows, q = _parse_rows(lines, cell_types_idx, fa, P)
        conn.send(("queries", q))
        r1, r2 = conn.recv()
        conn.send(("lines", "".join(_format_rows(rows, r1, r2, P)), len(rows)))
    except BaseException as e:  # surfaced in the parent
        import traceback
        conn.send(("error", "%r\n%s" % (e, traceback.format_exc())))
    finally:
        conn.close()


def _line_aligned_ranges(path, start, n):
    """n byte ranges [lo, hi) covering [start, EOF), each ending at a line break."""
    size = os.path.getsize(path)
    cuts = [start]
    with open(path, 'rb') as f:
        for k in range(1, n):
            f.seek(max(start, start + (size - start) * k // n))
            f.readline()
            cuts.append(min(max(f.tell(), cuts[-1]), size))
    cuts.append(size)
    return [(cuts[i], cuts[i + 1]) for i in range(n) if cuts[i + 1] > cuts[i]]


def variant_calling_step1(infile, outfile, fasta, alpha1, beta1, alpha2, beta2, min_ac_cells, min_ac_reads, min_cells,
                          min_reads, min_cell_types, max_cell_types, fisher_cutoff, engine, procs=None):
    P = _Params(min_ac_cells, min_ac_reads, min_cells, min_reads, min_cell_types, max_cell_types, fisher_cutoff)
    out_lines = []          # header lines written verbatim
    cell_types_idx = None
    body_start = 0
    # header: '##' lines and the first '#CHROM' line, split the way text mode splits them (see _text_lines)
    for pos, line in _header_lines(infile):
        body_start = pos
        if line is None:
            break
        if line.startswith('##'):
            out_lines.append(line)
            continue
        if line.startswith('#CHROM') and cell_types_idx is None:
            elements = line.rstrip('\n').split('\t')
            cell_types_idx = {x: elements[x] for x in range(len(elements)) if x > 4}
            for _, text in INFO_HEADER:
                out_lines.append(text + '\n')
            elements.insert(4, "\t".join(k for k, _ in INFO_HEADER))
            out_lines.append('\t'.join(elements) + '\n')
            continue
        break
    body_bytes = os.path.getsize(infile) - body_start
    native = _native_ok(P) and cell_types_idx is not None and body_bytes > 0
    if procs is None:
        procs = int(os.environ.get("LONGSOM_PROCS", "0") or 0)   # an explicit setting is honoured as is
        if procs <= 0:
            procs = 1 if body_bytes < (8 << 20) else min(16, _available_cpus())   # small tables: not worth forking

    warm = {}

    def get_engine():
        # `engine` may be a factory: the CUDA context is then created after the workers have been forked (a forked
        # child must never inherit a live context) and, in the multi-process path, while they parse
        if "thread" in warm:
            warm.pop("thread").join()
            if "error" in warm:
                raise warm["error"]
        if "engine" not in warm:
            warm["engine"] = engine() if callable(engine) else engine
        return warm["engine"]

    def tails(q):
        eng = get_engine()
        p1 = eng.betabinom_sf(q[0], q[1], alpha1, beta1)
        p2 = eng.betabinom_sf(q[2], q[3], alpha2, beta2)
        # == round(np.float64, 4) of the reference, element-wise
        return np.round(p1, 4), np.round(p2, 4)

    if native:
        # Native row passes, in byte ranges so that the memory in flight does not grow with the table.  With the CUDA
        # engine every range is called on the device (_device_ranges); otherwise the ranges go in waves through the
        # host passes: parsed on threads (the library releases the GIL), the wave's queries through K2 in one call,
        # formatted on threads and appended to the output.  A range the host parser refuses discards what has been
        # written and leaves the whole table to the Python passes below (whose exceptions are the reference's).
        from concurrent.futures import ThreadPoolExecutor
        nthr = 1 if body_bytes < (4 << 20) else min(16, _available_cpus())
        chunk = int(float(os.environ.get("LONGSOM_STEP1_CHUNK_MB", "64")) * (1 << 20))
        n_ranges = max(nthr, -(-body_bytes // max(chunk, 1 << 16)))
        ranges = _line_aligned_ranges(infile, body_start, int(n_ranges))
        fa = bamio.Fasta(fasta) if fasta is not None else None
        tmp_out = outfile + ".native.%d.tmp" % os.getpid()
        n_rows = n_queries = 0
        ok = False

        def read(rng):
            with open(infile, 'rb') as f:
                f.seek(rng[0])
                return f.read(rng[1] - rng[0])

        def parse(rng):
            return _NativeRange(read(rng), cell_types_idx, P)
        try:
            with open(tmp_out, 'wb') as out:
                out.write("".join(out_lines).encode())
                # the device path needs the CUDA engine; stand-in engines (the CPU tests' scipy tails) keep the host passes
                if hasattr(Engine if callable(engine) else engine, "step1_load"):
                    n_rows, n_queries = _device_ranges(get_engine(), out, ranges, read, cell_types_idx, fa, P,
                                                       (alpha1, beta1, alpha2, beta2), tails)
                else:
                    with ThreadPoolExecutor(nthr) as ex:
                        for w0 in range(0, len(ranges), nthr):
                            wave = []
                            try:
                                for r in ex.map(parse, ranges[w0:w0 + nthr]):   # (a refusal surfaces here as ValueError)
                                    wave.append(r)
                                qs = [r.q for r in wave]
                                r1, r2 = tails(tuple(np.concatenate([q[j] for q in qs]) for j in range(4)))
                                o1 = np.concatenate([[0], np.cumsum([len(q[0]) for q in qs])]).astype(np.int64)
                                o2 = np.concatenate([[0], np.cumsum([len(q[2]) for q in qs])]).astype(np.int64)
                                if fa is not None:     # contigs are loaded once, before the threads share the reader
                                    for r in wave:
                                        for ci in range(r.lib.ls_s1_n_chroms(r.h)):
                                            try:
                                                fa.contig(r.lib.ls_s1_chrom(r.h, ci).decode())
                                            except Exception:
                                                pass
                                texts = list(ex.map(lambda kr: kr[1].format(r1[o1[kr[0]]:o1[kr[0] + 1]],
                                                                            r2[o2[kr[0]]:o2[kr[0] + 1]], fa, P),
                                                    enumerate(wave)))
                                for t in texts:
                                    out.write(t)
                                n_rows += sum(r.n_rows for r in wave)
                                n_queries += len(r1) + len(r2)
                            finally:
                                for r in wave:
                                    r.close()
            os.replace(tmp_out, outfile)
            ok = True
        except ValueError:
            pass   # fall through to the Python passes
        finally:
            if fa is not None:
                fa.close()
            if not ok and os.path.exists(tmp_out):
                os.remove(tmp_out)
        if ok:
            return n_rows, n_queries
        if "engine" in warm:
            procs = 1   # a wave has already created the CUDA context: the Python passes must not fork below it

    if procs <= 1:
        fa = bamio.Fasta(fasta) if fasta is not None else None
        with open(infile, 'rb') as f:
            f.seek(body_start)
            data_lines = _text_lines(f.read())
        if cell_types_idx is None and data_lines:
            raise TypeError("'NoneType' object is not iterable")  # data before any #CHROM line: the reference fails here too
        rows, q = _parse_rows(data_lines, cell_types_idx, fa, P)
        r1, r2 = tails(q)
        with open(outfile, 'w') as out:
            out.writelines(out_lines)
            out.writelines(_format_rows(rows, r1, r2, P))
        if fa is not None:
            fa.close()
        return len(rows), len(q[0]) + len(q[2])

    import multiprocessing as mp
    ctx = mp.get_context("fork")
    workers = []
    for lo, hi in _line_aligned_ranges(infile, body_start, procs):
        parent, child = ctx.Pipe()
        pr = ctx.Process(target=_worker, args=(child, infile, lo, hi, cell_types_idx, fasta, P), daemon=True)
        pr.start()
        child.close()
        workers.append((pr, parent))

    if callable(engine):
        import threading

        def make():
            try:
                warm["engine"] = engine()
            except Exception as e:
                warm["error"] = e
        warm["thread"] = threading.Thread(target=make, daemon=True)
        warm["thread"].start()

    def receive(conn, kind):
        msg = conn.recv()
        if msg[0] == "error":
            raise RuntimeError("step1 worker failed: " + msg[1])
        assert msg[0] == kind
        return msg[1:]
    queries = [receive(conn, "queries")[0] for _, conn in workers]
    r1, r2 = tails(tuple(np.concatenate([q[j] for q in queries]) for j in range(4)))
    o1 = o2 = 0
    for (_, conn), q in zip(workers, queries):
        conn.send((r1[o1:o1 + len(q[0])], r2[o2:o2 + len(q[2])]))
        o1 += len(q[0])
        o2 += len(q[2])
    n_rows = 0
    with open(outfile, 'w') as out:
        out.writelines(out_lines)
        for pr, conn in workers:
            text, n = receive(conn, "lines")
            out.write(text)
            n_rows += n
            pr.join()
    return n_rows, len(r1) + len(r2)


def initialize_parser():
    # flags, types and defaults of step1.py:585-604
    p = argparse.ArgumentParser(description='Script to perform the scRNA somatic variant calling')
    p.add_argument('--infile', type=str, help='Input file with all samples merged in a single tsv', required=True)
    p.add_argument('--outfile', type=str, help='Output file prefix', required=True)
    p.add_argument('--ref', type=str, help='Reference fasta file (*fai must exist)', required=True)
    p.add_argument('--editing', type=str, help='RNA editing file to be used to remove RNA-diting sites', required=False)
    p.add_argument('--pon', type=str, help='Panel of normals (PoN) file to be used to remove germline and false positive calls', required=False)
    p.add_argument('--min_cov', type=int, default=5, help='Minimum depth of coverage to consider a sample. [Default: 5]', required=False)
    p.add_argument('--min_cells', type=int, default=5, help='Minimum number of cells covering a site to consider a sample. [Default: 5]', required=False)
    p.add_argument('--min_ac_cells', type=int, default=2, help='Minimum number of cells supporting the alternative allele to consider a mutation. [Default: 2]', required=False)
    p.add_argument('--min_ac_reads', type=int, default=3, help='Minimum number of reads supporting the alternative allele to consider a mutation. [Default: 3]', required=False)
    p.add_argument('--max_cell_types', type=int, default=1, help='Maximum number of cell types carrying a mutation to make a somatic call. [Default: 1]', required=False)
    p.add_argument('--min_cell_types', type=int, default=2, help='Minimum number of cell types with enough coverage and cell to consider a site as callable [Default: 2]', required=False)
    p.add_argument('--fisher_cutoff', type=float, default=1, help='P-value cutoff for the Fisher exact test performed to detect strand bias. By default, this test is switched off with a value of 1 [Default: 1]', required=False)
    p.add_argument('--min_distance', type=int, default=5, help='Minimum distance allowed between potential somatic variants [Default: 5]', required=False)
    p.add_argument('--alpha1', type=float, default=0.21356677091082193, help='Alpha parameter for Beta-binomial distribution of read counts.', required=False)
    p.add_argument('--beta1', type=float, default=104.95163748636298, help='Beta parameter for Beta-binomial distribution of read counts.', required=False)
    p.add_argument('--alpha2', type=float, default=0.2474528917555431, help='Alpha parameter for Beta-binomial distribution of cell counts.', required=False)
    p.add_argument('--beta2', type=float, default=162.03696139428595, help='Beta parameter for Beta-binomial distribution of cell counts.', required=False)
    return p


def main(argv=None):
    args = initialize_parser().parse_args(argv)
    start = timeit.default_timer()
    print('\n------------------------------')
    print('Variant calling')
    print('------------------------------\n')
    print('- Variant calling step 1\n')
    outfile1 = args.outfile + ".calling.step1.tsv"
    made = []

    def make_engine():  # created lazily: after the worker processes have been forked, while they parse
        made.append(Engine(devices_from_env()[0]))
        return made[-1]
    try:
        n_rows, n_q = variant_calling_step1(args.infile, outfile1, args.ref, args.alpha1, args.beta1, args.alpha2,
                                            args.beta2, args.min_ac_cells, args.min_ac_reads, args.min_cells,
                                            args.min_cov, args.min_cell_types, args.max_cell_types, args.fisher_cutoff,
                                            make_engine)
    finally:
        for eng in made:
            eng.close()
    print('Step 1 variant calling: %d positions processed, %d beta-binomial tails on the GPU' % (n_rows, n_q))
    print('\nTotal computing time: ' + str(round(timeit.default_timer() - start, 2)) + ' seconds')


if __name__ == '__main__':
    main(sys.argv[1:])
