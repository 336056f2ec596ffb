"""Python face of the C-ABI: one Engine == one ls_ctx == one B200 + one stream.

Mirrors the reference's unit operations:
  Engine.pileup_count     <-> BaseCellCounter.run_interval          (BaseCellCounter.py:182-320)
  Engine.genotype_count   <-> SingleCellGenotype.run_interval loop  (SingleCellGenotype.py:114-178)
  Engine.genotype_sparse  <-> the same loop + its betabinom.sf calls (SingleCellGenotype.py:114-218), touched pairs only
  Engine.betabinom_sf     <-> scipy.stats.betabinom.sf call sites   (BaseCellCalling.step1.py:196,201)
  Engine.site_mask        <-> step2.build_dict / GetExtraFilters    (BaseCellCalling.step2.py:124-221)
  Engine.geno_matrix_*    <-> the pandas pivots of SingleCellGenotype (SingleCellGenotype.py:351-379)
  Engine.geno_long_*      <-> the long-table row loops of both genotype scripts (SingleCellGenotype.py:128-214)
Every method runs on the GPU; there is no CPU path behind any of them.
"""
import ctypes as C

import numpy as np

from . import _lib as L
from .batch import ReadBatch, SiteCounts, Windows


class CountParams:
    """Thresholds of BaseCellCounter (CLI defaults BaseCellCounter.py:334-339; the workflow passes min_mq 60)."""

    def __init__(self, min_bq=20, min_mq=255, min_dp=5, min_cc=5, min_ac=0, max_depth=200000):
        self.min_bq, self.min_mq, self.min_dp, self.min_cc, self.min_ac, self.max_depth = (
            int(min_bq), int(min_mq), int(min_dp), int(min_cc), int(min_ac), int(max_depth))

    def as_struct(self):
        return L.LsCountParams(self.min_bq, self.min_mq, self.min_dp, self.min_cc, self.min_ac, self.max_depth)


class Engine:
    def __init__(self, device=0):
        self._lib = L.load()
        self._ctx = C.c_void_p()
        rc = self._lib.ls_ctx_create(int(device), C.byref(self._ctx))
        if rc != L.LS_OK:
            self._ctx = None
            raise L.LongSomError("ls_ctx_create(device=%d) failed with %d: no usable CUDA device; "
                                 "longsom_b200 has no CPU fallback" % (device, rc))
        self.device = device
        self.last_stats = None
        self._keep = None

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.ls_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, what):
        if rc != L.LS_OK:
            msg = self._lib.ls_last_error(self._ctx)
            err = L.LongSomError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else ""))
            err.code = rc
            raise err

    # ---- K1 ------------------------------------------------------------------------------
    def upload(self, batch: ReadBatch, windows: Windows = None):
        bs = batch.as_struct()
        ws = windows.as_struct() if windows is not None else L.LsWindows()
        self._keep = (batch, windows)
        self._check(self._lib.ls_pileup_upload(self._ctx, C.byref(bs), C.byref(ws)), "ls_pileup_upload")

    def run(self, params: CountParams):
        ps = params.as_struct()
        n = C.c_int64(0)
        st = L.LsRunStats()
        self._check(self._lib.ls_pileup_run(self._ctx, C.byref(ps), C.byref(n), C.byref(st)), "ls_pileup_run")
        self.last_stats = st.as_dict()
        return int(n.value)

    def compact(self):
        """Passing sites of the last run into output order, on the device (the second half of a bench step)."""
        st = L.LsRunStats()
        self._check(self._lib.ls_pileup_compact(self._ctx, C.byref(st)), "ls_pileup_compact")
        self.last_stats = st.as_dict()

    def fetch(self, n_sites):
        out = SiteCounts.empty(n_sites)
        s = out.as_struct()
        self._check(self._lib.ls_pileup_fetch(self._ctx, C.byref(s)), "ls_pileup_fetch")
        return out.head(int(s.n_sites))

    def pileup_count(self, batch: ReadBatch, windows: Windows, params: CountParams) -> SiteCounts:
        """upload + run + fetch.  Sites ordered by (window order, pos)."""
        self.upload(batch, windows)
        n = self.run(params)
        return self.fetch(n)

    def pileup_count_e2e(self, batch: ReadBatch, windows: Windows, params: CountParams, out: SiteCounts):
        """Single C-ABI call with host buffers (the end-to-end entry point); out must be large enough."""
        bs, ws, ps, st = batch.as_struct(), windows.as_struct(), params.as_struct(), L.LsRunStats()
        s = out.as_struct()
        self._check(self._lib.ls_pileup_count(self._ctx, C.byref(bs), C.byref(ws), C.byref(ps), C.byref(s),
                                              C.byref(st)), "ls_pileup_count")
        self.last_stats = st.as_dict()
        return int(s.n_sites)

    # ---- K1' -----------------------------------------------------------------------------
    def genotype_count(self, site_tid, site_pos, alt_class, n_cells, min_bq=30, min_mq=255, max_depth=200000,
                       alt_only=False, bin_size=50000):
        """Dp / Alt per (site, cell) for the batch of the last upload()."""
        site_tid = np.ascontiguousarray(site_tid, np.int32)
        site_pos = np.ascontiguousarray(site_pos, np.int32)
        alt_class = np.ascontiguousarray(alt_class, np.uint8)
        n = site_pos.shape[0]
        dp = np.zeros((n, n_cells), np.int32)
        alt = np.zeros((n, n_cells), np.int32)
        gp = L.LsGenoParams(int(min_bq), int(min_mq), int(max_depth), 1 if alt_only else 0, int(bin_size), 0)
        st = L.LsRunStats()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self._check(self._lib.ls_genotype_count(self._ctx, vp(site_tid), vp(site_pos), vp(alt_class), n, int(n_cells),
                                                C.byref(gp), vp(dp), vp(alt), C.byref(st)), "ls_genotype_count")
        self.last_stats = st.as_dict()
        return dp, alt

    def genotype_sparse(self, site_tid, site_pos, alt_class, n_cells, alpha, beta, skip_p=None, min_bq=30, min_mq=255,
                        max_depth=200000, alt_only=False, bin_size=50000, fetch=True):
        """Touched (site, cell) pairs only, sorted by (site, cell): (site, cell, dp, alt, p) arrays, p = beta-binomial
        tail of pairs with alt > 0 at sites with skip_p == 0 (NaN elsewhere), evaluated on the device.
        fetch=False leaves the tuples in HBM and returns their number (bench: device-resident rate)."""
        site_tid = np.ascontiguousarray(site_tid, np.int32)
        site_pos = np.ascontiguousarray(site_pos, np.int32)
        alt_class = np.ascontiguousarray(alt_class, np.uint8)
        n = site_pos.shape[0]
        sk = None if skip_p is None else np.ascontiguousarray(skip_p, np.uint8)
        gp = L.LsGenoParams(int(min_bq), int(min_mq), int(max_depth), 1 if alt_only else 0, int(bin_size), 0)
        st, nt = L.LsRunStats(), C.c_int64(0)
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None
        self._check(self._lib.ls_genotype_sparse_run(self._ctx, vp(site_tid), vp(site_pos), vp(alt_class), vp(sk), n,
                                                     int(n_cells), C.byref(gp), float(alpha), float(beta), C.byref(nt),
                                                     C.byref(st)), "ls_genotype_sparse_run")
        self.last_stats = st.as_dict()
        m = int(nt.value)
        if not fetch:
            return m
        site, cell, dp, alt = (np.zeros(m, np.int32) for _ in range(4))
        p = np.zeros(m, np.float64)
        t = L.LsGenoTuples(m, 0, vp(site), vp(cell), vp(dp), vp(alt), vp(p))
        self._check(self._lib.ls_genotype_sparse_fetch(self._ctx, C.byref(t)), "ls_genotype_sparse_fetch")
        return site, cell, dp, alt, p

    # ---- genotype matrices ---------------------------------------------------------------
    def geno_matrix_load(self, row, col, dp, alt, p, labels, row_flags, n_cols, col_absent=None, float_mode=False,
                         pvalue=0.01):
        """Pairs of the Dp / Alt / VAF / Binary matrices in matrix coordinates (row rank, column rank), kept on the
        device for geno_matrix_text.  labels: the printed row labels (bytes), in row order; row_flags: LS_GENO_ROW_*;
        col_absent: 1 for the columns SNV rows do not have; p: the beta-binomial tail rounded to four places."""
        row, col = np.ascontiguousarray(row, np.int32), np.ascontiguousarray(col, np.int32)
        dp, alt = np.ascontiguousarray(dp, np.int32), np.ascontiguousarray(alt, np.int32)
        p = np.ascontiguousarray(p, np.float64)
        row_flags = np.ascontiguousarray(row_flags, np.uint8)
        lens = np.fromiter((len(x) for x in labels), np.int64, len(labels))
        label_off = np.zeros(len(labels) + 1, np.int64)
        np.cumsum(lens, out=label_off[1:])
        blob = b"".join(labels)
        absent = None if col_absent is None else np.ascontiguousarray(col_absent, np.uint8)
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None
        s = L.LsGenoMatrixIn(len(labels), row.shape[0], int(n_cols), 1 if float_mode else 0, vp(row), vp(col), vp(dp),
                             vp(alt), vp(p), C.cast(C.c_char_p(blob), C.c_void_p), vp(label_off), vp(row_flags),
                             vp(absent), float(pvalue))
        self._check(self._lib.ls_geno_matrix_load(self._ctx, C.byref(s)), "ls_geno_matrix_load")

    def geno_matrix_text(self, kind, row_lo, out, capacity):
        """Text of the whole rows row_lo.. of matrix `kind` (LS_GENO_MATRIX_*) that fit in `capacity` bytes at address
        `out`: (rows written, bytes)."""
        rows, nb = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.ls_geno_matrix_text(self._ctx, int(kind), int(row_lo), out, int(capacity), C.byref(rows),
                                                  C.byref(nb)), "ls_geno_matrix_text")
        return int(rows.value), int(nb.value)

    # ---- genotype long table -------------------------------------------------------------
    def geno_long_load(self, cell, dp, alt, p, hit_lo, hit_hi, site_flags, prefix, index, cell_text, hccv=False,
                       pvalue=0.01):
        """The long table's layout, kept on the device for geno_long_text: the touched pairs (cell, dp, alt, p rounded
        to four places; sorted by cell inside each site's range), and per output site, in row order, its pair range
        hit_lo .. hit_hi, LS_GENO_ROW_CHRM flag, prefix (the seven leading columns, bytes) and index (the INDEX column,
        bytes; None when hccv).  cell_text: b"barcode\\tcell type" of each cell."""
        cell, dp, alt = (np.ascontiguousarray(x, np.int32) for x in (cell, dp, alt))
        p = np.ascontiguousarray(p, np.float64)
        hit_lo, hit_hi = np.ascontiguousarray(hit_lo, np.int64), np.ascontiguousarray(hit_hi, np.int64)
        site_flags = np.ascontiguousarray(site_flags, np.uint8)

        def packed(texts):
            off = np.zeros(len(texts) + 1, np.int64)
            np.cumsum(np.fromiter((len(x) for x in texts), np.int64, len(texts)), out=off[1:])
            return b"".join(texts), off
        pre, pre_off = packed(prefix)
        idx, idx_off = packed(index) if not hccv else (b"", None)
        ct, ct_off = packed(cell_text)
        vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None
        bp = lambda b: C.cast(C.c_char_p(b), C.c_void_p)
        s = L.LsGenoLongIn(len(hit_lo), len(cell_text), 1 if hccv else 0, cell.shape[0], vp(cell), vp(dp), vp(alt), vp(p),
                           vp(hit_lo), vp(hit_hi), vp(site_flags), bp(pre), vp(pre_off), bp(idx) if not hccv else None,
                           vp(idx_off), bp(ct), vp(ct_off), float(pvalue))
        self._check(self._lib.ls_geno_long_load(self._ctx, C.byref(s)), "ls_geno_long_load")

    def geno_long_text(self, site_lo, out, capacity):
        """Text of the whole sites site_lo.. of the loaded long table that fit in `capacity` bytes at address `out`:
        (sites written, bytes)."""
        sites, nb = C.c_int64(0), C.c_int64(0)
        self._check(self._lib.ls_geno_long_text(self._ctx, int(site_lo), out, int(capacity), C.byref(sites),
                                                C.byref(nb)), "ls_geno_long_text")
        return int(sites.value), int(nb.value)

    def geno_long_times(self):
        """Device time of the geno_long_text calls since the last load, from events: {ms_text, ms_copy, blocks,
        bytes}."""
        t, c, n, b = C.c_double(0), C.c_double(0), C.c_int64(0), C.c_int64(0)
        self._check(self._lib.ls_geno_long_times(self._ctx, C.byref(t), C.byref(c), C.byref(n), C.byref(b)),
                    "ls_geno_long_times")
        return dict(ms_text=t.value, ms_copy=c.value, blocks=n.value, bytes=b.value)

    def geno_long_release(self):
        """Frees the device buffers of the loaded long table."""
        self._check(self._lib.ls_geno_long_release(self._ctx), "ls_geno_long_release")

    # ---- K2 ------------------------------------------------------------------------------
    def betabinom_sf(self, k, n, a, b):
        """p[i] = scipy.stats.betabinom.sf(k[i] - eps, n[i], a, b) for any 0 < eps < 1 (integer k)."""
        k = np.ascontiguousarray(k, np.int32)
        n = np.ascontiguousarray(n, np.int32)
        m = k.shape[0]
        p = np.zeros(m, np.float64)
        st = L.LsRunStats()
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        if m:
            self._check(self._lib.ls_betabinom_sf(self._ctx, vp(k), vp(n), float(a), float(b), vp(p), m, C.byref(st)),
                        "ls_betabinom_sf")
        self.last_stats = st.as_dict()
        return p

    # ---- K3 ------------------------------------------------------------------------------
    def site_mask(self, keys, query):
        keys = np.ascontiguousarray(keys, np.uint64)
        query = np.ascontiguousarray(query, np.uint64)
        hit = np.zeros(query.shape[0], np.uint8)
        st = L.LsRunStats()
        vp = lambda x: x.ctypes.data_as(C.c_void_p) if x.size else None
        if query.shape[0]:
            self._check(self._lib.ls_site_mask(self._ctx, vp(keys), keys.shape[0], vp(query), query.shape[0], vp(hit),
                                               C.byref(st)), "ls_site_mask")
        self.last_stats = st.as_dict()
        return hit

    def site_table_load(self, table, keys):
        """Sort a (tid<<32 | pos) key table into resident slot `table`; look it up with site_table_lookup."""
        keys = np.ascontiguousarray(keys, np.uint64)
        st = L.LsRunStats()
        self._check(self._lib.ls_site_table_load(self._ctx, int(table), keys.ctypes.data_as(C.c_void_p) if keys.size else None,
                                                 keys.shape[0], C.byref(st)), "ls_site_table_load")
        self.last_stats = st.as_dict()

    def site_table_lookup(self, table, query):
        query = np.ascontiguousarray(query, np.uint64)
        hit = np.zeros(query.shape[0], np.uint8)
        st = L.LsRunStats()
        vp = lambda x: x.ctypes.data_as(C.c_void_p) if x.size else None
        self._check(self._lib.ls_site_table_lookup(self._ctx, int(table), vp(query), query.shape[0], vp(hit), C.byref(st)),
                    "ls_site_table_lookup")
        self.last_stats = st.as_dict()
        return hit

    def flush_l2(self):
        self._check(self._lib.ls_flush_l2(self._ctx), "ls_flush_l2")

    def synchronize(self):
        self._check(self._lib.ls_device_synchronize(self._ctx), "ls_device_synchronize")
