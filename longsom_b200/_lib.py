"""ctypes binding of include/longsom_b200.h (the C-ABI of the CUDA library).

There is no CPU fallback: if liblongsom_b200.so is missing the import of the product path
fails loudly, and ls_ctx_create fails when no CUDA device is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblongsom_b200.so")

LS_OK, LS_E_CUDA, LS_E_ARG, LS_E_STATE, LS_E_CAPACITY = 0, -1, -2, -3, -4
LS_SITE_WORDS = 26
LS_BASE_ALIGN = 16
CLASS_NAMES = ["A", "C", "T", "G", "I", "D", "N", "O"]
CLASS_ID = {c: i for i, c in enumerate(CLASS_NAMES)}
LS_CLASS_NA = 8

# every symbol include/longsom_b200.h declares (checked by tests/test_cpu.py::test_abi_exports_every_declared_symbol)
ABI_SYMBOLS = [
    "ls_abi_version", "ls_ctx_create", "ls_ctx_destroy", "ls_last_error", "ls_host_alloc", "ls_host_free",
    "ls_pileup_upload", "ls_pileup_run", "ls_pileup_compact", "ls_pileup_fetch", "ls_pileup_count", "ls_genotype_count",
    "ls_genotype_sparse_run", "ls_genotype_sparse_fetch",
    "ls_betabinom_sf", "ls_site_mask", "ls_site_table_load", "ls_site_table_lookup", "ls_device_synchronize", "ls_device_pci_bus_id", "ls_flush_l2",
    "ls_geno_matrix_load", "ls_geno_matrix_text", "ls_geno_long_load", "ls_geno_long_text", "ls_geno_long_times",
    "ls_geno_long_release",
]
LS_GENO_MATRIX_DP, LS_GENO_MATRIX_ALT, LS_GENO_MATRIX_VAF, LS_GENO_MATRIX_BINARY = 0, 1, 2, 3
LS_GENO_ROW_CHRM, LS_GENO_ROW_FUSION = 1, 2


class LsReadBatch(C.Structure):
    _fields_ = [
        ("n_reads", C.c_int64), ("n_cigar", C.c_int64), ("n_bases", C.c_int64),
        ("tid", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p),
        ("cell", C.c_void_p), ("cigar_off", C.c_void_p), ("cigar", C.c_void_p), ("base_off", C.c_void_p),
        ("l_qseq", C.c_void_p), ("seq4", C.c_void_p), ("qual", C.c_void_p),
    ]


class LsWindows(C.Structure):
    _fields_ = [
        ("n_windows", C.c_int64), ("tid", C.c_void_p), ("start", C.c_void_p), ("end", C.c_void_p),
        ("ref_off", C.c_void_p), ("ref", C.c_void_p),
    ]


class LsCountParams(C.Structure):
    _fields_ = [("min_bq", C.c_int32), ("min_mq", C.c_int32), ("min_dp", C.c_int32), ("min_cc", C.c_int32),
                ("min_ac", C.c_int32), ("max_depth", C.c_int32)]


class LsGenoParams(C.Structure):
    _fields_ = [("min_bq", C.c_int32), ("min_mq", C.c_int32), ("max_depth", C.c_int32), ("alt_only", C.c_int32),
                ("bin_size", C.c_int32), ("reserved", C.c_int32)]


class LsGenoTuples(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n_tuples", C.c_int64), ("site", C.c_void_p), ("cell", C.c_void_p),
                ("dp", C.c_void_p), ("alt", C.c_void_p), ("p", C.c_void_p)]


class LsRunStats(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_segments", C.c_float), ("ms_sort", C.c_float), ("ms_count", C.c_float),
                ("ms_compact", C.c_float), ("n_segments", C.c_int64), ("n_tiles", C.c_int64),
                ("n_aligned", C.c_int64), ("n_events", C.c_int64), ("count_launches", C.c_int32),
                ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class LsSiteCounts(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("n_sites", C.c_int64), ("tid", C.c_void_p), ("pos", C.c_void_p),
                ("ref", C.c_void_p), ("counts", C.c_void_p)]


class LsGenoMatrixIn(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_pairs", C.c_int64), ("n_cols", C.c_int32), ("float_mode", C.c_int32),
                ("row", C.c_void_p), ("col", C.c_void_p), ("dp", C.c_void_p), ("alt", C.c_void_p), ("p", C.c_void_p),
                ("labels", C.c_void_p), ("label_off", C.c_void_p), ("row_flags", C.c_void_p), ("col_absent", C.c_void_p),
                ("pvalue", C.c_double)]


class LsGenoLongIn(C.Structure):
    _fields_ = [("n_sites", C.c_int64), ("n_cells", C.c_int32), ("hccv", C.c_int32), ("n_pairs", C.c_int64),
                ("cell", C.c_void_p), ("dp", C.c_void_p), ("alt", C.c_void_p), ("p", C.c_void_p), ("hit_lo", C.c_void_p),
                ("hit_hi", C.c_void_p), ("site_flags", C.c_void_p), ("prefix", C.c_void_p), ("prefix_off", C.c_void_p),
                ("index", C.c_void_p), ("index_off", C.c_void_p), ("cell_text", C.c_void_p), ("cell_off", C.c_void_p),
                ("pvalue", C.c_double)]


class LongSomError(RuntimeError):
    pass


_lib = None


def load():
    """Load liblongsom_b200.so and declare prototypes.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LongSomError(
            "longsom_b200: %s not found -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C longsom_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    lib.ls_abi_version.restype = C.c_int
    lib.ls_ctx_create.argtypes = [C.c_int, P(C.c_void_p)]
    lib.ls_ctx_destroy.argtypes = [C.c_void_p]
    lib.ls_last_error.argtypes = [C.c_void_p]
    lib.ls_last_error.restype = C.c_char_p
    lib.ls_host_alloc.argtypes = [C.c_size_t, P(C.c_void_p)]
    lib.ls_host_free.argtypes = [C.c_void_p]
    lib.ls_pileup_upload.argtypes = [C.c_void_p, P(LsReadBatch), P(LsWindows)]
    lib.ls_pileup_run.argtypes = [C.c_void_p, P(LsCountParams), P(C.c_int64), P(LsRunStats)]
    lib.ls_pileup_compact.argtypes = [C.c_void_p, P(LsRunStats)]
    lib.ls_pileup_fetch.argtypes = [C.c_void_p, P(LsSiteCounts)]
    lib.ls_pileup_count.argtypes = [C.c_void_p, P(LsReadBatch), P(LsWindows), P(LsCountParams), P(LsSiteCounts),
                                    P(LsRunStats)]
    lib.ls_genotype_count.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                      P(LsGenoParams), C.c_void_p, C.c_void_p, P(LsRunStats)]
    lib.ls_genotype_sparse_run.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                           P(LsGenoParams), C.c_double, C.c_double, P(C.c_int64), P(LsRunStats)]
    lib.ls_genotype_sparse_fetch.argtypes = [C.c_void_p, P(LsGenoTuples)]
    lib.ls_betabinom_sf.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p,
                                    C.c_int64, P(LsRunStats)]
    lib.ls_device_pci_bus_id.argtypes = [C.c_int, C.c_char_p, C.c_int]
    lib.ls_site_table_load.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
    lib.ls_site_table_lookup.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.ls_site_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                 P(LsRunStats)]
    lib.ls_geno_matrix_load.argtypes = [C.c_void_p, P(LsGenoMatrixIn)]
    lib.ls_geno_matrix_text.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64, P(C.c_int64), P(C.c_int64)]
    lib.ls_geno_long_load.argtypes = [C.c_void_p, P(LsGenoLongIn)]
    lib.ls_geno_long_text.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, P(C.c_int64), P(C.c_int64)]
    lib.ls_geno_long_times.argtypes = [C.c_void_p, P(C.c_double), P(C.c_double), P(C.c_int64), P(C.c_int64)]
    lib.ls_geno_long_release.argtypes = [C.c_void_p]
    lib.ls_device_synchronize.argtypes = [C.c_void_p]
    lib.ls_flush_l2.argtypes = [C.c_void_p]
    for name in ABI_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("ls_last_error",):
            fn.restype = C.c_int
    _lib = lib
    return lib
