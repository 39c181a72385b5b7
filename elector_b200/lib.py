"""Locates and loads the in-tree C-ABI library (elector_b200/libelector_poa.so)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class LibraryNotBuilt(RuntimeError):
    pass


def library_path():
    # ELECTOR_POA_LIB selects another build of the same library (A/B runs of kernel variants)
    return os.environ.get("ELECTOR_POA_LIB") or os.path.join(_HERE, "libelector_poa.so")


def poa_binary_path():
    return os.path.join(_HERE, "bin", "poa")


def splitter_binary_path():
    return os.path.join(_HERE, "bin", "masterSplitter")


def load_library():
    """Returns the ctypes handle; raises LibraryNotBuilt (never falls back) if it is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise LibraryNotBuilt(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback." % path)
    lib = ctypes.CDLL(path)
    c = ctypes
    i64p, i32p = c.POINTER(c.c_int64), c.POINTER(c.c_int32)
    vp = c.c_void_p
    lib.elector_poa_init.argtypes = [c.c_int, c.c_char_p, c.POINTER(vp)]
    lib.elector_poa_init.restype = c.c_int
    lib.elector_poa_free.argtypes = [vp]
    lib.elector_poa_free.restype = None
    lib.elector_last_error.argtypes = [vp]
    lib.elector_last_error.restype = c.c_char_p
    lib.elector_poa_run.argtypes = [vp, c.c_int64, vp, vp, vp, vp, vp, vp, vp, c.c_int64, vp, vp, vp, vp, vp, vp]
    lib.elector_poa_run.restype = c.c_int
    lib.elector_poa_rows_bound.argtypes = [c.c_int64, vp, vp, vp]
    lib.elector_poa_rows_bound.restype = c.c_int64
    lib.elector_poa_run_device.argtypes = [vp, c.c_int64] + [vp] * 9 + [vp, c.c_int64] + [vp] * 7
    lib.elector_poa_run_device.restype = c.c_int
    lib.elector_poa_files.argtypes = [vp, c.c_char_p, c.c_char_p, c.c_char_p, c.c_char_p, c.c_int]
    lib.elector_poa_files.restype = c.c_int
    lib.elector_tally_run.argtypes = [vp, c.c_int64, vp, vp, vp, vp, vp]
    lib.elector_tally_run.restype = c.c_int
    lib.elector_unpack_columns.argtypes = [vp, c.c_int64, vp, vp, vp]
    lib.elector_unpack_columns.restype = None
    lib.elector_merge_run.argtypes = [vp, c.c_int64, vp, c.c_int64, vp, c.c_int64, vp, vp, vp, vp, vp, vp, c.c_int64, vp, vp]
    lib.elector_merge_run.restype = c.c_int
    lib.elector_merge_tally_device.argtypes = [vp, c.c_int64, vp, c.c_int64, vp, c.c_int64, vp, vp, vp, vp]
    lib.elector_merge_tally_device.restype = c.c_int
    lib.elector_pipeline_run.argtypes = [vp, c.c_int64, vp, vp, vp, vp, vp, vp, c.c_int64, vp, vp, c.c_int64] + [vp] * 8
    lib.elector_pipeline_run.restype = c.c_int
    lib.elector_pipeline_run2.argtypes = [vp, vp]
    lib.elector_pipeline_run2.restype = c.c_int
    lib.elector_pack_letters.argtypes = [vp, c.c_int64, vp, vp, vp, c.c_int64]
    lib.elector_pack_letters.restype = c.c_int64
    lib.elector_merged_bound.argtypes = [c.c_int64, c.c_int64, vp, vp, vp]
    lib.elector_merged_bound.restype = c.c_int64
    lib.elector_split_bounds.argtypes = [c.c_int64, vp, vp, vp, vp, vp, vp, vp]
    lib.elector_split_bounds.restype = c.c_int
    lib.elector_split_run.argtypes = [vp, c.c_int64] + [vp] * 7 + [c.c_double, vp, vp, vp, c.c_int64, vp, vp, vp, vp, c.c_int64, vp, c.c_int64, vp, c.c_int64, vp]
    lib.elector_split_run.restype = c.c_int
    lib.elector_reads_run.argtypes = [vp, c.c_int64] + [vp] * 7 + [c.c_double] + [vp] * 9 + [c.c_int64, vp, vp]
    lib.elector_reads_run.restype = c.c_int
    lib.elector_reads_pipeline_run.argtypes = [vp, vp]
    lib.elector_reads_pipeline_run.restype = c.c_int
    lib.elector_last_reads_ms.argtypes = [vp, c.POINTER(c.c_float), c.POINTER(c.c_float), c.POINTER(c.c_float)]
    lib.elector_last_reads_ms.restype = c.c_int
    lib.elector_last_stretches.argtypes = [vp, c.c_int64, vp]
    lib.elector_last_stretches.restype = c.c_int
    rep_tail = [c.c_int, c.c_int, c.c_double, c.c_int, c.c_int, c.c_char_p, c.c_char_p, c.c_char_p, c.c_char_p, vp, vp, c.c_int64, vp, c.c_int64]
    lib.elector_report_write.argtypes = [c.c_int64, vp, vp, vp, vp, vp, vp, vp] + rep_tail
    lib.elector_report_write.restype = c.c_int
    lib.elector_report_run.argtypes = [vp, c.c_int64, vp, vp, vp, vp, vp, vp] + rep_tail
    lib.elector_report_run.restype = c.c_int
    lib.elector_sort_fasta.argtypes = [c.c_char_p, c.c_char_p, vp]
    lib.elector_sort_fasta.restype = c.c_int
    lib.elector_duplicate_reads.argtypes = [c.c_char_p] * 5 + [vp]
    lib.elector_duplicate_reads.restype = c.c_int
    lib.elector_tally_sum_device.argtypes = [vp, c.c_int64, vp, vp]
    lib.elector_tally_sum_device.restype = c.c_int
    lib.elector_last_phase_ms.argtypes = [vp, c.POINTER(c.c_float), c.POINTER(c.c_float)]
    lib.elector_last_phase_ms.restype = c.c_int
    lib.elector_last_kernel_ms.argtypes = [vp, c.POINTER(c.c_float), c.POINTER(c.c_int)]
    lib.elector_last_kernel_ms.restype = c.c_int
    lib.elector_event_record.argtypes = [vp, c.c_int]
    lib.elector_event_record.restype = c.c_int
    lib.elector_event_elapsed_ms.argtypes = [vp, c.POINTER(c.c_float)]
    lib.elector_event_elapsed_ms.restype = c.c_int
    lib.elector_int32_peak.argtypes = [vp, c.POINTER(c.c_double), c.POINTER(c.c_double)]
    lib.elector_int32_peak.restype = c.c_int
    _LIB = lib
    return lib
