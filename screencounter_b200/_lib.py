"""ctypes loader for the C-ABI library (include/scg.h).  No torch types cross this boundary."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libscg.so")

_lib = None


class ScgSource(C.Structure):
    _fields_ = [("path", C.c_char_p), ("data", C.c_void_p), ("size", C.c_size_t)]


class ScgSynthSpec(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("first_read", C.c_longlong),
        ("n_reads", C.c_longlong),
        ("read_len", C.c_int),
        ("constant", C.c_char_p),
        ("n_pools", C.c_int),
        ("pools", C.POINTER(C.c_char_p) * 2),
        ("n_choices", C.c_int * 2),
        ("paired_rows", C.c_int),
        ("strand", C.c_int),
        ("construct_permille", C.c_int),
        ("sub_per_10k", C.c_int),
        ("n_per_10k", C.c_int),
        ("random_space", C.c_longlong),
    ]


def lib():
    """The loaded library.  There is no fallback: a missing build is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "screencounter_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C screencounter_b200/csrc`. There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.scg_last_error.restype = C.c_char_p
        L.scg_last_error.argtypes = [C.c_void_p]
        L.scg_version.restype = C.c_char_p
        L.scg_timing_json.restype = C.c_char_p
        L.scg_timing_json.argtypes = [C.c_void_p]
        L.scg_kernel_launches.restype = C.c_longlong
        L.scg_kernel_launches.argtypes = [C.c_void_p]
        L.scg_ctx_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        L.scg_ctx_create_multi.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int]
        L.scg_ctx_devices.argtypes = [C.c_void_p]
        L.scg_result_columns.argtypes = [C.c_void_p]
        L.scg_result_copy_matrix.argtypes = [C.c_void_p, C.c_void_p]
        L.scg_bgzf_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.scg_bgzf_inflate.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_double)]
        L.scg_ctx_destroy.argtypes = [C.c_void_p]
        L.scg_ctx_destroy.restype = None
        L.scg_result_rows.restype = C.c_size_t
        L.scg_result_rows.argtypes = [C.c_void_p]
        L.scg_result_reads.restype = C.c_size_t
        L.scg_result_reads.argtypes = [C.c_void_p]
        L.scg_result_width.argtypes = [C.c_void_p]
        L.scg_result_trace_width.argtypes = [C.c_void_p]
        L.scg_result_copy_table.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.scg_result_copy_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.scg_result_free.argtypes = [C.c_void_p]
        L.scg_result_free.restype = None
        L.scg_reads_count.restype = C.c_longlong
        L.scg_reads_count.argtypes = [C.c_void_p]
        L.scg_reads_device_bytes.restype = C.c_longlong
        L.scg_reads_device_bytes.argtypes = [C.c_void_p]
        L.scg_reads_free.argtypes = [C.c_void_p]
        L.scg_reads_free.restype = None
        L.scg_table_rows.restype = C.c_longlong
        L.scg_table_rows.argtypes = [C.c_void_p]
        L.scg_table_key_len.argtypes = [C.c_void_p]
        L.scg_table_key_words.argtypes = [C.c_void_p]
        L.scg_table_keys.restype = C.c_void_p
        L.scg_table_keys.argtypes = [C.c_void_p]
        L.scg_table_counts.restype = C.c_void_p
        L.scg_table_counts.argtypes = [C.c_void_p]
        L.scg_table_free.restype = None
        L.scg_table_free.argtypes = [C.c_void_p]
        L.scg_table_from_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(C.c_void_p)]
        L.scg_table_merge.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.scg_table_render.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.scg_plan_free.argtypes = [C.c_void_p]
        L.scg_plan_free.restype = None
        L.scg_plan_kernel.restype = C.c_char_p
        L.scg_plan_kernel.argtypes = [C.c_void_p]
        _lib = L
    return _lib


# every symbol include/scg.h declares (checked by tests/test_host.py::test_abi_exports_every_declared_symbol)
EXPORTS = [
    "scg_ctx_create", "scg_ctx_create_multi", "scg_ctx_devices", "scg_ctx_destroy", "scg_last_error", "scg_version", "scg_timing_json", "scg_kernel_launches",
    "scg_result_rows", "scg_result_width", "scg_result_reads", "scg_result_copy_table", "scg_result_trace_width",
    "scg_result_copy_trace", "scg_result_free",
    "scg_count_single", "scg_count_random", "scg_count_combo_single", "scg_count_dual_single_end", "scg_count_dual",
    "scg_count_combo_paired", "scg_count_single_paired", "scg_match_barcodes",
    "scg_count_single_many", "scg_count_combo_many", "scg_count_random_many", "scg_result_columns", "scg_result_copy_matrix",
    "scg_bgzf_compress", "scg_bgzf_inflate",
    "scg_reads_from_source", "scg_reads_count", "scg_reads_device_bytes", "scg_reads_free",
    "scg_reads_synthesize", "scg_synth_fastq",
    "scg_single_plan_create", "scg_single_plan_run", "scg_plan_free", "scg_plan_kernel",
    "scg_dual_plan_create", "scg_dual_plan_run", "scg_combo_plan_create", "scg_combo_plan_run",
    "scg_random_plan_create", "scg_random_plan_run", "scg_plan_reset", "scg_plan_harvest",
    "scg_plan_sorted_table", "scg_plan_dense_tally", "scg_table_rows", "scg_table_key_len", "scg_table_key_words", "scg_table_keys", "scg_table_counts",
    "scg_table_from_device", "scg_table_merge", "scg_table_render", "scg_table_free",
    "scg_host_pack_roundtrip", "scg_jit_selftest", "scg_jit_selftest_uniform", "scg_jit_selftest_handler",
    "scg_device_alloc", "scg_device_free", "scg_device_zero", "scg_device_to_host", "scg_synchronize",
    "scg_host_alloc", "scg_host_free", "scg_search_segmented",
]
