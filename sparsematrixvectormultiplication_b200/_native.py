"""ctypes binding of ``libspmv_b200.so`` -- the C-ABI declared in ``include/*.h``.

The library is built IN-TREE by ``__graft_entry__.build()`` / ``make -C csrc``.  There is no
Python, PyTorch or CPU fallback for the product: if the library is missing, importing anything that
needs it raises ``NativeLibraryMissing``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
# SPMV_B200_LIB: another build of the SAME library (tools/ab_variants.py compares compile-time variants on one box)
LIB_PATH = Path(os.environ.get("SPMV_B200_LIB") or PKG_DIR / "libspmv_b200.so")
HACK_SIZE = 32

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)
c_ll_p = C.POINTER(C.c_longlong)


class NativeLibraryMissing(RuntimeError):
    pass


class SpmvError(RuntimeError):
    """A C-ABI call returned a negative status."""

    def __init__(self, code: int, message: str):
        super().__init__(f"spmv_b200 error {code}: {message}")
        self.code = code


# ---- structs of the drop-in host API (same field order as the reference headers) ---------------
class PreMatrixStruct(C.Structure):  # include/matrix_parser.h  <- reference libs/matrix_parser.h:6-14
    _fields_ = [("M", C.c_int), ("N", C.c_int), ("nz", C.c_int), ("I", c_int_p), ("J", c_int_p),
                ("val", c_dbl_p), ("type", C.c_char * 4)]


class CSRMatrixStruct(C.Structure):  # include/csr_matrix.h  <- reference libs/csr_matrix.h:8-16
    _fields_ = [("M", C.c_int), ("N", C.c_int), ("nz", C.c_int), ("row_ptr", c_int_p),
                ("col_idx", c_int_p), ("values", c_dbl_p), ("type", C.c_char * 4)]


class ELLPACKBlockStruct(C.Structure):  # include/hll_matrix.h  <- reference libs/hll_matrix.h:15-21
    _fields_ = [("M", C.c_int), ("N", C.c_int), ("MAXNZ", C.c_int), ("JA", c_int_p), ("AS", c_dbl_p)]


class HLLMatrixStruct(C.Structure):  # reference libs/hll_matrix.h:24-27
    _fields_ = [("num_blocks", C.c_int), ("blocks", C.POINTER(ELLPACKBlockStruct))]


class DiffMetricsStruct(C.Structure):  # reference libs/performance_calculate.h:33-37
    _fields_ = [("mean_abs_err", C.c_double), ("mean_rel_err", C.c_double), ("significant_diffs", C.c_int)]


class CsrInfo(C.Structure):  # include/spmv_b200.h spmv_b200_csr_info_t
    _fields_ = [("M", C.c_int), ("N", C.c_int), ("nnz", C.c_longlong), ("num_tiles", C.c_int),
                ("num_long_rows", C.c_int), ("num_fragments", C.c_int), ("threads_per_row", C.c_int),
                ("tile_items", C.c_int), ("long_threshold", C.c_int), ("algorithmic_bytes", C.c_longlong),
                ("max_row_nnz", C.c_int), ("auto_algo", C.c_int), ("row_batch", C.c_int), ("fused_batch", C.c_int),
                ("flat_batch", C.c_int), ("flat_chunks", C.c_int), ("image_bytes", C.c_longlong), ("image_form", C.c_int),
                ("image_index_bytes", C.c_int), ("image_device_bytes", C.c_longlong),
                ("image_value_bytes", C.c_int), ("image_patterns", C.c_int),
                ("image_windows", C.c_int)]


class HllInfo(C.Structure):  # include/spmv_b200.h spmv_b200_hll_info_t
    _fields_ = [("M", C.c_int), ("N", C.c_int), ("num_hacks", C.c_int), ("max_maxnz", C.c_int),
                ("slots", C.c_longlong), ("nnz_reference_slots", C.c_longlong),
                ("algorithmic_bytes", C.c_longlong), ("auto_kernel", C.c_int), ("row_batch", C.c_int),
                ("fused_batch", C.c_int), ("flat_batch", C.c_int), ("flat_chunks", C.c_int)]


class Peers(C.Structure):  # include/spmv_b200.h spmv_b200_peers_t
    _fields_ = [("count", C.c_int), ("dst", C.c_void_p * 7), ("lo", C.c_int * 7), ("hi", C.c_int * 7)]


class Mail(C.Structure):  # include/spmv_b200.h spmv_b200_mail_t
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("iteration", C.c_ulonglong), ("box", C.c_void_p * 8),
                ("counter", C.c_void_p), ("status", C.c_void_p)]


class Async(C.Structure):  # include/spmv_b200.h spmv_b200_async_t
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("iteration", C.c_ulonglong), ("box", C.c_void_p * 8),
                ("num_recv", C.c_int), ("recv_from", C.c_int * 7), ("send_to", C.c_int * 7),
                ("counter", C.c_void_p), ("bcounter", C.c_void_p), ("status", C.c_void_p)]


class MultiInfo(C.Structure):  # include/spmv_b200.h spmv_b200_multi_info_t
    _fields_ = [("ngpus", C.c_int), ("format", C.c_int), ("M", C.c_longlong), ("N", C.c_longlong), ("nnz", C.c_longlong),
                ("stride", C.c_longlong), ("fused_ok", C.c_int), ("row_begin", C.c_longlong * 8), ("row_end", C.c_longlong * 8),
                ("nnz_part", C.c_longlong * 8), ("halo_doubles", C.c_longlong * 8)]


MAILBOX_BYTES = 2 * 8 * 16
ASYNC_MAILBOX_BYTES = 4 * 8 * 16 + 8 * 8

_V = C.c_void_p
_I = C.c_int
_LL = C.c_longlong
_ULL = C.c_ulonglong
_D = C.c_double

# name -> (restype, argtypes).  Every symbol that include/*.h declares is listed here;
# tests/test_abi_symbols.py checks the headers against the built library.
SIGNATURES = {
    # ---- spmv_b200.h ----
    "spmv_b200_last_error": (C.c_char_p, []),
    "spmv_b200_clear_error": (None, []),
    "spmv_b200_version": (_I, []),
    "spmv_b200_device_count": (_I, [c_int_p]),
    "spmv_b200_device_info": (_I, [C.c_char_p, _I, c_int_p, c_ll_p, c_ll_p]),
    "spmv_b200_csr_upload": (_I, [_I, _I, _LL, _V, _V, _V, C.POINTER(_V)]),
    "spmv_b200_csr_wrap_device": (_I, [_I, _I, _LL, _V, _V, _V, _V, C.POINTER(_V)]),
    "spmv_b200_csr_replan": (_I, [_V, _I, _I, _I, _V]),
    "spmv_b200_csr_info": (_I, [_V, C.POINTER(CsrInfo)]),
    "spmv_b200_csr_device_arrays": (_I, [_V, C.POINTER(_V), C.POINTER(_V), C.POINTER(_V)]),
    "spmv_b200_csr_download": (_I, [_V, _V, _V, _V]),
    "spmv_b200_csr_spmv": (_I, [_V, _V, _V, _I, _I, _V]),
    "spmv_b200_csr_spmv_host": (_I, [_V, _V, _V, _I, _I]),
    "spmv_b200_csr_from_coo": (_I, [_I, _I, _LL, _V, _V, _V, C.POINTER(_V)]),
    "spmv_b200_csr_from_coo_device": (_I, [_I, _I, _LL, _V, _V, _V, _V, C.POINTER(_V)]),
    "spmv_b200_csr_spmv_rows": (_I, [_V, _I, _I, _V, _V, _V]),
    "spmv_b200_csr_set_image": (_I, [_V, _I, _V]),
    "spmv_b200_csr_partials_count": (_I, [_V]),
    "spmv_b200_csr_remap_columns": (_I, [_V, _I, c_ll_p, _LL, _V]),
    "spmv_b200_csr_interior_rows": (_I, [_V, _LL, _LL, c_int_p, c_int_p, _V]),
    "spmv_b200_csr_spmv_fused": (_I, [_V, _V, _V, _V, _V, C.POINTER(Peers), _V]),
    "spmv_b200_csr_spmv_fused_mail": (_I, [_V, _V, _V, _V, C.POINTER(Peers), C.POINTER(Mail), _V]),
    "spmv_b200_csr_flat_partials_count": (_I, [_V]),
    "spmv_b200_csr_spmv_fused_flat": (_I, [_V, _V, _V, _V, _V, C.POINTER(Peers), _V]),
    "spmv_b200_mail_exchange": (_I, [_V, _I, C.POINTER(Mail), _V, _V]),
    "spmv_b200_hll_flat_partials_count": (_I, [_V]),
    "spmv_b200_hll_spmv_fused_flat": (_I, [_V, _V, _V, _V, _V, C.POINTER(Peers), _V]),
    "spmv_b200_csr_spmv_fused_async": (_I, [_V, _V, _V, _V, C.POINTER(Peers), C.POINTER(Async), _V]),
    "spmv_b200_vec_sum": (_I, [_V, _I, _V, _V]),
    "spmv_b200_ipc_alloc": (_I, [_LL, C.POINTER(_V), C.c_char * 64]),
    "spmv_b200_ipc_open": (_I, [C.c_char * 64, C.POINTER(_V)]),
    "spmv_b200_ipc_close": (_I, [_V]),
    "spmv_b200_ipc_free": (_I, [_V]),
    "spmv_b200_csr_free": (None, [_V]),
    "spmv_b200_csr_spmv_raw": (_I, [_I, _LL, _V, _V, _V, _V, _V, _I, _V]),
    "spmv_b200_hll_upload": (_I, [C.POINTER(HLLMatrixStruct), _I, _I, C.POINTER(_V)]),
    "spmv_b200_hll_from_csr": (_I, [_V, _V, C.POINTER(_V)]),
    "spmv_b200_hll_info": (_I, [_V, C.POINTER(HllInfo)]),
    "spmv_b200_hll_download": (_I, [_V, C.POINTER(HLLMatrixStruct)]),
    "spmv_b200_hll_device_arrays": (_I, [_V, C.POINTER(_V), C.POINTER(_V), C.POINTER(_V)]),
    "spmv_b200_hll_spmv": (_I, [_V, _V, _V, _V]),
    "spmv_b200_hll_spmv_slice": (_I, [_V, _V, _V, _V]),
    "spmv_b200_hll_spmv_stream": (_I, [_V, _V, _V, _V]),
    "spmv_b200_hll_spmv_host": (_I, [_V, _V, _V]),
    "spmv_b200_hll_spmv_rows": (_I, [_V, _V, _V, _V]),
    "spmv_b200_csr_enable_f32": (_I, [_V, _V]),
    "spmv_b200_csr_spmv_f32": (_I, [_V, _V, _V, _I, _I, _V]),
    "spmv_b200_csr_spmv_host_f32": (_I, [_V, _V, _V]),
    "spmv_b200_hll_enable_f32": (_I, [_V, _V]),
    "spmv_b200_hll_spmv_f32": (_I, [_V, _V, _V, _V]),
    "spmv_b200_hll_spmv_host_f32": (_I, [_V, _V, _V]),
    "spmv_b200_csr_row_form_f32": (_I, [_V]),
    "spmv_b200_hll_row_form_f32": (_I, [_V]),
    "spmv_b200_hll_row_form": (_I, [_V]),
    "spmv_b200_row_forms": (_I, [_I]),
    "spmv_b200_row_form_describe": (_I, [_I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "spmv_b200_resident_cache": (_I, [_I]),
    "spmv_b200_autotune": (_I, [_I]),
    "spmv_b200_resident_drop": (None, []),
    "spmv_b200_csr_time": (_I, [_V, _V, _V, _I, _I, _I, c_dbl_p, c_dbl_p]),
    "spmv_b200_hll_time": (_I, [_V, _V, _V, _I, _I, _I, c_dbl_p, c_dbl_p]),
    "spmv_b200_hll_spmv_hacks": (_I, [_V, _I, _I, _V, _V, _V]),
    "spmv_b200_hll_free": (None, [_V]),
    "spmv_b200_csr_spmm": (_I, [_V, _I, _V, _LL, _V, _LL, _I, _V]),
    "spmv_b200_hll_spmm": (_I, [_V, _I, _V, _LL, _V, _LL, _V]),
    "spmv_b200_csr_spmm_f32": (_I, [_V, _I, _V, _LL, _V, _LL, _I, _V]),
    "spmv_b200_hll_spmm_f32": (_I, [_V, _I, _V, _LL, _V, _LL, _V]),
    "spmv_b200_csr_spmm_host": (_I, [_V, _I, _V, _LL, _V, _LL, _I]),
    "spmv_b200_hll_spmm_host": (_I, [_V, _I, _V, _LL, _V, _LL]),
    "spmv_b200_csr_spmm_host_f32": (_I, [_V, _I, _V, _LL, _V, _LL, _I]),
    "spmv_b200_hll_spmm_host_f32": (_I, [_V, _I, _V, _LL, _V, _LL]),
    "spmv_b200_hll_partials_count": (_I, [_V]),
    "spmv_b200_hll_spmv_fused": (_I, [_V, _V, _V, _V, _V, C.POINTER(Peers), _V]),
    "spmv_b200_hll_spmv_fused_mail": (_I, [_V, _V, _V, _V, C.POINTER(Peers), C.POINTER(Mail), _V]),
    "spmv_b200_synth_csr": (_I, [_I, _LL, _LL, _I, _ULL, _LL, _LL, _V, C.POINTER(_V)]),
    "spmv_b200_synth_row_offset": (_LL, [_I, _LL, _LL, _I, _LL]),
    "spmv_b200_synth_vector": (_I, [_V, _LL, _ULL, _V]),
    "spmv_b200_vec_fill": (_I, [_V, _LL, _D, _V]),
    "spmv_b200_vec_ws_doubles": (_I, []),
    "spmv_b200_vec_sumsq": (_I, [_V, _LL, _V, _V, _V]),
    "spmv_b200_vec_scale_by_inv_norm": (_I, [_V, _V, _LL, _V, _V]),
    "spmv_b200_vec_push": (_I, [_V, _LL, _I, C.POINTER(_V), _I, _V]),
    "spmv_b200_multi_init_synth": (_I, [_I, _I, _I, _LL, _LL, _I, _ULL, C.POINTER(_V)]),
    "spmv_b200_multi_init_csr": (_I, [_I, _I, _I, _I, _LL, _V, _V, _V, C.POINTER(_V)]),
    "spmv_b200_multi_info": (_I, [_V, C.POINTER(MultiInfo)]),
    "spmv_b200_multi_reset": (_I, [_V, _V]),
    "spmv_b200_multi_iterate": (_I, [_V, _I, _I, c_dbl_p, c_dbl_p]),
    "spmv_b200_multi_get_x": (_I, [_V, _V]),
    "spmv_b200_multi_spmv": (_I, [_V, _V, _V]),
    "spmv_b200_multi_free": (None, [_V]),
    # ---- matrix_parser.h ----
    "init_pre_matrix": (None, [C.POINTER(PreMatrixStruct)]),
    "free_pre_matrix": (None, [C.POINTER(PreMatrixStruct)]),
    "read_matrix_market": (_I, [C.c_char_p, C.POINTER(PreMatrixStruct)]),
    "print_pre_matrix": (None, [C.POINTER(PreMatrixStruct), C.c_bool]),
    # ---- csr_matrix.h ----
    "init_csr_matrix": (None, [C.POINTER(CSRMatrixStruct)]),
    "free_csr_matrix": (None, [C.POINTER(CSRMatrixStruct)]),
    "convert_in_csr": (_I, [C.POINTER(PreMatrixStruct), C.POINTER(CSRMatrixStruct), C.c_char_p]),
    "print_csr_matrix": (None, [C.POINTER(CSRMatrixStruct)]),
    "write_memory_stats_to_csv": (None, [C.c_char_p, _I, C.c_size_t]),
    "csr_matrix_vector_mult": (None, [_I, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p]),
    "prepare_thread_distribution": (_I, [_I, c_int_p, _I, _LL, C.POINTER(c_int_p), C.POINTER(c_int_p)]),
    "spvm_csr_parallel": (None, [c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, _I, c_int_p, c_int_p]),
    "spvm_csr_parallel_simd": (None, [c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, _I, c_int_p, c_int_p]),
    # ---- hll_matrix.h ----
    "init_hll_matrix": (None, [C.POINTER(HLLMatrixStruct)]),
    "convert_to_hll": (_I, [C.POINTER(PreMatrixStruct), C.POINTER(HLLMatrixStruct)]),
    "free_hll_matrix": (None, [C.POINTER(HLLMatrixStruct)]),
    "printHLLMatrix": (None, [C.POINTER(HLLMatrixStruct)]),
    "spmv_hll_serial": (None, [_I, C.POINTER(ELLPACKBlockStruct), c_dbl_p, c_dbl_p]),
    "prepare_thread_distribution_hll": (_I, [C.POINTER(HLLMatrixStruct), _I, C.POINTER(c_int_p), C.POINTER(c_int_p)]),
    "spmv_hll": (None, [C.POINTER(ELLPACKBlockStruct), c_dbl_p, c_dbl_p, _I, c_int_p, c_int_p]),
    "spmv_hll_simd": (None, [C.POINTER(ELLPACKBlockStruct), c_dbl_p, c_dbl_p, _I, c_int_p, c_int_p]),
    # ---- performance_calculate.h ----
    "computeDifferenceMetrics": (DiffMetricsStruct, [c_dbl_p, c_dbl_p, _I, _D, _D, C.c_bool]),
    "initialize_metrics": (None, []),
    "cleanup_metrics": (None, []),
    "get_metric_value": (_D, [_I]),
    "get_relative_error": (_D, [_I]),
    "get_absolute_error": (_D, [_I]),
    "update_medium_metric": (None, [_I, _D]),
    "reset_medium_time_metrics": (None, []),
    "computeAverageErrors": (DiffMetricsStruct, [_I]),
    "accumulateErrors": (None, [C.POINTER(DiffMetricsStruct), _I]),
    "calculate_flops": (_D, [_I, _D]),
    "print_flops": (None, [_D]),
    "get_metric_min": (_D, [_I]),
    "get_metric_max": (_D, [_I]),
    "get_metric_median": (_D, [_I]),
    "calculate_csr_bytes": (_LL, [_I, _I, _LL, _I]),
    "calculate_hll_bytes": (_LL, [_I, _I, _LL, _I, _I]),
    "calculate_bandwidth_gbs": (_D, [_LL, _D]),
    "calculate_roofline_fraction": (_D, [_LL, _D, _D]),
    # ---- utility.h ----
    "init_vector_at_one": (None, [c_dbl_p, _I]),
    "swap": (None, [c_int_p, c_int_p]),
    "swap_double": (None, [c_dbl_p, c_dbl_p]),
    "partition": (C.c_size_t, [c_int_p, c_dbl_p, C.c_size_t, C.c_size_t]),
    "sort_row": (None, [c_int_p, c_dbl_p, C.c_size_t, C.c_size_t]),
    "clear_cache": (None, [C.c_size_t]),
    "process_matrix_file": (_I, [C.c_char_p, C.POINTER(PreMatrixStruct)]),
    "create_directory": (None, [C.c_char_p]),
    "write_results_to_csv": (None, [C.c_char_p, _I, _I, _I, _I] + [_D] * 6 + [DiffMetricsStruct] * 4 + [_D] * 14 + [C.c_char_p]),
    # ---- mmio.h ----
    "mm_read_banner": (_I, [_V, C.POINTER(C.c_char * 4)]),
    "mm_read_mtx_crd_size": (_I, [_V, c_int_p, c_int_p, c_int_p]),
    "mm_write_banner": (_I, [_V, C.c_char * 4]),
    "mm_write_mtx_crd_size": (_I, [_V, _I, _I, _I]),
    "mm_is_valid": (_I, [C.c_char * 4]),
    "mm_typecode_to_str": (_V, [C.c_char * 4]),
}

_lib = None


def build(verbose: bool = False) -> Path:
    """Compile libspmv_b200.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", str(PKG_DIR / "csrc"), "-j8"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libspmv_b200.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return LIB_PATH


def lib() -> C.CDLL:
    """The loaded library.  Raises NativeLibraryMissing -- loudly -- when it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise NativeLibraryMissing(
                f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                f"or `make -C {PKG_DIR / 'csrc'}`. There is no Python/CPU fallback for the SpMV path.")
        handle = C.CDLL(str(LIB_PATH))
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def clear_error() -> None:
    lib().spmv_b200_clear_error()


def last_error() -> str:
    return lib().spmv_b200_last_error().decode("utf-8", "replace")


def check(code: int) -> None:
    if code != 0:
        raise SpmvError(code, last_error())
