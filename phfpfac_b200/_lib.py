"""ctypes loader for phfpfac_b200/_build/libpfac_b200.so (the C ABI of include/pfac_b200.h).

The library is the product: there is no Python or CPU implementation of the scan behind it.
If the shared object is missing, importing fails loudly with the build command.
"""
import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
# PFAC_B200_LIB: another build of the same library (development: kernel variants side by side)
LIB_PATH = os.environ.get("PFAC_B200_LIB") or os.path.join(PKG_DIR, "_build", "libpfac_b200.so")

# every symbol include/pfac_b200.h declares
ABI_SYMBOLS = [
    "pfac_last_error", "pfac_abi_version",
    "pfac_tables_build_file", "pfac_tables_build_mem", "pfac_tables_build_file_ext", "pfac_tables_build_mem_ext",
    "pfac_tables_build_file_rules", "pfac_tables_build_mem_rules", "pfac_tables_case_rules", "pfac_pattern_file_hash_rules",
    "pfac_tables_from_arrays", "pfac_tables_save", "pfac_tables_load", "pfac_tables_destroy",
    "pfac_tables_source_hash", "pfac_pattern_file_hash",
    "pfac_tables_n_parts", "pfac_tables_n_patterns", "pfac_tables_max_pat_len", "pfac_tables_width",
    "pfac_tables_flags", "pfac_tables_part_info", "pfac_tables_s0", "pfac_tables_r", "pfac_tables_HT", "pfac_tables_val",
    "pfac_tables_idmap", "pfac_tables_lookup", "pfac_tables_pattern_lengths", "pfac_tables_derive_check",
    "pfac_tables_filter_profile",
    "pfac_device_count", "pfac_ctx_create", "pfac_ctx_destroy", "pfac_ctx_device",
    "pfac_scan_device", "pfac_scan_device_sync", "pfac_scan_batch_device", "pfac_scan_batch_device_sync",
    "pfac_flows_create", "pfac_flows_destroy", "pfac_flows_reset", "pfac_flows_position", "pfac_scan_flows_device_sync",
    "pfac_scan_host", "pfac_host_alloc", "pfac_host_free", "pfac_host_register", "pfac_host_unregister",
    "pfac_ctx_last_scan_info", "pfac_ctx_derived_info", "pfac_ctx_set_timing", "pfac_ctx_kernel_time",
    "pfac_job_create", "pfac_job_destroy", "pfac_job_run", "pfac_job_run_file", "pfac_job_n_segments", "pfac_job_segment",
    "pfac_job_last_timing", "pfac_job_plan",
    "pfac_write_begin", "pfac_write_records", "pfac_write_end", "pfac_format_records",
    "pfac_sidecar_begin", "pfac_sidecar_records", "pfac_sidecar_end", "pfac_sidecar_read",
]

PFAC_OK = 0
PFAC_ERR_ARG = -5
PFAC_ERR_OUTPUT_FULL = -8
PFAC_ERR_NO_DEVICE = -9
PFAC_ERR_LIMIT = -10


class PfacError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pfac error {code}: {msg}")
        self.code = code


_i32p = C.POINTER(C.c_int32)
_vp = C.c_void_p


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make lib` (or __graft_entry__.build()). "
            "phfpfac_b200 has no fallback implementation.")
    lib = C.CDLL(LIB_PATH)
    lib.pfac_last_error.restype = C.c_char_p
    lib.pfac_tables_build_file.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(_vp)]
    lib.pfac_tables_build_mem.argtypes = [_vp, C.c_size_t, C.c_int, C.c_int, C.POINTER(_vp)]
    lib.pfac_tables_build_file_ext.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_uint, C.POINTER(_vp)]
    lib.pfac_tables_build_mem_ext.argtypes = [_vp, C.c_size_t, C.c_int, C.c_int, C.c_uint, C.POINTER(_vp)]
    lib.pfac_tables_build_file_rules.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_uint, _vp, C.c_uint32, C.POINTER(_vp)]
    lib.pfac_tables_build_mem_rules.argtypes = [_vp, C.c_size_t, C.c_int, C.c_int, C.c_uint, _vp, C.c_uint32, C.POINTER(_vp)]
    lib.pfac_tables_case_rules.argtypes = [_vp, _vp, C.c_uint32]
    lib.pfac_pattern_file_hash_rules.argtypes = [C.c_char_p, C.c_uint, _vp, C.c_uint32, C.POINTER(C.c_uint64)]
    lib.pfac_tables_save.argtypes = [_vp, C.c_char_p]
    lib.pfac_tables_source_hash.argtypes = [_vp]
    lib.pfac_tables_source_hash.restype = C.c_uint64
    lib.pfac_pattern_file_hash.argtypes = [C.c_char_p, C.c_uint, C.POINTER(C.c_uint64)]
    lib.pfac_tables_load.argtypes = [C.c_char_p, C.POINTER(_vp)]
    lib.pfac_tables_from_arrays.argtypes = [_vp, _vp, C.c_int32, _vp, _vp, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_int32, _vp, C.c_int32, C.POINTER(_vp)]
    lib.pfac_tables_destroy.argtypes = [_vp]
    lib.pfac_tables_destroy.restype = None
    for n in ("pfac_tables_n_parts", "pfac_tables_n_patterns", "pfac_tables_max_pat_len", "pfac_tables_width"):
        getattr(lib, n).argtypes = [_vp]
    lib.pfac_tables_flags.argtypes = [_vp]
    lib.pfac_tables_flags.restype = C.c_uint
    lib.pfac_tables_part_info.argtypes = [_vp, C.c_int, _i32p]
    for n in ("pfac_tables_s0", "pfac_tables_r", "pfac_tables_HT", "pfac_tables_val", "pfac_tables_idmap"):
        getattr(lib, n).argtypes = [_vp, C.c_int]
        getattr(lib, n).restype = _i32p
    lib.pfac_tables_derive_check.argtypes = [_vp, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
    lib.pfac_tables_filter_profile.argtypes = [_vp, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, _vp, C.c_uint64,
                                               C.POINTER(C.c_uint64)]
    lib.pfac_tables_lookup.argtypes = [_vp, C.c_int, C.c_int32, C.c_int32]
    lib.pfac_tables_lookup.restype = C.c_int32
    lib.pfac_tables_pattern_lengths.argtypes = [_vp, C.c_int, _vp, C.c_int32, C.POINTER(C.c_int32)]
    lib.pfac_device_count.argtypes = [C.POINTER(C.c_int)]
    lib.pfac_ctx_create.argtypes = [C.c_int, _vp, C.c_int, C.c_int, C.c_size_t, C.POINTER(_vp)]
    lib.pfac_ctx_destroy.argtypes = [_vp]
    lib.pfac_ctx_destroy.restype = None
    lib.pfac_ctx_device.argtypes = [_vp]
    lib.pfac_scan_device.argtypes = [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _vp, C.c_uint64, _vp, _vp]
    lib.pfac_scan_device_sync.argtypes = [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _vp, C.c_uint64,
                                          C.POINTER(C.c_uint64), _vp]
    lib.pfac_scan_batch_device.argtypes = [_vp, _vp, _vp, C.c_uint32, _vp, C.c_uint64, _vp, _vp, _vp]
    lib.pfac_scan_batch_device_sync.argtypes = [_vp, _vp, _vp, C.c_uint32, _vp, C.c_uint64, _vp,
                                                C.POINTER(C.c_uint64), _vp]
    lib.pfac_flows_create.argtypes = [_vp, C.c_uint32, C.POINTER(_vp)]
    lib.pfac_flows_destroy.argtypes = [_vp]
    lib.pfac_flows_destroy.restype = None
    lib.pfac_flows_reset.argtypes = [_vp, C.c_uint32]
    lib.pfac_flows_position.argtypes = [_vp, C.c_uint32, C.POINTER(C.c_uint64)]
    lib.pfac_scan_flows_device_sync.argtypes = [_vp, _vp, _vp, _vp, C.c_uint32, _vp, C.c_uint64, _vp, _vp,
                                                C.POINTER(C.c_uint64), _vp]
    lib.pfac_scan_host.argtypes = [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _vp, C.c_uint64,
                                   C.POINTER(C.c_uint64)]
    lib.pfac_host_alloc.argtypes = [C.POINTER(_vp), C.c_size_t]
    lib.pfac_host_free.argtypes = [_vp]
    lib.pfac_host_free.restype = None
    lib.pfac_host_register.argtypes = [_vp, C.c_size_t, C.c_int]
    lib.pfac_host_unregister.argtypes = [_vp]
    lib.pfac_host_unregister.restype = None
    lib.pfac_ctx_last_scan_info.argtypes = [_vp, C.POINTER(C.c_uint64)]
    lib.pfac_ctx_set_timing.argtypes = [_vp, C.c_int]
    lib.pfac_ctx_kernel_time.argtypes = [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    lib.pfac_ctx_derived_info.argtypes = [_vp, C.POINTER(C.c_uint64)]
    lib.pfac_job_create.argtypes = [_vp, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_size_t, C.POINTER(_vp)]
    lib.pfac_job_destroy.argtypes = [_vp]
    lib.pfac_job_destroy.restype = None
    lib.pfac_job_run.argtypes = [_vp, _vp, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.pfac_job_run_file.argtypes = [_vp, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.pfac_job_n_segments.argtypes = [_vp]
    lib.pfac_job_segment.argtypes = [_vp, C.c_int, C.POINTER(C.c_uint64), C.POINTER(_vp), C.POINTER(C.c_uint64)]
    lib.pfac_job_plan.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                  C.POINTER(C.c_uint64)]
    lib.pfac_job_last_timing.argtypes = [_vp, C.POINTER(C.c_double)]
    lib.pfac_write_begin.argtypes = [C.c_char_p, C.POINTER(_vp)]
    lib.pfac_write_records.argtypes = [_vp, C.c_uint64, _vp, C.c_uint64]
    lib.pfac_write_end.argtypes = [_vp]
    lib.pfac_format_records.argtypes = [C.c_uint64, _vp, C.c_uint64, _vp, C.c_size_t]
    lib.pfac_format_records.restype = C.c_size_t
    lib.pfac_sidecar_begin.argtypes = [C.c_char_p, C.POINTER(_vp)]
    lib.pfac_sidecar_records.argtypes = [_vp, C.c_uint64, _vp, C.c_uint64]
    lib.pfac_sidecar_end.argtypes = [_vp]
    lib.pfac_sidecar_read.argtypes = [C.c_char_p, _vp, _vp, C.c_uint64, C.POINTER(C.c_uint64)]
    return lib


lib = _load()


def check(rc):
    if rc != PFAC_OK:
        raise PfacError(rc, lib.pfac_last_error().decode(errors="replace"))
    return rc
