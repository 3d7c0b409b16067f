"""ctypes binding of librecoup_b200.so (include/recoup_b200.h).

The library is the product; this module only declares its C signatures.  There is no fallback:
if the shared object is missing the import fails, and if no sm_100 GPU can be bound every compute
call raises `RecoupError` (RCP_ERR_NOGPU).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RCP_LIB_PATH") or os.path.join(_HERE, "librecoup_b200.so")     # RCP_LIB_PATH: A/B builds

RCP_OK, RCP_ERR_CUDA, RCP_ERR_ARG, RCP_ERR_HANDLE, RCP_ERR_NOGPU, RCP_ERR_UNSUPPORTED, RCP_ERR_DATA = range(7)
MEM_HOST, MEM_DEVICE = 0, 1
STRAND_ANY = 2
WHERE = {"whole": 0, "center": 1, "upstream": 2, "downstream": 3}
STAT = {"mean": 0, "median": 1}
INTERP = {"auto": 0, "spline": 1, "linear": 2, "neighborhood": 3}
SAMPLE_KIND = {"Rejection": 0, "Rounding": 1}
COVERAGE_PATH = {"auto": 0, "index": 1, "buckets": 2, "blocks": 3, "split": 4}
VALUE_INT32, VALUE_FLOAT32 = 0, 1

_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_i8p = C.POINTER(C.c_int8)
_u8p = C.POINTER(C.c_uint8)
_f64p = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p   # used for arrays that may live on the host or on the device

# name -> (restype, argtypes); exactly the declarations of include/recoup_b200.h
SIGNATURES = {
    "rcp_last_error": (C.c_char_p, []),
    "rcp_abi_version": (C.c_int, []),
    "rcp_init": (C.c_int, [C.c_int]),
    "rcp_shutdown": (C.c_int, []),
    "rcp_device_info": (C.c_int, [_ip, _ip, _ip, _ip, _i64p]),
    "rcp_stream": (C.c_void_p, []),
    "rcp_sync": (C.c_int, []),
    "rcp_launch_count": (C.c_int64, [C.c_int]),
    "rcp_set_coverage_path": (C.c_int, [C.c_int]),
    "rcp_set_deferred_validation": (C.c_int, [C.c_int]),
    "rcp_host_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p)]),
    "rcp_host_free": (C.c_int, [C.c_void_p]),
    "rcp_timing_enable": (C.c_int, [C.c_int]),
    "rcp_timing_read": (C.c_int, [C.c_int, C.c_int, _f64p, _i64p]),
    "rcp_timing_stage_name": (C.c_char_p, [C.c_int]),
    "rcp_r_sample": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, _ip]),
    "rcp_r_rank_table": (C.c_int, [C.c_int, C.c_int, C.c_int, _ip]),
    "rcp_reads_load": (C.c_int, [C.c_int64, _vp, _vp, _vp, _vp, C.c_int, _i64p, C.c_int, C.c_int, _ip]),
    "rcp_matrix_col_profile": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int,
                                         _vp, _vp]),
    "rcp_matrix_group_col_profile": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int, C.c_int, C.c_int,
                                               C.c_int, _vp, _vp]),
    "rcp_matrix_row_stat": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, _vp]),
    "rcp_order": (C.c_int, [_vp, C.c_int64, C.c_int, C.c_int, _vp, _i64p]),
    "rcp_matrix_quantile": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int, C.c_int, _vp]),
    "rcp_reads_width_quantile": (C.c_int, [C.c_int64, _vp, _vp, C.c_double, C.c_int, _f64p, _i64p]),
    "rcp_r_sample_sorted": (C.c_int, [C.c_int, C.c_int, C.c_int, _i64p, _i64p, _vp]),
    "rcp_reads_load_select": (C.c_int, [C.c_int64, _vp, _vp, _vp, _vp, C.c_double, C.c_int64, _vp, C.c_int,
                                        _i64p, C.c_int, C.c_int, _i64p, _ip]),
    "rcp_coverage_path_info": (C.c_int, [C.c_int, _ip, _i64p]),
    "rcp_rows_put": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_int64, _vp]),
    "rcp_reads_route_count": (C.c_int, [C.c_int64, _vp, _vp, _vp, C.c_int, C.c_int, _i32p, _i64p]),
    "rcp_reads_route_pack": (C.c_int, [C.c_int64, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _i32p, _i64p, _vp, _vp, _vp,
                                       _vp]),
    "rcp_reads_load_width": (C.c_int, [C.c_int64, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp, C.c_int, _i64p,
                                       C.c_int, C.c_int, _ip]),
    "rcp_reads_load_rle": (C.c_int, [C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int, _i64p,
                                     C.c_int, C.c_int, _ip]),
    "rcp_bgzf_size": (C.c_int, [_vp, C.c_int64, _i64p, _i64p]),
    "rcp_bgzf_inflate": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int]),
    "rcp_bam_index": (C.c_int, [_vp, C.c_int64, _i64p, _vp, C.c_int64]),
    "rcp_bam_decode": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, _i64p, C.c_int, C.c_int, _ip, _i64p]),
    "rcp_bam_decode_param": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, _i64p, C.c_int, C.c_int, _i32p,
                                       C.c_int, C.c_int, C.c_int, _i32p, _i32p, _i32p, C.c_int, C.c_char_p, _i32p,
                                       _i32p, _i64p, C.POINTER(C.c_char_p), _ip, _i64p]),
    "rcp_bed_decode": (C.c_int, [_vp, C.c_int64, C.c_int, C.POINTER(C.c_char_p), C.c_int, _ip, _i64p]),
    "rcp_decoded_fetch": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, C.c_int64]),
    "rcp_decoded_free": (C.c_int, [C.c_int]),
    "rcp_reads_load_decoded": (C.c_int, [C.c_int, C.c_int, _i64p, C.c_int, _ip]),
    "rcp_decoded_width_quantile": (C.c_int, [C.c_int, C.c_double, _f64p, _i64p]),
    "rcp_reads_load_decoded_select": (C.c_int, [C.c_int, C.c_double, C.c_int64, _vp, C.c_int, _i64p, C.c_int,
                                                _i64p, _ip]),
    "rcp_reads_info": (C.c_int, [C.c_int, _i64p, _ip, _i64p]),
    "rcp_reads_free": (C.c_int, [C.c_int]),
    "rcp_coverage": (C.c_int, [C.c_int, C.c_int64, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _ip]),
    "rcp_coverage_list": (C.c_int, [C.c_int, C.c_int64, _i64p, _vp, _vp, _vp, _vp, C.c_int, C.c_int,
                                    C.c_int, _ip]),
    "rcp_coverage_concat3": (C.c_int, [C.c_int, C.c_int, C.c_int, _ip]),
    "rcp_coverage_set_scale": (C.c_int, [C.c_int, C.c_double]),
    "rcp_coverage_info": (C.c_int, [C.c_int, _i64p, _i64p, _i64p, _f64p]),
    "rcp_coverage_lengths": (C.c_int, [C.c_int, _i32p]),
    "rcp_coverage_fetch": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _i32p, C.c_int64]),
    "rcp_coverage_rle": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _i64p, _i32p, _i32p, C.c_int64]),
    "rcp_coverage_free": (C.c_int, [C.c_int]),
    "rcp_bigwig_load": (C.c_int, [_vp, C.c_int64, C.c_int, _ip]),
    "rcp_signal_info": (C.c_int, [C.c_int, _ip, _i64p, _i64p]),
    "rcp_signal_chroms": (C.c_int, [C.c_int, C.c_char_p, _i64p]),
    "rcp_signal_fetch": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, C.c_int64]),
    "rcp_signal_free": (C.c_int, [C.c_int]),
    "rcp_signal_coverage": (C.c_int, [C.c_int, C.c_int64, _i64p, _vp, _vp, _vp, _vp, C.c_int, _ip]),
    "rcp_coverage_value_type": (C.c_int, [C.c_int, _ip]),
    "rcp_coverage_storage_bytes": (C.c_int, [C.c_int, _ip]),
    "rcp_coverage_fetch_f32": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _vp, C.c_int64]),
    "rcp_coverage_rle_f32": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _i64p, _vp, _i32p, C.c_int64]),
    "rcp_bin_matrix": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_int, _vp, C.c_int64, C.c_int]),
    "rcp_base_matrix": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _vp, C.c_int64, C.c_int]),
    "rcp_profile_ncols": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _i64p]),
    "rcp_profile_matrix": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int, _vp, C.c_int64, C.c_int]),
    "rcp_coverage_profile": (C.c_int, [C.c_int, C.c_int64, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_double, _vp, C.c_int64, _vp, C.c_int]),
    "rcp_sort_keys_u32": (C.c_int, [_vp, C.c_int64, C.c_int, C.c_int]),
    "rcp_shared_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]),
    "rcp_shared_open": (C.c_int, [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "rcp_shared_close": (C.c_int, [C.c_void_p]),
    "rcp_shared_free": (C.c_int, [C.c_void_p]),
    "rcp_rows_scatter": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, _vp, _vp, C.c_int64]),
    "rcp_kmeans": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_int, C.c_int, _vp, _vp, _vp, _vp, _f64p, _ip, _ip, _ip]),
    "rcp_r_sample_int": (C.c_int, [C.c_int, C.c_int, C.c_int, _i64p, _i64p, _vp]),
    "rcp_hclust": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp]),
}


class RecoupError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("librecoup_b200 error %d: %s" % (code, message))
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). recoup_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()
_initialised_device = None


def check(rc):
    if rc != RCP_OK:
        raise RecoupError(rc, lib.rcp_last_error().decode("utf-8", "replace"))


def init(device=None):
    """Bind this process to one GPU (default: LOCAL_RANK or 0).  Raises without a B200."""
    global _initialised_device
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _initialised_device == device:
        return
    check(lib.rcp_init(int(device)))
    _initialised_device = device


def shutdown():
    global _initialised_device
    lib.rcp_shutdown()
    _initialised_device = None


def set_coverage_path(path):
    """"auto" | "split" | "buckets" | "index" ("blocks" is a retired name for "buckets"): how
    rcp_coverage finds each region's reads (same results; see include/recoup_b200.h).  Applies to
    every later coverage call; "index" also sorts reads at load time from then on."""
    ensure_init()
    check(lib.rcp_set_coverage_path(COVERAGE_PATH[path]))


def ensure_init():
    if _initialised_device is None:
        init()
