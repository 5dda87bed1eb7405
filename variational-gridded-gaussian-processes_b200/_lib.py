"""ctypes binding of libvggp.so (include/vggp.h).  There is no fallback: a missing library is an ImportError at
first use, a non-zero status is a RuntimeError carrying vggp_last_error()."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvggp.so")

B1_ASVGP, B0_GRIDDED, SVGP_GRID, VFF_GRID, SVGP_MARKOV = 0, 1, 2, 3, 4
F32, F64 = 0, 1
MEANOPT_JACOBI, MEANOPT_KRONECKER = 0, 1
PROBE_RADEMACHER, PROBE_UNIT = 0, 1
LOGDET_FIELDS, CT_FIELDS = 6, 5
ABI_VERSION = 5

WS_K, WS_P, WS_R, WS_Q, WS_S, WS_ALPHA, WS_SCAL, WS_KRAW, WS_QBAND = range(9)

_vp = C.c_void_p
_i64 = C.c_int64
_dp = C.c_void_p   # device pointers travel as integers


class BinnedDesc(C.Structure):
    """vggp_binned_desc (include/vggp.h): layout of one binned data set."""
    _fields_ = [("bytes", _i64), ("n", _i64), ("n_inside", _i64), ("n_tasks", _i64), ("n_runs", _i64),
                ("data_elems", _i64), ("off_task_off", _i64), ("off_task_R", _i64), ("off_run_cell", _i64),
                ("off_run_n", _i64), ("off_run_start", _i64), ("off_data", _i64),
                ("run_cap", C.c_int32), ("D", C.c_int32)]


class EpochDesc(C.Structure):
    """vggp_epoch_desc (include/vggp.h): layout of one epoch of binned minibatches."""
    _fields_ = [("bytes", _i64), ("n", _i64), ("batch_size", _i64), ("n_batches", _i64), ("n_tasks", _i64),
                ("n_runs", _i64), ("data_elems", _i64), ("seed", C.c_uint64), ("epoch", C.c_uint64),
                ("rank", C.c_int32), ("run_cap", C.c_int32), ("D", C.c_int32), ("elem_size", C.c_int32)]


EPOCH_TOTALS = 5


class ArDesc(C.Structure):
    """vggp_ar_desc (include/vggp.h): peer addresses of the symmetric gradient buffers and signal pads."""
    _fields_ = [("mc_ptr", C.c_void_p), ("buf_ptrs", C.c_void_p * 8), ("pad_ptrs", C.c_void_p * 8),
                ("rank", C.c_int32), ("world", C.c_int32)]


# name -> (restype, argtypes); every symbol declared in include/vggp.h
SIGNATURES = {
    "vggp_abi_version": (C.c_int, []),
    "vggp_last_error": (C.c_char_p, []),
    "vggp_launch_count": (C.c_uint64, []),
    "vggp_plan_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.POINTER(C.c_int),
                                   C.POINTER(C.POINTER(C.c_float)), C.c_int, C.c_int]),
    "vggp_plan_destroy": (C.c_int, [_vp]),
    "vggp_plan_dims": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(_i64)]),
    "vggp_gbuf_layout": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "vggp_grid_forward": (C.c_int, [_vp, _dp, _dp, _dp, _vp]),
    "vggp_obs_pack_geometry": (C.c_int, [_vp, _i64, C.POINTER(_i64), C.POINTER(C.c_int)]),
    "vggp_obs_pack": (C.c_int, [_vp, C.POINTER(_vp), _dp, _i64, C.c_int, C.POINTER(_vp), _dp, _vp]),
    "vggp_obs_fwd_bwd_packed": (C.c_int, [_vp, C.POINTER(_vp), _dp, _i64, _dp, _vp]),
    "vggp_obs_fwd_bwd": (C.c_int, [_vp, C.POINTER(_vp), _dp, _i64, _dp, _vp]),
    "vggp_obs_bin_prepare": (C.c_int, [_vp, C.POINTER(_vp), _i64, C.c_int, C.POINTER(BinnedDesc), _vp]),
    "vggp_obs_bin_pack": (C.c_int, [_vp, C.POINTER(BinnedDesc), C.POINTER(_vp), _dp, _dp, _vp]),
    "vggp_obs_fwd_bwd_binned": (C.c_int, [_vp, C.POINTER(BinnedDesc), _dp, _dp, _vp]),
    "vggp_epoch_bin_prepare": (C.c_int, [_vp, C.POINTER(_vp), _i64, _i64, _i64, C.c_int, C.c_uint64, C.c_uint64, C.c_int,
                                         C.POINTER(EpochDesc), C.POINTER(_i64), _vp]),
    "vggp_epoch_bin_pack": (C.c_int, [_vp, C.POINTER(EpochDesc), C.POINTER(_i64), C.POINTER(_vp), _dp, _dp, _vp]),
    "vggp_epoch_batch": (C.c_int, [C.POINTER(EpochDesc), C.POINTER(_i64), _i64, C.POINTER(BinnedDesc), C.POINTER(_i64)]),
    "vggp_set_binned_stream": (C.c_int, [C.c_int]),
    "vggp_set_deterministic": (C.c_int, [_vp, C.c_int]),
    "vggp_workspace_bytes": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "vggp_grid_backward": (C.c_int, [_vp, _dp, _dp, _dp, _dp, C.c_double, _dp, _dp, _dp, _dp, _vp]),
    "vggp_read_info": (C.c_int, [_vp, C.POINTER(C.c_int), _vp]),
    "vggp_info_async": (C.c_int, [_vp, _vp, _vp]),
    "vggp_allreduce_gbuf": (C.c_int, [_vp, C.POINTER(ArDesc), _dp, _vp]),
    "vggp_k1_timing": (C.c_int, [_vp, C.c_int]),
    "vggp_k1_time_read": (C.c_int, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "vggp_k1_graph_time_read": (C.c_int, [_vp, C.POINTER(C.c_float)]),
    "vggp_predict": (C.c_int, [_vp, C.POINTER(_vp), _i64, _dp, _dp, _vp]),
    "vggp_metrics": (C.c_int, [C.c_int, _dp, _dp, _i64, _dp, _vp]),
    "vggp_predict_metrics": (C.c_int, [_vp, C.POINTER(_vp), _dp, _i64, _dp, _vp]),
    "vggp_minmax": (C.c_int, [C.c_int, _dp, _i64, _dp, _vp]),
    "vggp_minmax_scale": (C.c_int, [C.c_int, _dp, _i64, _dp, C.c_int, _dp, _vp]),
    "vggp_generate_tracks": (C.c_int, [C.c_int, C.c_int, _i64, _i64, _i64, _i64, C.c_int, C.c_double, C.POINTER(_vp), _vp, _vp]),
    "vggp_elbo_host": (C.c_int, [_vp, C.POINTER(_vp), _vp, _i64, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _vp, _vp]),
    "vggp_meanopt_assemble": (C.c_int, [_vp, C.POINTER(BinnedDesc), _dp, _vp]),
    "vggp_meanopt_solve": (C.c_int, [_vp, C.c_double, C.c_int, _dp, C.POINTER(C.c_int), C.POINTER(C.c_double), _vp]),
    "vggp_meanopt_solve_pc": (C.c_int, [_vp, C.c_int, C.c_double, C.c_int, _dp, C.POINTER(C.c_int), C.POINTER(C.c_double),
                                        _vp]),
    "vggp_logdet_system": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_double, _vp, _vp, _vp]),
    "vggp_collapsed_terms": (C.c_int, [_vp, C.POINTER(BinnedDesc), _dp, _dp, _vp]),
    "vggp_covopt_update": (C.c_int, [_vp, C.c_int, _dp, C.c_double, _dp, _dp, _dp, _vp]),
    "vggp_b1_stencil": (C.c_int, [_vp, C.c_int, _dp, _i64, _dp, _dp, _dp, _vp]),
    "vggp_features_dense": (C.c_int, [_vp, C.c_int, _dp, _i64, _dp, _dp, _vp]),
    "vggp_workspace_ptr": (C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp), C.POINTER(_i64)]),
    "vggp_gemm_f64": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                _dp, _i64, _i64, _i64, _dp, _i64, _i64, _i64, C.c_double,
                                _dp, _i64, _i64, _i64, C.c_int, _vp]),
    "vggp_mode_product": (C.c_int, [_vp, C.c_int, _dp, _dp, _dp, _vp]),
    "vggp_set_gemm_mode": (C.c_int, [C.c_int]),
}

_lib = None


def load():
    """Load libvggp.so and bind every declared symbol (raises if the library or a symbol is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.vggp_abi_version() != ABI_VERSION:
        raise ImportError("libvggp.so ABI version mismatch: rebuild the library")
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load().vggp_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libvggp status {status}: {msg}")
