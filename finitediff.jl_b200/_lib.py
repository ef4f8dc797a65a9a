"""ctypes binding of the C ABI in include/fdjac_b200.h (libfdjac_b200.so) and of the harness library
include/fdjac_synth.h (libfdjac_synth.so).

There is NO fallback: if the shared library is missing or cannot be loaded this module raises — the product path
never routes through PyTorch eager code or the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "libfdjac_b200.so"
SYNTH_PATH = HERE / "libfdjac_synth.so"

FDB_OK, FDB_ERR_INVALID, FDB_ERR_CUDA, FDB_ERR_CALLBACK, FDB_ERR_NOMEM, FDB_ERR_UNSUPPORTED, FDB_ERR_NO_DEVICE = range(7)
FDB_FORWARD, FDB_CENTRAL, FDB_COMPLEX, FDB_HCENTRAL = 0, 1, 2, 3
FDB_J_CSC_NZVAL, FDB_J_DENSE, FDB_J_BAND, FDB_J_SLOTS = 0, 1, 2, 3
# FDB_STEP_DEFAULT: relstep / absstep keyword not given (any other value, 0 included, is used as passed)
STEP_DEFAULT = float("nan")

# int (*fdb_fn)(void* ctx, double* d_fx, const double* d_x, int64 batch, int64 ldfx, int64 ldx, void* stream)
FDB_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p)


class PlanOpts(C.Structure):
    _fields_ = [
        ("fdtype", C.c_int32), ("device", C.c_int32), ("use_current_device", C.c_int32), ("no_drift", C.c_int32),
        ("max_batch", C.c_int64), ("scratch_bytes", C.c_int64),
        ("rank", C.c_int32), ("world", C.c_int32), ("partition", C.c_int32), ("strategy", C.c_int32),
        ("use_graph", C.c_int32), ("shared_j", C.c_int32),
    ]


class PlanInfo(C.Structure):
    _fields_ = [
        ("m", C.c_int64), ("n", C.c_int64), ("n_entries", C.c_int64), ("j_len", C.c_int64),
        ("n_colors", C.c_int64), ("n_local_colors", C.c_int64), ("n_groups", C.c_int64), ("slabs", C.c_int64),
        ("fcalls_per_jacobian", C.c_int64), ("device_bytes", C.c_int64),
        ("fdtype", C.c_int32), ("jkind", C.c_int32), ("sp_kind", C.c_int32), ("color_bits", C.c_int32),
        ("alg_bytes_scatter", C.c_int64), ("strategy", C.c_int32), ("lanes", C.c_int32), ("mean_row_jump", C.c_double),
        ("moved_bytes_scatter", C.c_int64), ("staged", C.c_int32), ("lists_resident", C.c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Counters(C.Structure):
    _fields_ = [("jacobians", C.c_int64), ("f_points", C.c_int64), ("f_invocations", C.c_int64),
                ("kernel_launches", C.c_int64), ("scatter_launches", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/fdjac_b200.h declares: name -> (restype, argtypes)
_vp, _i64, _i32, _f64, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_int
_PP = C.POINTER(C.c_void_p)
ABI_SYMBOLS = {
    "fdb_abi_version": (_int, []),
    "fdb_last_error": (C.c_char_p, []),
    "fdb_device_count": (_int, []),
    "fdb_default_relstep": (_f64, [_int]),
    "fdb_compute_epsilon": (_f64, [_int, _f64, _f64, _f64, _f64]),
    "fdb_plan_create_csc": (_int, [_PP, _i64, _i64, _vp, _vp, _int, _vp, _vp, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_plan_create_coo": (_int, [_PP, _i64, _i64, _i64, _vp, _vp, _int, _vp, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_plan_create_banded": (_int, [_PP, _i64, _i64, _i64, _i64, _int, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_plan_create_dense": (_int, [_PP, _i64, _i64, _i64, C.POINTER(PlanOpts)]),
    "fdb_plan_create_dense_colorvec": (_int, [_PP, _i64, _i64, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_plan_destroy": (_int, [_vp]),
    "fdb_plan_info": (_int, [_vp, C.POINTER(PlanInfo)]),
    "fdb_plan_counters": (_int, [_vp, C.POINTER(Counters)]),
    "fdb_plan_dense_range": (_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "fdb_plan_color_owner": (_int, [_vp, C.POINTER(_i32), _i64]),
    "fdb_plan_get_eps": (_int, [_vp, C.POINTER(_f64), _i64, _vp]),
    "fdb_plan_set_peers": (_int, [_vp, _int, C.POINTER(_vp)]),
    "fdb_plan_enable_timing": (_int, [_vp, _int]),
    "fdb_plan_read_timing": (_int, [_vp, C.POINTER(_f64), C.POINTER(_i64)]),
    "fdb_jacobian": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f64, _f64, _f64, _vp]),
    "fdb_jacobian_complex": (_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "fdb_jacobian_host": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f64, _f64, _f64]),
    "fdb_eps_plan_create": (_int, [_PP, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_color_eps": (_int, [_vp, _vp, _f64, _f64, _f64, _vp, _vp]),
    "fdb_plan_set_external_eps": (_int, [_vp, _vp]),
    "fdb_group_create_csc": (_int, [_PP, _int, C.POINTER(_int), _i64, _i64, _vp, _vp, _int, _vp, _vp, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_group_create_banded": (_int, [_PP, _int, C.POINTER(_int), _i64, _i64, _i64, _i64, _int, _i64, _vp, C.POINTER(PlanOpts)]),
    "fdb_group_create_dense": (_int, [_PP, _int, C.POINTER(_int), _i64, _i64, _i64, C.POINTER(PlanOpts)]),
    "fdb_group_destroy": (_int, [_vp]),
    "fdb_group_size": (_int, [_vp, C.POINTER(_int)]),
    "fdb_group_plan": (_int, [_vp, _int, _PP]),
    "fdb_group_jacobian": (_int, [_vp, _vp, C.POINTER(_vp), _vp, _vp, _vp, _vp, _f64, _f64, _f64, _vp]),
    "fdb_sync_create": (_int, [_PP, _int, _int, _int]),
    "fdb_sync_flags": (_int, [_vp, _PP]),
    "fdb_sync_set_peers": (_int, [_vp, C.POINTER(_vp)]),
    "fdb_sync_barrier": (_int, [_vp, _vp]),
    "fdb_sync_destroy": (_int, [_vp]),
    "fdb_matrix_colors_banded": (_int, [_i64, _i64, _i64, _vp, _vp]),
    "fdb_matrix_colors_csc": (_int, [_i64, _i64, _vp, _vp, _vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "fdb_check_coloring_csc": (_int, [_i64, _i64, _vp, _vp, _vp, C.POINTER(_i64)]),
    "fdb_jvp_plan_create": (_int, [_PP, _i64, _i64, C.POINTER(PlanOpts)]),
    "fdb_jvp": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f64, _f64, _f64, _vp]),
    "fdb_hessian_plan_create": (_int, [_PP, _i64, C.POINTER(PlanOpts)]),
    "fdb_hessian": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f64, _f64, _vp]),
    "fdb_host_alloc": (_int, [_PP, C.c_size_t]),
    "fdb_host_free": (_int, [_vp]),
    "fdb_device_alloc": (_int, [_PP, C.c_size_t]),
    "fdb_device_free": (_int, [_vp]),
    "fdb_memcpy_h2d": (_int, [_vp, _vp, C.c_size_t, _vp]),
    "fdb_memcpy_d2h": (_int, [_vp, _vp, C.c_size_t, _vp]),
    "fdb_stream_sync": (_int, [_vp]),
    "fdb_ipc_get_handle": (_int, [_vp, C.c_char_p]),
    "fdb_ipc_open": (_int, [C.c_char_p, _PP]),
    "fdb_ipc_close": (_int, [_vp]),
}

SYNTH_SYMBOLS = {
    "fdbs_tridiag": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_tridiag_c": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_tridiag_rows": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_store_probe": (_int, [_vp, _i64, _int, _int, _vp]),
    "fdbs_lap5": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_ellrows": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_rank1": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_hess_poly": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_fail": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "fdbs_fill_x": (_int, [_vp, _i64, C.c_uint64, _vp]),
    "fdbs_flush_l2": (_int, [_vp, _i64, _vp]),
}


class TridiagCtx(C.Structure):
    _fields_ = [("n", _i64), ("calls", _i64)]


class TridiagRowsCtx(C.Structure):
    _fields_ = [("n", _i64), ("row0", _i64), ("nrows", _i64), ("x0", _i64), ("calls", _i64)]


class Lap5Ctx(C.Structure):
    _fields_ = [("g", _i64), ("calls", _i64)]


class EllCtx(C.Structure):
    _fields_ = [("m", _i64), ("K", _i64), ("d_cols", _vp), ("d_coef", _vp), ("calls", _i64)]


class Rank1Ctx(C.Structure):
    _fields_ = [("n", _i64), ("d_w", _vp), ("d_block_sums", _vp), ("max_batch", _i64), ("calls", _i64)]


class HessPolyCtx(C.Structure):
    _fields_ = [("n", _i64), ("d_w", _vp), ("calls", _i64)]


class FdbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libfdjac_b200 status {status}: {message}")
        self.status = status


_lib = None
_synth = None


def _bind(lib, table):
    for name, (res, args) in table.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


def lib():
    """Load libfdjac_b200.so (built in-tree by build.py).  Fails loudly when it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python finitediff.jl_b200/build.py` "
                "(__graft_entry__.build()).  There is no CPU/PyTorch fallback for this path.")
        _lib = _bind(C.CDLL(str(LIB_PATH)), ABI_SYMBOLS)
    return _lib


def synth():
    global _synth
    if _synth is None:
        if not SYNTH_PATH.exists():
            raise ImportError(f"{SYNTH_PATH} is missing: run `python finitediff.jl_b200/build.py`")
        _synth = _bind(C.CDLL(str(SYNTH_PATH)), SYNTH_SYMBOLS)
    return _synth


def check(status: int):
    if status != FDB_OK:
        msg = lib().fdb_last_error()
        raise FdbError(status, msg.decode() if msg else "")


def fn_address(cfunc) -> int:
    return C.cast(cfunc, C.c_void_p).value
