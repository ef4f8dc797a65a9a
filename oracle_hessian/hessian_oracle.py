"""ctypes binding of the Hessian CPU oracle (oracle_hessian/libfd_hessian_oracle.so).

TEST INFRASTRUCTURE ONLY — see fd_hessian_oracle.h.  Only tests/, __graft_entry__.smoke() and profiles/hessian_bench.py
import this module; the product package (finitediff.jl_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libfd_hessian_oracle.so"

_f64p = C.POINTER(C.c_double)
FDO_SFN = C.CFUNCTYPE(C.c_double, C.c_void_p, _f64p)


class SynthHessPolyCtx(C.Structure):
    _fields_ = [("n", C.c_int64), ("w", _f64p)]


def build(force: bool = False) -> Path:
    """Compile the oracle with the committed Makefile (gcc, no GPU needed)."""
    srcs = [_HERE / "fd_hessian_oracle.c", _HERE / "synth_scalar.c", _HERE / "fd_hessian_oracle.h", _HERE / "Makefile"]
    if force or not _LIB_PATH.exists() or any(s.stat().st_mtime > _LIB_PATH.stat().st_mtime for s in srcs):
        env = dict(os.environ)
        env.pop("CC", None)
        subprocess.run(["make", "-C", str(_HERE)], check=True, env=env, capture_output=True)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            build()
        L = C.CDLL(str(_LIB_PATH))
        L.fdo_hcentral_default_relstep.restype = C.c_double
        L.fdo_hcentral_default_relstep.argtypes = []
        L.fdo_hcentral_compute_epsilon.restype = C.c_double
        L.fdo_hcentral_compute_epsilon.argtypes = [C.c_double, C.c_double, C.c_double]
        L.fdo_finite_difference_hessian.restype = C.c_int
        L.fdo_finite_difference_hessian.argtypes = [_f64p, C.c_int64, C.c_void_p, C.c_void_p, _f64p, C.c_int64,
                                                    C.c_double, C.c_double, _f64p, C.POINTER(C.c_int64)]
        L.fdo_finite_difference_hessian_cached.restype = C.c_int
        L.fdo_finite_difference_hessian_cached.argtypes = [_f64p, C.c_int64, C.c_void_p, C.c_void_p, _f64p, C.c_int64,
                                                           _f64p, _f64p, _f64p, _f64p, C.c_double, C.c_double, _f64p,
                                                           C.POINTER(C.c_int64)]
        L.synth_hess_poly.restype = C.c_double
        L.synth_hess_poly.argtypes = [C.c_void_p, _f64p]
        _lib = L
    return _lib


def default_relstep() -> float:
    return lib().fdo_hcentral_default_relstep()


def compute_epsilon(x: float, relstep: float, absstep: float) -> float:
    return lib().fdo_hcentral_compute_epsilon(float(x), float(relstep), float(absstep))


def _p(a):
    return None if a is None else a.ctypes.data_as(_f64p)


def hessian(f, x, *, relstep=None, absstep=None, cache=None, ctx=None):
    """finite_difference_hessian!(H, f, x, cache; relstep, absstep) (src/hessians.jl:202-292) on the CPU.

    f: Python callable f(x: ndarray) -> float, or a native fdo_sfn (e.g. lib().synth_hess_poly) with `ctx`.
    cache: None (HessianCache(x)) or a tuple of four float64 arrays (xpp, xpm, xmp, xmm), written in place.
    Returns dict(H=(n, n) ndarray, eps=ndarray[n], fcalls=int)."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1)
    n = x.size
    H = np.zeros((max(n, 1), max(n, 1)), order="F")
    eps = np.zeros(max(n, 1))
    calls = C.c_int64(0)
    if ctx is None:
        def tramp(_ctx, px):
            return float(f(np.ctypeslib.as_array(px, shape=(n,)).copy() if n else np.zeros(0)))
        keep = FDO_SFN(tramp)
        fptr, cptr = C.cast(keep, C.c_void_p), None
    else:
        fptr, cptr, keep = C.cast(f, C.c_void_p), C.cast(C.pointer(ctx), C.c_void_p), None
    rs = float("nan") if relstep is None else float(relstep)
    ab = float("nan") if absstep is None else float(absstep)
    if cache is None:
        rc = L.fdo_finite_difference_hessian(_p(H), max(n, 1), fptr, cptr, _p(x), n, rs, ab, _p(eps), C.byref(calls))
    else:
        arrs = [np.asarray(a) for a in cache]
        for a in arrs:
            if a.dtype != np.float64 or not a.flags.c_contiguous or a.size < n:
                raise TypeError("cache arrays must be contiguous float64 of length(x)")
        rc = L.fdo_finite_difference_hessian_cached(_p(H), max(n, 1), fptr, cptr, _p(x), n, *map(_p, arrs), rs, ab,
                                                    _p(eps), C.byref(calls))
    del keep
    if rc != 0:
        raise RuntimeError(f"oracle returned {rc}")
    return {"H": H[:n, :n].copy(), "eps": eps[:n].copy(), "fcalls": int(calls.value)}


def hess_poly(x, w, *, relstep=None, absstep=None):
    """The oracle's Hessian of the synthetic f (synth_hess_poly, twin of fdbs_hess_poly)."""
    w = np.ascontiguousarray(w, dtype=np.float64)
    ctx = SynthHessPolyCtx(len(w), w.ctypes.data_as(_f64p))
    r = hessian(lib().synth_hess_poly, x, relstep=relstep, absstep=absstep, ctx=ctx)
    r["_keep"] = w
    return r


def hess_poly_value(x, w) -> float:
    w = np.ascontiguousarray(w, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    ctx = SynthHessPolyCtx(len(w), w.ctypes.data_as(_f64p))
    return lib().synth_hess_poly(C.cast(C.pointer(ctx), C.c_void_p), _p(x))
