"""finitediff.jl_b200 — B200 (sm_100a) drop-in for FiniteDiff.jl's coloured sparse-Jacobian hot path.

Layout (only what the path needs):
    csrc/      hand-written CUDA kernels + the C ABI (libfdjac_b200.so; include/fdjac_b200.h)
    api.py     host-side mirror of the reference interface (JacobianCache / finite_difference_jacobian!, JVPCache,
               HessianCache / finite_difference_hessian!)
    distributed.py  multi-GPU plumbing over the C ABI's fdb_group_* / fdb_sync_* (colour shards, column blocks)
    julia/     the `ccall` wrapper a Julia host would load (not executable in this image: no julia)
    _lib.py    ctypes binding of the C ABI (fails loudly if the .so is missing)
    build.py   nvcc recipe (sm_100a only)

The directory name contains a dot, so it is imported through /root/repo/_bootstrap.py under the alias
`finitediff_jl_b200`.
"""
from . import _lib  # noqa: F401
from .api import (BandedBlockBandedMatrix, BandedMatrix, BlockBandedMatrix, DenseColumnBlock, HessianCache, JacobianCache, JVPCache, NativeFn, Plan, SparseMatrixCSC, Tridiagonal, compute_epsilon,
                  default_relstep, finite_difference_hessian, finite_difference_hessian_, finite_difference_jacobian_,
                  finite_difference_jacobian_b, finite_difference_jvp_, check_coloring, make_plan, matrix_colors,
                  pinned_empty, resize_, zeros_colmajor)

__all__ = ["BandedBlockBandedMatrix", "BandedMatrix", "BlockBandedMatrix", "DenseColumnBlock", "HessianCache",
           "finite_difference_hessian", "finite_difference_hessian_", "JacobianCache", "JVPCache", "finite_difference_jvp_", "NativeFn", "Plan", "SparseMatrixCSC", "Tridiagonal", "compute_epsilon",
           "default_relstep", "finite_difference_jacobian_", "finite_difference_jacobian_b", "make_plan", "matrix_colors", "check_coloring",
           "pinned_empty", "resize_", "zeros_colmajor"]
