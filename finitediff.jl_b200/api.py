"""Host-side mirror of the reference interface for the coloured-Jacobian path, over the C ABI.

The reference is Julia and this image has no `julia`, so the executable host side is this Python mirror (the Julia
`ccall` wrapper with the same surface is shipped, unexecuted, in julia/FiniteDiffB200.jl).  Names, argument meaning
and error behaviour follow src/jacobians.jl:

    JacobianCache(x[, fx[, fx1]], fdtype="forward", returntype=float64; colorvec=1:length(x), sparsity=nothing)
                                                                       (jacobians.jl:11-17, :50-57, :94-102)
    finite_difference_jacobian_(J, f, x, cache, f_in=None; relstep, absstep, colorvec, sparsity, dir)   (:504-514)
    finite_difference_jacobian_(J, f, x, fdtype="forward", returntype, f_in; relstep, absstep, colorvec, sparsity)
                                                                       (cache-less, :446-455)
    resize_(cache, i)                                                  (:655-661)
    default_relstep / compute_epsilon                                  (epsilons.jl:26-29,50-53,74-77,134-144)
    JVPCache / finite_difference_jvp_                                  (src/jvp.jl)
    HessianCache / finite_difference_hessian_ / finite_difference_hessian   (src/hessians.jl:67-292)

(`!` is not a Python identifier character: `finite_difference_jacobian!` is spelled with a trailing underscore.)
Index arrays keep Julia's convention: Int64, 1-based.  PyTorch is used only for device memory and streams.
All compute happens in libfdjac_b200.so; there is no eager/CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import weakref
import zlib
from typing import Callable, Optional

import numpy as np
import torch

from . import _lib as L

__all__ = [
    "SparseMatrixCSC", "BandedMatrix", "Tridiagonal", "BandedBlockBandedMatrix", "DenseColumnBlock", "NativeFn", "JacobianCache", "Plan",
    "finite_difference_jacobian_", "finite_difference_jacobian_b", "resize_", "default_relstep", "compute_epsilon",
    "zeros_colmajor", "pinned_empty", "JVPCache", "finite_difference_jvp_", "HessianCache",
    "finite_difference_hessian_", "finite_difference_hessian",
]

_DEFAULT = object()

_FDTYPES = {"forward": L.FDB_FORWARD, "central": L.FDB_CENTRAL, "complex": L.FDB_COMPLEX, L.FDB_FORWARD: L.FDB_FORWARD,
            L.FDB_CENTRAL: L.FDB_CENTRAL, L.FDB_COMPLEX: L.FDB_COMPLEX}


def _fdtype_code(fdtype) -> int:
    if isinstance(fdtype, str):
        fdtype = fdtype.lstrip(":")
    if fdtype not in _FDTYPES:
        # epsilons.jl:159-167 fdtype_error
        raise ValueError("Unrecognized fdtype: valid values are 'forward', 'central' and 'complex'.")
    return _FDTYPES[fdtype]


def _step_fdtype_code(fdtype) -> int:
    """_fdtype_code, plus the Hessian's 'hcentral' (a step-size type only: no Jacobian plan takes it)."""
    if (isinstance(fdtype, str) and fdtype.lstrip(":") == "hcentral") or (isinstance(fdtype, int) and fdtype == L.FDB_HCENTRAL):
        return L.FDB_HCENTRAL
    return _fdtype_code(fdtype)


def default_relstep(fdtype, T=torch.float64) -> float:
    """src/epsilons.jl:134-144 ("hcentral": eps(Float64)^(1/4) = 2^-13)"""
    return L.lib().fdb_default_relstep(_step_fdtype_code(fdtype))


def compute_epsilon(fdtype, x: float, relstep: float, absstep: float, dir: float = 1.0) -> float:
    """src/epsilons.jl:26-29 (forward) / :50-53 (central) / :74-77 (hcentral)"""
    return L.lib().fdb_compute_epsilon(_step_fdtype_code(fdtype), float(x), float(relstep), float(absstep), float(dir))


# ------------------------------------------------------------------------------------------------ array helpers
class PeerValues:
    """J value storage that lives in ANOTHER process / on another GPU and is only mapped here (CUDA IPC, peer access): a
    raw device pointer + length, deliberately NOT a torch tensor — torch would attribute the mapping to the exporting
    device and copy it on any device mismatch, and stores into a copy never reach the owner."""
    is_cuda = True
    dtype = torch.float64

    def __init__(self, ptr: int, numel: int):
        self._ptr, self._numel = int(ptr), int(numel)

    def data_ptr(self) -> int:
        return self._ptr

    def numel(self) -> int:
        return self._numel


def _is_cuda(t) -> bool:
    return (isinstance(t, torch.Tensor) and t.is_cuda) or isinstance(t, PeerValues)


def _index_ptr(a):
    """(pointer, keepalive) of an Int64 index array living on the host (numpy / CPU tensor) or the device."""
    if a is None:
        return None, None
    if isinstance(a, torch.Tensor):
        if a.dtype != torch.int64:
            raise TypeError("index arrays must be Int64 (as SparseMatrixCSC{Float64,Int64} stores them)")
        a = a.contiguous()
        return a.data_ptr(), a
    if isinstance(a, range):
        a = np.arange(a.start, a.stop, a.step, dtype=np.int64)
    arr = np.ascontiguousarray(a, dtype=np.int64)
    return arr.ctypes.data, arr


def _is_identity_colorvec(colorvec, n: int) -> bool:
    """colorvec == 1:n (the JacobianCache default, jacobians.jl:16), whatever container holds it."""
    if colorvec is None:
        return True
    if isinstance(colorvec, range):
        return colorvec == range(1, n + 1)
    if isinstance(colorvec, torch.Tensor):
        return colorvec.numel() == n and bool(torch.equal(colorvec.reshape(-1).cpu().to(torch.int64),
                                                          torch.arange(1, n + 1, dtype=torch.int64)))
    arr = np.asarray(colorvec).reshape(-1)
    return arr.size == n and bool(np.array_equal(arr, np.arange(1, n + 1)))


def _index_key(a):
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        return ("t", a.data_ptr(), a.numel(), a._version, str(a.device))
    if isinstance(a, range):
        return ("r", a.start, a.stop, a.step)
    arr = np.asarray(a)
    if arr.size <= 4096:
        return ("v", arr.shape, arr.astype(np.int64).tobytes())
    # large host arrays: identity + a strided content sample (4096 elements, first and last included), so that an
    # in-place edit of colorvec / colptr / rowval is noticed in all but contrived cases without an O(n) pass on every
    # call.  The plan holds a private compressed copy: after an in-place edit that the sample cannot see, call
    # cache.invalidate() (documented in JacobianCache).
    flat = arr.reshape(-1)
    step = max(1, flat.size // 4096)
    sample = np.ascontiguousarray(flat[::step]).tobytes() + np.ascontiguousarray(flat[-1:]).tobytes()
    return ("n", arr.__array_interface__["data"][0], arr.size, zlib.crc32(sample))


def zeros_colmajor(m: int, n: int, device="cuda") -> torch.Tensor:
    """A Julia-style dense Matrix{Float64}: logical (m, n), column-major storage (stride (1, m))."""
    return torch.zeros((n, m), dtype=torch.float64, device=device).t()


def pinned_empty(count: int) -> np.ndarray:
    """float64 host array in pinned memory (fdb_host_alloc) — what fdb_jacobian_host needs to reach PCIe speed."""
    p = C.c_void_p()
    L.check(L.lib().fdb_host_alloc(C.byref(p), max(int(count), 1) * 8))
    buf = (C.c_double * max(int(count), 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.float64, count=int(count))
    weakref.finalize(buf, L.lib().fdb_host_free, p)
    return arr


class _DevArray:
    """Zero-copy view of raw device memory for torch.as_tensor (CUDA array interface v3)."""

    def __init__(self, ptr: int, shape, strides=None, typestr: str = "<f8"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": strides}


# ------------------------------------------------------------------------------------------------ matrix types
class SparseMatrixCSC:
    """Mirror of SparseArrays.SparseMatrixCSC{Float64,Int64}: m, n, colptr[n+1], rowval[nnz] (Int64, 1-based),
    nzval[nnz] (float64; CUDA tensor for the device path, numpy array for the host path)."""

    def __init__(self, m, n, colptr, rowval, nzval):
        self.m, self.n = int(m), int(n)
        self.colptr, self.rowval, self.nzval = colptr, rowval, nzval

    @property
    def shape(self):
        return (self.m, self.n)

    @property
    def nnz(self):
        return int(self.rowval.shape[0]) if hasattr(self.rowval, "shape") else len(self.rowval)

    @staticmethod
    def from_scipy(A, device="cuda", index_device=None):
        import scipy.sparse as sp
        A = sp.csc_matrix(A)
        A.sort_indices()
        colptr = torch.from_numpy(A.indptr.astype(np.int64) + 1)
        rowval = torch.from_numpy(A.indices.astype(np.int64) + 1)
        if index_device is not None:
            colptr, rowval = colptr.to(index_device), rowval.to(index_device)
        nz = torch.zeros(A.nnz, dtype=torch.float64, device=device) if device != "host" else np.zeros(A.nnz)
        return SparseMatrixCSC(A.shape[0], A.shape[1], colptr, rowval, nz)

    def similar(self):
        nz = torch.empty_like(self.nzval) if isinstance(self.nzval, torch.Tensor) else np.empty_like(self.nzval)
        return SparseMatrixCSC(self.m, self.n, self.colptr, self.rowval, nz)

    def to_dense(self) -> np.ndarray:
        cp = np.asarray(self.colptr.cpu() if isinstance(self.colptr, torch.Tensor) else self.colptr) - 1
        rv = np.asarray(self.rowval.cpu() if isinstance(self.rowval, torch.Tensor) else self.rowval) - 1
        nz = self.nzval.cpu().numpy() if isinstance(self.nzval, torch.Tensor) else np.asarray(self.nzval)
        import scipy.sparse as sp
        return sp.csc_matrix((nz, rv, cp), shape=(self.m, self.n)).toarray()


class BandedMatrix:
    """Mirror of BandedMatrices.BandedMatrix: data is the (l+u+1) x n column-major band storage (flat float64),
    entry (r,c) at data[u+r-c+1, c] (1-based; ext/FiniteDiffBandedMatricesExt.jl:22)."""

    def __init__(self, m, n, l, u, data=None, device="cuda"):
        self.m, self.n, self.l, self.u = int(m), int(n), int(l), int(u)
        if data is None:
            data = torch.zeros((self.l + self.u + 1) * self.n, dtype=torch.float64, device=device)
        self.data = data

    @property
    def shape(self):
        return (self.m, self.n)

    def to_dense(self) -> np.ndarray:
        d = self.data.cpu().numpy() if isinstance(self.data, torch.Tensor) else np.asarray(self.data)
        w = self.l + self.u + 1
        J = np.zeros((self.m, self.n))
        for c in range(1, self.n + 1):
            for r in range(max(1, c - self.u), min(self.m, c + self.l) + 1):
                J[r - 1, c - 1] = d[(c - 1) * w + (self.u + r - c)]
        return J


class Tridiagonal:
    """Mirror of LinearAlgebra.Tridiagonal(dl, d, du): one buffer [dl; d; du]; its structural nonzeros are
    enumerated band by band like ArrayInterface.findstructralnz does (order is irrelevant to the result)."""

    def __init__(self, n, buf=None, device="cuda"):
        self.n = int(n)
        if buf is None:
            buf = torch.zeros(max(3 * self.n - 2, 0), dtype=torch.float64, device=device)
        self.buf = buf

    @property
    def shape(self):
        return (self.n, self.n)

    @property
    def dl(self):
        return self.buf[: self.n - 1]

    @property
    def d(self):
        return self.buf[self.n - 1: 2 * self.n - 1]

    @property
    def du(self):
        return self.buf[2 * self.n - 1:]

    def findstructralnz(self):
        n = self.n
        rows = np.concatenate([np.arange(2, n + 1), np.arange(1, n + 1), np.arange(1, n)]).astype(np.int64)
        cols = np.concatenate([np.arange(1, n), np.arange(1, n + 1), np.arange(2, n + 1)]).astype(np.int64)
        slots = np.arange(1, 3 * n - 1, dtype=np.int64)
        return rows, cols, slots

    def to_dense(self) -> np.ndarray:
        b = self.buf.cpu().numpy()
        n = self.n
        return np.diag(b[n - 1: 2 * n - 1]) + np.diag(b[: n - 1], -1) + np.diag(b[2 * n - 1:], 1)


class BandedBlockBandedMatrix:
    """Mirror of BlockBandedMatrices.BandedBlockBandedMatrix: square blocks structure given by `rowblocks` / `colblocks`
    (block lengths), block bandwidths (l, u) and sub-block bandwidths (lam, mu).  The decompression hook
    ext/FiniteDiffBlockBandedMatricesExt.jl:16-42 writes, for every column j of block-column J and every block-row
    K in blockcolrange(J) = max(1,J-u):min(N,J+l), the in-sub-band rows k in max(1,j-mu):min(m_K, j+lam).
    Storage here: one band-data column of (l+u+1)*(lam+mu+1) slots per matrix column — slot
    (K-J+u)*(lam+mu+1) + (mu+k-j) for entry (k, j) of block (K, J) (the BlockBandedMatrices layout as documented; the
    package source is not vendored in the reference tree, so the LAYOUT is this mirror's own — the ENTRY SET and the
    values are what parity is about, coloring_tests.jl:99-119)."""

    def __init__(self, rowblocks, colblocks, blockbandwidths, subblockbandwidths, data=None, device="cuda"):
        self.rb, self.cb = [int(b) for b in rowblocks], [int(b) for b in colblocks]
        (self.l, self.u), (self.lam, self.mu) = blockbandwidths, subblockbandwidths
        self.m, self.n = sum(self.rb), sum(self.cb)
        self.w = (self.l + self.u + 1) * (self.lam + self.mu + 1)
        if data is None:
            data = torch.zeros(self.w * self.n, dtype=torch.float64, device=device)
        self.data = data
        self._nz = None

    @property
    def shape(self):
        return (self.m, self.n)

    def findstructralnz(self):
        """(rows, cols, slots), 1-based, in the order the reference's hook visits them."""
        if self._nz is None:
            ro = np.concatenate([[0], np.cumsum(self.rb)])
            co = np.concatenate([[0], np.cumsum(self.cb)])
            sw = self.lam + self.mu + 1
            rows, cols, slots = [], [], []
            N_r, N_c = len(self.rb), len(self.cb)
            for J in range(1, N_c + 1):
                for K in range(max(1, J - self.u), min(N_r, J + self.l) + 1):
                    mK = self.rb[K - 1]
                    for j in range(1, self.cb[J - 1] + 1):
                        k = np.arange(max(1, j - self.mu), min(mK, j + self.lam) + 1)
                        if len(k) == 0:
                            continue
                        gc = co[J - 1] + j
                        rows.append(ro[K - 1] + k)
                        cols.append(np.full(len(k), gc))
                        slots.append((gc - 1) * self.w + (K - J + self.u) * sw + (self.mu + k - j) + 1)
            cat = lambda a: np.concatenate(a).astype(np.int64) if a else np.zeros(0, np.int64)
            self._nz = (cat(rows), cat(cols), cat(slots))
        return self._nz

    def to_dense(self) -> np.ndarray:
        rows, cols, slots = self.findstructralnz()
        d = self.data.cpu().numpy() if isinstance(self.data, torch.Tensor) else np.asarray(self.data)
        J = np.zeros((self.m, self.n))
        J[rows - 1, cols - 1] = d[slots - 1]
        return J

    def matrix_colors(self) -> np.ndarray:
        """A valid colouring for the full structure: block colour (cycle l+u+1) x sub-band colour (cycle lam+mu+1)
        — the scheme of ArrayInterface.matrix_colors(::BandedBlockBandedMatrix) for uniform blocks."""
        sw, bw = self.lam + self.mu + 1, self.l + self.u + 1
        out = []
        for J, nb in enumerate(self.cb):
            out.append((J % bw) * sw + (np.arange(nb) % sw) + 1)
        return np.concatenate(out).astype(np.int64)


class BlockBandedMatrix(BandedBlockBandedMatrix):
    """Mirror of BlockBandedMatrices.BlockBandedMatrix: dense blocks inside the block band.  Hook
    ext/FiniteDiffBlockBandedMatricesExt.jl:44-68: for every column j of block-column J, ALL rows of every block-row K
    in blockcolrange(J).  Expressed as a BandedBlockBandedMatrix whose sub-block bandwidths cover the whole block."""

    def __init__(self, rowblocks, colblocks, blockbandwidths, data=None, device="cuda"):
        full = max(max(rowblocks), max(colblocks)) - 1 if len(rowblocks) and len(colblocks) else 0
        super().__init__(rowblocks, colblocks, blockbandwidths, (full, full), data=data, device=device)


class DenseColumnBlock:
    """Columns [col0, col0+ncols) of a dense m x n Jacobian held by ONE rank (north_star config 5: the dense Jacobian is
    column-partitioned over the GPUs and may stay that way): `slab` is the rank's own column-major (m, ncols) storage.
    Use it as J with a JacobianCache built with rank=, world= and sparsity=None; the plan's column range must be the
    block (checked on first use)."""

    def __init__(self, m, n, col0, ncols, device="cuda", slab=None):
        self.m, self.n, self.col0, self.ncols = int(m), int(n), int(col0), int(ncols)
        self.slab = zeros_colmajor(self.m, max(self.ncols, 1), device) if slab is None else slab

    @property
    def shape(self):
        return (self.m, self.n)


def _findstructralnz_dense(A):
    """src/jacobians.jl:473-488: column-major scan of a dense 0/1 prototype."""
    A = np.asarray(A.cpu() if isinstance(A, torch.Tensor) else A)
    if A.ndim == 1:
        A = A.reshape(1, -1)
    c, r = np.nonzero(A.T)
    return (r + 1).astype(np.int64), (c + 1).astype(np.int64)


# ------------------------------------------------------------------------------------------------ user functions
class NativeFn:
    """A native fdb_fn (function address + context struct), e.g. the synthetic f! of libfdjac_synth.so."""

    def __init__(self, address: int, ctx=None, max_batch: int = 1, keepalive=None):
        self.address = int(address)
        self.ctx = ctx
        self.max_batch = int(max_batch)
        self._keepalive = keepalive

    @property
    def ctx_ptr(self):
        return C.cast(C.pointer(self.ctx), C.c_void_p) if self.ctx is not None else None


class _PyFn:
    """Wraps a Python f!(fx, x) working on CUDA tensors as an fdb_fn.  `batched=True` callables receive 2-D
    (batch, m) / (batch, n) tensors; otherwise they are called once per point with 1-D tensors."""

    def __init__(self, f: Callable, m: int, n: int, device: torch.device, batched: bool, complex_: bool = False):
        self.f, self.m, self.n, self.device, self.batched = f, m, n, device, batched
        self.exc: Optional[BaseException] = None
        self.calls = 0
        # complex-step callbacks (fdb_fn_c) see complex128 tensors; ld* then count complex elements
        self.typestr, self.esize = ("<c16", 16) if complex_ else ("<f8", 8)
        self.cfunc = L.FDB_FN(self._tramp)

    def _tramp(self, _ctx, p_fx, p_x, batch, ldfx, ldx, stream):
        try:
            cur = torch.cuda.current_stream(self.device)
            ctx = None
            if (stream or 0) != cur.cuda_stream:
                ctx = torch.cuda.stream(torch.cuda.ExternalStream(stream or 0, device=self.device))
                ctx.__enter__()
            try:
                es = self.esize
                fx2 = torch.as_tensor(_DevArray(p_fx, (batch, self.m), (ldfx * es, es), self.typestr), device=self.device)
                x2 = torch.as_tensor(_DevArray(p_x, (batch, self.n), (ldx * es, es), self.typestr), device=self.device)
                if self.batched:
                    self.calls += int(batch)
                    self.f(fx2, x2)
                else:
                    for b in range(int(batch)):
                        self.calls += 1
                        self.f(fx2[b], x2[b])
            finally:
                if ctx is not None:
                    ctx.__exit__(None, None, None)
            return 0
        except BaseException as e:  # never let an exception cross the C ABI
            self.exc = e
            return 1


# ------------------------------------------------------------------------------------------------ plans
class Plan:
    """Owner of an fdb_plan* (the per-(pattern, colorvec, fdtype) state)."""

    def __init__(self, handle: int, keep=(), owned: bool = True):
        self._h = C.c_void_p(handle)
        self._keep = keep
        # members of an fdb_group are owned (and destroyed) by the group: owned=False gives a plain view
        self._fin = weakref.finalize(self, L.lib().fdb_plan_destroy, C.c_void_p(handle)) if owned else (lambda: None)

    @property
    def handle(self):
        return self._h

    def info(self) -> dict:
        i = L.PlanInfo()
        L.check(L.lib().fdb_plan_info(self._h, C.byref(i)))
        return i.as_dict()

    def counters(self) -> dict:
        c = L.Counters()
        L.check(L.lib().fdb_plan_counters(self._h, C.byref(c)))
        return c.as_dict()

    def eps(self, stream=None) -> np.ndarray:
        i = self.info()
        count = i["n_local_colors"] if i["sp_kind"] == 0 else i["n_colors"]
        out = np.zeros(max(count, 1))
        L.check(L.lib().fdb_plan_get_eps(self._h, out.ctypes.data_as(C.POINTER(C.c_double)), len(out),
                                         C.c_void_p(stream or 0)))
        return out[:count]

    def color_owner(self) -> np.ndarray:
        i = self.info()
        out = np.zeros(max(i["n_colors"], 1), np.int32)
        L.check(L.lib().fdb_plan_color_owner(self._h, out.ctypes.data_as(C.POINTER(C.c_int32)), len(out)))
        return out[: i["n_colors"]]

    def dense_range(self):
        b, e = C.c_int64(), C.c_int64()
        L.check(L.lib().fdb_plan_dense_range(self._h, C.byref(b), C.byref(e)))
        return b.value, e.value

    def set_peers(self, ptrs):
        arr = (C.c_void_p * max(len(ptrs), 1))(*ptrs)
        L.check(L.lib().fdb_plan_set_peers(self._h, len(ptrs), arr))

    def enable_timing(self, on=True):
        L.check(L.lib().fdb_plan_enable_timing(self._h, int(bool(on))))

    def read_timing(self):
        """(summed scatter milliseconds, scatter launches) since the last read; synchronises the recorded events."""
        ms, cnt = C.c_double(), C.c_int64()
        L.check(L.lib().fdb_plan_read_timing(self._h, C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    def destroy(self):
        self._fin()


def _opts(fdtype, device_index, *, no_drift=False, max_batch=1, scratch_bytes=0, rank=0, world=1, partition=0,
          strategy=0, use_graph=False, shared_j=False):
    return L.PlanOpts(fdtype=fdtype, device=device_index, use_current_device=0, no_drift=int(bool(no_drift)),
                      max_batch=int(max_batch), scratch_bytes=int(scratch_bytes), rank=int(rank), world=int(world),
                      partition=int(partition), strategy=int(strategy), use_graph=int(bool(use_graph)), shared_j=int(bool(shared_j)))


def _device_index(device) -> int:
    d = torch.device(device)
    return d.index if d.index is not None else torch.cuda.current_device()


def _dense_ld(J: torch.Tensor):
    """(m, n, ldJ) of a column-major dense J (Julia Matrix).  Row-major tensors are rejected loudly."""
    if isinstance(J, DenseColumnBlock):
        return J.m, J.n, max(int(J.slab.stride(1)) if J.slab.dim() == 2 and J.slab.shape[1] > 1 else J.m, J.m, 1)
    if J.dim() == 1:
        return J.shape[0], 1, max(J.shape[0], 1)
    m, n = J.shape
    if J.dtype != torch.float64:
        raise TypeError("J must be float64")
    if m > 1 and J.stride(0) != 1:
        raise ValueError("dense J must be column-major (Julia Matrix layout): use zeros_colmajor(m, n) or X.t()")
    ld = J.stride(1) if n > 1 else max(m, 1)
    if m == 1 and n > 1:
        ld = J.stride(1)
    return m, n, max(int(ld), m, 1)


def make_plan(J, sparsity, colorvec, fdtype, x_len: int, device, **plan_kw) -> Plan:
    """Create the fdb_plan for (typeof(J), sparsity, colorvec, fdtype) — the dispatch the reference performs with
    _use_findstructralnz / _use_sparseCSC_common_sparsity / typeof(J) (jacobians.jl:522-535)."""
    lib = L.lib()
    fd = _fdtype_code(fdtype)
    o = _opts(fd, _device_index(device), **plan_kw)
    h = C.c_void_p()
    cv_ptr, cv_keep = _index_ptr(colorvec)
    keep = [cv_keep]
    if sparsity is None:
        # dense column branch (jacobians.jl:548-557): column i of J from perturbing component i, colorvec = 1:n.
        # With sparsity === nothing and any OTHER colorvec the reference loops color_i in 1:maximum(colorvec) and
        # perturbs COMPONENT color_i (the colour id used as an index), writing only those leading columns of J (J is
        # not zero-filled on this branch) — reproduced as written by fdb_plan_create_dense_colorvec.
        m, n, ld = _dense_ld(J)
        if colorvec is not None and not _is_identity_colorvec(colorvec, n):
            L.check(lib.fdb_plan_create_dense_colorvec(C.byref(h), m, n, ld, cv_ptr, C.byref(o)))
        else:
            L.check(lib.fdb_plan_create_dense(C.byref(h), m, n, ld, C.byref(o)))
    elif isinstance(sparsity, SparseMatrixCSC):
        cp, k1 = _index_ptr(sparsity.colptr)
        rv, k2 = _index_ptr(sparsity.rowval)
        keep += [k1, k2]
        if isinstance(J, SparseMatrixCSC):
            if J is sparsity or (J.colptr is sparsity.colptr and J.rowval is sparsity.rowval):
                jcp = jrv = None
            else:
                jcp, k3 = _index_ptr(J.colptr)
                jrv, k4 = _index_ptr(J.rowval)
                keep += [k3, k4]
            L.check(lib.fdb_plan_create_csc(C.byref(h), sparsity.m, sparsity.n, cp, rv, L.FDB_J_CSC_NZVAL, jcp, jrv, 0,
                                            cv_ptr, C.byref(o)))
        elif isinstance(J, torch.Tensor):
            m, n, ld = _dense_ld(J)
            if (m, n) != (sparsity.m, sparsity.n):
                raise ValueError("size(J) != size(sparsity)")
            L.check(lib.fdb_plan_create_csc(C.byref(h), m, n, cp, rv, L.FDB_J_DENSE, None, None, ld, cv_ptr, C.byref(o)))
        else:
            raise TypeError(f"unsupported J type {type(J)} for a SparseMatrixCSC sparsity")
    elif isinstance(sparsity, BandedMatrix):
        if isinstance(J, BandedMatrix):
            if (J.l, J.u) != (sparsity.l, sparsity.u):
                raise ValueError("J and sparsity must have the same bandwidths")
            L.check(lib.fdb_plan_create_banded(C.byref(h), sparsity.m, sparsity.n, sparsity.l, sparsity.u, L.FDB_J_BAND,
                                               0, cv_ptr, C.byref(o)))
        elif isinstance(J, torch.Tensor):
            m, n, ld = _dense_ld(J)
            L.check(lib.fdb_plan_create_banded(C.byref(h), m, n, sparsity.l, sparsity.u, L.FDB_J_DENSE, ld, cv_ptr,
                                               C.byref(o)))
        else:
            raise TypeError(f"unsupported J type {type(J)} for a BandedMatrix sparsity")
    elif isinstance(sparsity, Tridiagonal):
        rows, cols, slots = sparsity.findstructralnz()
        n = sparsity.n
        if isinstance(J, Tridiagonal):
            L.check(lib.fdb_plan_create_coo(C.byref(h), n, n, len(rows), rows.ctypes.data, cols.ctypes.data,
                                            L.FDB_J_SLOTS, slots.ctypes.data, 3 * n - 2, cv_ptr, C.byref(o)))
        elif isinstance(J, torch.Tensor):
            m, nn, ld = _dense_ld(J)
            L.check(lib.fdb_plan_create_coo(C.byref(h), m, nn, len(rows), rows.ctypes.data, cols.ctypes.data,
                                            L.FDB_J_DENSE, None, ld, cv_ptr, C.byref(o)))
        else:
            raise TypeError(f"unsupported J type {type(J)} for a Tridiagonal sparsity")
        keep += [rows, cols, slots]
    elif isinstance(sparsity, BandedBlockBandedMatrix):
        # ext/FiniteDiffBlockBandedMatricesExt.jl:16-42: the hook's (block-row, sub-band) entry set, written by slot
        rows, cols, slots = sparsity.findstructralnz()
        if isinstance(J, BandedBlockBandedMatrix):
            if (J.rb, J.cb, J.l, J.u, J.lam, J.mu) != (sparsity.rb, sparsity.cb, sparsity.l, sparsity.u, sparsity.lam, sparsity.mu):
                raise ValueError("J and sparsity must have the same block structure")
            L.check(lib.fdb_plan_create_coo(C.byref(h), sparsity.m, sparsity.n, len(rows), rows.ctypes.data, cols.ctypes.data,
                                            L.FDB_J_SLOTS, slots.ctypes.data, sparsity.w * sparsity.n, cv_ptr, C.byref(o)))
        elif isinstance(J, torch.Tensor):
            m, nn, ld = _dense_ld(J)
            L.check(lib.fdb_plan_create_coo(C.byref(h), m, nn, len(rows), rows.ctypes.data, cols.ctypes.data,
                                            L.FDB_J_DENSE, None, ld, cv_ptr, C.byref(o)))
        else:
            raise TypeError(f"unsupported J type {type(J)} for a BandedBlockBandedMatrix sparsity")
        keep += [rows, cols, slots]
    elif isinstance(sparsity, (torch.Tensor, np.ndarray, list)):
        # dense 0/1 prototype: rows/cols from _findstructralnz (jacobians.jl:526-527), J must be dense
        rows, cols = _findstructralnz_dense(sparsity)
        if not isinstance(J, torch.Tensor):
            raise TypeError("a dense prototype sparsity needs a dense J")
        m, n, ld = _dense_ld(J)
        L.check(lib.fdb_plan_create_coo(C.byref(h), m, n, len(rows), rows.ctypes.data, cols.ctypes.data, L.FDB_J_DENSE,
                                        None, ld, cv_ptr, C.byref(o)))
        keep += [rows, cols]
    else:
        raise TypeError(f"unsupported sparsity type {type(sparsity)}")
    return Plan(h.value, tuple(keep))


def _has_sparsestruct(J) -> bool:
    """ArrayInterface.has_sparsestruct(J) as used at jacobians.jl:455."""
    return isinstance(J, (SparseMatrixCSC, BandedMatrix, Tridiagonal, BandedBlockBandedMatrix))


def _j_values(J):
    if isinstance(J, SparseMatrixCSC):
        return J.nzval
    if isinstance(J, BandedMatrix):
        return J.data
    if isinstance(J, Tridiagonal):
        return J.buf
    if isinstance(J, BandedBlockBandedMatrix):
        return J.data
    if isinstance(J, DenseColumnBlock):
        return J.slab
    return J


def _j_key(J):
    if isinstance(J, SparseMatrixCSC):
        return ("csc", J.m, J.n, _index_key(J.colptr), _index_key(J.rowval))
    if isinstance(J, BandedMatrix):
        return ("band", J.m, J.n, J.l, J.u)
    if isinstance(J, Tridiagonal):
        return ("tri", J.n)
    if isinstance(J, BandedBlockBandedMatrix):
        return ("bbb", tuple(J.rb), tuple(J.cb), J.l, J.u, J.lam, J.mu)
    if isinstance(J, torch.Tensor):
        return ("dense", tuple(J.shape), tuple(J.stride()))
    if isinstance(J, DenseColumnBlock):
        return ("denseblock", J.m, J.n, J.col0, J.ncols, tuple(J.slab.stride()))
    if isinstance(J, np.ndarray):
        return ("hdense", J.shape, J.strides)
    return ("obj", id(J))


def _sp_key(sp):
    if sp is None:
        return None
    if isinstance(sp, (SparseMatrixCSC, BandedMatrix, Tridiagonal, BandedBlockBandedMatrix)):
        return _j_key(sp)
    if isinstance(sp, torch.Tensor):
        return ("proto", sp.data_ptr(), tuple(sp.shape), sp._version)
    a = np.asarray(sp)
    return ("protov", a.shape, a.tobytes())


# ------------------------------------------------------------------------------------------------ JacobianCache
class JacobianCache:
    """Mirror of FiniteDiff.JacobianCache (jacobians.jl:1-9) with its three constructors:

        JacobianCache(x, fdtype=..)                 allocating, square (x1=copy(x), fx=copy(x), fx1=copy(x))   :11-36
        JacobianCache(x, fx, fdtype=..)             allocating (fx1 = copy(fx))                               :50-80
        JacobianCache(x1, fx, fx1, fdtype=..)       non-allocating: ALIASES the arrays passed in              :94-128

    Fields x1, x2, fx, fx1, colorvec, sparsity keep their names.  The B200 path keeps the perturbed points and the
    stacked f! outputs in plan-owned scratch; of the cache arrays only `fx` is written (forward mode: fx = f(x),
    jacobians.jl:540-542).  x1/x2/fx1 are not touched (documented drop: in the reference they end as x (with drift),
    the last colour's mask*x, and the last colour's divided difference).
    Extra keywords (B200-specific): max_batch, scratch_bytes, no_drift, rank, world, partition.
    Plans are cached per (typeof(J), sparsity, colorvec, fdtype) and hold private compressed copies of the index arrays:
    index arrays are treated as immutable while cached (torch tensors are tracked by their version counter, large numpy
    arrays by identity + a content sample); after editing one in place call `cache.invalidate()`.
    """

    def __init__(self, x1, fx=None, fx1=None, fdtype="forward", returntype=torch.float64, *, colorvec=None,
                 sparsity=None, inplace=True, **plan_kw):
        if isinstance(fx, str):          # JacobianCache(x, "central")
            fdtype, fx = fx, None
        if isinstance(fx1, str):         # JacobianCache(x, fx, "central")
            fdtype, fx1 = fx1, None
        self.fdtype = fdtype.lstrip(":") if isinstance(fdtype, str) else fdtype
        _fdtype_code(self.fdtype)
        if returntype not in (torch.float64, float, np.float64):
            raise TypeError("only Float64 is supported by the B200 path")
        if not _is_cuda(x1):
            raise TypeError("JacobianCache needs CUDA float64 tensors (this path has no CPU implementation)")
        if _fdtype_code(self.fdtype) == L.FDB_COMPLEX:
            # complex step: x1 and fx are complex (`false .* im .* x`), fx1 === nothing  (:20-32, :60-76, :105-117)
            fx_like = x1 if fx is None else fx
            self.x1 = torch.zeros(x1.shape, dtype=torch.complex128, device=x1.device)
            self.fx = torch.zeros(fx_like.shape, dtype=torch.complex128, device=x1.device)
            self.fx1 = None
        elif fx is None and fx1 is None:
            self.x1, self.fx, self.fx1 = x1.clone(), x1.clone(), x1.clone()           # :25-33
        elif fx1 is None:
            self.x1, self.fx, self.fx1 = x1.clone(), fx.clone(), fx.clone()           # :62-76
        else:
            if fx.dtype != torch.float64 or fx1.dtype != torch.float64:              # @assert eltype :120-121
                raise AssertionError("eltype(fx) == eltype(fx1) == returntype")
            self.x1, self.fx, self.fx1 = x1, fx, fx1                                  # aliases :118-122
        self.x2 = torch.zeros_like(self.x1)                                           # :124
        n = self.x1.numel()
        self.colorvec = range(1, n + 1) if colorvec is None else colorvec             # :16
        self.sparsity = sparsity
        self._plan_kw = plan_kw
        self._plans = {}

    def plan_for(self, J, sparsity, colorvec, x_len) -> Plan:
        default_cv = isinstance(colorvec, range) and colorvec == range(1, x_len + 1)
        key = (_j_key(J), _sp_key(sparsity), None if default_cv else _index_key(colorvec), self.fdtype)
        p = self._plans.get(key)
        if p is None:
            p = make_plan(J, sparsity, None if default_cv else colorvec, self.fdtype, x_len, self.x1.device,
                          **self._plan_kw)
            self._plans[key] = p
        return p

    def invalidate(self):
        for p in self._plans.values():
            p.destroy()
        self._plans.clear()


def resize_(cache: JacobianCache, i: int):
    """resize!(cache, i)  jacobians.jl:655-661: resizes x1, fx, fx1 and resets colorvec to 1:i."""
    i = int(i)

    def rs(t):
        out = torch.zeros(i, dtype=t.dtype, device=t.device)
        k = min(i, t.numel())
        out[:k] = t.reshape(-1)[:k]
        return out

    cache.x1 = rs(cache.x1)
    cache.x2 = torch.zeros_like(cache.x1)
    cache.fx = rs(cache.fx)
    if cache.fx1 is not None:
        cache.fx1 = rs(cache.fx1)
    cache.colorvec = range(1, i + 1)
    cache.invalidate()
    return None


# ------------------------------------------------------------------------------------------------ colouring
def matrix_colors(A, device=None) -> torch.Tensor:
    """ArrayInterface.matrix_colors(A) on the device: an Int64 CUDA tensor of 1-based colours, ready to be passed as
    `colorvec`.  Tridiagonal -> 1,2,3,...; BandedMatrix(l,u) -> cycle 1:(l+u+1) (ArrayInterface's closed forms);
    SparseMatrixCSC -> a valid distance-2 column colouring (deterministic Jones-Plassmann, fdb_matrix_colors_csc);
    dense tensors -> 1:n (ArrayInterface: eachindex of the columns)."""
    lib = L.lib()
    if isinstance(A, Tridiagonal):
        n, l, u = A.n, 1, 1
        dev = A.buf.device if device is None else torch.device(device)
    elif isinstance(A, BandedMatrix):
        n, l, u = A.n, A.l, A.u
        dev = (A.data.device if isinstance(A.data, torch.Tensor) and A.data.is_cuda else torch.device("cuda")) if device is None else torch.device(device)
    elif isinstance(A, SparseMatrixCSC):
        dev = torch.device("cuda") if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        out = torch.zeros(max(A.n, 1), dtype=torch.int64, device=dev)
        cp, k1 = _index_ptr(A.colptr)
        rv, k2 = _index_ptr(A.rowval)
        nc, nr = C.c_int64(), C.c_int64()
        with torch.cuda.device(dev):
            L.check(lib.fdb_matrix_colors_csc(A.m, A.n, cp, rv, out.data_ptr(), C.byref(nc), C.byref(nr)))
        out = out[: A.n]
        out.n_colors, out.n_rounds = nc.value, nr.value
        return out
    elif isinstance(A, BandedBlockBandedMatrix):
        return torch.from_numpy(A.matrix_colors()).to(torch.device("cuda") if device is None else torch.device(device))
    elif isinstance(A, torch.Tensor):
        n = A.shape[1] if A.dim() == 2 else 1
        return torch.arange(1, n + 1, dtype=torch.int64, device=A.device if A.is_cuda else (device or "cuda"))
    else:
        raise TypeError(f"matrix_colors: unsupported type {type(A)}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    out = torch.zeros(max(n, 1), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        L.check(lib.fdb_matrix_colors_banded(n, l, u, out.data_ptr(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
    return out[:n]


def check_coloring(A: "SparseMatrixCSC", colorvec) -> int:
    """Number of (row, colour) collisions of `colorvec` on the CSC pattern (0 = valid for the decompression)."""
    cp, k1 = _index_ptr(A.colptr)
    rv, k2 = _index_ptr(A.rowval)
    cv, k3 = _index_ptr(colorvec)
    out = C.c_int64()
    L.check(L.lib().fdb_check_coloring_csc(A.m, A.n, cp, rv, cv, C.byref(out)))
    return out.value


# ------------------------------------------------------------------------------------------------ the public call
def _as_fn(f, m, n, device, plan_batch, complex_=False):
    if isinstance(f, NativeFn):
        return f.address, f.ctx_ptr, None
    w = _PyFn(f, m, n, device, bool(getattr(f, "batched", False)), complex_)
    return L.fn_address(w.cfunc), None, w


def finite_difference_jacobian_(J, f, x, cache=None, f_in=None, returntype=None, *, fdtype=None, relstep=None,
                                absstep=None, colorvec=None, sparsity=_DEFAULT, dir=True, stream=None):
    """finite_difference_jacobian!(J, f, x, cache::JacobianCache, f_in=nothing; relstep, absstep, colorvec, sparsity, dir)
    (jacobians.jl:504-514), or — when `cache` is None or an fdtype string — the cache-less form
    finite_difference_jacobian!(J, f, x, fdtype, returntype, f_in; relstep, absstep, colorvec, sparsity) (:446-455).

    J: SparseMatrixCSC | BandedMatrix | Tridiagonal | column-major dense CUDA tensor (zeros_colmajor).
    f: Python callable f(fx, x) on CUDA tensors (set f.batched=True for 2-D batches) or a NativeFn.
    x: float64 CUDA tensor (any shape; flattened like Julia's vec).  Never modified.
    Returns None.
    """
    if isinstance(cache, str) or cache is None:
        # cache-less entry :446-471
        fd = cache if isinstance(cache, str) else (fdtype or "forward")
        if isinstance(f_in, torch.dtype):
            f_in = None
        if sparsity is _DEFAULT:
            sparsity = J if _has_sparsestruct(J) else None                              # :455
        xv = x.reshape(-1)
        m = _shape_of(J)[0]
        if f_in is None and _fdtype_code(fd) == L.FDB_FORWARD:
            fx = torch.zeros_like(xv) if m == xv.numel() else torch.zeros(m, dtype=torch.float64, device=x.device)
            c = JacobianCache(xv, fx, fd)                                                # :456-463 (f(fx,x) runs inside)
            # the reference evaluates f(fx,x) here and passes cache.fx as f_in; the plan does the same evaluation
            # first thing inside fdb_jacobian (same call count, same order)
            return finite_difference_jacobian_(J, f, x, c, None, relstep=relstep, absstep=absstep,
                                               colorvec=range(1, xv.numel() + 1) if colorvec is None else colorvec,
                                               sparsity=sparsity, stream=stream)
        if f_in is None:
            c = JacobianCache(xv, fd)                                                    # :464-465
        else:
            c = JacobianCache(xv, f_in.reshape(-1), fd)                                  # :466-467
        return finite_difference_jacobian_(J, f, x, c, c.fx if f_in is not None else None, relstep=relstep,
                                           absstep=absstep,
                                           colorvec=range(1, xv.numel() + 1) if colorvec is None else colorvec,
                                           sparsity=sparsity, stream=stream)

    if not isinstance(cache, JacobianCache):
        raise TypeError("cache must be a JacobianCache, an fdtype string, or None")
    if not _is_cuda(x) or x.dtype != torch.float64:
        raise TypeError("x must be a float64 CUDA tensor: the B200 path has no CPU implementation")
    fd = _fdtype_code(cache.fdtype)
    colorvec = cache.colorvec if colorvec is None else colorvec                          # :511
    sparsity = cache.sparsity if sparsity is _DEFAULT else sparsity                 # :512
    xv = x.reshape(-1)
    if not xv.is_contiguous():
        xv = xv.contiguous()
    n = xv.numel()
    m, ncols = _shape_of(J)                                                              # :515
    if ncols != n:
        raise ValueError(f"size(J,2)={ncols} != length(x)={n}")
    plan = cache.plan_for(J, sparsity, colorvec, n)
    if isinstance(J, DenseColumnBlock) and plan.dense_range() != (J.col0, J.col0 + J.ncols):
        raise ValueError(f"DenseColumnBlock [{J.col0}, {J.col0 + J.ncols}) is not this rank's column block {plan.dense_range()}")
    jv = _j_values(J)
    if not _is_cuda(jv) or jv.dtype != torch.float64:
        raise TypeError("J's value storage must be a float64 CUDA tensor")
    if cache.fx.numel() != m:
        raise ValueError(f"length(cache.fx)={cache.fx.numel()} != size(J,1)={m} (use the 3-array constructor)")
    addr, ctx, pyfn = _as_fn(f, m, n, x.device, 1, fd == L.FDB_COMPLEX)
    if stream is None:
        stream = torch.cuda.current_stream(x.device).cuda_stream
    if fd == L.FDB_COMPLEX:
        # jacobians.jl:623-648: one complex evaluation per colour, J = imag(f(x + im*eps*e_k))/eps, eps = eps(Float64)
        with torch.cuda.device(x.device):
            st = L.lib().fdb_jacobian_complex(plan.handle, addr, ctx, xv.data_ptr(), jv.data_ptr(), C.c_void_p(stream))
        if st == L.FDB_ERR_CALLBACK and pyfn is not None and pyfn.exc is not None:
            exc, pyfn.exc = pyfn.exc, None
            raise exc
        L.check(st)
        cache._last_plan = plan
        return None
    fin_ptr = None
    if f_in is not None and fd == L.FDB_FORWARD:
        f_in = f_in.reshape(-1)
        if not _is_cuda(f_in) or f_in.dtype != torch.float64 or f_in.numel() != m:
            raise TypeError("f_in must be a float64 CUDA tensor of length size(J,1)")
        fin_ptr = f_in.data_ptr()
    with torch.cuda.device(x.device):
        st = L.lib().fdb_jacobian(plan.handle, addr, ctx, xv.data_ptr(), jv.data_ptr(), cache.fx.data_ptr(), fin_ptr,
                                  L.STEP_DEFAULT if relstep is None else float(relstep),
                                  L.STEP_DEFAULT if absstep is None else float(absstep), float(dir), C.c_void_p(stream))
    if st == L.FDB_ERR_CALLBACK and pyfn is not None and pyfn.exc is not None:
        exc, pyfn.exc = pyfn.exc, None
        raise exc                                          # user f threw: propagate like Julia does
    L.check(st)
    cache._last_plan = plan
    return None


finite_difference_jacobian_b = finite_difference_jacobian_  # alias ("bang")


# ------------------------------------------------------------------------------------------------ JVP (src/jvp.jl)
class JVPCache:
    """Mirror of FiniteDiff.JVPCache{X1, FX1, fdtype} (src/jvp.jl:14-17): fields x1, fx1.

        JVPCache(x, fdtype="forward")          allocating: x1 = copy(x), fx1 = copy(x)      (:39-44)
        JVPCache(x, fx1, fdtype="forward")     non-allocating: aliases the arrays passed in (:73-80)
    """

    def __init__(self, x, fx1=None, fdtype="forward"):
        if isinstance(fx1, str):
            fdtype, fx1 = fx1, None
        self.fdtype = fdtype.lstrip(":") if isinstance(fdtype, str) else fdtype
        code = _fdtype_code(self.fdtype)
        if not _is_cuda(x):
            raise TypeError("JVPCache needs CUDA float64 tensors (this path has no CPU implementation)")
        if fx1 is None:
            self.x1, self.fx1 = x.clone(), x.clone()
        else:
            self.x1, self.fx1 = x, fx1
        self._code = code
        self._plan = None

    def plan(self, m: int, n: int) -> "Plan":
        if self._plan is None or self._plan_key != (m, n):
            if self._code == L.FDB_COMPLEX:
                # jvp.jl:248-250
                raise ValueError("finite_difference_jvp doesn't support :complex-mode finite diff")
            h = C.c_void_p()
            o = _opts(self._code, _device_index(self.x1.device))
            L.check(L.lib().fdb_jvp_plan_create(C.byref(h), m, n, C.byref(o)))
            self._plan, self._plan_key = Plan(h.value), (m, n)
        return self._plan


def finite_difference_jvp_(jvp, f, x, v, cache=None, f_in=None, *, relstep=None, absstep=None, dir=True, stream=None):
    """finite_difference_jvp!(jvp, f, x, v, cache::JVPCache, f_in=nothing; relstep, absstep, dir) (src/jvp.jl:238-274), or
    — when `cache` is None or an fdtype string — the cache-less form (:198-216).
    jvp[m], x[n], v[n]: float64 CUDA tensors; f(fx, x) as for the Jacobian.  Returns None."""
    if isinstance(cache, str) or cache is None:
        fd = cache if isinstance(cache, str) else "forward"
        xv = x.reshape(-1)
        if f_in is not None:
            c = JVPCache(xv.clone(), f_in.reshape(-1).clone(), fd)                      # JVPCache(x, f_in, fdtype)  :209
            return finite_difference_jvp_(jvp, f, x, v, c, c.fx1, relstep=relstep, absstep=absstep, stream=stream)
        c = JVPCache(xv, fd)                                                            # :210-215 (f(fx,x) runs inside)
        if jvp.numel() != xv.numel():
            c.fx1 = torch.zeros(jvp.numel(), dtype=torch.float64, device=x.device)
        return finite_difference_jvp_(jvp, f, x, v, c, None, relstep=relstep, absstep=absstep, stream=stream)
    if not isinstance(cache, JVPCache):
        raise TypeError("cache must be a JVPCache, an fdtype string, or None")
    for t in (jvp, x, v):
        if not _is_cuda(t) or t.dtype != torch.float64:
            raise TypeError("jvp, x, v must be float64 CUDA tensors: the B200 path has no CPU implementation")
    xv, vv, jv = x.reshape(-1), v.reshape(-1), jvp.reshape(-1)
    if not (xv.is_contiguous() and vv.is_contiguous() and jv.is_contiguous()):
        raise ValueError("jvp, x, v must be contiguous")
    n, m = xv.numel(), jv.numel()
    if vv.numel() != n:
        raise ValueError("length(v) != length(x)")
    plan = cache.plan(m, n)
    if cache.x1.numel() != n or cache.fx1.numel() != m:
        raise ValueError("JVPCache arrays do not match length(x) / length(jvp)")
    addr, ctx, pyfn = _as_fn(f, m, n, x.device, 1)
    if stream is None:
        stream = torch.cuda.current_stream(x.device).cuda_stream
    fin_ptr = None
    if f_in is not None and cache._code == L.FDB_FORWARD:
        fin_ptr = f_in.reshape(-1).data_ptr()
    with torch.cuda.device(x.device):
        st = L.lib().fdb_jvp(plan.handle, addr, ctx, jv.data_ptr(), xv.data_ptr(), vv.data_ptr(), cache.x1.data_ptr(),
                             cache.fx1.data_ptr(), fin_ptr, L.STEP_DEFAULT if relstep is None else float(relstep),
                             L.STEP_DEFAULT if absstep is None else float(absstep), float(dir), C.c_void_p(stream))
    if st == L.FDB_ERR_CALLBACK and pyfn is not None and pyfn.exc is not None:
        exc, pyfn.exc = pyfn.exc, None
        raise exc
    L.check(st)
    cache._last_plan = plan
    return None


def _shape_of(J):
    if isinstance(J, (SparseMatrixCSC, BandedMatrix, Tridiagonal, BandedBlockBandedMatrix, DenseColumnBlock)):
        return J.shape
    if isinstance(J, torch.Tensor):
        if J.dim() == 1:
            return (J.shape[0], 1)
        return tuple(J.shape)
    raise TypeError(f"unsupported J type {type(J)}")


# ------------------------------------------------------------------------------------------------ Hessian (src/hessians.jl)
class _PyScalarFn:
    """Wraps a scalar Python f(x) -> number on CUDA tensors as an fdb_fn with m = 1.  `batched=True` callables receive
    the (batch, n) points at once and return `batch` values; otherwise f is called once per point with a 1-D tensor."""

    def __init__(self, f: Callable, n: int, device: torch.device, batched: bool):
        self.f, self.n, self.device, self.batched = f, n, device, batched
        self.exc: Optional[BaseException] = None
        self.calls = 0
        self.cfunc = L.FDB_FN(self._tramp)

    def _tramp(self, _ctx, p_fx, p_x, batch, ldfx, ldx, stream):
        try:
            cur = torch.cuda.current_stream(self.device)
            ctx = None
            if (stream or 0) != cur.cuda_stream:
                ctx = torch.cuda.stream(torch.cuda.ExternalStream(stream or 0, device=self.device))
                ctx.__enter__()
            try:
                fx = torch.as_tensor(_DevArray(p_fx, (batch,), (ldfx * 8,)), device=self.device)
                x2 = torch.as_tensor(_DevArray(p_x, (batch, self.n), (ldx * 8, 8)), device=self.device)
                if self.batched:
                    self.calls += int(batch)
                    out = torch.as_tensor(self.f(x2), dtype=torch.float64, device=self.device).reshape(-1)
                    if out.numel() != batch:
                        raise ValueError(f"batched f returned {out.numel()} values for {batch} points")
                    fx.copy_(out)
                else:
                    for b in range(int(batch)):
                        self.calls += 1
                        fx[b] = self.f(x2[b])
            finally:
                if ctx is not None:
                    ctx.__exit__(None, None, None)
            return 0
        except BaseException as e:  # never let an exception cross the C ABI
            self.exc = e
            return 1


_NO_INPLACE = object()


class HessianCache:
    """Mirror of FiniteDiff.HessianCache{T, fdtype, inplace} (src/hessians.jl:1-6): fields xpp, xpm, xmp, xmm.

        HessianCache(x, fdtype="hcentral", inplace=True)               allocating: four copies of x          (:83-89)
        HessianCache(xpp, xpm, xmp, xmm, fdtype="hcentral", inplace)   non-allocating: aliases the arrays    (:67-73)

    The four-array form without `inplace` throws, as the reference does: its default `_hessian_inplace(x)` (:69) names
    a variable that does not exist there.  The B200 path builds its points in plan-owned memory and never writes the
    cache arrays (their end state in the reference, x again, is dropped), so a cache built from another x of the same
    length gives the same Hessian (finitedifftests.jl:608-614).  The immutable branch (inplace=False) computes the same
    values.  Extra keywords (B200-specific): max_batch (points per callback; default: NativeFn.max_batch for a native f,
    1024 for a Python f) and scratch_bytes (cap on the B copies of x)."""

    def __init__(self, *args, fdtype=None, inplace=_NO_INPLACE, max_batch=None, scratch_bytes=0):
        if len(args) >= 4 and all(isinstance(a, torch.Tensor) for a in args[:4]):
            self.xpp, self.xpm, self.xmp, self.xmm = args[:4]
            rest = list(args[4:])
            if rest:
                fdtype = rest.pop(0)
            if rest:
                inplace = rest.pop(0)
            if inplace is _NO_INPLACE:
                raise TypeError("HessianCache(xpp, xpm, xmp, xmm, fdtype) needs `inplace`: the reference's default "
                                "_hessian_inplace(x) refers to an undefined `x` (hessians.jl:69)")
            x = self.xpp
        elif len(args) >= 1:
            x = args[0]
            rest = list(args[1:])
            if rest:
                fdtype = rest.pop(0)
            if rest:
                inplace = rest.pop(0)
            if rest:
                raise TypeError("HessianCache(x, fdtype, inplace) takes at most three positional arguments")
            if not _is_cuda(x):
                raise TypeError("HessianCache needs a CUDA float64 tensor (this path has no CPU implementation)")
            self.xpp, self.xpm, self.xmp, self.xmm = x.clone(), x.clone(), x.clone(), x.clone()
        else:
            raise TypeError("HessianCache(x[, fdtype, inplace]) or HessianCache(xpp, xpm, xmp, xmm, fdtype, inplace)")
        if not _is_cuda(x):
            raise TypeError("HessianCache needs CUDA float64 tensors (this path has no CPU implementation)")
        fdtype = "hcentral" if fdtype is None else fdtype
        self.fdtype = fdtype.lstrip(":") if isinstance(fdtype, str) else fdtype
        _step_fdtype_code(self.fdtype)
        self.inplace = True if inplace is _NO_INPLACE else bool(inplace)
        self.max_batch = None if max_batch is None else int(max_batch)
        self.scratch_bytes = int(scratch_bytes)
        self._plan = None
        self._plan_key = None

    def plan(self, n: int, device, max_batch: int) -> Plan:
        key = (n, str(device), max_batch)
        if self._plan is None or self._plan_key != key:
            h = C.c_void_p()
            o = _opts(_step_fdtype_code(self.fdtype), _device_index(device), max_batch=max_batch,
                      scratch_bytes=self.scratch_bytes)
            L.check(L.lib().fdb_hessian_plan_create(C.byref(h), n, C.byref(o)))
            self._plan, self._plan_key = Plan(h.value), key
        return self._plan


def _hessian_ld(H: torch.Tensor, n: int) -> int:
    """Leading dimension of an (n, n) float64 CUDA view with one unit stride.  H is symmetric bit for bit, so a
    row-major view is filled as the column-major matrix it is the transpose of."""
    if not isinstance(H, torch.Tensor) or not H.is_cuda or H.dtype != torch.float64:
        raise TypeError("H must be a float64 CUDA tensor")
    if H.dim() != 2 or tuple(H.shape) != (n, n):
        raise ValueError(f"size(H) = {tuple(H.shape)} != ({n}, {n})")
    if n <= 1:
        return max(n, 1)
    if H.stride(0) == 1:
        return int(H.stride(1))
    if H.stride(1) == 1:
        return int(H.stride(0))
    raise ValueError("H needs one unit stride (a column- or row-major view)")


def finite_difference_hessian_(H, f, x, cache=None, *, relstep=None, absstep=None, stream=None):
    """finite_difference_hessian!(H, f, x, cache::HessianCache; relstep, absstep) (src/hessians.jl:202-292), or — when
    `cache` is None or an fdtype string — the cache-less form (:181-189).

    H: (n, n) float64 CUDA tensor with one unit stride; every entry is written.
    f: scalar function of a 1-D float64 CUDA tensor (called once per point), a callable with f.batched = True taking
       the (B, n) points and returning B values, or a NativeFn (an fdb_fn writing one scalar per point).
    x: float64 CUDA tensor (any shape; flattened like Julia's vec).  Never modified.  Returns None."""
    if isinstance(cache, str) or cache is None:
        cache = HessianCache(x, "hcentral" if cache is None else cache)                   # :187
    if not isinstance(cache, HessianCache):
        raise TypeError("cache must be a HessianCache, an fdtype string, or None")
    if cache.fdtype != "hcentral":
        raise AssertionError("fdtype == Val(:hcentral)")                                  # :206
    if not _is_cuda(x) or x.dtype != torch.float64:
        raise TypeError("x must be a float64 CUDA tensor: the B200 path has no CPU implementation")
    xv = x.reshape(-1)
    if not xv.is_contiguous():
        xv = xv.contiguous()
    n = xv.numel()
    if cache.xpp.numel() != n:
        raise ValueError(f"length(cache.xpp) = {cache.xpp.numel()} != length(x) = {n}")
    ldH = _hessian_ld(H, n)
    if isinstance(f, NativeFn):
        addr, ctx, pyfn = f.address, f.ctx_ptr, None
        batch = cache.max_batch or f.max_batch
    else:
        pyfn = _PyScalarFn(f, n, x.device, bool(getattr(f, "batched", False)))
        addr, ctx = L.fn_address(pyfn.cfunc), None
        batch = cache.max_batch or 1024
    plan = cache.plan(n, x.device, batch)
    if stream is None:
        stream = torch.cuda.current_stream(x.device).cuda_stream
    with torch.cuda.device(x.device):
        st = L.lib().fdb_hessian(plan.handle, addr, ctx, xv.data_ptr(), H.data_ptr(), ldH,
                                 L.STEP_DEFAULT if relstep is None else float(relstep),
                                 L.STEP_DEFAULT if absstep is None else float(absstep), C.c_void_p(stream))
    if st == L.FDB_ERR_CALLBACK and pyfn is not None and pyfn.exc is not None:
        exc, pyfn.exc = pyfn.exc, None
        raise exc                                          # user f threw: propagate like Julia does
    L.check(st)
    cache._last_plan = plan
    return None


def finite_difference_hessian(f, x, cache=None, *, relstep=None, absstep=None, stream=None) -> torch.Tensor:
    """finite_difference_hessian(f, x[, cache]; relstep, absstep) (src/hessians.jl:140-167): a new (n, n) float64
    tensor, symmetric bit for bit (the reference wraps it in Symmetric)."""
    n = x.numel()
    H = torch.zeros((n, n), dtype=torch.float64, device=x.device)                        # mutable_zeromatrix(x) :164
    finite_difference_hessian_(H, f, x, cache, relstep=relstep, absstep=absstep, stream=stream)
    return H
