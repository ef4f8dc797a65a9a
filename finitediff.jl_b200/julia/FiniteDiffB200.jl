# FiniteDiffB200.jl — Julia host side of the B200 drop-in for FiniteDiff.jl's coloured Jacobian path.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no `julia` binary (SURVEY.md §8c).  The file is the binding a
# maintainer adds; the same C ABI (include/fdjac_b200.h) is exercised end-to-end through the Python/ctypes mirror
# (finitediff.jl_b200/api.py), which keeps the same names and argument meaning.  tests/test_julia_binding_cpu.py checks
# this file against the header without running it: struct layouts (field order / widths), every ccall's symbol and
# argument count, block balance.
#
# What it does: adds METHODS to FiniteDiff.finite_difference_jacobian! (src/jacobians.jl:504-514) and
# FiniteDiff.finite_difference_jvp! (src/jvp.jl:238-247) that dispatch on device arrays (CUDA.CuVector{Float64}) and forward
# the WHOLE colour loop to libfdjac_b200.so with one ccall — not the per-colour hooks (`_colorediteration!`), because a
# host round trip per colour would forfeit the device residency.  Covered: every (J, sparsity) combination the reference's
# hooks serve on this path —
#     DeviceCSC J + CSC sparsity            ext/FiniteDiffSparseArraysExt.jl:38-47 (same pattern) / :20-28 (other pattern)
#     CuMatrix J  + CSC sparsity            ext/FiniteDiffSparseArraysExt.jl:20-28
#     DeviceBanded J or CuMatrix J + Banded ext/FiniteDiffBandedMatricesExt.jl:13-27
#     DeviceTridiagonal J (structured, COO) src/iteration_utils.jl:25-32 with ArrayInterface.findstructralnz
#     CuMatrix J + dense 0/1 prototype      src/jacobians.jl:473-488, 526-527
#     CuMatrix J, sparsity === nothing      src/jacobians.jl:548-557, 590-598 (dense column branch, colorvec quirk included)
#   for Val(:forward), Val(:central) and Val(:complex) (src/jacobians.jl:623-648), plus the JVP, the multi-GPU group and
#   the Hessian of a scalar function (finite_difference_hessian!, src/hessians.jl:202-292: the stock cache-less and
#   out-of-place forms reach it through HessianCache(x) / mutable_zeromatrix(x) on a CuVector).
# Everything else of FiniteDiff.jl (CPU arrays, gradients, out-of-place Jacobians) keeps using the stock package.
module FiniteDiffB200

using FiniteDiff, SparseArrays, CUDA
import FiniteDiff: finite_difference_jacobian!, finite_difference_jvp!, finite_difference_hessian!, JacobianCache, JVPCache,
                  HessianCache

const libfdjac = get(ENV, "FDJAC_B200_LIB", "libfdjac_b200.so")

const FDB_FORWARD, FDB_CENTRAL, FDB_COMPLEX, FDB_HCENTRAL = Cint(0), Cint(1), Cint(2), Cint(3)
const FDB_J_CSC_NZVAL, FDB_J_DENSE, FDB_J_BAND, FDB_J_SLOTS = Cint(0), Cint(1), Cint(2), Cint(3)
const FDB_STEP_DEFAULT = NaN            # relstep / absstep keyword not given (include/fdjac_b200.h)

# mirror of fdb_plan_opts (include/fdjac_b200.h) — field order and widths are checked by tests/test_julia_binding_cpu.py
struct PlanOpts
    fdtype::Int32
    device::Int32
    use_current_device::Int32
    no_drift::Int32
    max_batch::Int64
    scratch_bytes::Int64
    rank::Int32
    world::Int32
    partition::Int32
    strategy::Int32
    use_graph::Int32
    shared_j::Int32
end
PlanOpts(fd; max_batch = 1, rank = 0, world = 1, use_graph = false, shared_j = false) =
    PlanOpts(fd, 0, 1, 0, max_batch, 0, rank, world, 0, 0, use_graph ? 1 : 0, shared_j ? 1 : 0)

# mirror of fdb_plan_info_t
struct PlanInfo
    m::Int64
    n::Int64
    n_entries::Int64
    j_len::Int64
    n_colors::Int64
    n_local_colors::Int64
    n_groups::Int64
    slabs::Int64
    fcalls_per_jacobian::Int64
    device_bytes::Int64
    fdtype::Int32
    jkind::Int32
    sp_kind::Int32
    color_bits::Int32
    alg_bytes_scatter::Int64
    strategy::Int32
    lanes::Int32
    mean_row_jump::Float64
    moved_bytes_scatter::Int64
    staged::Int32
    lists_resident::Int32
end

struct FdbError <: Exception
    status::Cint
    msg::String
end
function check(st::Cint)
    st == 0 && return nothing
    throw(FdbError(st, unsafe_string(ccall((:fdb_last_error, libfdjac), Cstring, ()))))
end

fdcode(::Val{:forward}) = FDB_FORWARD
fdcode(::Val{:central}) = FDB_CENTRAL
fdcode(::Val{:complex}) = FDB_COMPLEX
fdcode(::Val{T}) where {T} = FiniteDiff.fdtype_error(Float64)   # src/epsilons.jl:159-167

# ---- device-side J / sparsity wrappers: the index structure stays on the host exactly as the reference's types hold
#      it (that is what dispatch sees), the VALUES live on the device.
struct DeviceCSC
    host::SparseMatrixCSC{Float64, Int64}   # pattern (colptr / rowval)
    nzval::CuVector{Float64}                # values on the device
end
Base.size(J::DeviceCSC) = size(J.host)
Base.size(J::DeviceCSC, d) = size(J.host, d)

struct DeviceBanded                          # BandedMatrices.BandedMatrix: data[(l+u+1) x n], slot [u+r-c+1, c]
    m::Int
    n::Int
    l::Int
    u::Int
    data::CuVector{Float64}                  # (l+u+1)*n, column-major (ext/FiniteDiffBandedMatricesExt.jl:22)
end
Base.size(J::DeviceBanded) = (J.m, J.n)
Base.size(J::DeviceBanded, d) = d == 1 ? J.m : J.n

struct DeviceTridiagonal                     # LinearAlgebra.Tridiagonal(dl, d, du): one buffer [dl; d; du]
    n::Int
    buf::CuVector{Float64}                   # 3n - 2
end
Base.size(J::DeviceTridiagonal) = (J.n, J.n)
Base.size(J::DeviceTridiagonal, d) = J.n

# ArrayInterface.findstructralnz(::Tridiagonal): band by band (order is irrelevant to the result); slots into [dl; d; du]
function tridiagonal_structure(n::Int)
    rows = vcat(collect(Int64, 2:n), collect(Int64, 1:n), collect(Int64, 1:(n - 1)))
    cols = vcat(collect(Int64, 1:(n - 1)), collect(Int64, 1:n), collect(Int64, 2:n))
    slots = collect(Int64, 1:(3n - 2))
    rows, cols, slots
end

# src/jacobians.jl:473-488 — column-major scan of a dense 0/1 prototype
function dense_prototype_structure(A::AbstractMatrix)
    rows, cols = Int64[], Int64[]
    for j in axes(A, 2), i in axes(A, 1)
        if !iszero(A[i, j])
            push!(rows, i)
            push!(cols, j)
        end
    end
    rows, cols
end

# ---- plans: the per-(pattern, colorvec, fdtype) state the reference rebuilds on every call (jacobians.jl:515-535).
# Cached per index array: a WeakKeyDict keyed on the (mutable) anchor array of the pattern — when the caller drops the
# pattern the entry and its plans go away (finalizer -> fdb_plan_destroy); nothing is pinned forever.
mutable struct Plan
    handle::Ptr{Cvoid}
    roots::Any                     # host index arrays the plan was built from (kept alive for the plan's lifetime)
    function Plan(h, roots = nothing)
        p = new(h, roots)
        finalizer(q -> ccall((:fdb_plan_destroy, libfdjac), Cint, (Ptr{Cvoid},), q.handle), p)
        p
    end
end
const PLANS = WeakKeyDict{Any, Dict{Any, Plan}}()
const PLANS_LOCK = ReentrantLock()

function cached_plan(make::Function, anchor, key)
    lock(PLANS_LOCK) do
        d = get!(() -> Dict{Any, Plan}(), PLANS, anchor)
        get!(make, d, key)
    end
end

# colorvec as the ABI wants it: (pointer, root).  The ROOT must stay referenced (GC.@preserve) across the ccall:
# a freshly collected Vector is returned together with its pointer, never a pointer to a temporary.
function color_arg(cv::AbstractUnitRange, n::Integer)
    (first(cv) == 1 && length(cv) == n) && return (Ptr{Int64}(C_NULL), nothing)      # NULL => 1:n (jacobians.jl:16)
    v = collect(Int64, cv)
    (pointer(v), v)
end
function color_arg(cv::Vector{Int64}, n::Integer)
    (pointer(cv), cv)
end
function color_arg(cv::AbstractVector{<:Integer}, n::Integer)
    v = collect(Int64, cv)
    (pointer(v), v)
end
color_key(cv::AbstractUnitRange) = (:range, first(cv), last(cv))
color_key(cv) = (:vec, objectid(cv), length(cv))

function info(plan::Plan)
    r = Ref{PlanInfo}()
    check(ccall((:fdb_plan_info, libfdjac), Cint, (Ptr{Cvoid}, Ref{PlanInfo}), plan.handle, r))
    r[]
end

# sparsity::SparseMatrixCSC — J is a DeviceCSC (nzval slots) or a dense CuMatrix (ldJ)
function plan_csc(sp::SparseMatrixCSC{Float64, Int64}, Jhost, ldJ::Integer, colorvec, fd::Cint; kw...)
    jk = Jhost === nothing ? FDB_J_DENSE : FDB_J_CSC_NZVAL
    same = Jhost === nothing || Jhost === sp || (Jhost.colptr === sp.colptr && Jhost.rowval === sp.rowval)
    key = (:csc, objectid(sp.rowval), same ? 0 : objectid(Jhost.rowval), jk, ldJ, color_key(colorvec), fd, values(kw))
    cached_plan(sp.colptr, key) do
        h = Ref{Ptr{Cvoid}}(C_NULL)
        opts = Ref(PlanOpts(fd; kw...))
        m, n = size(sp)
        cptr, croot = color_arg(colorvec, n)
        GC.@preserve sp Jhost croot begin
            check(ccall((:fdb_plan_create_csc, libfdjac), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Cint, Ptr{Int64}, Ptr{Int64}, Int64, Ptr{Int64}, Ref{PlanOpts}),
                h, m, n, pointer(sp.colptr), pointer(sp.rowval), jk,
                same ? Ptr{Int64}(C_NULL) : pointer(Jhost.colptr), same ? Ptr{Int64}(C_NULL) : pointer(Jhost.rowval), ldJ,
                cptr, opts))
        end
        Plan(h[], (sp, Jhost, croot))
    end
end

# structural-nonzero lists (Tridiagonal / dense prototype): generic hook src/iteration_utils.jl:25-32
# `structure()` returns (rows, cols, slots-or-nothing); it runs only when the plan is not cached yet, so a cached call does
# no O(nnz) host work (the reference rebuilds these lists on every call, jacobians.jl:522-528)
function plan_coo(structure::Function, anchor, m::Integer, n::Integer, tag, jk::Cint, ld_or_len::Integer, colorvec, fd::Cint; kw...)
    key = (:coo, m, n, tag, jk, ld_or_len, color_key(colorvec), fd, values(kw))
    cached_plan(anchor, key) do
        rows, cols, slots = structure()
        h = Ref{Ptr{Cvoid}}(C_NULL)
        opts = Ref(PlanOpts(fd; kw...))
        cptr, croot = color_arg(colorvec, n)
        GC.@preserve rows cols slots croot begin
            check(ccall((:fdb_plan_create_coo, libfdjac), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Cint, Ptr{Int64}, Int64, Ptr{Int64}, Ref{PlanOpts}),
                h, m, n, length(rows), pointer(rows), pointer(cols), jk,
                slots === nothing ? Ptr{Int64}(C_NULL) : pointer(slots), ld_or_len, cptr, opts))
        end
        Plan(h[], (rows, cols, slots, croot))
    end
end

# sparsity::BandedMatrix(l, u): ext/FiniteDiffBandedMatricesExt.jl:13-27 (whole band)
function plan_banded(anchor, m::Integer, n::Integer, l::Integer, u::Integer, jk::Cint, ldJ::Integer, colorvec, fd::Cint; kw...)
    key = (:banded, m, n, l, u, jk, ldJ, color_key(colorvec), fd, values(kw))
    cached_plan(anchor, key) do
        h = Ref{Ptr{Cvoid}}(C_NULL)
        opts = Ref(PlanOpts(fd; kw...))
        cptr, croot = color_arg(colorvec, n)
        GC.@preserve croot begin
            check(ccall((:fdb_plan_create_banded, libfdjac), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Cint, Int64, Ptr{Int64}, Ref{PlanOpts}),
                h, m, n, l, u, jk, ldJ, cptr, opts))
        end
        Plan(h[], croot)
    end
end

# sparsity === nothing: dense column branch; a non-default colorvec reproduces jacobians.jl:547-557 as written
function plan_dense(anchor, m::Integer, n::Integer, ldJ::Integer, colorvec, fd::Cint; kw...)
    key = (:dense, m, n, ldJ, color_key(colorvec), fd, values(kw))
    cached_plan(anchor, key) do
        h = Ref{Ptr{Cvoid}}(C_NULL)
        opts = Ref(PlanOpts(fd; kw...))
        cptr, croot = color_arg(colorvec, n)
        GC.@preserve croot begin
            check(ccall((:fdb_plan_create_dense_colorvec, libfdjac), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Ptr{Int64}, Ref{PlanOpts}), h, m, n, ldJ, cptr, opts))
        end
        Plan(h[], croot)
    end
end

# ---- user function: a Julia closure f!(fx::CuVector, x::CuVector) behind the fdb_fn C signature
# int f(void* ctx, double* d_fx, const double* d_x, int64 batch, int64 ldfx, int64 ldx, void* stream)
mutable struct FnState
    f::Any
    m::Int
    n::Int
    err::Any
end

function f_trampoline(ctx::Ptr{Cvoid}, fx::CuPtr{Float64}, x::CuPtr{Float64}, batch::Int64, ldfx::Int64, ldx::Int64,
        stream::Ptr{Cvoid})::Cint
    st = unsafe_pointer_to_objref(ctx)::FnState
    try
        for b in 0:(batch - 1)          # plans are created with max_batch = 1 for plain closures
            fxv = unsafe_wrap(CuArray, fx + b * ldfx * sizeof(Float64), st.m)
            xv = unsafe_wrap(CuArray, x + b * ldx * sizeof(Float64), st.n)
            st.f(fxv, xv)               # must only enqueue on the task-local CUDA.jl stream (== `stream`)
        end
        return Cint(0)
    catch err
        st.err = err                    # never unwind through C: report, rethrow on the Julia side
        return Cint(1)
    end
end

# complex-step callback (fdb_fn_c): complex128 arrays, ld* count COMPLEX elements
function f_trampoline_c(ctx::Ptr{Cvoid}, fx::CuPtr{ComplexF64}, x::CuPtr{ComplexF64}, batch::Int64, ldfx::Int64, ldx::Int64,
        stream::Ptr{Cvoid})::Cint
    st = unsafe_pointer_to_objref(ctx)::FnState
    try
        for b in 0:(batch - 1)
            fxv = unsafe_wrap(CuArray, fx + b * ldfx * sizeof(ComplexF64), st.m)
            xv = unsafe_wrap(CuArray, x + b * ldx * sizeof(ComplexF64), st.n)
            st.f(fxv, xv)
        end
        return Cint(0)
    catch err
        st.err = err
        return Cint(1)
    end
end

stepval(::Nothing) = FDB_STEP_DEFAULT
stepval(v::Real) = Float64(v)

# the one place the hot path is entered: fdb_jacobian / fdb_jacobian_complex on the current CUDA.jl stream
function run_plan!(plan::Plan, jvals::CuArray{Float64}, f, x::CuVector{Float64}, fx, f_in, m::Integer, fdtype, relstep, absstep, dir)
    st = FnState(f, m, length(x), nothing)
    rc = Cint(0)
    if fdtype == Val(:complex)
        cf = @cfunction(f_trampoline_c, Cint, (Ptr{Cvoid}, CuPtr{ComplexF64}, CuPtr{ComplexF64}, Int64, Int64, Int64, Ptr{Cvoid}))
        GC.@preserve st x jvals begin
            rc = ccall((:fdb_jacobian_complex, libfdjac), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Ptr{Cvoid}),
                plan.handle, cf, pointer_from_objref(st), pointer(x), pointer(jvals), CUDA.stream().handle)
        end
    else
        cf = @cfunction(f_trampoline, Cint, (Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Int64, Int64, Ptr{Cvoid}))
        GC.@preserve st x jvals fx f_in begin
            rc = ccall((:fdb_jacobian, libfdjac), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64},
                    Float64, Float64, Float64, Ptr{Cvoid}),
                plan.handle, cf, pointer_from_objref(st), pointer(x), pointer(jvals),
                (fx === nothing || eltype(fx) != Float64) ? CU_NULL : pointer(fx),
                f_in === nothing ? CU_NULL : pointer(f_in), stepval(relstep), stepval(absstep), Float64(dir),
                CUDA.stream().handle)
        end
    end
    st.err === nothing || throw(st.err)     # an exception inside f! propagates like in the reference
    check(rc)
    nothing                                  # jacobians.jl:652
end

const DeviceJ = Union{DeviceCSC, DeviceBanded, DeviceTridiagonal, CuMatrix{Float64}}

ld(J::CuMatrix) = max(stride(J, 2), size(J, 1), 1)

# dispatch on (typeof(J), typeof(sparsity)) — what _use_findstructralnz / _use_sparseCSC_common_sparsity / the ext
# methods decide in the reference (jacobians.jl:522-535)
function plan_for(J::DeviceCSC, sp, colorvec, fd)
    sph = sp isa DeviceCSC ? sp.host : sp
    sph isa SparseMatrixCSC || throw(ArgumentError("a DeviceCSC Jacobian needs a SparseMatrixCSC sparsity"))
    (plan_csc(sph, J.host, 0, colorvec, fd), J.nzval)
end
function plan_for(J::DeviceBanded, sp, colorvec, fd)
    (sp isa DeviceBanded && (sp.l, sp.u) == (J.l, J.u)) || throw(ArgumentError("J and sparsity must have the same bandwidths"))
    (plan_banded(J.data, J.m, J.n, J.l, J.u, FDB_J_BAND, 0, colorvec, fd), J.data)
end
function plan_for(J::DeviceTridiagonal, sp, colorvec, fd)
    (plan_coo(() -> tridiagonal_structure(J.n), J.buf, J.n, J.n, :tridiagonal, FDB_J_SLOTS, 3 * J.n - 2, colorvec, fd), J.buf)
end
function plan_for(J::CuMatrix{Float64}, sp, colorvec, fd)
    m, n = size(J)
    if sp === nothing                                                   # jacobians.jl:548-557
        return (plan_dense(J, m, n, ld(J), colorvec, fd), J)
    elseif sp isa DeviceCSC || sp isa SparseMatrixCSC                   # ext/..SparseArraysExt.jl:20-28
        sph = sp isa DeviceCSC ? sp.host : sp
        return (plan_csc(sph, nothing, ld(J), colorvec, fd), J)
    elseif sp isa DeviceBanded                                          # ext/..BandedMatricesExt.jl:13-27, dense target
        return (plan_banded(J, m, n, sp.l, sp.u, FDB_J_DENSE, ld(J), colorvec, fd), J)
    elseif sp isa DeviceTridiagonal
        return (plan_coo(J, m, n, :tridiagonal, FDB_J_DENSE, ld(J), colorvec, fd) do
                rows, cols, _ = tridiagonal_structure(sp.n)
                (rows, cols, nothing)
            end, J)
    elseif sp isa AbstractMatrix                                        # dense 0/1 prototype, jacobians.jl:526-527
        # keyed on the prototype's identity: editing it in place needs a new array (as for every cached pattern)
        return (plan_coo(J, m, n, (:prototype, objectid(sp)), FDB_J_DENSE, ld(J), colorvec, fd) do
                rows, cols = dense_prototype_structure(sp)
                (rows, cols, nothing)
            end, J)
    end
    throw(ArgumentError("unsupported sparsity type $(typeof(sp))"))
end

"""
    finite_difference_jacobian!(J, f!, x::CuVector{Float64}, cache::JacobianCache, f_in = nothing;
                                relstep, absstep, colorvec, sparsity, dir)

Same signature and keyword meaning as `src/jacobians.jl:504-514`.  `J` is a `DeviceCSC`, `DeviceBanded`,
`DeviceTridiagonal` or a dense `CuMatrix{Float64}`; `x`, `cache.fx`, `f_in` are `CuVector{Float64}`.
`relstep` / `absstep` left at their defaults are passed as FDB_STEP_DEFAULT; explicit values (0 included) as given.
"""
function finite_difference_jacobian!(J::DeviceJ, f, x::CuVector{Float64},
        cache::JacobianCache{T1, T2, T3, T4, cType, sType, fdtype, returntype}, f_in = nothing;
        relstep = nothing, absstep = relstep,
        colorvec = cache.colorvec, sparsity = cache.sparsity, dir = true) where {T1, T2, T3, T4, cType, sType, fdtype, returntype}
    size(J, 2) == length(x) || throw(DimensionMismatch("size(J,2) != length(x)"))
    plan, jvals = plan_for(J, sparsity, colorvec, fdcode(fdtype))
    run_plan!(plan, jvals, f, x, cache.fx, f_in, size(J, 1), fdtype, relstep, absstep, dir)
end

# ---- JVP: finite_difference_jvp!(jvp, f, x, v, cache::JVPCache, f_in; relstep, absstep, dir)   src/jvp.jl:238-274
const JVP_PLANS = Dict{Tuple{Int, Int, Cint}, Plan}()

function jvp_plan(m::Integer, n::Integer, fd::Cint)
    lock(PLANS_LOCK) do
        get!(JVP_PLANS, (Int(m), Int(n), fd)) do
            h = Ref{Ptr{Cvoid}}(C_NULL)
            opts = Ref(PlanOpts(fd))
            check(ccall((:fdb_jvp_plan_create, libfdjac), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ref{PlanOpts}), h, m, n, opts))
            Plan(h[])
        end
    end
end

function finite_difference_jvp!(jvp::CuVector{Float64}, f, x::CuVector{Float64}, v::CuVector{Float64},
        cache::JVPCache{X1, FX1, fdtype}, f_in = nothing;
        relstep = nothing, absstep = relstep, dir = true) where {X1, FX1, fdtype}
    fdtype == Val(:complex) && error("finite_difference_jvp doesn't support :complex-mode finite diff")   # jvp.jl:248-250
    plan = jvp_plan(length(jvp), length(x), fdcode(fdtype))
    st = FnState(f, length(jvp), length(x), nothing)
    cf = @cfunction(f_trampoline, Cint, (Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Int64, Int64, Ptr{Cvoid}))
    rc = Cint(0)
    GC.@preserve st jvp x v cache f_in begin
        rc = ccall((:fdb_jvp, libfdjac), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64},
                CuPtr{Float64}, Float64, Float64, Float64, Ptr{Cvoid}),
            plan.handle, cf, pointer_from_objref(st), pointer(jvp), pointer(x), pointer(v), pointer(cache.x1), pointer(cache.fx1),
            f_in === nothing ? CU_NULL : pointer(f_in), stepval(relstep), stepval(absstep), Float64(dir), CUDA.stream().handle)
    end
    st.err === nothing || throw(st.err)
    check(rc)
    nothing
end

# ---- Hessian: finite_difference_hessian!(H, f, x, cache::HessianCache; relstep, absstep)   src/hessians.jl:202-292
# f(x::CuVector) returns a number and is called once per point; wrap it in BatchedScalar(f, max_batch) when it can take
# the points of a batch at once: f(X) with X an n x B CuMatrix view (column b = point b) returning B numbers.
struct BatchedScalar{F}
    f::F
    max_batch::Int
end

const HESSIAN_PLANS = Dict{Tuple{Int, Int}, Plan}()

function hessian_plan(n::Integer, max_batch::Integer)
    lock(PLANS_LOCK) do
        get!(HESSIAN_PLANS, (Int(n), Int(max_batch))) do
            h = Ref{Ptr{Cvoid}}(C_NULL)
            opts = Ref(PlanOpts(FDB_HCENTRAL; max_batch = max_batch))
            check(ccall((:fdb_hessian_plan_create, libfdjac), Cint, (Ref{Ptr{Cvoid}}, Int64, Ref{PlanOpts}), h, n, opts))
            Plan(h[])
        end
    end
end

# fdb_fn with m = 1: point b's scalar goes to fx[b*ldfx]
function scalar_trampoline(ctx::Ptr{Cvoid}, fx::CuPtr{Float64}, x::CuPtr{Float64}, batch::Int64, ldfx::Int64, ldx::Int64,
        stream::Ptr{Cvoid})::Cint
    st = unsafe_pointer_to_objref(ctx)::FnState
    try
        if st.f isa BatchedScalar
            X = view(unsafe_wrap(CuArray, x, (Int(ldx), Int(batch))), 1:st.n, :)
            vals = st.f.f(X)
            copyto!(unsafe_wrap(CuArray, fx, Int(batch)), Float64.(vals))       # ldfx == 1
        else
            for b in 0:(batch - 1)
                xv = unsafe_wrap(CuArray, x + b * ldx * sizeof(Float64), st.n)
                fill!(unsafe_wrap(CuArray, fx + b * ldfx * sizeof(Float64), 1), Float64(st.f(xv)))
            end
        end
        return Cint(0)
    catch err
        st.err = err
        return Cint(1)
    end
end

"""
    finite_difference_hessian!(H::CuMatrix{Float64}, f, x::CuVector{Float64}, cache::HessianCache; relstep, absstep)

Same signature and keyword meaning as `src/hessians.jl:202-205`; `fdtype` must be `Val(:hcentral)` (`:206`).  The cache
arrays are not used (the points are built in plan-owned memory) and keep their contents.  Every entry of `H` is
written; `H[j,i]` is a bit copy of `H[i,j]` (`copytri!`, `:291`).
"""
function finite_difference_hessian!(H::CuMatrix{Float64}, f, x::CuVector{Float64},
        cache::HessianCache{T, fdtype, inplace};
        relstep = nothing, absstep = relstep) where {T, fdtype, inplace}
    @assert fdtype == Val(:hcentral)
    n = length(x)
    size(H) == (n, n) || throw(DimensionMismatch("size(H) != (length(x), length(x))"))
    plan = hessian_plan(n, f isa BatchedScalar ? f.max_batch : 1)
    st = FnState(f, 1, n, nothing)
    cf = @cfunction(scalar_trampoline, Cint, (Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Int64, Int64, Ptr{Cvoid}))
    rc = Cint(0)
    GC.@preserve st H x begin
        rc = ccall((:fdb_hessian, libfdjac), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Float64, Float64, Ptr{Cvoid}),
            plan.handle, cf, pointer_from_objref(st), pointer(x), pointer(H), Int64(ld(H)), stepval(relstep),
            stepval(absstep), CUDA.stream().handle)
    end
    st.err === nothing || throw(st.err)
    check(rc)
    nothing
end

# ---- several GPUs from ONE call: fdb_group_* (colours / dense column blocks partitioned over `devices`; devices[1] is the
#      root and owns x, J, cache.fx; every member's scatter kernel stores its entries straight into the root's J).
mutable struct Group
    handle::Ptr{Cvoid}
    n::Int
    roots::Any
    function Group(h, n, roots)
        g = new(h, n, roots)
        finalizer(q -> ccall((:fdb_group_destroy, libfdjac), Cint, (Ptr{Cvoid},), q.handle), g)
        g
    end
end

function group_csc(J::DeviceCSC, colorvec, fdtype, devices::Vector{Cint}; kw...)
    sp = J.host
    h = Ref{Ptr{Cvoid}}(C_NULL)
    opts = Ref(PlanOpts(fdcode(fdtype); kw...))
    m, n = size(sp)
    cptr, croot = color_arg(colorvec, n)
    GC.@preserve sp croot devices begin
        check(ccall((:fdb_group_create_csc, libfdjac), Cint,
            (Ref{Ptr{Cvoid}}, Cint, Ptr{Cint}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Cint, Ptr{Int64}, Ptr{Int64}, Int64, Ptr{Int64},
                Ref{PlanOpts}),
            h, length(devices), pointer(devices), m, n, pointer(sp.colptr), pointer(sp.rowval), FDB_J_CSC_NZVAL,
            Ptr{Int64}(C_NULL), Ptr{Int64}(C_NULL), 0, cptr, opts))
    end
    Group(h[], length(devices), (sp, croot))
end

function group_banded(J::DeviceBanded, colorvec, fdtype, devices::Vector{Cint}; kw...)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    opts = Ref(PlanOpts(fdcode(fdtype); kw...))
    cptr, croot = color_arg(colorvec, J.n)
    GC.@preserve croot devices begin
        check(ccall((:fdb_group_create_banded, libfdjac), Cint,
            (Ref{Ptr{Cvoid}}, Cint, Ptr{Cint}, Int64, Int64, Int64, Int64, Cint, Int64, Ptr{Int64}, Ref{PlanOpts}),
            h, length(devices), pointer(devices), J.m, J.n, J.l, J.u, FDB_J_BAND, 0, cptr, opts))
    end
    Group(h[], length(devices), croot)
end

function group_dense(J::CuMatrix{Float64}, fdtype, devices::Vector{Cint}; kw...)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    opts = Ref(PlanOpts(fdcode(fdtype); kw...))
    m, n = size(J)
    GC.@preserve devices begin
        check(ccall((:fdb_group_create_dense, libfdjac), Cint,
            (Ref{Ptr{Cvoid}}, Cint, Ptr{Cint}, Int64, Int64, Int64, Ref{PlanOpts}),
            h, length(devices), pointer(devices), m, n, ld(J), opts))
    end
    Group(h[], length(devices), nothing)
end

# fs[i]: the closure member i calls (its arrays live on devices[i]); x, jvals, fx, f_in live on devices[1]
function group_jacobian!(g::Group, jvals::CuArray{Float64}, fs::Vector, x::CuVector{Float64}, m::Integer;
        fx = nothing, f_in = nothing, relstep = nothing, absstep = relstep, dir = true)
    states = [FnState(f, m, length(x), nothing) for f in fs]
    ctxs = Ptr{Cvoid}[pointer_from_objref(s) for s in states]
    cf = @cfunction(f_trampoline, Cint, (Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Int64, Int64, Ptr{Cvoid}))
    rc = Cint(0)
    GC.@preserve states ctxs x jvals fx f_in begin
        rc = ccall((:fdb_group_jacobian, libfdjac), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Ptr{Cvoid}}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64}, CuPtr{Float64},
                Float64, Float64, Float64, Ptr{Cvoid}),
            g.handle, cf, pointer(ctxs), pointer(x), pointer(jvals), fx === nothing ? CU_NULL : pointer(fx),
            f_in === nothing ? CU_NULL : pointer(f_in), stepval(relstep), stepval(absstep), Float64(dir), CUDA.stream().handle)
    end
    for s in states
        s.err === nothing || throw(s.err)
    end
    check(rc)
    nothing
end

# ---- column-block shards (few-colour problems on several GPUs): one process per GPU, each owning the columns c0+1:c1.
# `sub` is the block's pattern (colptr slice rebased to 1, rows rebased to the block's first row), `f_rows!` computes
# that row range from the x slice the rows depend on, `eps` holds the step sizes of the FULL x (color_eps! below).
function color_eps!(eps::CuVector{Float64}, epsplan::Plan, x::CuVector{Float64}; relstep = nothing, absstep = relstep, dir = true)
    check(ccall((:fdb_color_eps, libfdjac), Cint,
        (Ptr{Cvoid}, CuPtr{Float64}, Float64, Float64, Float64, CuPtr{Float64}, Ptr{Cvoid}),
        epsplan.handle, pointer(x), stepval(relstep), stepval(absstep), Float64(dir), pointer(eps), CUDA.stream().handle))
    eps
end

function eps_plan(n::Integer, colorvec::Vector{Int64}, fd::Cint)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    opts = Ref(PlanOpts(fd))
    GC.@preserve colorvec begin
        check(ccall((:fdb_eps_plan_create, libfdjac), Cint, (Ref{Ptr{Cvoid}}, Int64, Ptr{Int64}, Ref{PlanOpts}),
            h, n, pointer(colorvec), opts))
    end
    Plan(h[], colorvec)
end

set_external_eps!(plan::Plan, eps::CuVector{Float64}) =
    check(ccall((:fdb_plan_set_external_eps, libfdjac), Cint, (Ptr{Cvoid}, CuPtr{Float64}), plan.handle, pointer(eps)))

end # module
