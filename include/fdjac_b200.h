/*
 * fdjac_b200.h — C ABI of libfdjac_b200.so: the B200 (sm_100a) drop-in for ONE path of
 * FiniteDiff.jl — the cached, in-place, graph-coloured Jacobian
 *     finite_difference_jacobian!(J, f!, x, cache::JacobianCache; colorvec, sparsity)
 *     (reference: src/jacobians.jl:504-653 and the hooks it dispatches to).
 *
 * Boundary rules
 *   - plain C, extern "C"; pointers + sizes only; no C++/torch types; never throws.
 *   - every entry point returns an fdb_status; fdb_last_error() gives the thread-local message.
 *   - index arrays cross the ABI exactly as Julia stores them: Int64, 1-BASED
 *     (SparseMatrixCSC{Float64,Int64}.colptr / .rowval, Vector{Int} colorvec), and may live in
 *     HOST or DEVICE memory (detected with cudaPointerGetAttributes) — pointer(J.colptr) can be
 *     passed with no conversion.  The plan keeps private, compressed device copies.
 *   - x, fx, J value buffers are DEVICE pointers (fdb_jacobian) or HOST pointers
 *     (fdb_jacobian_host, which stages H2D/D2H itself).  Caller owns every buffer it passes.
 *   - one in-flight call per plan; calls are stream-ordered and asynchronous (no host sync
 *     inside fdb_jacobian).  Different plans may be used concurrently from different threads.
 *
 * Each entry point cites the reference interface it replaces; the Julia-side binding is in
 * finitediff.jl_b200/julia/FiniteDiffB200.jl and INTEGRATION.md.
 */
#ifndef FDJAC_B200_H
#define FDJAC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDB_ABI_VERSION 2

/* "keyword not given" for relstep / absstep (jacobians.jl:508-510 defaults: relstep = default_relstep(fdtype, T),
 * absstep = relstep).  Any other value, 0 included, is used as passed: relstep = 0 is a pure absolute step,
 * absstep = 0 a pure relative one, as in the reference. */
#define FDB_STEP_DEFAULT (__builtin_nan(""))

typedef enum {
  FDB_OK = 0,
  FDB_ERR_INVALID = 1,     /* bad argument / inconsistent pattern (the reference would throw / @assert) */
  FDB_ERR_CUDA = 2,        /* a CUDA runtime call failed (message has the cudaError string) */
  FDB_ERR_CALLBACK = 3,    /* user f! returned non-zero: the colour loop was aborted (Julia: exception in f) */
  FDB_ERR_NOMEM = 4,
  FDB_ERR_UNSUPPORTED = 5, /* e.g. fdtype other than forward/central (epsilons.jl:159-167 fdtype_error) */
  FDB_ERR_NO_DEVICE = 6    /* no CUDA device: this library has NO CPU fallback */
} fdb_status;

/* fdtype — the Val(:forward)/Val(:central)/Val(:complex) type parameter of JacobianCache (jacobians.jl:1-9).
 * FDB_COMPLEX is the complex-step colour loop (jacobians.jl:623-648): x + im*eps, J = imag(f)/eps, eps = eps(Float64);
 * plans of that type are driven through fdb_jacobian_complex with a complex128 callback.
 * FDB_HCENTRAL is the Val(:hcentral) parameter of HessianCache (hessians.jl:1-6): only Hessian plans take it
 * (fdb_hessian_plan_create), and the Hessian plan takes nothing else (hessians.jl:206). */
enum { FDB_FORWARD = 0, FDB_CENTRAL = 1, FDB_COMPLEX = 2, FDB_HCENTRAL = 3 };

/* Where `J[row, col] = v` lands — what the reference decides by dispatch on typeof(J). */
typedef enum {
  FDB_J_CSC_NZVAL = 0, /* J::SparseMatrixCSC with the sparsity's pattern: nzval[p]   (ext/FiniteDiffSparseArraysExt.jl:38-47) */
  FDB_J_DENSE = 1,     /* J::Matrix column-major, leading dimension ldJ              (ext/..SparseArraysExt.jl:20-28, iteration_utils.jl:25-32) */
  FDB_J_BAND = 2,      /* J::BandedMatrix data[(l+u+1) x n], slot [u+r-c+1, c]        (ext/FiniteDiffBandedMatricesExt.jl:13-27) */
  FDB_J_SLOTS = 3      /* structured J (e.g. Tridiagonal): explicit 1-based slot per structural entry (iteration_utils.jl:25-32) */
} fdb_jkind;

/*
 * User function f!(fx, x) — replaces the Julia closure called at jacobians.jl:563,605-606.
 * Evaluate `batch` points: for b in [0,batch):  d_fx[b*ldfx .. +m) = f(d_x[b*ldx .. +n)).
 * Must only ENQUEUE work on `stream` (a cudaStream_t) and must not synchronise.  Return 0 on
 * success; any other value aborts the Jacobian and is reported as FDB_ERR_CALLBACK.
 * From Julia: @cfunction(f_trampoline, Cint, (Ptr{Cvoid}, CuPtr{Float64}, CuPtr{Float64}, Int64, Int64, Int64, Ptr{Cvoid})).
 * The plan is created with max_batch = 1 for callbacks that can only do one point per call.
 */
typedef int (*fdb_fn)(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx,
                      void *stream);

/* Complex-step variant of the callback (fdtype = FDB_COMPLEX): d_fx / d_x are complex128 arrays (re, im interleaved:
 * cuDoubleComplex / ComplexF64); ldfx / ldx count COMPLEX elements.  Same rules as fdb_fn. */
typedef int (*fdb_fn_c)(void *ctx, void *d_fx, const void *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);

/* Plan options (all fields have a usable zero default). */
typedef struct {
  int32_t fdtype;          /* FDB_FORWARD (default, as jacobians.jl:13) or FDB_CENTRAL */
  int32_t device;          /* CUDA device ordinal; -1 or 0-initialised+use_current => current device */
  int32_t use_current_device; /* 1: ignore `device`, use cudaGetDevice() */
  int32_t no_drift;        /* 0 (default): replay the reference's (x1+eps)-eps drift of earlier colours bit-exactly
                              (jacobians.jl:562,584); 1: perturb from the pristine x */
  int64_t max_batch;       /* points per f! callback invocation; 0/1 => one point per call */
  int64_t scratch_bytes;   /* budget for the stacked f! outputs; 0 => 8 GiB */
  int32_t rank, world;     /* colour partition over GPUs (one process per GPU): this plan handles the colours
                              owned by `rank` of `world`; world<=1 => all colours */
  int32_t partition;       /* 0: round-robin colours; 1: nnz-balanced (LPT) */
  int32_t strategy;        /* CSC scatter: 0 auto; 1 one fused pass over J's storage order; 2 colour-major entry lists, a
                              launch per group of L2-resident f! outputs, overlapped with the next group's f!; 3 colour-major
                              lists with every f! output resident: one launch at the end (see fdb_plan_info_t.strategy) */
  int32_t use_graph;       /* 1: capture the whole call (library kernels + the callback's launches) into a CUDA graph on
                              first use and replay it while (f, ctx, buffers, scalars) stay the same.  The callback must
                              be capture-safe: enqueue-only on the given stream, no allocation, no host-side state. */
  int32_t shared_j;        /* 1: the J passed to fdb_jacobian is SHARED with other ranks' plans (a peer-mapped pointer to one
                              buffer, e.g. rank 0's): this plan only stores the entries / columns it owns and never zero-fills
                              J — the owner of the buffer zero-fills it (when the scatter is not self-defining) and orders
                              the ranks (fdb_sync_barrier / fdb_group_jacobian do both) */
} fdb_plan_opts;

typedef struct fdb_plan fdb_plan;

typedef struct {
  int64_t m, n;
  int64_t n_entries;       /* structural entries the scatter writes per Jacobian (nnz; in-band slots for banded) */
  int64_t j_len;           /* doubles in J's value storage */
  int64_t n_colors;        /* maximum(colorvec) */
  int64_t n_local_colors;  /* colours this rank evaluates */
  int64_t n_groups;        /* scatter launches per Jacobian (1 => fully fused single pass) */
  int64_t slabs;           /* colours whose f! outputs are resident at once */
  int64_t fcalls_per_jacobian; /* f! evaluations (points) per call: 1+C fwd, 2C central (local colours only) */
  int64_t device_bytes;    /* device memory held by the plan */
  int32_t fdtype, jkind, sp_kind, color_bits;
  int64_t alg_bytes_scatter; /* SURVEY.md §8(d) algorithmic bytes of the diff+scatter per Jacobian */
  int32_t strategy;        /* chosen scatter strategy: 0 fused single pass, 1 per-colour column lists */
  int32_t lanes;           /* lanes per column of the column-list kernel */
  double mean_row_jump;    /* mean |row[e+1]-row[e]| over consecutive entries (gather locality metric) */
  int64_t moved_bytes_scatter; /* COMPULSORY bytes of the shipped diff+scatter formulation per Jacobian (this rank): every
                              index / slab / fx / J byte it must move once — the roofline numerator.  CSC fused pass:
                              E*(4 + |colour| + 8*slabs_read + 8) [+ 8m fx, forward]; colour-major lists: E*(4 + |slot| +
                              8*slabs_read + 8) [+ 8m]; explicit destinations: + 8 per entry; banded / dense: = alg_bytes;
                              TMA-staged fused pass: E*(2 + |colour| + 8) + 8m*(slabs_read*C [+ 1]) */
  int32_t staged;          /* 1: the fused pass runs in its TMA-staged form (row-local pattern: slab windows staged through
                              shared memory by cp.async.bulk, 16-bit row offsets) */
  int32_t lists_resident;  /* 1: colour-major lists with every local colour's f! output resident (one launch) */
} fdb_plan_info_t;

typedef struct {
  int64_t jacobians;       /* completed fdb_jacobian calls */
  int64_t f_points;        /* f! points evaluated */
  int64_t f_invocations;   /* callback invocations */
  int64_t kernel_launches; /* library kernels launched (excludes the user's f!) */
  int64_t scatter_launches;
} fdb_counters_t;

/* ---- library ---- */
int fdb_abi_version(void);
/* thread-local message of the last failing call on this thread */
const char *fdb_last_error(void);
/* number of usable CUDA devices (0 => every compute entry point returns FDB_ERR_NO_DEVICE) */
int fdb_device_count(void);

/* ---- step size: src/epsilons.jl:134-144 / :26-29,50-53,74-77 (host-side scalars, for callers and tests).
 *      FDB_HCENTRAL: default relstep eps(Float64)^(1/4) = 2^-13; the step is max(relstep*|x|, absstep), no dir. ---- */
double fdb_default_relstep(int fdtype);
double fdb_compute_epsilon(int fdtype, double x, double relstep, double absstep, double dir);

/* ---- plans: the per-(pattern, colorvec, fdtype) state the reference rebuilds on every call
 *      (jacobians.jl:515-535: colour reshape, findstructralnz, same-pattern test) ---- */

/* sparsity::SparseMatrixCSC (m x n, colptr[n+1], rowval[nnz]).
 *   jkind = FDB_J_CSC_NZVAL: J is a CSC with pattern (j_colptr, j_rowval); NULL,NULL => same arrays as the sparsity.
 *           Same pattern (ext/..SparseArraysExt.jl:51-52) => fast path nzval[p]; a different pattern is accepted when every
 *           sparsity entry exists in J (the generic J[r,c]= path of :20-28), else FDB_ERR_UNSUPPORTED (would need insertion).
 *   jkind = FDB_J_DENSE: J is a dense column-major matrix with leading dimension ldJ (coloring_tests.jl:51-64).
 * colorvec: n colours, 1-based; NULL => 1:n (jacobians.jl:16). */
fdb_status fdb_plan_create_csc(fdb_plan **plan, int64_t m, int64_t n, const int64_t *colptr, const int64_t *rowval,
                               int jkind, const int64_t *j_colptr, const int64_t *j_rowval, int64_t ldJ,
                               const int64_t *colorvec, const fdb_plan_opts *opts);

/* sparsity given as structural-nonzero lists rows_index/cols_index (ArrayInterface.findstructralnz of a structured
 * matrix, or _findstructralnz of a dense 0/1 prototype, jacobians.jl:473-488,522-528) — generic hook iteration_utils.jl:25-32.
 *   jkind = FDB_J_DENSE (ldJ) or FDB_J_SLOTS (slots[nnz] 1-based into a J value buffer of j_len doubles). */
fdb_status fdb_plan_create_coo(fdb_plan **plan, int64_t m, int64_t n, int64_t nnz, const int64_t *rows_index,
                               const int64_t *cols_index, int jkind, const int64_t *slots, int64_t ldJ_or_jlen,
                               const int64_t *colorvec, const fdb_plan_opts *opts);

/* sparsity::BandedMatrix with bandwidths (l,u): ext/FiniteDiffBandedMatricesExt.jl:13-27 (writes the WHOLE band).
 *   jkind = FDB_J_BAND (J is the (l+u+1) x n band data) or FDB_J_DENSE (ldJ). */
fdb_status fdb_plan_create_banded(fdb_plan **plan, int64_t m, int64_t n, int64_t l, int64_t u, int jkind, int64_t ldJ,
                                  const int64_t *colorvec, const fdb_plan_opts *opts);

/* sparsity === nothing: dense column branch jacobians.jl:548-557,590-598 (colorvec = 1:n; per-component step).
 * With world>1 the columns are block-partitioned: this rank computes columns [col_begin, col_end) (0-based, see
 * fdb_plan_info) and d_J passed to fdb_jacobian points at THAT column slab (ldJ x ncols_local). */
fdb_status fdb_plan_create_dense(fdb_plan **plan, int64_t m, int64_t n, int64_t ldJ, const fdb_plan_opts *opts);
/* sparsity === nothing WITH a caller-supplied colorvec, as jacobians.jl:547-557 is written: the loop runs color_i in
 * 1:maximum(colorvec), perturbs COMPONENT color_i and writes J[:, color_i] (J is not zero-filled; later columns keep
 * their contents).  maximum(colorvec) > n (BoundsError in the reference) => FDB_ERR_INVALID.  colorvec NULL => 1:n. */
fdb_status fdb_plan_create_dense_colorvec(fdb_plan **plan, int64_t m, int64_t n, int64_t ldJ, const int64_t *colorvec,
                                          const fdb_plan_opts *opts);

fdb_status fdb_plan_destroy(fdb_plan *plan);
fdb_status fdb_plan_info(const fdb_plan *plan, fdb_plan_info_t *info);
fdb_status fdb_plan_counters(const fdb_plan *plan, fdb_counters_t *out);
/* dense plans: the [begin,end) 0-based column range this rank owns */
fdb_status fdb_plan_dense_range(const fdb_plan *plan, int64_t *col_begin, int64_t *col_end);
/* colour ownership (0-based colour index -> owning rank), n_colors entries */
fdb_status fdb_plan_color_owner(const fdb_plan *plan, int32_t *owner_out, int64_t cap);
/* Copy the step sizes used by the most recent call to the host (synchronises `stream`): eps per colour
 * (coloured plans, n_colors entries) or per local column (dense plans).  For tests / diagnostics. */
fdb_status fdb_plan_get_eps(fdb_plan *plan, double *h_eps, int64_t cap, void *stream);
/* Multi-GPU fused gather: besides d_J, the scatter also stores every value it owns into these peer J buffers
 * (device pointers valid on this device: cudaIpcOpenMemHandle / peer-enabled allocations).  n_peers = 0 clears. */
fdb_status fdb_plan_set_peers(fdb_plan *plan, int n_peers, double *const *peer_J);

/* Device-side timing of the diff+scatter launches (CUDA events recorded on the call's stream around every scatter
 * launch).  Off by default.  fdb_plan_read_timing synchronises the recorded events, returns the summed scatter time in
 * milliseconds and the number of launches since the last read, and resets the accumulators. */
fdb_status fdb_plan_enable_timing(fdb_plan *plan, int enable);
fdb_status fdb_plan_read_timing(fdb_plan *plan, double *scatter_ms, int64_t *scatter_launches);

/*
 * The hot path — replaces finite_difference_jacobian!(J, f, x, cache, f_in; relstep, absstep, colorvec, sparsity, dir)
 * (jacobians.jl:504-514) for the plan's (sparsity, colorvec, fdtype).
 *   d_x    : n doubles (device). NEVER modified (the reference perturbs it in place in central mode and restores it,
 *            jacobians.jl:604,620; here the minus points are built in plan-owned scratch).
 *   d_J    : J's value storage (device): nzval / dense / band data / slots buffer.  Fully defined on return
 *            (fill_matrix!(J,0) + scatter semantics of jacobians.jl:530-532,566-572).
 *   d_fx   : m doubles (device) — cache.fx.  Forward mode: receives f(x) unless d_f_in is given.  May be NULL
 *            (plan-owned buffer is used).  Central mode: unused.
 *   d_f_in : forward mode only: precomputed f(x) (`f_in`, jacobians.jl:540-545) or NULL.
 *   relstep, absstep: FDB_STEP_DEFAULT (NaN) => defaults (default_relstep(fdtype); absstep = relstep); other values as passed.
 *   dir    : forward only (epsilons.jl:28); pass 1.0 for the default `dir=true`.
 *   stream : cudaStream_t (NULL = legacy default stream).
 * f!-call count and order match the reference: forward f(x) first (unless f_in) then colours ascending;
 * central f(x+eps e_k) then f(x-eps e_k) per colour; a colour with no columns still triggers its call(s).
 */
fdb_status fdb_jacobian(fdb_plan *plan, fdb_fn f, void *ctx, const double *d_x, double *d_J, double *d_fx,
                        const double *d_f_in, double relstep, double absstep, double dir, void *stream);

/* Complex-step Jacobian (jacobians.jl:623-648) for plans created with fdtype = FDB_COMPLEX: per colour ONE evaluation
 * f(fx, x + im*eps*(color==k)) on complex128 device arrays, J = imag(fx)/eps with eps = eps(Float64); no f(x) baseline,
 * no cancellation (the reference's tests bound the error by 1e-14, finitedifftests.jl:462).  x and J stay real. */
fdb_status fdb_jacobian_complex(fdb_plan *plan, fdb_fn_c f, void *ctx, const double *d_x, double *d_J, void *stream);

/* Same call with HOST buffers (the reference-facing form: Array x, host J storage): copies x to the device, runs
 * fdb_jacobian on an internal stream, copies J's value storage (and fx when h_fx != NULL) back, then synchronises.
 * Pageable memory works; pinned memory (fdb_host_alloc) is what reaches PCIe speed. */
fdb_status fdb_jacobian_host(fdb_plan *plan, fdb_fn f, void *ctx, const double *h_x, double *h_J, double *h_fx,
                             const double *h_f_in, double relstep, double absstep, double dir);

/* ---- Column-block sharding (SURVEY §8f row 4: problems with fewer colours than GPUs) -------------------------------
 * A shard is a plan over a contiguous block of columns of the sparsity (its colptr slice rebased to 1, row indices
 * rebased to the first row the block touches), evaluated on the slice of x that those rows depend on, with a
 * slice-aware f! (the callback's ctx carries the row / x offsets).  The reference takes every colour's step size from
 * the norm over ALL colour-k components of x (jacobians.jl:559-561), so a shard must not derive it from its slice:
 *   fdb_eps_plan_create   plan that only knows (n, colorvec) of the FULL problem,
 *   fdb_color_eps         eps[k] of every colour for a full-length device x (the K2 pass alone), left in the plan
 *                         (fdb_plan_get_eps) and optionally copied to d_eps_out (device, n_colors doubles); also valid
 *                         on any coloured Jacobian plan,
 *   fdb_plan_set_external_eps   makes a Jacobian plan copy its step sizes from d_eps (device, at least the plan's
 *                         n_colors entries, read on the call's stream) instead of running its own K2 pass; NULL
 *                         restores the built-in pass.  With the same eps the shard's values are bit-identical to the
 *                         corresponding segment of the unsharded Jacobian. */
fdb_status fdb_eps_plan_create(fdb_plan **plan, int64_t n, const int64_t *colorvec, const fdb_plan_opts *opts);
fdb_status fdb_color_eps(fdb_plan *plan, const double *d_x, double relstep, double absstep, double dir,
                         double *d_eps_out, void *stream);
fdb_status fdb_plan_set_external_eps(fdb_plan *plan, const double *d_eps);

/* ---- Multi-GPU behind the C ABI (SURVEY §8e) — no NCCL on the data path ---------------------------------------------
 * Colours (dense plans: column blocks) are independent given x: every GPU evaluates its share and its diff+scatter
 * kernel stores the entries it owns straight into ONE Jacobian buffer (the root's) through peer-mapped memory over
 * NVLink — the final gather is the kernel's own store.
 *
 * (1) ONE process, n devices — what a Julia host needs to reach several GPUs from a single
 *     finite_difference_jacobian!(J, f, x, cache) call (jacobians.jl:504-514): fdb_group_create_* builds one plan per
 *     device (rank i of n; devices[0] is the root and owns x, J, fx), enables peer access to the root, and
 *     fdb_group_jacobian pushes x to the members, runs every member's colour loop on its own stream and joins them on
 *     the caller's stream with CUDA events (asynchronous; no host synchronisation).  ctx[i] is the callback context of
 *     member i (f! is invoked with device-i pointers and stream).  Device ordinals may repeat (two members on one GPU).
 *     Dense groups: member i fills its column block of the root's J.  Forward / central plans. */
typedef struct fdb_group fdb_group;
fdb_status fdb_group_create_csc(fdb_group **group, int n_devices, const int *devices, int64_t m, int64_t n,
                                const int64_t *colptr, const int64_t *rowval, int jkind, const int64_t *j_colptr,
                                const int64_t *j_rowval, int64_t ldJ, const int64_t *colorvec, const fdb_plan_opts *opts);
fdb_status fdb_group_create_banded(fdb_group **group, int n_devices, const int *devices, int64_t m, int64_t n, int64_t l,
                                   int64_t u, int jkind, int64_t ldJ, const int64_t *colorvec, const fdb_plan_opts *opts);
fdb_status fdb_group_create_dense(fdb_group **group, int n_devices, const int *devices, int64_t m, int64_t n, int64_t ldJ,
                                  const fdb_plan_opts *opts);
fdb_status fdb_group_destroy(fdb_group *group);
fdb_status fdb_group_size(const fdb_group *group, int *n_members);
/* member i's plan (owned by the group): fdb_plan_info / fdb_plan_counters / fdb_plan_get_eps / fdb_plan_color_owner */
fdb_status fdb_group_plan(const fdb_group *group, int member, fdb_plan **plan);
/* arguments as fdb_jacobian; d_x, d_J, d_fx, d_f_in live on devices[0], `stream` is a stream of devices[0] */
fdb_status fdb_group_jacobian(fdb_group *group, fdb_fn f, void *const *ctx, const double *d_x, double *d_J, double *d_fx,
                              const double *d_f_in, double relstep, double absstep, double dir, void *stream);

/* (2) one process per GPU (torchrun / MPI style): create the plan with opts.rank / opts.world and opts.shared_j = 1, map
 *     the root's J with fdb_ipc_open and pass THAT pointer as d_J (or keep a private J and name the root's buffer with
 *     fdb_plan_set_peers).  fdb_sync is the device-side barrier that orders the ranks: a flag block per rank in peer
 *     memory, fdb_sync_barrier enqueues one tiny kernel that signals every peer (st.release.sys) and waits for every
 *     peer's signal (ld.acquire.sys) — stream-ordered, no host involvement, replayable inside a CUDA graph.
 *     Typical call:  barrier (root finished reading J, and zero-filled it if needed)  ->  fdb_jacobian  ->  barrier.
 *       fdb_sync_flags      this rank's flag block (a dedicated allocation: export it with fdb_ipc_get_handle)
 *       fdb_sync_set_peers  every rank's flag block as mapped on this device (fdb_ipc_open), indexed by rank */
typedef struct fdb_sync fdb_sync;
fdb_status fdb_sync_create(fdb_sync **sync, int rank, int world, int device /* -1: current */);
fdb_status fdb_sync_flags(fdb_sync *sync, void **d_flags);
fdb_status fdb_sync_set_peers(fdb_sync *sync, void *const *d_flags_by_rank);
fdb_status fdb_sync_barrier(fdb_sync *sync, void *stream);
fdb_status fdb_sync_destroy(fdb_sync *sync);

/* ---- Colouring on the device: the ArrayInterface.matrix_colors(A) step callers run before this path
 *      (test/coloring_tests.jl:112,117).  d_colorvec is a caller-owned DEVICE array of n Int64 (1-based colours), ready to
 *      be passed to fdb_plan_create_* — a solver that resize!s its problem can recolour and re-plan without a host round
 *      trip of the pattern.
 *        banded   closed form ArrayInterface uses for BandedMatrix / Tridiagonal (l=u=1) / Bidiagonal: cycle 1:(l+u+1)
 *        csc      a valid distance-2 colouring of the columns (no two columns of one colour share a row) by a
 *                 deterministic Jones-Plassmann sweep; the result depends on the pattern alone.  colptr / rowval: Int64,
 *                 1-based, host or device.  n_colors / n_rounds (host, nullable) receive maximum(colorvec) / sweeps.
 *        check    number of (row, colour) collisions of a colouring (0 = valid for this path's decompression). */
fdb_status fdb_matrix_colors_banded(int64_t n, int64_t l, int64_t u, int64_t *d_colorvec, void *stream);
fdb_status fdb_matrix_colors_csc(int64_t m, int64_t n, const int64_t *colptr, const int64_t *rowval, int64_t *d_colorvec,
                                 int64_t *n_colors, int64_t *n_rounds);
fdb_status fdb_check_coloring_csc(int64_t m, int64_t n, const int64_t *colptr, const int64_t *rowval, const int64_t *colorvec,
                                  int64_t *n_conflicts);

/* ---- Jacobian-vector product: finite_difference_jvp!(jvp, f, x, v, cache::JVPCache, f_in; relstep, absstep, dir)
 *      src/jvp.jl:238-274 — eps from sqrt(abs(dot(x, v))) (computed on the device), forward: f(fx1,x), f(jvp,x+eps v);
 *      central: f(fx1, x-eps v) then f(jvp, x+eps v).  opts->fdtype selects forward/central (complex is rejected like
 *      in the reference).  d_x1 / d_fx1 are the JVPCache arrays (n / m doubles; NULL => plan-owned scratch);
 *      d_f_in: forward only, precomputed f(x). ---- */
fdb_status fdb_jvp_plan_create(fdb_plan **plan, int64_t m, int64_t n, const fdb_plan_opts *opts);
fdb_status fdb_jvp(fdb_plan *plan, fdb_fn f, void *ctx, double *d_jvp, const double *d_x, const double *d_v, double *d_x1,
                   double *d_fx1, const double *d_f_in, double relstep, double absstep, double dir, void *stream);

/* ---- Hessian of a scalar function: finite_difference_hessian!(H, f, x, cache::HessianCache; relstep, absstep)
 *      src/hessians.jl:202-292.  The reference makes 2n^2+1 scalar calls one at a time; here they are batched points:
 *        p = 0                      f(x)
 *        row i (0-based) at R(i) = 1 + 2i(2n-i):  x+e_i*E_i, x-e_i*E_i, then for j = i+1..n-1 the four points with
 *                                   components (i, j) moved by (+,+), (+,-), (-,+), (-,-)       (:226-227, :239-260)
 *      every other component is exactly x (the reference restores by assignment, :272-275, :284-289).  Step
 *      e_k = max(relstep*|x_k|, absstep) for the diagonal and the off-diagonal alike (:223, :234, :252).
 *        H[i,i] = ((F[R] - 2 F[0]) + F[R+1]) / (e_i*e_i)                                          (:233)
 *        H[i,j] = (((F[q] - F[q+1]) - F[q+2]) + F[q+3]) / ((4 e_i)*e_j),  q = R(i)+2+4(j-i-1)      (:268-269)
 *        H[j,i] = H[i,j] bit for bit                                                              (copytri!, :291)
 *   fdb_hessian_plan_create: opts->fdtype must be FDB_HCENTRAL (anything else: FDB_ERR_UNSUPPORTED, as :206 asserts);
 *      opts->max_batch = points per callback (0/1: one); opts->scratch_bytes caps the B copies of x (0: 8 GiB);
 *      world > 1 and use_graph = 1 are FDB_ERR_UNSUPPORTED.  The plan owns the 2n^2+1 values F (16 n^2 bytes,
 *      allocated here: FDB_ERR_NOMEM when that fails).
 *   fdb_hessian: f is an fdb_fn with m = 1: point b's scalar goes to d_fx[b*ldfx] (ldfx = 1; d_fx is 8-byte aligned).
 *      d_x: n doubles (device), never written.  d_H: dense column-major n x n, leading dimension ldH >= n (device);
 *      every one of the n^2 entries is written, rows [n, ldH) of each column are not touched.  relstep / absstep:
 *      FDB_STEP_DEFAULT as for fdb_jacobian.  Stream-ordered, no host synchronisation.
 *   Other entry points: fdb_jacobian / fdb_jvp / fdb_color_eps / fdb_plan_set_external_eps reject a Hessian plan
 *      (FDB_ERR_INVALID) and fdb_hessian rejects every other plan; fdb_plan_get_eps returns the n steps of the last call;
 *      fdb_plan_info: m = 1, n_colors = n, fcalls_per_jacobian = 2n^2+1, moved_bytes_scatter = the combine kernel's
 *      compulsory bytes (F read once, eps, H written once); fdb_plan_counters / fdb_plan_enable_timing count and time
 *      the combine launch as the scatter launch. ---- */
fdb_status fdb_hessian_plan_create(fdb_plan **plan, int64_t n, const fdb_plan_opts *opts);
fdb_status fdb_hessian(fdb_plan *plan, fdb_fn f, void *ctx, const double *d_x, double *d_H, int64_t ldH, double relstep,
                       double absstep, void *stream);

/* ---- helpers for hosts without their own CUDA bindings ---- */
fdb_status fdb_host_alloc(void **p, size_t bytes);  /* pinned host memory */
fdb_status fdb_host_free(void *p);
fdb_status fdb_device_alloc(void **p, size_t bytes);
fdb_status fdb_device_free(void *p);
fdb_status fdb_memcpy_h2d(void *d, const void *h, size_t bytes, void *stream);
fdb_status fdb_memcpy_d2h(void *h, const void *d, size_t bytes, void *stream);
fdb_status fdb_stream_sync(void *stream);
/* CUDA IPC, for the one-process-per-GPU fused gather (handle is CUDA_IPC_HANDLE_SIZE = 64 bytes) */
fdb_status fdb_ipc_get_handle(void *d_ptr, unsigned char handle[64]);
fdb_status fdb_ipc_open(const unsigned char handle[64], void **d_ptr);
fdb_status fdb_ipc_close(void *d_ptr);

#ifdef __cplusplus
}
#endif
#endif /* FDJAC_B200_H */
