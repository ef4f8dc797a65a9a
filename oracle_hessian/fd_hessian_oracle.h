/*
 * fd_hessian_oracle.h — CPU ORACLE for the Hessian path (fdb_hessian).
 *
 * TEST INFRASTRUCTURE ONLY, with the status of oracle/fd_oracle.h: only tests/, __graft_entry__.smoke() and
 * profiles/hessian_bench.py load it, as the checker / reported baseline.  It is a library of its own so that the
 * Jacobian oracle the existing parity tests are pinned against stays byte for byte what it is.
 *
 * What it is: a plain-C restatement of FiniteDiff.jl v2.31.1
 *   src/hessians.jl:202-292   cached finite_difference_hessian!  (in-place branch: the four cache arrays and their
 *                             restores; the immutable branch computes the same values)
 *   src/hessians.jl:67-89     HessianCache constructors (the arrays are caller-owned here)
 *   src/epsilons.jl:74-77,134-144   compute_epsilon(::Val{:hcentral}) / default_relstep(:hcentral)
 * Pinned by the reference's own Hessian known answers (test/finitedifftests.jl:561-576, 593-598, 608-614,
 * test/cache_reuse_tests.jl:130-139) and, bit for bit, by an independent Python transcription (tests/test_hessian.py).
 */
#ifndef FD_HESSIAN_ORACLE_H
#define FD_HESSIAN_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* scalar user function f(x)  (hessians.jl:209 `fx = f(x)`) */
typedef double (*fdo_sfn)(void *ctx, const double *x);

/* epsilons.jl:134-144: eps(Float64)^(1/4) */
double fdo_hcentral_default_relstep(void);
/* epsilons.jl:74-77: max(relstep*abs(x), absstep) */
double fdo_hcentral_compute_epsilon(double x, double relstep, double absstep);

/* finite_difference_hessian!(H, f, x, cache; relstep, absstep) hessians.jl:202-292 with HessianCache(x) (:83-89).
 *   H: column-major n x n, leading dimension ldH >= n; all n^2 entries are written, rows [n, ldH) are not.
 *   relstep / absstep: NaN = keyword not given (relstep = default_relstep(:hcentral), absstep = relstep).
 *   eps_out (n, nullable): the step of every component.  fcalls (nullable): number of f calls (2n^2+1).
 * Returns 0, or nonzero on invalid arguments. */
int fdo_finite_difference_hessian(double *H, int64_t ldH, fdo_sfn f, void *ctx, const double *x, int64_t n,
                                  double relstep, double absstep, double *eps_out, int64_t *fcalls);

/* The same with caller-supplied cache arrays xpp, xpm, xmp, xmm (n each): HessianCache(xpp, xpm, xmp, xmm, fdtype,
 * inplace) (:67-73).  Their contents on entry do not matter (:213-216 copies x into them). */
int fdo_finite_difference_hessian_cached(double *H, int64_t ldH, fdo_sfn f, void *ctx, const double *x, int64_t n,
                                         double *xpp, double *xpm, double *xmp, double *xmm, double relstep,
                                         double absstep, double *eps_out, int64_t *fcalls);

#ifdef __cplusplus
}
#endif
#endif
