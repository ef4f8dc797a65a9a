/*
 * fdjac_synth.h — libfdjac_synth.so: device implementations of the SYNTHETIC f!(dx, x) functions the benchmark
 * and the parity tests differentiate (bench/test harness, not part of the product ABI).  Each is an fdb_fn
 * (include/fdjac_b200.h): batched, enqueue-only on the given stream.  Arithmetic is written with explicit
 * __dadd_rn/__dmul_rn so it is bit-identical to the CPU twins in oracle/synth_fns.c.
 *
 *   fdbs_tridiag : test/coloring_tests.jl:5-13    dx[i] = x[i-1] - 2x[i] + x[i+1]
 *   fdbs_tridiag_rows : the same stencil for a row range of the problem, reading a slice of x (column-block shards)
 *   fdbs_lap5    : test/coloring_tests.jl:99-108  clamped 5-point stencil on a g x g grid (column-major)
 *   fdbs_ellrows : dx[i] = sum_p coef[p,i]*x[cols[p,i]] + 0.1*x[cols[0,i]]^2, ELL layout [K][m]   (SURVEY.md §8d config C4)
 *   fdbs_rank1   : dx[i] = x[i]^2 + w[i]*S, S = blocked-sum(x)/n                (SURVEY.md §8d config C5 variant)
 *   fdbs_hess_poly : SCALAR f(x) = sum w_i x_i^3 + sum x_i x_{i+1} + (sum x_i)^2/(2n)  (m = 1; fdb_hessian's callback).
 *                  Hessian in closed form: diagonal 6 w_i x_i + 1/n, (i, i+-1) 1 + 1/n, every other entry 1/n.
 *                  Fixed summation order (one warp per point): lane l sums the terms of components l, l+32, l+64, ...
 *                  in ascending order, then the xor butterfly p[l] += p[l^o], o = 16..1, for each of the three sums;
 *                  f = (A + B) + (S*S)/(2n).  Its CPU twin is oracle_hessian/synth_scalar.c.
 */
#ifndef FDJAC_SYNTH_H
#define FDJAC_SYNTH_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct { int64_t n; int64_t calls; } fdbs_tridiag_ctx;
/* slice-aware variant: rows [row0, row0+nrows) of the n-row stencil; d_x[0] is global component x0 */
typedef struct { int64_t n; int64_t row0; int64_t nrows; int64_t x0; int64_t calls; } fdbs_tridiag_rows_ctx;
typedef struct { int64_t g; int64_t calls; } fdbs_lap5_ctx;
typedef struct { int64_t m; int64_t K; const int32_t *d_cols; const double *d_coef; int64_t calls; } fdbs_ell_ctx;
typedef struct { int64_t n; const double *d_w; double *d_block_sums; int64_t max_batch; int64_t calls; } fdbs_rank1_ctx;
typedef struct { int64_t n; const double *d_w; int64_t calls; } fdbs_hess_poly_ctx;

int fdbs_tridiag(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
int fdbs_tridiag_rows(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
/* complex128 twin of fdbs_tridiag (an fdb_fn_c): the stencil on real and imaginary parts, for the complex-step path */
int fdbs_tridiag_c(void *ctx, void *d_fx, const void *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
int fdbs_lap5(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
int fdbs_ellrows(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
int fdbs_rank1(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
/* scalar function for fdb_hessian: d_fx[b*ldfx] = f(point b) */
int fdbs_hess_poly(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);
/* a callback that always fails (error-path tests) */
int fdbs_fail(void *ctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream);

/* x[i] = 0.5 + u_i, u_i from splitmix64(seed, i): same generator as oracle/synth_fns.c:synth_fill_x */
int fdbs_fill_x(double *d_x, int64_t n, uint64_t seed, void *stream);
/* write a buffer larger than L2 (flushes L2 between timed iterations) */
/* store-only bandwidth probe (profiles/write_bw_probe.py): mode 0 constant data, mode 1 a distinct value per element */
int fdbs_store_probe(double *d_out, int64_t n, int mode, int blocks, void *stream);
int fdbs_flush_l2(void *d_buf, int64_t bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif
