/*
 * synth_scalar.c — CPU twin of the synthetic scalar function fdbs_hess_poly (finitediff.jl_b200/csrc/synth_fns.cu),
 * TEST INFRASTRUCTURE like fd_hessian_oracle.c.  Same evaluation order as the CUDA twin, no FMA contraction
 * (-ffp-contract=off here; __dadd_rn/__dmul_rn there), so the two agree bit for bit.
 *
 *   f(x) = sum w_i x_i^3 + sum x_i x_{i+1} + (sum x_i)^2/(2n)
 *   Hessian: diagonal 6 w_i x_i + 1/n, (i, i+-1) 1 + 1/n, every other entry 1/n.
 */
#include <stdint.h>

typedef struct { int64_t n; const double *w; } synth_hess_poly_ctx;

double synth_hess_poly(void *vctx, const double *x) {
  const synth_hess_poly_ctx *c = (const synth_hess_poly_ctx *)vctx;
  const int64_t n = c->n;
  if (n <= 0) return 0.0;
  /* lane l of a warp: components l, l+32, ... in ascending order */
  double a[32], b[32], s[32], qa[32], qb[32], qs[32];
  for (int l = 0; l < 32; ++l) {
    double ta = 0.0, tb = 0.0, ts = 0.0;
    for (int64_t i = l; i < n; i += 32) {
      const double xi = x[i];
      ta = ta + c->w[i] * ((xi * xi) * xi);
      if (i + 1 < n) tb = tb + xi * x[i + 1];
      ts = ts + xi;
    }
    a[l] = ta;
    b[l] = tb;
    s[l] = ts;
  }
  /* xor butterfly p[l] = p[l] + p[l^o], o = 16, 8, 4, 2, 1 */
  for (int o = 16; o > 0; o >>= 1) {
    for (int l = 0; l < 32; ++l) {
      qa[l] = a[l] + a[l ^ o];
      qb[l] = b[l] + b[l ^ o];
      qs[l] = s[l] + s[l ^ o];
    }
    for (int l = 0; l < 32; ++l) {
      a[l] = qa[l];
      b[l] = qb[l];
      s[l] = qs[l];
    }
  }
  return (a[0] + b[0]) + (s[0] * s[0]) / (double)(2 * n);
}
