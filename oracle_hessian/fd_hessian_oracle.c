/*
 * fd_hessian_oracle.c — CPU restatement of finite_difference_hessian! (src/hessians.jl:202-292).  See the header.
 * Compiled with -ffp-contract=off: every operation rounds on its own, in the order the reference writes it.
 */
#include "fd_hessian_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* epsilons.jl:134-144: `eps(T)^(1/4)` for T = Float64 */
double fdo_hcentral_default_relstep(void) { return pow(2.220446049250313e-16, 0.25); }

/* Base.max for Float64: NaN wins, and +0.0 > -0.0 */
static double jl_max(double a, double b) {
  if (isnan(a) || isnan(b)) return a + b;
  if (b > a || (signbit(a) && !signbit(b))) return b;
  return a;
}

/* epsilons.jl:74-77 */
double fdo_hcentral_compute_epsilon(double x, double relstep, double absstep) {
  return jl_max(relstep * fabs(x), absstep);
}

int fdo_finite_difference_hessian_cached(double *H, int64_t ldH, fdo_sfn f, void *ctx, const double *x, int64_t n,
                                         double *xpp, double *xpm, double *xmp, double *xmm, double relstep,
                                         double absstep, double *eps_out, int64_t *fcalls) {
  if (n < 0 || ldH < n || !f) return 1;
  if (n > 0 && (!H || !x || !xpp || !xpm || !xmp || !xmm)) return 1;
  /* keyword defaults :204-205 */
  if (isnan(relstep)) relstep = fdo_hcentral_default_relstep();
  if (isnan(absstep)) absstep = relstep;
  int64_t calls = 0;
  /* fx = f(x)   :209 */
  const double fx = f(ctx, x);
  calls += 1;
  /* copyto!(xpp, x) ... copyto!(xmm, x)   :213-216 */
  if (n > 0) {
    memcpy(xpp, x, (size_t)n * sizeof(double));
    memcpy(xpm, x, (size_t)n * sizeof(double));
    memcpy(xmp, x, (size_t)n * sizeof(double));
    memcpy(xmm, x, (size_t)n * sizeof(double));
  }
  /* for i in 1:n   :221 */
  for (int64_t i = 0; i < n; ++i) {
    const double xi = x[i];                                                    /* :222 */
    const double epsilon = fdo_hcentral_compute_epsilon(xi, relstep, absstep); /* :223 Val(:hcentral) */
    if (eps_out) eps_out[i] = epsilon;
    xpp[i] = xi + epsilon;                                                     /* :226 */
    xmm[i] = xi - epsilon;                                                     /* :227 */
    {
      const double fpp = f(ctx, xpp);                                          /* :233, arguments left to right */
      const double fmm = f(ctx, xmm);
      calls += 2;
      H[i + i * ldH] = ((fpp - 2 * fx) + fmm) / (epsilon * epsilon);           /* :233  epsilon^2 = epsilon*epsilon */
    }
    const double epsiloni = fdo_hcentral_compute_epsilon(xi, relstep, absstep); /* :234 Val(:central), same steps */
    const double xp = xi + epsiloni;                                           /* :235 */
    const double xm = xi - epsiloni;                                           /* :236 */
    xpp[i] = xp;                                                               /* :239-242 */
    xpm[i] = xp;
    xmp[i] = xm;
    xmm[i] = xm;
    /* for j in (i+1):n   :250 */
    for (int64_t j = i + 1; j < n; ++j) {
      const double xj = x[j];                                                  /* :251 */
      const double epsilonj = fdo_hcentral_compute_epsilon(xj, relstep, absstep); /* :252 */
      const double xjp = xj + epsilonj;                                        /* :253 */
      const double xjm = xj - epsilonj;                                        /* :254 */
      xpp[j] = xjp;                                                            /* :257-260 */
      xpm[j] = xjm;
      xmp[j] = xjp;
      xmm[j] = xjm;
      const double fpp = f(ctx, xpp);                                          /* :269, arguments left to right */
      const double fpm = f(ctx, xpm);
      const double fmp = f(ctx, xmp);
      const double fmm = f(ctx, xmm);
      calls += 4;
      H[i + j * ldH] = (((fpp - fpm) - fmp) + fmm) / ((4 * epsiloni) * epsilonj);   /* :268-269 */
      xpp[j] = xj;                                                             /* :272-275 */
      xpm[j] = xj;
      xmp[j] = xj;
      xmm[j] = xj;
    }
    xpp[i] = xi;                                                               /* :285-288 */
    xpm[i] = xi;
    xmp[i] = xi;
    xmm[i] = xi;
  }
  /* LinearAlgebra.copytri!(H, 'U')   :291 */
  for (int64_t j = 0; j < n; ++j)
    for (int64_t i = j + 1; i < n; ++i) H[i + j * ldH] = H[j + i * ldH];
  if (fcalls) *fcalls = calls;
  return 0;
}

/* HessianCache(x) :83-89 (cx = copy(x), copy(x), copy(x), copy(x)), then the cached call */
int fdo_finite_difference_hessian(double *H, int64_t ldH, fdo_sfn f, void *ctx, const double *x, int64_t n,
                                  double relstep, double absstep, double *eps_out, int64_t *fcalls) {
  if (n < 0) return 1;
  const size_t len = (size_t)(n > 0 ? n : 1);
  double *buf = (double *)malloc(4 * len * sizeof(double));
  if (!buf) return 2;
  const int rc = fdo_finite_difference_hessian_cached(H, ldH, f, ctx, x, n, buf, buf + len, buf + 2 * len, buf + 3 * len,
                                                      relstep, absstep, eps_out, fcalls);
  free(buf);
  return rc;
}
