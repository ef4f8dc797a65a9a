// synth_fns.cu — libfdjac_synth.so: synthetic f!(dx, x) device functions for the bench / parity harness
// (include/fdjac_synth.h).  Bit-identical to oracle/synth_fns.c: explicit __dadd_rn/__dmul_rn, same evaluation order.
#include "../../include/fdjac_synth.h"

#include <cuda_runtime.h>
#include <cstdint>

namespace {
constexpr int kT = 256;

__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }

// dx[i] = (x[i-1] - 2*x[i]) + x[i+1];  dx[0] = -2*x[0] + x[1];  dx[n-1] = x[n-2] - 2*x[n-1]
__global__ void __launch_bounds__(kT) k_tridiag(double *__restrict__ fx, const double *__restrict__ x, int64_t n,
                                                int64_t ldfx, int64_t ldx) {
  const double *xb = x + (int64_t)blockIdx.y * ldx;
  double *fb = fx + (int64_t)blockIdx.y * ldfx;
  const int64_t stride = (int64_t)gridDim.x * kT * 2;
  for (int64_t i0 = (blockIdx.x * (int64_t)kT + threadIdx.x) * 2; i0 < n; i0 += stride) {
    // two rows per thread: one 16-byte load of (x[i0], x[i0+1]) plus the two neighbours
    if (i0 + 1 < n) {
      const double2 c = *reinterpret_cast<const double2 *>(xb + i0);
      const double lft = i0 > 0 ? __ldg(xb + i0 - 1) : 0.0;
      const double rgt = i0 + 2 < n ? __ldg(xb + i0 + 2) : 0.0;
      double a, b;
      if (i0 == 0) a = add(mul(-2.0, c.x), c.y);
      else a = add(sub(lft, mul(2.0, c.x)), c.y);
      if (i0 + 1 == n - 1) b = sub(c.x, mul(2.0, c.y));
      else b = add(sub(c.x, mul(2.0, c.y)), rgt);
      __stcs(reinterpret_cast<double2 *>(fb + i0), make_double2(a, b));
    } else {
      // last row of an odd-length vector
      const double c = xb[i0];
      fb[i0] = n == 1 ? mul(-2.0, c) : sub(__ldg(xb + i0 - 1), mul(2.0, c));
    }
  }
}

__global__ void __launch_bounds__(kT) k_lap5(double *__restrict__ out, const double *__restrict__ x, int64_t g,
                                             int64_t ldfx, int64_t ldx) {
  const double *xb = x + (int64_t)blockIdx.z * ldx;
  double *ob = out + (int64_t)blockIdx.z * ldfx;
  const int64_t j = blockIdx.y;  // grid column
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < g; i += (int64_t)gridDim.x * kT) {
    const int64_t im = i > 0 ? i - 1 : 0, ip = i + 1 < g ? i + 1 : g - 1;
    const int64_t jm = j > 0 ? j - 1 : 0, jp = j + 1 < g ? j + 1 : g - 1;
    double s = xb[i + j * g];
    s = add(s, xb[im + j * g]);
    s = add(s, xb[ip + j * g]);
    s = add(s, xb[i + jm * g]);
    s = add(s, xb[i + jp * g]);
    ob[i + j * g] = s;
  }
}

// ELL layout [K][m]: entry p of row i at p*m + i -> the index / coefficient streams are read fully coalesced
__global__ void __launch_bounds__(kT) k_ellrows(double *__restrict__ fx, const double *__restrict__ x, int64_t m, int K,
                                                const int32_t *__restrict__ cols, const double *__restrict__ coef,
                                                int64_t ldfx, int64_t ldx) {
  const double *xb = x + (int64_t)blockIdx.y * ldx;
  double *fb = fx + (int64_t)blockIdx.y * ldfx;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < m; i += (int64_t)gridDim.x * kT) {
    const double x0 = __ldg(xb + __ldcs(cols + i));
    double s = mul(__ldcs(coef + i), x0);
    for (int p = 1; p < K; ++p) s = add(s, mul(__ldcs(coef + (int64_t)p * m + i), __ldg(xb + __ldcs(cols + (int64_t)p * m + i))));
    s = add(s, mul(0.1, mul(x0, x0)));
    fb[i] = s;
  }
}

// blocked sum: blocks of 1024 summed sequentially (one thread each — tiny), then block sums sequentially
__global__ void __launch_bounds__(kT) k_block_sums(const double *__restrict__ x, int64_t n, int64_t ldx,
                                                   double *__restrict__ bs, int64_t nblk) {
  // one warp per 1024-block: lane l sums x[b + l + 32 j] (j ascending, coalesced), xor butterfly — the order of
  // oracle/synth_fns.c:synth_blocked_sum
  const double *xb = x + (int64_t)blockIdx.y * ldx;
  const int lane = threadIdx.x & 31;
  for (int64_t b = blockIdx.x * (int64_t)(kT / 32) + (threadIdx.x >> 5); b < nblk; b += (int64_t)gridDim.x * (kT / 32)) {
    const int64_t s0 = b * 1024;
    double s = 0.0;
#pragma unroll 8
    for (int j = 0; j < 32; ++j) {
      const int64_t idx = s0 + lane + 32 * j;
      s = add(s, idx < n ? xb[idx] : 0.0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = add(s, __shfl_xor_sync(0xffffffffu, s, o));
    if (lane == 0) bs[(int64_t)blockIdx.y * nblk + b] = s;
  }
}

// S[p] = (block sums of point p added in block order) / n, left in bs[p*nblk] (only thread p touches row p)
__global__ void __launch_bounds__(kT) k_point_sums(double *__restrict__ bs, int64_t nblk, int64_t n, int64_t batch) {
  const int64_t p = blockIdx.x * (int64_t)kT + threadIdx.x;
  if (p >= batch) return;
  double t = 0.0;
  for (int64_t b = 0; b < nblk; ++b) t = add(t, bs[p * nblk + b]);
  bs[p * nblk] = __ddiv_rn(t, (double)n);
}

__global__ void __launch_bounds__(kT) k_rank1(double *__restrict__ fx, const double *__restrict__ x, int64_t n,
                                              const double *__restrict__ w, const double *__restrict__ bs, int64_t nblk,
                                              int64_t ldfx, int64_t ldx, int vec_ok) {
  const double *xb = x + (int64_t)blockIdx.y * ldx;
  double *fb = fx + (int64_t)blockIdx.y * ldfx;
  const double s = __ldg(bs + (int64_t)blockIdx.y * nblk);
  const int64_t stride = (int64_t)gridDim.x * kT;
  if (vec_ok) {
    // two rows per lane, two independent 16-byte loads of x in flight; x and f are read / written once (streaming), w is
    // shared by every point of the batch (cacheable)
    const int64_t n2 = n >> 1;
    const double2 *x2 = reinterpret_cast<const double2 *>(xb), *w2 = reinterpret_cast<const double2 *>(w);
    double2 *f2 = reinterpret_cast<double2 *>(fb);
    int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x;
    for (; i + stride < n2; i += 2 * stride) {
      const double2 a = __ldcs(x2 + i), b = __ldcs(x2 + i + stride);
      const double2 wa = __ldg(w2 + i), wb = __ldg(w2 + i + stride);
      __stcs(f2 + i, make_double2(add(mul(a.x, a.x), mul(wa.x, s)), add(mul(a.y, a.y), mul(wa.y, s))));
      __stcs(f2 + i + stride, make_double2(add(mul(b.x, b.x), mul(wb.x, s)), add(mul(b.y, b.y), mul(wb.y, s))));
    }
    for (; i < n2; i += stride) {
      const double2 a = __ldcs(x2 + i), wa = __ldg(w2 + i);
      __stcs(f2 + i, make_double2(add(mul(a.x, a.x), mul(wa.x, s)), add(mul(a.y, a.y), mul(wa.y, s))));
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) { const double v = xb[n - 1]; fb[n - 1] = add(mul(v, v), mul(w[n - 1], s)); }
    return;
  }
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < n; i += stride) {
    const double v = xb[i];
    fb[i] = add(mul(v, v), mul(w[i], s));
  }
}

// Slice-aware tridiagonal stencil (column-block sharded runs): rows [row0, row0+nrows) of the n-row problem, reading a
// slice of x whose element 0 is global component x0.  Same expression per row as k_tridiag => bit-identical values.
__global__ void __launch_bounds__(kT) k_tridiag_rows(double *__restrict__ fx, const double *__restrict__ x, int64_t n,
                                                     int64_t row0, int64_t nrows, int64_t x0, int64_t ldfx, int64_t ldx) {
  const double *xb = x + (int64_t)blockIdx.y * ldx - x0;     // xb[global index]
  double *fb = fx + (int64_t)blockIdx.y * ldfx;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < nrows; i += (int64_t)gridDim.x * kT) {
    const int64_t r = row0 + i;
    const double c = xb[r];
    double o;
    if (n == 1) o = mul(-2.0, c);
    else if (r == 0) o = add(mul(-2.0, c), xb[1]);
    else if (r == n - 1) o = sub(xb[r - 1], mul(2.0, c));
    else o = add(sub(xb[r - 1], mul(2.0, c)), xb[r + 1]);
    fb[i] = o;
  }
}

// complex twin of k_tridiag (complex-step path): complex128 arrays as double2; the stencil on re and im separately
__global__ void __launch_bounds__(kT) k_tridiag_c(double2 *__restrict__ fx, const double2 *__restrict__ x, int64_t n,
                                                  int64_t ldfx, int64_t ldx) {
  const double2 *xb = x + (int64_t)blockIdx.y * ldx;
  double2 *fb = fx + (int64_t)blockIdx.y * ldfx;
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < n; i += (int64_t)gridDim.x * kT) {
    const double2 c = xb[i];
    double2 o;
    if (n == 1) { o.x = mul(-2.0, c.x); o.y = mul(-2.0, c.y); }
    else if (i == 0) { const double2 r = xb[1]; o.x = add(mul(-2.0, c.x), r.x); o.y = add(mul(-2.0, c.y), r.y); }
    else if (i == n - 1) { const double2 l = xb[i - 1]; o.x = sub(l.x, mul(2.0, c.x)); o.y = sub(l.y, mul(2.0, c.y)); }
    else {
      const double2 l = xb[i - 1], r = xb[i + 1];
      o.x = add(sub(l.x, mul(2.0, c.x)), r.x);
      o.y = add(sub(l.y, mul(2.0, c.y)), r.y);
    }
    fb[i] = o;
  }
}

// Scalar f(x) = sum w_i x_i^3 + sum x_i x_{i+1} + (sum x_i)^2/(2n), one warp per point.  Lane l sums the terms of
// components l, l+32, ... in ascending order; xor butterfly; lane 0 forms (A + B) + (S*S)/(2n) — the order of
// oracle_hessian/synth_scalar.c:synth_hess_poly.
__global__ void __launch_bounds__(kT) k_hess_poly(double *__restrict__ fx, const double *__restrict__ x, int64_t n,
                                                 const double *__restrict__ w, int64_t batch, int64_t ldfx, int64_t ldx) {
  const int64_t p = blockIdx.x * (int64_t)(kT / 32) + (threadIdx.x >> 5);
  if (p >= batch) return;
  const int lane = threadIdx.x & 31;
  const double *xb = x + p * ldx;
  double a = 0.0, b = 0.0, s = 0.0;
  for (int64_t i = lane; i < n; i += 32) {
    const double xi = xb[i];
    a = add(a, mul(__ldg(w + i), mul(mul(xi, xi), xi)));
    if (i + 1 < n) b = add(b, mul(xi, xb[i + 1]));
    s = add(s, xi);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a = add(a, __shfl_xor_sync(0xffffffffu, a, o));
    b = add(b, __shfl_xor_sync(0xffffffffu, b, o));
    s = add(s, __shfl_xor_sync(0xffffffffu, s, o));
  }
  if (lane == 0) fx[p * ldfx] = add(add(a, b), __ddiv_rn(mul(s, s), (double)(2 * n)));
}

__device__ __forceinline__ uint64_t splitmix64_at(uint64_t seed, uint64_t i) {
  uint64_t z = seed + (i + 1) * 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

__global__ void __launch_bounds__(kT) k_fill_x(double *__restrict__ x, int64_t n, uint64_t seed) {
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < n; i += (int64_t)gridDim.x * kT)
    x[i] = __dadd_rn(0.5, __dmul_rn((double)(splitmix64_at(seed, (uint64_t)i) >> 11), 1.0 / 9007199254740992.0));
}

__global__ void __launch_bounds__(kT) k_flush(double *__restrict__ p, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)kT + threadIdx.x; i < n; i += (int64_t)gridDim.x * kT) p[i] = 0.0;
}

inline int blocks_for(int64_t items, int64_t cap = 148 * 8) {
  int64_t b = (items + kT - 1) / kT;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}
}  // namespace

// Store-only bandwidth probe: n doubles written once with 16-byte streaming stores, grid-stride in address order.
// mode 0: one constant; mode 1: a different value per element (rules out constant-data effects in the memory system)
__global__ void __launch_bounds__(kT) k_store_probe(double *__restrict__ out, int64_t n, int mode) {
  const int64_t stride = (int64_t)gridDim.x * kT * 2;
  for (int64_t i = (blockIdx.x * (int64_t)kT + threadIdx.x) * 2; i + 1 < n; i += stride) {
    const double v0 = mode ? (double)i * 1.0000001 + 0.5 : 1.0;
    const double v1 = mode ? (double)(i + 1) * 1.0000001 + 0.5 : 1.0;
    __stcs(reinterpret_cast<double2 *>(out + i), make_double2(v0, v1));
  }
}

extern "C" {

int fdbs_tridiag(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_tridiag_ctx *c = (fdbs_tridiag_ctx *)vctx;
  if (!c || batch < 1 || batch > 65535) return 1;
  c->calls += batch;
  if (c->n <= 0) return 0;
  // the 16-byte path needs 16-byte aligned rows (plan buffers are; ldx/ldfx are even)
  if (((uintptr_t)d_x & 15) || ((uintptr_t)d_fx & 15) || (ldx & 1) || (ldfx & 1)) return 2;
  dim3 grid((unsigned)blocks_for((c->n + 1) / 2), (unsigned)batch);
  k_tridiag<<<grid, kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->n, ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_tridiag_rows(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_tridiag_rows_ctx *c = (fdbs_tridiag_rows_ctx *)vctx;
  if (!c || batch < 1 || batch > 65535) return 1;
  c->calls += batch;
  if (c->nrows <= 0) return 0;
  dim3 grid((unsigned)blocks_for(c->nrows), (unsigned)batch);
  k_tridiag_rows<<<grid, kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->n, c->row0, c->nrows, c->x0, ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_tridiag_c(void *vctx, void *d_fx, const void *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_tridiag_ctx *c = (fdbs_tridiag_ctx *)vctx;
  if (!c || batch < 1 || batch > 65535) return 1;
  c->calls += batch;
  if (c->n <= 0) return 0;
  dim3 grid((unsigned)blocks_for(c->n), (unsigned)batch);
  k_tridiag_c<<<grid, kT, 0, (cudaStream_t)stream>>>((double2 *)d_fx, (const double2 *)d_x, c->n, ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_lap5(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_lap5_ctx *c = (fdbs_lap5_ctx *)vctx;
  if (!c || batch < 1 || batch > 65535 || c->g > 65535) return 1;
  c->calls += batch;
  if (c->g <= 0) return 0;
  dim3 grid((unsigned)blocks_for(c->g, 8), (unsigned)c->g, (unsigned)batch);
  k_lap5<<<grid, kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->g, ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_ellrows(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_ell_ctx *c = (fdbs_ell_ctx *)vctx;
  if (!c || batch < 1 || batch > 65535) return 1;
  c->calls += batch;
  if (c->m <= 0) return 0;
  dim3 grid((unsigned)blocks_for(c->m, 148 * 16), (unsigned)batch);
  k_ellrows<<<grid, kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->m, (int)c->K, c->d_cols, c->d_coef, ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_rank1(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_rank1_ctx *c = (fdbs_rank1_ctx *)vctx;
  if (!c || batch < 1 || batch > c->max_batch || batch > 65535) return 1;
  c->calls += batch;
  if (c->n <= 0) return 0;
  const int64_t nblk = (c->n + 1023) / 1024;
  dim3 g1((unsigned)blocks_for(nblk * 32, 64), (unsigned)batch);   // one warp per 1024-block
  k_block_sums<<<g1, kT, 0, (cudaStream_t)stream>>>(d_x, c->n, ldx, c->d_block_sums, nblk);
  k_point_sums<<<(unsigned)((batch + kT - 1) / kT), kT, 0, (cudaStream_t)stream>>>(c->d_block_sums, nblk, c->n, batch);
  // 16-byte path: every point / output / w base 16-byte aligned (even leading dimensions)
  const int vec_ok = (((uintptr_t)d_x | (uintptr_t)d_fx | (uintptr_t)c->d_w) & 15) == 0 && (ldx & 1) == 0 && (ldfx & 1) == 0;
  dim3 g2((unsigned)blocks_for((c->n + 3) / 4, 128), (unsigned)batch);
  k_rank1<<<g2, kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->n, c->d_w, c->d_block_sums, nblk, ldfx, ldx, vec_ok);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_hess_poly(void *vctx, double *d_fx, const double *d_x, int64_t batch, int64_t ldfx, int64_t ldx, void *stream) {
  fdbs_hess_poly_ctx *c = (fdbs_hess_poly_ctx *)vctx;
  if (!c || batch < 1) return 1;
  c->calls += batch;
  if (c->n <= 0) {   // f of the empty vector: every sum is 0
    if (cudaMemset2DAsync(d_fx, (size_t)ldfx * 8, 0, 8, (size_t)batch, (cudaStream_t)stream) != cudaSuccess) return 3;
    return 0;
  }
  k_hess_poly<<<(unsigned)((batch + kT / 32 - 1) / (kT / 32)), kT, 0, (cudaStream_t)stream>>>(d_fx, d_x, c->n, c->d_w, batch,
                                                                                            ldfx, ldx);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_fail(void *, double *, const double *, int64_t, int64_t, int64_t, void *) { return 42; }

int fdbs_fill_x(double *d_x, int64_t n, uint64_t seed, void *stream) {
  if (n <= 0) return 0;
  k_fill_x<<<blocks_for(n), kT, 0, (cudaStream_t)stream>>>(d_x, n, seed);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_store_probe(double *d_out, int64_t n, int mode, int blocks, void *stream) {
  if (n <= 0 || blocks <= 0) return 1;
  k_store_probe<<<blocks, kT, 0, (cudaStream_t)stream>>>(d_out, n, mode);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

int fdbs_flush_l2(void *d_buf, int64_t bytes, void *stream) {
  if (bytes <= 0) return 0;
  k_flush<<<blocks_for(bytes / 8), kT, 0, (cudaStream_t)stream>>>((double *)d_buf, bytes / 8);
  return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

}  // extern "C"
