// kernels_hessian.cuh — Hessian of a scalar function: finite_difference_hessian!(H, f, x, cache) src/hessians.jl:202-292.
// The reference evaluates its 2n^2+1 points one f call at a time.  Here the points are laid out in the reference's call
// order p = 0 .. 2n^2 and evaluated in batches of B by the caller's f (one scalar per point, into F[p]):
//     p = 0                          f(x)                                                         (:209)
//     row i at R(i) = 1 + 2i(2n-i):  x_i + e_i, x_i - e_i                                          (:226-227, :233)
//                                    then for j = i+1..n-1: (i, j) moved by (+,+), (+,-), (-,+), (-,-)   (:239-260, :269)
// Every other component is exactly x (the reference restores by assignment :272-275, :284-289; nothing drifts).
// The steps (component_eps, kernels_eps.cuh), B copies of x once per call, the per-batch point update below (O(B)
// stores: a slot only differs from x in <= 2 components), and one combine pass that turns F into H.
#pragma once
#include "common.cuh"

namespace fdb {

// first point of row i (0-based)
__device__ __forceinline__ int64_t hess_row_start(int64_t i, int64_t n) { return 1 + 2 * i * (2 * n - i); }

// p (>= 1) -> (i, j, si, sj): component i moved by si*e_i, and (j >= 0) component j moved by sj*e_j
__device__ __forceinline__ void hess_decode(int64_t p, int64_t n, int64_t &i, int64_t &j, int &si, int &sj) {
  // largest i with R(i) <= p: the root of 2i^2 - 4ni + (p-1) = 0, then an exact integer fix-up
  const double disc = (double)n * (double)n - 0.5 * (double)(p - 1);
  int64_t r = n - (int64_t)ceil(sqrt(disc > 0.0 ? disc : 0.0));
  if (r < 0) r = 0;
  if (r > n - 1) r = n - 1;
  while (r > 0 && hess_row_start(r, n) > p) --r;
  while (r + 1 < n && hess_row_start(r + 1, n) <= p) ++r;
  i = r;
  const int64_t o = p - hess_row_start(r, n);
  if (o < 2) {                       // diagonal pair: xpp[i] = xi + epsilon, xmm[i] = xi - epsilon   (:226-227)
    j = -1;
    si = o == 0 ? 1 : -1;
    sj = 0;
    return;
  }
  const int64_t k = (o - 2) >> 2;
  const int s = (int)((o - 2) & 3);  // f(_xpp), f(_xpm), f(_xmp), f(_xmm) in argument order (:269)
  j = r + 1 + k;
  si = s < 2 ? 1 : -1;
  sj = (s & 1) ? -1 : 1;
}

__device__ __forceinline__ double hess_moved(double xk, double ek, int s) {
  return s > 0 ? __dadd_rn(xk, ek) : __dsub_rn(xk, ek);   // xi + epsilon / xi - epsilon   (:226-227, :235-236, :253-254)
}

// X[b][:] = x for b < B, one element per thread: B may be far larger than n here (the dense branch's replicate_x gives
// each thread one component and loops over B, which serialises a small n with a large B)
__global__ void __launch_bounds__(kThreads)
hess_replicate(const double *__restrict__ x, int64_t n, int64_t ldx, int64_t B, double *__restrict__ X) {
  const int64_t total = n * B, stride = (int64_t)gridDim.x * kThreads;
  for (int64_t k = blockIdx.x * (int64_t)kThreads + threadIdx.x; k < total; k += stride) {
    const int64_t b = k / n, j = k - b * n;
    X[b * ldx + j] = __ldg(x + j);
  }
}

// Slot b of the point buffer X holds point p0 + b (b < kc).  It held point prev_p0 + b (b < prevB): restore the <= 2
// components that point moved, then move this point's.  Same thread, so the restore lands before the new value.
__global__ void __launch_bounds__(kThreads)
hess_points(const double *__restrict__ x, const double *__restrict__ eps, int64_t n, int64_t p0, int64_t kc,
            int64_t prev_p0, int64_t prevB, int64_t ldx, double *__restrict__ X) {
  const int64_t b = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  double *slot = X + b * ldx;
  int64_t i, j;
  int si, sj;
  if (b < prevB && prev_p0 + b > 0) {
    hess_decode(prev_p0 + b, n, i, j, si, sj);
    slot[i] = x[i];
    if (j >= 0) slot[j] = x[j];
  }
  if (b < kc && p0 + b > 0) {
    hess_decode(p0 + b, n, i, j, si, sj);
    slot[i] = hess_moved(x[i], eps[i], si);
    if (j >= 0) slot[j] = hess_moved(x[j], eps[j], sj);
  }
}

// One 32 x 32 tile (I, J), I <= J, of the upper triangle per block: the entries i <= j are formed from their F runs
// (contiguous along j for a fixed i: the warp of row i reads 4 x 32 consecutive values), staged through shared memory
// and stored twice — H[i, j] and its mirror H[j, i] — so both halves of the column-major H are written by warps walking
// down a column.  F is passed so that F[1] is 16-byte aligned: every run starts at an odd index (R(i) is odd), which
// makes each entry's four values two aligned 16-byte loads.  Explicit _rn operations in the reference's order (:233,
// :268-269): no contraction can change the bits.
constexpr int kHessTile = 32;

__global__ void __launch_bounds__(kThreads)
hess_combine(const double *__restrict__ F, const double *__restrict__ eps, int64_t n, double *__restrict__ H,
             int64_t ldH) {
  const int64_t I = blockIdx.y, J = blockIdx.x;
  if (I > J) return;
  __shared__ double tile[kHessTile][kHessTile + 1];
  __shared__ double e_row[kHessTile], e_col[kHessTile];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  constexpr int kRowsPerPass = kThreads / 32;
  const int64_t i0 = I * kHessTile, j0 = J * kHessTile;
  if (ty == 0) e_row[tx] = i0 + tx < n ? eps[i0 + tx] : 0.0;
  if (ty == 1) e_col[tx] = j0 + tx < n ? eps[j0 + tx] : 0.0;
  const double two_fx = __dmul_rn(2.0, __ldg(F));                       // 2*fx
  __syncthreads();
  for (int r = ty; r < kHessTile; r += kRowsPerPass) {
    const int64_t i = i0 + r, j = j0 + tx;
    double v = 0.0;
    if (i < n && j < n && i <= j) {
      const int64_t R = hess_row_start(i, n);
      if (i == j) {
        const double2 pm = __ldcs(reinterpret_cast<const double2 *>(F + R));                   // f(_xpp), f(_xmm)
        const double ei = e_row[r];
        v = __ddiv_rn(__dadd_rn(__dsub_rn(pm.x, two_fx), pm.y), __dmul_rn(ei, ei));           // :233
      } else {
        const int64_t q = R + 2 + 4 * (j - i - 1);
        const double2 a = __ldcs(reinterpret_cast<const double2 *>(F + q));                   // f(_xpp), f(_xpm)
        const double2 c = __ldcs(reinterpret_cast<const double2 *>(F + q + 2));               // f(_xmp), f(_xmm)
        v = __ddiv_rn(__dadd_rn(__dsub_rn(__dsub_rn(a.x, a.y), c.x), c.y),
                      __dmul_rn(__dmul_rn(4.0, e_row[r]), e_col[tx]));                         // :268-269
      }
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  // H[i, j], i <= j: column j = j0 + r, the warp walks rows i = i0 + tx
  for (int r = ty; r < kHessTile; r += kRowsPerPass) {
    const int64_t j = j0 + r, i = i0 + tx;
    if (i < n && j < n && i <= j) H[i + j * ldH] = tile[tx][r];
  }
  // H[j, i] = H[i, j], i < j (copytri!(H, 'U') :291): column i = i0 + r, the warp walks rows j = j0 + tx
  for (int r = ty; r < kHessTile; r += kRowsPerPass) {
    const int64_t i = i0 + r, j = j0 + tx;
    if (i < n && j < n && i < j) H[j + i * ldH] = tile[r][tx];
  }
}

}  // namespace fdb
