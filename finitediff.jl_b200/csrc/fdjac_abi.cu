// fdjac_abi.cu — libfdjac_b200.so: plan management + the C ABI declared in include/fdjac_b200.h.
// B200 / sm_100a only.  There is NO CPU fallback: without a CUDA device every compute entry point fails with
// FDB_ERR_NO_DEVICE.  Nothing here includes, links or calls anything under oracle/.
#include "../../include/fdjac_b200.h"

#include <algorithm>
#include <climits>
#include <cstdarg>
#include <cmath>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <numeric>
#include <string>
#include <type_traits>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "kernels_eps.cuh"
#include "kernels_perturb.cuh"
#include "kernels_plan.cuh"
#include "kernels_scatter.cuh"
#include "kernels_staged.cuh"
#include "kernels_jvp.cuh"
#include "kernels_color.cuh"
#include "kernels_hessian.cuh"

using namespace fdb;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;

static fdb_status fail(fdb_status st, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return st;
}

#define CU(expr)                                                                                       \
  do {                                                                                                 \
    cudaError_t e__ = (expr);                                                                          \
    if (e__ != cudaSuccess)                                                                            \
      return fail(FDB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define TRY(expr)                    \
  do {                               \
    fdb_status s__ = (expr);         \
    if (s__ != FDB_OK) return s__;   \
  } while (0)

enum { SP_NONE = 0, SP_CSC = 1, SP_COO = 3, SP_BANDED = 4, SP_JVP = 5, SP_EPS = 6, SP_HESS = 7 };

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess) {
      if (prev == dev) ok = true;
      else ok = cudaSetDevice(dev) == cudaSuccess;
    }
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// identity of a captured call: same function, buffers and scalar arguments => same launch sequence
struct GraphKey {
  void *f = nullptr, *ctx = nullptr;
  const void *x = nullptr, *J = nullptr, *fx = nullptr, *f_in = nullptr;
  double relstep = 0, absstep = 0, dir = 0;
  int n_peers = 0;
  long long peer_generation = 0;
  const void *ext_eps = nullptr;
  bool operator==(const GraphKey &o) const {
    return f == o.f && ctx == o.ctx && x == o.x && J == o.J && fx == o.fx && f_in == o.f_in && relstep == o.relstep &&
           absstep == o.absstep && dir == o.dir && n_peers == o.n_peers && peer_generation == o.peer_generation &&
           ext_eps == o.ext_eps;
  }
};

// ------------------------------------------------------------------------------------------------ plan
struct fdb_plan {
  int device = 0, sm_count = 148;
  int fdtype = FDB_FORWARD, sp_kind = SP_CSC, jkind = FDB_J_CSC_NZVAL;
  int no_drift = 0;
  int rank = 0, world = 1;
  int64_t m = 0, n = 0, E = 0, j_len = 0, ldJ = 0, l = 0, u = 0;
  int32_t C = 0;
  int color_bits = 8;
  bool has_invalid = false;
  // compressed index streams (device)
  void *jcolor = nullptr;     // [n] CT
  int32_t *row32 = nullptr;   // [E]
  void *ecolor = nullptr;     // [E] CT
  int64_t *dest = nullptr;    // [E] or null (identity)
  int32_t *local_of = nullptr;      // [C] device
  int32_t *d_local_colors = nullptr;// [n_local] device (global colour ids, ascending)
  std::vector<int32_t> local_colors, owner;
  // step sizes
  double *eps = nullptr, *sumsq = nullptr, *partial = nullptr;
  int eps_blocks = 0;
  int64_t eps_chunk = 0;
  int32_t eps_group = 1;   // largest aligned lane group without a repeated colour (color_lane_conflicts)
  const double *ext_eps = nullptr;   // step sizes supplied by the caller (fdb_plan_set_external_eps), device, >= C entries
  unsigned int *ticket = nullptr;   // last-block-done counter of color_sumsq_reg
  // eps from the per-colour column lists (CSC plans with more than kEpsRegColors colours)
  bool eps_lists = false;
  int64_t *bucket_start_d = nullptr, *chunk_base_d = nullptr;
  double *eps_list_partial = nullptr;
  int64_t eps_list_max_chunks = 0;
  bool peers_aligned = true;
  bool shared_J = false;            // member of an fdb_group: J is shared with the other members (root zero-fills it)
  // scratch
  double *fx_own = nullptr, *Fp = nullptr, *Fm = nullptr, *xp = nullptr, *xm = nullptr;
  int64_t slabs = 0, ldF = 0, ldx = 0, batch = 1, n_groups = 0;
  int64_t pbatch = 1;   // perturbed points built per perturb pass (>= batch): x is read once for all of them
  // scatter form of a CSC plan (internal; opts->strategy 0..3 is mapped onto it in fdb_plan_create_csc):
  // 0 = one fused pass over J's storage order, 1 = colour-major entry lists (per group of resident colours)
  int strategy = 0;
  bool strategy_auto = true;
  bool lists_resident = false;         // lists with every local colour's f! output resident: ONE launch over them
  // A/B switches (environment, read ONCE when the plan is created — never on the hot path; DESIGN.md §4)
  struct Tunables {
    bool no_staged = false, no_eps_lists = false, no_eps_overlap = false, cm_prefetch = false, force_overlap = false;
    bool no_fx_cm = false, force_fx_cm = false, no_pack = false;
    int hi_stream = -1;                // -1: by pattern (random => evict-first slab gathers), 0 / 1: forced
    // walk direction (r2 A/B 9, C2 step forward / central: 0.2790 / 0.3961 -> 0.2757 / 0.3916 ms): bit 0 the staged scatter
    // starts at the END of J's storage, bit 1 the perturbation pass at the end of x — each reads first what the kernel
    // before it streamed last (still in L2), and the first f! finds the heads of the points the perturbation wrote last
    int reverse = 3;
    int cm_slab_stream = 1;            // colour-major scatter, forward: slab gathers evict-first (CmArgs::slab_stream)
    int eps_depth = 2;                 // color_sumsq_reg: tiles of loads in flight per thread (same summation order, same bits)
    int cols_depth = 0, cols_gx = 64;  // diff_columns: loads in flight per thread (0 = by mode) / cap on the row blocks per column
    int stages = 2;
    char staged_variant[3] = {'6', 'n', 0};
  } tune;
  bool double_buffer = false;          // two output buffers so a group's scatter overlaps the next group's f!
  cudaStream_t side = nullptr;
  cudaEvent_t ev_f[2] = {nullptr, nullptr}, ev_scat[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_eps = nullptr;   // forward mode: the eps pass runs beside f(x) on the side stream
  int32_t *colptr32 = nullptr, *cols_by_color = nullptr;
  // colour-major entry lists of this rank's colours (strategy 1; built by build_cm_lists)
  int32_t *cm_row = nullptr;
  void *cm_slot = nullptr;            // int32 (nzval slot) or int64 (explicit destination: dest != nullptr)
  int64_t *cm_start = nullptr;        // device [n_local + 1]
  double *fx_cm = nullptr;            // forward: f(x) in colour-major order (rebuilt by every Jacobian)
  std::vector<int64_t> cm_start_h;    // host copy; [n_local] .. cm_invalid_end = entries of columns without a valid colour
  int64_t cm_invalid_end = 0;
  // TMA-staged form of the fused pass (row-local patterns; kernels_staged.cuh)
  uint16_t *row16 = nullptr;
  int32_t *tile_w0 = nullptr;
  int32_t stage_W = 0;
  bool staged = false, stage_packed = false;
  std::vector<int64_t> bucket_start;   // [C+2] offsets into cols_by_color; bucket C = columns without a valid colour
  int lanes = 1;
  double mean_row_jump = 0.0;
  // peers (multi-GPU fused gather)
  double **d_peers = nullptr;
  int n_peers = 0;
  // dense-column plans
  int64_t col_begin = 0, col_end = 0;
  double *eps_cols = nullptr;
  // Hessian plans: the 2n^2+1 point values, F[p] at hess_F[p + 1] (so F[1] is 16-byte aligned, see hess_combine)
  double *hess_F = nullptr;
  int64_t hess_points = 0;
  // host-buffer path
  cudaStream_t hstream = nullptr;
  double *h_dx = nullptr, *h_dJ = nullptr, *h_dfx = nullptr, *h_dfin = nullptr;
  // bookkeeping
  std::vector<void *> allocs;
  size_t device_bytes = 0;
  fdb_counters_t cnt{};
  int64_t alg_bytes = 0;
  int64_t last_eps_count = 0;
  bool complex_entry = false;   // set while fdb_jacobian_complex drives the call
  // optional CUDA-graph replay of the whole call
  bool use_graph = false;
  cudaStream_t cstream = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  GraphKey graph_key;
  fdb_counters_t graph_delta{};
  long long peer_generation = 0;
  // optional device-side timing of the scatter launches
  bool timing = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pending, ev_pool;

  fdb_status alloc(void **p, size_t bytes) {
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
      *p = nullptr;
      return fail(FDB_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    }
    allocs.push_back(*p);
    device_bytes += bytes;
    return FDB_OK;
  }
  template <typename T> fdb_status alloc_t(T **p, size_t count) { return alloc((void **)p, count * sizeof(T)); }
  int grid(int64_t items, int per_block = kThreads, int waves = 8) const {
    int64_t b = (items + per_block - 1) / per_block;
    const int64_t cap = (int64_t)sm_count * waves;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
  }
};

// A caller-supplied Int64 array that may live on the host or the device: make it readable by kernels.
struct I64View {
  const int64_t *d = nullptr;
  int64_t *owned = nullptr;
  ~I64View() { if (owned) cudaFree(owned); }
};

static fdb_status view_i64(const int64_t *p, int64_t count, I64View &v) {
  if (!p || count <= 0) { v.d = nullptr; return FDB_OK; }
  cudaPointerAttributes at{};
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); at.type = cudaMemoryTypeUnregistered; }
  if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) { v.d = p; return FDB_OK; }
  CU(cudaMalloc((void **)&v.owned, (size_t)count * sizeof(int64_t)));
  CU(cudaMemcpy(v.owned, p, (size_t)count * sizeof(int64_t), cudaMemcpyHostToDevice));
  v.d = v.owned;
  return FDB_OK;
}

static fdb_status check_device(const fdb_plan_opts *o, int *dev) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return fail(FDB_ERR_NO_DEVICE, "no CUDA device available (%s): libfdjac_b200 has no CPU fallback",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  }
  int d = 0;
  if (!o || o->use_current_device || o->device < 0) { CU(cudaGetDevice(&d)); }
  else d = o->device;
  if (d >= count) return fail(FDB_ERR_INVALID, "device %d out of range (%d devices)", d, count);
  *dev = d;
  return FDB_OK;
}

template <typename F> static fdb_status dispatch_ct(int bits, F &&fn) {
  if (bits == 8) return fn((uint8_t)0);
  if (bits == 16) return fn((uint16_t)0);
  return fn((int32_t)0);
}

static const char *plan_err_text(uint32_t e) {
  if (e & kErrColptr) return "colptr is not a valid CSC column pointer (must start at 1, be non-decreasing, end at nnz+1)";
  if (e & kErrRowRange) return "row index outside 1..m";
  if (e & kErrColRange) return "column index outside 1..n";
  if (e & kErrSlotRange) return "slot outside 1..j_len";
  if (e & kErrMissingInJ) return "a sparsity entry is absent from J's CSC pattern (the reference would insert a new stored entry; unsupported)";
  return "invalid pattern";
}

// colours: max/min, narrow type, per-column colour array
static fdb_status setup_colors(fdb_plan *P, const int64_t *colorvec /*host or device or null*/, I64View &cv) {
  const int64_t n = P->n;
  TRY(view_i64(colorvec, n, cv));
  long long mx = n, mn = n > 0 ? 1 : 0;
  if (cv.d && n > 0) {
    long long *d_mm = nullptr;
    CU(cudaMalloc((void **)&d_mm, 2 * sizeof(long long)));
    long long init[2] = {LLONG_MIN, LLONG_MAX};
    CU(cudaMemcpy(d_mm, init, sizeof init, cudaMemcpyHostToDevice));
    color_minmax<<<P->grid(n), kThreads>>>(cv.d, n, d_mm, d_mm + 1);
    long long out[2];
    cudaError_t e = cudaMemcpy(out, d_mm, sizeof out, cudaMemcpyDeviceToHost);
    cudaFree(d_mm);
    if (e != cudaSuccess) return fail(FDB_ERR_CUDA, "colour min/max failed: %s", cudaGetErrorString(e));
    mx = out[0];
    mn = out[1];
  }
  if (n == 0) mx = 0;
  if (mx < 0) mx = 0;                       // maximum(colorvec) < 1: the colour loop 1:max is empty
  if (mx > 0x7FFFFFF0LL) return fail(FDB_ERR_UNSUPPORTED, "maximum(colorvec) = %lld exceeds 2^31", mx);
  P->C = (int32_t)mx;
  P->has_invalid = n > 0 && mn < 1;
  P->color_bits = mx <= 255 ? 8 : (mx <= 65535 ? 16 : 32);
  TRY(P->alloc(&P->jcolor, (size_t)std::max<int64_t>(n, 1) * (P->color_bits / 8)));
  if (n > 0) {
    uint32_t *d_flags = nullptr;
    const bool window_path = P->C > kEpsRegColors;
    if (window_path) {
      CU(cudaMalloc((void **)&d_flags, sizeof(uint32_t)));
      CU(cudaMemset(d_flags, 0, sizeof(uint32_t)));
    }
    fdb_status st = dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      convert_colors<CT><<<P->grid(n), kThreads>>>(cv.d, n, (CT *)P->jcolor);
      if (window_path) color_lane_conflicts<CT><<<P->grid(n), kThreads>>>((const CT *)P->jcolor, n, P->C, d_flags);
      CU(cudaGetLastError());
      return FDB_OK;
    });
    if (st == FDB_OK && window_path) {
      uint32_t flags = 0;
      cudaError_t e = cudaMemcpy(&flags, d_flags, sizeof flags, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) st = fail(FDB_ERR_CUDA, "colour conflict flags: %s", cudaGetErrorString(e));
      P->eps_group = 1;
      for (int lg = 1; lg <= 5 && !(flags & (1u << lg)); ++lg) P->eps_group = 1 << lg;
    }
    if (d_flags) cudaFree(d_flags);
    if (st != FDB_OK) return st;
  }
  return FDB_OK;
}

// step-size buffers of a coloured plan: eps / sumsq per colour, block partials of the one-pass reduction
static fdb_status alloc_eps_buffers(fdb_plan *P) {
  const int32_t C = P->C;
  TRY(P->alloc_t(&P->eps, std::max<int32_t>(C, 1)));
  TRY(P->alloc_t(&P->sumsq, std::max<int32_t>(C, 1)));
  {
    int64_t nb = (P->n + 2047) / 2048;
    // window path: 64 bytes of shared memory per window colour and block (<= 32 KB) -> one resident wave
    nb = std::max<int64_t>(1, std::min<int64_t>(nb, (int64_t)P->sm_count * (C <= 256 ? 8 : 6)));
    P->eps_blocks = (int)nb;
    int64_t chunk = (P->n + nb - 1) / nb;
    P->eps_chunk = (std::max<int64_t>(chunk, 1) + 31) & ~(int64_t)31;   // aligned 32-column steps on the window path
    const int64_t stride = C <= kEpsRegColors ? kEpsRegColors : std::min<int64_t>(C, kEpsWindow);
    TRY(P->alloc_t(&P->partial, (size_t)nb * stride));
    TRY(P->alloc_t(&P->ticket, 4));
    CU(cudaMemset(P->ticket, 0, 16));
  }

  return FDB_OK;
}

// colour ownership (multi-GPU), local colour list, scratch sizing
static fdb_status finish_colored_plan(fdb_plan *P, const fdb_plan_opts *o, const std::vector<unsigned long long> &count) {
  const int32_t C = P->C;
  P->owner.assign(C, 0);
  const int world = P->world;
  if (world > 1) {
    if (o && o->partition == 1) {
      // LPT: heaviest colour first onto the least-loaded rank (ties -> lowest rank), deterministic on every rank
      std::vector<int32_t> order(C);
      std::iota(order.begin(), order.end(), 0);
      std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return count[a] > count[b]; });
      std::vector<unsigned long long> load(world, 0);
      for (int32_t k : order) {
        int best = 0;
        for (int r = 1; r < world; ++r) if (load[r] < load[best]) best = r;
        P->owner[k] = best;
        load[best] += count[k] + 1;
      }
    } else {
      for (int32_t k = 0; k < C; ++k) P->owner[k] = k % world;
    }
  }
  std::vector<int32_t> local_of(C, -1);
  P->local_colors.clear();
  for (int32_t k = 0; k < C; ++k)
    if (P->owner[k] == P->rank) { local_of[k] = (int32_t)P->local_colors.size(); P->local_colors.push_back(k); }
  const int64_t n_local = (int64_t)P->local_colors.size();
  TRY(P->alloc_t(&P->local_of, std::max<int32_t>(C, 1)));
  TRY(P->alloc_t(&P->d_local_colors, std::max<int64_t>(n_local, 1)));
  if (C > 0) CU(cudaMemcpy(P->local_of, local_of.data(), (size_t)C * 4, cudaMemcpyHostToDevice));
  if (n_local > 0) CU(cudaMemcpy(P->d_local_colors, P->local_colors.data(), (size_t)n_local * 4, cudaMemcpyHostToDevice));

  TRY(alloc_eps_buffers(P));

  // scratch: stacked f! outputs (slabs) + perturbed points
  const bool central = P->fdtype == FDB_CENTRAL;
  const int64_t cw = P->fdtype == FDB_COMPLEX ? 2 : 1;     // doubles per element of the f! in/outputs
  P->ldF = (P->m + 1) & ~(int64_t)1;
  P->ldx = (P->n + 1) & ~(int64_t)1;
  if (P->ldF < 2) P->ldF = 2;
  if (P->ldx < 2) P->ldx = 2;
  int64_t budget = (o && o->scratch_bytes > 0) ? o->scratch_bytes : (int64_t)8 << 30;
  const int64_t per_slab = 8 * cw * P->ldF * (central ? 2 : 1);
  int64_t slabs = std::max<int64_t>(1, budget / per_slab);
  slabs = std::min<int64_t>(slabs, std::max<int64_t>(n_local, 1));
  if (P->sp_kind == SP_CSC && P->strategy == 0 && P->strategy_auto && slabs < n_local) P->strategy = 1;
  if (P->strategy == 1 && !P->lists_resident) {
    // per-colour lists: keep only as many f! outputs in flight as stay L2-resident until their scatter (~48 MB)
    const int64_t l2_slabs = std::max<int64_t>(1, (int64_t)48000000 / per_slab);
    slabs = std::min<int64_t>(slabs, l2_slabs);
  }
  if (P->strategy == 1) slabs = std::min<int64_t>(slabs, kCmMaxGroup);
  P->slabs = slabs;
  P->n_groups = n_local == 0 ? 0 : (n_local + slabs - 1) / slabs;
  int64_t batch = (o && o->max_batch > 1) ? o->max_batch : 1;
  batch = std::min<int64_t>(batch, slabs);
  P->batch = batch;
  // even when f! takes one point per call, build up to kPerturbMaxPoints points per pass over x (one read of x and
  // the colour stream instead of one per colour) when the point buffers fit in an eighth of the scratch budget
  int64_t pbatch = std::max<int64_t>(batch, std::min<int64_t>(kPerturbMaxPoints, std::max<int64_t>(n_local, 1)));
  while (pbatch > batch && pbatch * 8 * cw * P->ldx * (central ? 2 : 1) > budget / 8) --pbatch;
  P->pbatch = pbatch;
  // two output buffers + a side stream: a group's scatter (and its NVLink stores, when peers are set) overlaps the next
  // group's f! evaluations
  // Off by default since r2: the scatter and the next f! compete for the same L2 / DRAM, and the NVLink stores of a
  // 5 MB colour need no hiding.  C4, ms per Jacobian, sequence vs overlapped: 13.08 / 14.06 (1 GPU), 7.06 / 7.24 (2),
  // 3.65 / 3.72 (4), 2.08 / 2.17 (8).  FDB_FORCE_OVERLAP=1 switches the double-buffered side-stream form back on.
  P->double_buffer = false;
  if (P->tune.force_overlap && P->sp_kind == SP_CSC && P->strategy == 1 && (int64_t)P->local_colors.size() > slabs) P->double_buffer = true;
  const size_t nbuf = P->double_buffer ? 2 : 1;
  CU(cudaStreamCreateWithFlags(&P->side, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&P->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&P->ev_eps, cudaEventDisableTiming));
  if (P->double_buffer) {
    for (int b = 0; b < 2; ++b) {
      CU(cudaEventCreateWithFlags(&P->ev_f[b], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&P->ev_scat[b], cudaEventDisableTiming));
    }
  }
  TRY(P->alloc_t(&P->fx_own, (size_t)P->ldF));
  TRY(P->alloc_t(&P->Fp, nbuf * (size_t)slabs * P->ldF * cw));
  TRY(P->alloc_t(&P->xp, (size_t)pbatch * P->ldx * cw));
  if (central) {
    TRY(P->alloc_t(&P->Fm, nbuf * (size_t)slabs * P->ldF));
    TRY(P->alloc_t(&P->xm, (size_t)pbatch * P->ldx));
  }
  return FDB_OK;
}

// Per-colour column lists (cols_by_color, ascending inside a colour; P->bucket_start must be set) and, for more colours
// than the register path takes, the chunk tables of the list-based eps pass.
static fdb_status build_color_lists(fdb_plan *P) {
  const int64_t n = P->n;
  const int32_t C = P->C;
  if (!P->cols_by_color) TRY(P->alloc_t(&P->cols_by_color, (size_t)std::max<int64_t>(n, 1)));
  if (n > 0) {
    // a stable radix sort of the column ids by colour (deterministic: the list-based eps pass sums in list order, and
    // sharded and unsharded plans must produce the same bits)
    uint32_t *k_in = nullptr, *k_out = nullptr;
    int32_t *v_in = nullptr;
    void *d_tmp = nullptr;
    size_t tmp_bytes = 0;
    auto cleanup = [&]() { cudaFree(k_in); cudaFree(k_out); cudaFree(v_in); cudaFree(d_tmp); };
    cudaError_t e = cudaMalloc((void **)&k_in, (size_t)n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&k_out, (size_t)n * 4);
    if (e == cudaSuccess) e = cudaMalloc((void **)&v_in, (size_t)n * 4);
    if (e == cudaSuccess) {
      dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
        using CT = decltype(tag);
        color_sort_keys<CT><<<P->grid(n), kThreads>>>((const CT *)P->jcolor, n, C, k_in, v_in);
        return FDB_OK;
      });
      int end_bit = 1;
      while (end_bit < 32 && ((uint64_t)1 << end_bit) <= (uint64_t)C) ++end_bit;
      e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in, k_out, v_in, P->cols_by_color, (int)n, 0, end_bit);
      if (e == cudaSuccess) e = cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 16);
      if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, k_in, k_out, v_in, P->cols_by_color, (int)n, 0, end_bit);
      if (e == cudaSuccess) e = cudaDeviceSynchronize();
    }
    cleanup();
    if (e != cudaSuccess) return fail(FDB_ERR_CUDA, "column lists: %s", cudaGetErrorString(e));
  }
  // step sizes from the column lists (more colours than the register path takes)
  if (C > kEpsRegColors && C <= (1 << 22) && n > 0) {
    std::vector<int64_t> cb((size_t)C + 1, 0);
    int64_t maxc = 1;
    for (int32_t k = 0; k < C; ++k) {
      const int64_t len = P->bucket_start[(size_t)k + 1] - P->bucket_start[(size_t)k];
      const int64_t nc = (len + kEpsListChunk - 1) / kEpsListChunk;
      cb[(size_t)k + 1] = cb[(size_t)k] + nc;
      maxc = std::max(maxc, nc);
    }
    TRY(P->alloc_t(&P->bucket_start_d, (size_t)C + 2));
    TRY(P->alloc_t(&P->chunk_base_d, (size_t)C + 1));
    TRY(P->alloc_t(&P->eps_list_partial, (size_t)std::max<int64_t>(cb[(size_t)C], 1)));
    CU(cudaMemcpy(P->bucket_start_d, P->bucket_start.data(), ((size_t)C + 2) * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(P->chunk_base_d, cb.data(), ((size_t)C + 1) * 8, cudaMemcpyHostToDevice));
    P->eps_list_max_chunks = maxc;
    P->eps_lists = true;
  }
  return FDB_OK;
}

// host offsets of the per-colour column buckets from their device counts ([C+1]: bucket C = columns without a valid colour)
static fdb_status bucket_offsets(fdb_plan *P, const unsigned long long *d_bucket_counts) {
  const int32_t C = P->C;
  std::vector<unsigned long long> bc((size_t)C + 1, 0);
  CU(cudaMemcpy(bc.data(), d_bucket_counts, ((size_t)C + 1) * 8, cudaMemcpyDeviceToHost));
  P->bucket_start.assign((size_t)C + 2, 0);
  for (int32_t k = 0; k <= C; ++k) P->bucket_start[(size_t)k + 1] = P->bucket_start[(size_t)k] + (int64_t)bc[(size_t)k];
  return FDB_OK;
}

// gather kernel for build_cm_lists: block b copies the column bucket of local colour (or of the invalid bucket) b
__global__ void __launch_bounds__(kThreads)
cm_gather_cols(const int32_t *__restrict__ cols_by_color, const int64_t *__restrict__ src_start /* [nseg] */,
               const int64_t *__restrict__ dst_start /* [nseg+1] */, int64_t nseg, int32_t *__restrict__ list_cols) {
  for (int64_t sgm = blockIdx.x; sgm < nseg; sgm += gridDim.x) {
    const int64_t s0 = src_start[sgm], d0 = dst_start[sgm], cnt = dst_start[sgm + 1] - d0;
    for (int64_t i = threadIdx.x; i < cnt; i += kThreads) list_cols[d0 + i] = cols_by_color[s0 + i];
  }
}

// Colour-major entry lists of the colours this rank evaluates (CSC plans, strategy 1): see kernels_scatter.cuh.
static fdb_status build_cm_lists(fdb_plan *P, const std::vector<unsigned long long> &count /* entries per colour */) {
  const int64_t n_local = (int64_t)P->local_colors.size();
  const int32_t C = P->C;
  const bool zero_bucket = P->rank == 0 && P->bucket_start[(size_t)C + 1] > P->bucket_start[(size_t)C];
  const int64_t nseg = n_local + (zero_bucket ? 1 : 0);
  std::vector<int64_t> src(std::max<int64_t>(nseg, 1), 0), dst((size_t)nseg + 1, 0);
  P->cm_start_h.assign((size_t)n_local + 1, 0);
  unsigned long long valid_total = 0;
  for (int32_t k = 0; k < C; ++k) valid_total += count[(size_t)k];
  for (int64_t li = 0; li < n_local; ++li) {
    const int32_t k = P->local_colors[(size_t)li];
    src[(size_t)li] = P->bucket_start[(size_t)k];
    dst[(size_t)li + 1] = dst[(size_t)li] + (P->bucket_start[(size_t)k + 1] - P->bucket_start[(size_t)k]);
    P->cm_start_h[(size_t)li + 1] = P->cm_start_h[(size_t)li] + (int64_t)count[(size_t)k];
  }
  int64_t e_local = P->cm_start_h[(size_t)n_local];
  P->cm_invalid_end = e_local;
  if (zero_bucket) {
    src[(size_t)n_local] = P->bucket_start[(size_t)C];
    dst[(size_t)n_local + 1] = dst[(size_t)n_local] + (P->bucket_start[(size_t)C + 1] - P->bucket_start[(size_t)C]);
    e_local += P->E - (int64_t)valid_total;
    P->cm_invalid_end = e_local;
  }
  const int64_t ncols = dst[(size_t)nseg];
  TRY(P->alloc_t(&P->cm_start, (size_t)n_local + 1));
  CU(cudaMemcpy(P->cm_start, P->cm_start_h.data(), ((size_t)n_local + 1) * 8, cudaMemcpyHostToDevice));
  TRY(P->alloc_t(&P->cm_row, (size_t)std::max<int64_t>(e_local, 1)));
  {
    // only where f(x) would otherwise be dragged through DRAM once per launch: several launches per Jacobian (colours
    // sharded over GPUs, or more colours than resident slabs).  r2 A/B on C4, scatter ms per Jacobian: 64 per-colour launches
    // 1.56 -> 1.35; one launch over all colours 1.23 -> 1.22 (+ 320 MB): not used there.
    const bool want = P->n_groups > 1 || P->tune.force_fx_cm;
    if (P->fdtype == FDB_FORWARD && e_local > 0 && want && !P->tune.no_fx_cm) TRY(P->alloc_t(&P->fx_cm, (size_t)e_local));
  }
  const bool wide = P->dest != nullptr;
  TRY(P->alloc(&P->cm_slot, (size_t)std::max<int64_t>(e_local, 1) * (wide ? 8 : 4)));
  if (ncols == 0 || e_local == 0) return FDB_OK;
  // temporaries (freed below): column list, counts, offsets, scan scratch
  int64_t *d_src = nullptr, *d_dst = nullptr;
  int32_t *list_cols = nullptr, *list_cnt = nullptr, *list_off = nullptr;
  void *d_tmp = nullptr;
  size_t tmp_bytes = 0;
  auto cleanup = [&]() {
    cudaFree(d_src); cudaFree(d_dst); cudaFree(list_cols); cudaFree(list_cnt); cudaFree(list_off); cudaFree(d_tmp);
  };
#define CM_CU(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); \
    return fail(FDB_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e__)); } } while (0)
  CM_CU(cudaMalloc((void **)&d_src, (size_t)nseg * 8));
  CM_CU(cudaMalloc((void **)&d_dst, ((size_t)nseg + 1) * 8));
  CM_CU(cudaMalloc((void **)&list_cols, (size_t)ncols * 4));
  CM_CU(cudaMalloc((void **)&list_cnt, (size_t)ncols * 4));
  CM_CU(cudaMalloc((void **)&list_off, (size_t)ncols * 4));
  CM_CU(cudaMemcpy(d_src, src.data(), (size_t)nseg * 8, cudaMemcpyHostToDevice));
  CM_CU(cudaMemcpy(d_dst, dst.data(), ((size_t)nseg + 1) * 8, cudaMemcpyHostToDevice));
  cm_gather_cols<<<(int)std::min<int64_t>(nseg, (int64_t)P->sm_count * 16), kThreads>>>(P->cols_by_color, d_src, d_dst, nseg, list_cols);
  cm_column_counts<<<P->grid(ncols), kThreads>>>(list_cols, ncols, P->colptr32, list_cnt);
  CM_CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, list_cnt, list_off, (int)ncols));
  CM_CU(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 16));
  CM_CU(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, list_cnt, list_off, (int)ncols));
  {
    const int lanes = P->lanes;
    const int64_t blocks = (ncols + (kThreads / lanes) - 1) / (kThreads / lanes);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)P->sm_count * 16));
    if (wide) cm_expand<int64_t><<<grid, kThreads>>>(list_cols, list_off, ncols, P->colptr32, P->row32, P->dest, lanes, P->cm_row, (int64_t *)P->cm_slot);
    else cm_expand<int32_t><<<grid, kThreads>>>(list_cols, list_off, ncols, P->colptr32, P->row32, nullptr, lanes, P->cm_row, (int32_t *)P->cm_slot);
  }
  // consistency: the last column's end must be the entry total the per-colour counts promised
  int32_t last_off = 0, last_cnt = 0;
  CM_CU(cudaMemcpy(&last_off, list_off + (ncols - 1), 4, cudaMemcpyDeviceToHost));
  CM_CU(cudaMemcpy(&last_cnt, list_cnt + (ncols - 1), 4, cudaMemcpyDeviceToHost));
  CM_CU(cudaDeviceSynchronize());
#undef CM_CU
  cleanup();
  if ((int64_t)last_off + last_cnt != e_local)
    return fail(FDB_ERR_INVALID, "internal: colour-major list holds %lld entries, expected %lld", (long long)last_off + last_cnt,
                (long long)e_local);
  return FDB_OK;
}

// TMA-staged fused pass: eligible when the whole Jacobian is one resident group on one rank, the destination is the
// identity (CSC nzval) and every 1024-entry tile touches a short row window (row-local pattern).
static fdb_status try_stage_plan(fdb_plan *P) {
  P->staged = false;
  if (P->tune.no_staged) return FDB_OK;
  if (P->sp_kind != SP_CSC || P->dest != nullptr || P->strategy != 0 || P->world != 1 || P->n_groups != 1) return FDB_OK;
  if (P->fdtype == FDB_COMPLEX || P->C < 1) return FDB_OK;
  const int nwin = P->fdtype == FDB_CENTRAL ? 2 * P->C : P->C + 1;
  const int64_t ntiles = P->E / kTile;
  if (nwin > kStageMaxWin || ntiles < 1) return FDB_OK;
  unsigned int *d_span = nullptr;
  TRY(P->alloc_t(&d_span, 1));
  CU(cudaMemset(d_span, 0, 4));
  TRY(P->alloc_t(&P->tile_w0, (size_t)ntiles));
  TRY(P->alloc_t(&P->row16, (size_t)ntiles * kTile));
  const int pgrid = (int)std::min<int64_t>(ntiles, (int64_t)P->sm_count * 16);
  stage_prepare<uint8_t><<<pgrid, kThreads>>>(P->row32, ntiles, P->tile_w0, P->row16, d_span, nullptr, P->C);
  unsigned int span = 0;
  CU(cudaMemcpy(&span, d_span, 4, cudaMemcpyDeviceToHost));
  const int64_t W = ((int64_t)span + 1) & ~(int64_t)1;
  // few colours, short windows: pack the entry's colour into the top 4 bits of its row offset (no colour stream at all)
  P->stage_packed = P->C <= 14 && W <= 4096 && span > 0 && !P->tune.no_pack;
  if (P->stage_packed) {
    TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      stage_prepare<CT><<<pgrid, kThreads>>>(P->row32, ntiles, P->tile_w0, P->row16, d_span, (const CT *)P->ecolor, P->C);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
    CU(cudaDeviceSynchronize());
  }
  const size_t smem = (size_t)2 * nwin * W * 8 + 2 * kStagesMax * 8 + (size_t)P->C * 8;
  if (span == 0 || span > 65535 || smem > (size_t)kStageMaxSmem) return FDB_OK;   // not row-local enough: keep the gather form
  P->stage_W = (int32_t)W;
  P->staged = true;
  return FDB_OK;
}

static fdb_status read_plan_err(uint32_t *d_err, const char *what) {
  uint32_t h = 0;
  CU(cudaMemcpy(&h, d_err, 4, cudaMemcpyDeviceToHost));
  const uint32_t hard = h & ~(uint32_t)(kErrPatternDiff | kErrRowOrder);
  if (hard == kErrMissingInJ) return fail(FDB_ERR_UNSUPPORTED, "%s: %s", what, plan_err_text(hard));
  if (hard) return fail(FDB_ERR_INVALID, "%s: %s", what, plan_err_text(hard));
  return FDB_OK;
}

static bool env_is(const char *name, char c) {
  const char *v = getenv(name);
  return v && v[0] == c;
}

// r2 A/B on C2 (same box, 1965 MHz, scatter us forward / central): gather form 123.4 / 139.5; staged 8 blocks 112.5 / 137.5;
// 6 blocks + index prefetch 108.0 / 139.0; 6 blocks, no prefetch 105.6 / 130.6 (default "6n"); 5 / 4 blocks 106.5 / 108.6
static void read_tunables(fdb_plan *P) {
  auto &t = P->tune;
  t.no_staged = env_is("FDB_NO_STAGED", '1');
  t.no_eps_lists = env_is("FDB_NO_EPS_LISTS", '1');
  t.no_eps_overlap = env_is("FDB_NO_EPS_OVERLAP", '1');
  t.cm_prefetch = env_is("FDB_CM_PREFETCH", '1');
  t.force_overlap = env_is("FDB_FORCE_OVERLAP", '1');
  t.no_fx_cm = env_is("FDB_NO_FX_CM", '1');
  t.force_fx_cm = env_is("FDB_FORCE_FX_CM", '1');
  t.no_pack = env_is("FDB_NO_PACK", '1');
  if (const char *hs = getenv("FDB_HI_STREAM")) t.hi_stream = hs[0] == '1' ? 1 : 0;
  if (const char *v = getenv("FDB_REVERSE")) { if (v[0] >= '0' && v[0] <= '3') t.reverse = v[0] - '0'; }
  if (env_is("FDB_CM_HINT", '0')) t.cm_slab_stream = 0;
  if (env_is("FDB_STAGES", '3')) t.stages = 3;
  if (env_is("FDB_EPS_DEPTH", '1')) t.eps_depth = 1;   // C2 central step 396.4 -> 395.2 us with 2 (profiles/r2_ab8.txt); forward: noise
  if (env_is("FDB_COLS_DEPTH", '4')) t.cols_depth = 4;
  if (env_is("FDB_COLS_DEPTH", '2')) t.cols_depth = 2;
  if (env_is("FDB_COLS_DEPTH", '1')) t.cols_depth = 1;
  if (const char *v = getenv("FDB_COLS_GX")) { const int g = atoi(v); if (g >= 1 && g <= 4096) t.cols_gx = g; }
  if (const char *v = getenv("FDB_STAGED_VARIANT")) {
    if (v[0]) { t.staged_variant[0] = v[0]; t.staged_variant[1] = v[1] ? v[1] : 'n'; }
  }
}

static fdb_status new_plan(fdb_plan **out, const fdb_plan_opts *o, int64_t m, int64_t n) {
  if (!out) return fail(FDB_ERR_INVALID, "plan output pointer is NULL");
  *out = nullptr;
  if (m < 0 || n < 0) return fail(FDB_ERR_INVALID, "negative dimensions m=%lld n=%lld", (long long)m, (long long)n);
  if (m > 0x7FFFFFF0LL || n > 0x7FFFFFF0LL) return fail(FDB_ERR_UNSUPPORTED, "m, n must be < 2^31");
  if (o && o->fdtype != FDB_FORWARD && o->fdtype != FDB_CENTRAL && o->fdtype != FDB_COMPLEX)
    return fail(FDB_ERR_UNSUPPORTED, "Unrecognized fdtype: valid values are forward (0), central (1) and complex (2)");
  int dev = 0;
  TRY(check_device(o, &dev));
  fdb_plan *P = new (std::nothrow) fdb_plan();
  if (!P) return fail(FDB_ERR_NOMEM, "out of host memory");
  P->device = dev;
  P->m = m;
  P->n = n;
  P->fdtype = o ? o->fdtype : FDB_FORWARD;
  P->no_drift = o ? o->no_drift : 0;
  P->use_graph = o && o->use_graph != 0;
  P->shared_J = o && o->shared_j != 0;
  read_tunables(P);
  P->world = (o && o->world > 1) ? o->world : 1;
  P->rank = (o && o->world > 1) ? o->rank : 0;
  if (P->rank < 0 || P->rank >= P->world) {
    const int bad_rank = P->rank, bad_world = P->world;
    delete P;
    return fail(FDB_ERR_INVALID, "rank %d outside world %d", bad_rank, bad_world);
  }
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) { delete P; return fail(FDB_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)); }
  P->sm_count = prop.multiProcessorCount;
  *out = P;
  return FDB_OK;
}

static void free_plan(fdb_plan *P) {
  if (!P) return;
  DeviceGuard g(P->device);
  for (void *p : P->allocs) cudaFree(p);
  for (auto &ev : P->ev_pending) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  for (auto &ev : P->ev_pool) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  if (P->hstream) cudaStreamDestroy(P->hstream);
  if (P->side) cudaStreamDestroy(P->side);
  for (int b = 0; b < 2; ++b) { if (P->ev_f[b]) cudaEventDestroy(P->ev_f[b]); if (P->ev_scat[b]) cudaEventDestroy(P->ev_scat[b]); }
  if (P->ev_fork) cudaEventDestroy(P->ev_fork);
  if (P->ev_eps) cudaEventDestroy(P->ev_eps);
  if (P->graph_exec) cudaGraphExecDestroy(P->graph_exec);
  if (P->cstream) cudaStreamDestroy(P->cstream);
  delete P;
}

#define PLAN_TRY(expr)                                   \
  do {                                                   \
    fdb_status s__ = (expr);                             \
    if (s__ != FDB_OK) { free_plan(P); *plan = nullptr; return s__; } \
  } while (0)

// relstep / absstep keywords of jacobians.jl:508-510: `relstep = default_relstep(fdtype, eltype(x)), absstep = relstep`.
// FDB_STEP_DEFAULT (NaN) means "keyword not given"; every other value — 0 and negatives included — is used as passed
// (relstep = 0 is a pure absolute step, absstep = 0 a pure relative one, exactly as in the reference).
static inline void resolve_steps(int fdtype, double &relstep, double &absstep) {
  if (std::isnan(relstep)) relstep = fdb_default_relstep(fdtype);
  if (std::isnan(absstep)) absstep = relstep;
}

// ------------------------------------------------------------------------------------------------ exported: misc
extern "C" {

int fdb_abi_version(void) { return FDB_ABI_VERSION; }
const char *fdb_last_error(void) { return g_err.c_str(); }
int fdb_device_count(void) {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
  return c;
}

// src/epsilons.jl:134-144
double fdb_default_relstep(int fdtype) {
  if (fdtype == FDB_FORWARD) return sqrt(DBL_EPSILON);
  if (fdtype == FDB_CENTRAL) return cbrt(DBL_EPSILON);
  if (fdtype == FDB_HCENTRAL) return 0x1p-13;   // eps(T)^(1/4) = (2^-52)^(1/4): exactly 2^-13
  return 1.0;
}
// src/epsilons.jl:26-29 / :50-53 / :74-77 (central and hcentral take no dir)
double fdb_compute_epsilon(int fdtype, double x, double relstep, double absstep, double dir) {
  const double a = relstep * fabs(x);
  const double e = a > absstep ? a : absstep;
  return fdtype == FDB_FORWARD ? e * dir : e;
}

// ------------------------------------------------------------------------------------------------ plan creation
fdb_status fdb_plan_create_csc(fdb_plan **plan, int64_t m, int64_t n, const int64_t *colptr, const int64_t *rowval,
                               int jkind, const int64_t *j_colptr, const int64_t *j_rowval, int64_t ldJ,
                               const int64_t *colorvec, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, m, n));
  P = *plan;
  DeviceGuard g(P->device);
  if (!colptr) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "colptr is NULL"); }
  if (jkind != FDB_J_CSC_NZVAL && jkind != FDB_J_DENSE) {
    free_plan(P); *plan = nullptr;
    return fail(FDB_ERR_INVALID, "CSC sparsity supports J kinds CSC_NZVAL and DENSE");
  }
  P->sp_kind = SP_CSC;
  P->jkind = jkind;
  // nnz = colptr[n]-1 : read the last element wherever it lives
  I64View cp, rv, cv, jcp, jrv;
  PLAN_TRY(view_i64(colptr, n + 1, cp));
  int64_t last = 1;
  {
    cudaError_t e = cudaMemcpy(&last, cp.d + n, 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "reading colptr[n]: %s", cudaGetErrorString(e)); }
  }
  const int64_t nnz = last - 1;
  if (nnz < 0 || nnz > 0x7FFFFFF0LL) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_UNSUPPORTED, "nnz=%lld unsupported (must be in [0, 2^31))", (long long)nnz); }
  if (nnz > 0 && !rowval) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "rowval is NULL"); }
  P->E = nnz;
  PLAN_TRY(view_i64(rowval, nnz, rv));
  PLAN_TRY(setup_colors(P, colorvec, cv));

  uint32_t *d_err = nullptr;
  unsigned long long *d_cnt = nullptr;
  PLAN_TRY(P->alloc_t(&d_err, 1));
  PLAN_TRY(P->alloc_t(&d_cnt, std::max<int32_t>(P->C, 1)));
  cudaMemset(d_err, 0, 4);
  cudaMemset(d_cnt, 0, (size_t)std::max<int32_t>(P->C, 1) * 8);
  PLAN_TRY(P->alloc_t(&P->row32, std::max<int64_t>(nnz, 4)));
  PLAN_TRY(P->alloc(&P->ecolor, (size_t)std::max<int64_t>(nnz, 4) * (P->color_bits / 8) + 16));

  bool same_pattern = true;
  bool other_csc = false;
  if (jkind == FDB_J_CSC_NZVAL && j_colptr && j_rowval && (j_colptr != colptr || j_rowval != rowval)) {
    // ext/FiniteDiffSparseArraysExt.jl:51-52
    PLAN_TRY(view_i64(j_colptr, n + 1, jcp));
    int64_t jlast = 1;
    {
      cudaError_t e = cudaMemcpy(&jlast, jcp.d + n, 8, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "reading J.colptr[n]: %s", cudaGetErrorString(e)); }
    }
    if (jlast < 1 || jlast - 1 > 0x7FFFFFF0LL) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "J.colptr[n+1]=%lld is not a valid CSC end pointer", (long long)jlast); }
    const int64_t jnnz = jlast - 1;
    PLAN_TRY(view_i64(j_rowval, jnnz, jrv));
    if (jnnz != nnz) same_pattern = false;
    else {
      compare_i64<<<P->grid(n + 1), kThreads>>>(cp.d, jcp.d, n + 1, d_err);
      if (nnz > 0) compare_i64<<<P->grid(nnz), kThreads>>>(rv.d, jrv.d, nnz, d_err);
      uint32_t h = 0;
      cudaMemcpy(&h, d_err, 4, cudaMemcpyDeviceToHost);
      same_pattern = !(h & kErrPatternDiff);
      cudaMemset(d_err, 0, 4);
    }
    other_csc = !same_pattern;
    P->j_len = jnnz;
  } else if (jkind == FDB_J_CSC_NZVAL) {
    P->j_len = nnz;
  } else {
    if (ldJ < m) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "ldJ=%lld < m=%lld", (long long)ldJ, (long long)m); }
    P->ldJ = ldJ;
    P->j_len = ldJ * n;
  }
  const bool need_dest = jkind == FDB_J_DENSE || other_csc;
  int32_t *col32 = nullptr;
  if (need_dest) {
    PLAN_TRY(P->alloc_t(&col32, std::max<int64_t>(nnz, 1)));
    PLAN_TRY(P->alloc_t(&P->dest, std::max<int64_t>(nnz, 1)));
  }
  validate_colptr<<<P->grid(n + 1), kThreads>>>(cp.d, n, nnz, d_err);
  PLAN_TRY(read_plan_err(d_err, "CSC sparsity"));
  if (other_csc) {   // J's own column pointer is searched by dest_other_csc: it must be a valid one too
    validate_colptr<<<P->grid(n + 1), kThreads>>>(jcp.d, n, P->j_len, d_err);
    PLAN_TRY(read_plan_err(d_err, "J's CSC pattern"));
  }
  if (nnz > 0) {
    PLAN_TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      const size_t hsm = P->C <= kPlanSmemColors ? (size_t)std::max<int32_t>(P->C, 1) * sizeof(unsigned int) : 0;
      expand_csc<CT><<<P->grid(nnz), kThreads, hsm>>>(cp.d, rv.d, m, n, nnz, (const CT *)P->jcolor, P->C, P->row32,
                                                 (CT *)P->ecolor, col32, d_cnt, d_err);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
    if (jkind == FDB_J_DENSE) dest_dense_from_rc<<<P->grid(nnz), kThreads>>>(P->row32, col32, nnz, ldJ, P->dest);
    else if (other_csc) dest_other_csc<<<P->grid(nnz), kThreads>>>(P->row32, col32, nnz, jcp.d, jrv.d, P->dest, d_err);
  }
  PLAN_TRY(read_plan_err(d_err, "CSC sparsity"));
  std::vector<unsigned long long> cnt(std::max<int32_t>(P->C, 1), 0);
  if (P->C > 0) {
    cudaError_t e = cudaMemcpy(cnt.data(), d_cnt, (size_t)P->C * 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "colour counts: %s", cudaGetErrorString(e)); }
  }
  // ---- per-colour column lists + gather-locality metric -> scatter strategy
  {
    const int32_t C = P->C;
    unsigned long long *d_bucket = nullptr, *d_jump = nullptr;
    PLAN_TRY(P->alloc_t(&d_bucket, (size_t)C + 2));
    PLAN_TRY(P->alloc_t(&d_jump, 1));
    cudaMemset(d_bucket, 0, ((size_t)C + 2) * 8);
    cudaMemset(d_jump, 0, 8);
    PLAN_TRY(P->alloc_t(&P->colptr32, (size_t)n + 1));
    PLAN_TRY(P->alloc_t(&P->cols_by_color, (size_t)std::max<int64_t>(n, 1)));
    PLAN_TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      colptr32_and_count<CT><<<P->grid(n + 1), kThreads>>>(cp.d, n, (const CT *)P->jcolor, C, P->colptr32, d_bucket);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
    std::vector<unsigned long long> bc((size_t)C + 1, 0);
    {
      cudaError_t e = cudaMemcpy(bc.data(), d_bucket, ((size_t)C + 1) * 8, cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "column buckets: %s", cudaGetErrorString(e)); }
    }
    P->bucket_start.assign((size_t)C + 2, 0);
    for (int32_t k = 0; k <= C; ++k) P->bucket_start[(size_t)k + 1] = P->bucket_start[(size_t)k] + (int64_t)bc[(size_t)k];
    PLAN_TRY(build_color_lists(P));
    if (nnz > 1) {
      row_jump_sum<<<P->grid(nnz), kThreads>>>(P->row32, nnz, d_jump);
      unsigned long long js = 0;
      cudaMemcpy(&js, d_jump, 8, cudaMemcpyDeviceToHost);
      P->mean_row_jump = (double)js / (double)(nnz - 1);
    }
    int lanes = 1;
    const double avg = n > 0 ? (double)nnz / (double)n : 1.0;
    while (lanes < 32 && lanes < avg) lanes *= 2;
    P->lanes = lanes;
    // opts->strategy: 0 auto, 1 fused storage-order pass, 2 colour-major lists launched per group of resident colours,
    // 3 colour-major lists with every slab resident (one launch).  The lists are what a launch needs whenever it would
    // otherwise stream entries it does not own: several ranks sharing the colours, or more colours than resident slabs
    // (the latter is decided in finish_colored_plan).
    const int want = opts ? opts->strategy : 0;
    bool per_color = P->world > 1;
    if (want == 1) per_color = false;
    if (want == 2 || want == 3) per_color = true;
    P->lists_resident = want == 3;       // colour-major lists, all slabs resident, one launch at the end
    // auto, one GPU, random pattern with many colours: colour-major lists with every slab resident (one launch) — the
    // colour-by-colour order keeps the gathers of a launch phase inside one 8m-byte slab + f(x) instead of spreading them
    // over C slabs at once (C4, r2: 0.96 ms vs 1.18 ms for the storage-order pass; row-local patterns stay fused / staged)
    if (want == 0 && P->world == 1 && P->mean_row_jump > 4096.0 && C >= 16) { per_color = true; P->lists_resident = true; }
    P->strategy = per_color ? 1 : 0;
    P->strategy_auto = want == 0;
  }
  PLAN_TRY(finish_colored_plan(P, opts, cnt));
  if (P->strategy == 1) PLAN_TRY(build_cm_lists(P, cnt));
  PLAN_TRY(try_stage_plan(P));
  // SURVEY.md §8(d): B_alg = 32*nnz + 16*n + 8 (valid colouring; Int64 indices as at the ABI)
  P->alg_bytes = 32 * nnz + 16 * n + 8;
  {
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "plan build: %s", cudaGetErrorString(e)); }
  }
  return FDB_OK;
}

fdb_status fdb_plan_create_coo(fdb_plan **plan, int64_t m, int64_t n, int64_t nnz, const int64_t *rows_index,
                               const int64_t *cols_index, int jkind, const int64_t *slots, int64_t ldJ_or_jlen,
                               const int64_t *colorvec, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, m, n));
  P = *plan;
  DeviceGuard g(P->device);
  if (nnz < 0 || nnz > 0x7FFFFFF0LL) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_UNSUPPORTED, "nnz=%lld unsupported", (long long)nnz); }
  if (nnz > 0 && (!rows_index || !cols_index)) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "rows_index/cols_index NULL"); }
  if (jkind != FDB_J_DENSE && jkind != FDB_J_SLOTS) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "COO sparsity supports J kinds DENSE and SLOTS"); }
  if (jkind == FDB_J_SLOTS && nnz > 0 && !slots) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "slots is NULL"); }
  if (jkind == FDB_J_DENSE && ldJ_or_jlen < m) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "ldJ < m"); }
  P->sp_kind = SP_COO;
  P->jkind = jkind;
  P->E = nnz;
  if (jkind == FDB_J_DENSE) { P->ldJ = ldJ_or_jlen; P->j_len = ldJ_or_jlen * n; }
  else P->j_len = ldJ_or_jlen;
  I64View rv, cvw, sv, cv;
  PLAN_TRY(view_i64(rows_index, nnz, rv));
  PLAN_TRY(view_i64(cols_index, nnz, cvw));
  if (jkind == FDB_J_SLOTS) PLAN_TRY(view_i64(slots, nnz, sv));
  PLAN_TRY(setup_colors(P, colorvec, cv));
  uint32_t *d_err = nullptr;
  unsigned long long *d_cnt = nullptr;
  PLAN_TRY(P->alloc_t(&d_err, 1));
  PLAN_TRY(P->alloc_t(&d_cnt, std::max<int32_t>(P->C, 1)));
  cudaMemset(d_err, 0, 4);
  cudaMemset(d_cnt, 0, (size_t)std::max<int32_t>(P->C, 1) * 8);
  PLAN_TRY(P->alloc_t(&P->row32, std::max<int64_t>(nnz, 4)));
  PLAN_TRY(P->alloc(&P->ecolor, (size_t)std::max<int64_t>(nnz, 4) * (P->color_bits / 8) + 16));
  PLAN_TRY(P->alloc_t(&P->dest, std::max<int64_t>(nnz, 1)));
  if (nnz > 0) {
    PLAN_TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      const size_t hsm = P->C <= kPlanSmemColors ? (size_t)std::max<int32_t>(P->C, 1) * sizeof(unsigned int) : 0;
      prepare_coo<CT><<<P->grid(nnz), kThreads, hsm>>>(rv.d, cvw.d, jkind == FDB_J_SLOTS ? sv.d : nullptr, nnz, m, n, P->ldJ,
                                                  P->j_len, (const CT *)P->jcolor, P->C, P->row32, (CT *)P->ecolor,
                                                  P->dest, d_cnt, d_err);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
  }
  PLAN_TRY(read_plan_err(d_err, "COO sparsity"));
  std::vector<unsigned long long> cnt(std::max<int32_t>(P->C, 1), 0);
  if (P->C > 0) cudaMemcpy(cnt.data(), d_cnt, (size_t)P->C * 8, cudaMemcpyDeviceToHost);
  PLAN_TRY(finish_colored_plan(P, opts, cnt));
  P->alg_bytes = 32 * nnz + 16 * n + 8;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "plan build: %s", cudaGetErrorString(e)); }
  return FDB_OK;
}

fdb_status fdb_plan_create_banded(fdb_plan **plan, int64_t m, int64_t n, int64_t l, int64_t u, int jkind, int64_t ldJ,
                                  const int64_t *colorvec, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, m, n));
  P = *plan;
  DeviceGuard g(P->device);
  if (jkind != FDB_J_BAND && jkind != FDB_J_DENSE) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "banded sparsity supports J kinds BAND and DENSE"); }
  if (l + u + 1 < 1 || l < -n || u < -m) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "invalid bandwidths l=%lld u=%lld", (long long)l, (long long)u); }
  if (jkind == FDB_J_DENSE && ldJ < m) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "ldJ < m"); }
  P->sp_kind = SP_BANDED;
  P->jkind = jkind;
  P->l = l;
  P->u = u;
  P->ldJ = ldJ;
  P->j_len = jkind == FDB_J_BAND ? (l + u + 1) * n : ldJ * n;
  I64View cv;
  PLAN_TRY(setup_colors(P, colorvec, cv));
  unsigned long long *d_cnt = nullptr;
  PLAN_TRY(P->alloc_t(&d_cnt, std::max<int32_t>(P->C, 1)));
  cudaMemset(d_cnt, 0, (size_t)std::max<int32_t>(P->C, 1) * 8);
  if (n > 0 && P->C > 0) {
    PLAN_TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      count_band_colors<CT><<<P->grid(n), kThreads>>>((const CT *)P->jcolor, m, n, l, u, P->C, d_cnt);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
  }
  std::vector<unsigned long long> cnt(std::max<int32_t>(P->C, 1), 0);
  if (P->C > 0) cudaMemcpy(cnt.data(), d_cnt, (size_t)P->C * 8, cudaMemcpyDeviceToHost);
  unsigned long long total = 0;
  for (auto c : cnt) total += c;
  P->E = (int64_t)total;
  PLAN_TRY(finish_colored_plan(P, opts, cnt));
  // SURVEY.md §8(d) banded: 8*sum_c band_len(c) written + 16*m*C read
  P->alg_bytes = 8 * (int64_t)total + 16 * m * (int64_t)P->C;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_CUDA, "plan build: %s", cudaGetErrorString(e)); }
  return FDB_OK;
}

// dense column branch over the leading `ncols` components (ncols == n for the default colorvec = 1:n)
static fdb_status create_dense(fdb_plan **plan, int64_t m, int64_t n, int64_t ldJ, int64_t ncols, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, m, n));
  P = *plan;
  DeviceGuard g(P->device);
  if (ldJ < m) { free_plan(P); *plan = nullptr; return fail(FDB_ERR_INVALID, "ldJ < m"); }
  P->sp_kind = SP_NONE;
  P->jkind = FDB_J_DENSE;
  P->ldJ = ldJ;
  // contiguous column blocks per rank (SURVEY.md §8e)
  const int64_t per = (ncols + P->world - 1) / P->world;
  P->col_begin = std::min<int64_t>(ncols, per * P->rank);
  P->col_end = std::min<int64_t>(ncols, P->col_begin + per);
  const int64_t ncl = P->col_end - P->col_begin;
  P->j_len = ldJ * ncl;
  P->E = m * ncl;
  P->C = (int32_t)n;
  const bool central = P->fdtype == FDB_CENTRAL;
  P->ldF = std::max<int64_t>(2, (m + 1) & ~(int64_t)1);
  P->ldx = std::max<int64_t>(2, (n + 1) & ~(int64_t)1);
  int64_t batch = (opts && opts->max_batch > 1) ? opts->max_batch : 1;
  int64_t budget = (opts && opts->scratch_bytes > 0) ? opts->scratch_bytes : (int64_t)8 << 30;
  const int64_t cw = P->fdtype == FDB_COMPLEX ? 2 : 1;
  const int64_t per_point = 8 * cw * (P->ldx + P->ldF * (central ? 2 : 1));
  batch = std::max<int64_t>(1, std::min<int64_t>(batch, budget / per_point));
  batch = std::min<int64_t>(batch, std::max<int64_t>(ncl, 1));
  batch = std::min<int64_t>(batch, 65535);   // gridDim.y of diff_columns
  P->batch = batch;
  P->slabs = batch;
  P->n_groups = ncl == 0 ? 0 : (ncl + batch - 1) / batch;
  PLAN_TRY(P->alloc_t(&P->fx_own, (size_t)P->ldF));
  PLAN_TRY(P->alloc_t(&P->Fp, (size_t)batch * P->ldF * cw));
  if (central) PLAN_TRY(P->alloc_t(&P->Fm, (size_t)batch * P->ldF));
  PLAN_TRY(P->alloc_t(&P->xp, (size_t)batch * P->ldx * cw));
  PLAN_TRY(P->alloc_t(&P->eps_cols, (size_t)std::max<int64_t>(ncl, 1)));
  // SURVEY.md §8(d) dense: 24*m per column
  P->alg_bytes = 24 * m * ncl;
  return FDB_OK;
}

fdb_status fdb_plan_create_dense(fdb_plan **plan, int64_t m, int64_t n, int64_t ldJ, const fdb_plan_opts *opts) {
  return create_dense(plan, m, n, ldJ, n, opts);
}

// sparsity === nothing with a caller-supplied colorvec, exactly as jacobians.jl:547-557 / :589-598 / :625-631 are written:
// `for color_i in 1:maximum(colorvec)` perturbs COMPONENT color_i (the colour id is used as an index) and writes
// J[:, color_i]; J is not zero-filled (:530 only fills when sparsity !== nothing), so columns beyond maximum(colorvec)
// keep their contents.  maximum(colorvec) > n indexes x1 out of bounds in the reference (BoundsError) -> FDB_ERR_INVALID.
fdb_status fdb_plan_create_dense_colorvec(fdb_plan **plan, int64_t m, int64_t n, int64_t ldJ, const int64_t *colorvec,
                                          const fdb_plan_opts *opts) {
  if (!plan) return fail(FDB_ERR_INVALID, "plan output pointer is NULL");
  *plan = nullptr;
  if (!colorvec) return create_dense(plan, m, n, ldJ, n, opts);
  if (n < 0 || m < 0) return fail(FDB_ERR_INVALID, "negative dimensions");
  int dev = 0;
  TRY(check_device(opts, &dev));
  DeviceGuard g(dev);
  long long mx = 0;
  if (n > 0) {
    I64View cv;
    TRY(view_i64(colorvec, n, cv));
    long long *d_mm = nullptr;
    CU(cudaMalloc((void **)&d_mm, 2 * sizeof(long long)));
    const long long init[2] = {LLONG_MIN, LLONG_MAX};
    cudaMemcpy(d_mm, init, sizeof init, cudaMemcpyHostToDevice);
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + kThreads - 1) / kThreads, 148 * 8));
    color_minmax<<<blocks, kThreads>>>(cv.d, n, d_mm, d_mm + 1);
    long long out[2] = {0, 0};
    const cudaError_t e = cudaMemcpy(out, d_mm, sizeof out, cudaMemcpyDeviceToHost);
    cudaFree(d_mm);
    if (e != cudaSuccess) return fail(FDB_ERR_CUDA, "colour maximum failed: %s", cudaGetErrorString(e));
    mx = out[0];
  }
  if (mx > n) return fail(FDB_ERR_INVALID, "sparsity=nothing: maximum(colorvec)=%lld indexes x beyond length(x)=%lld "
                                           "(BoundsError in the reference, jacobians.jl:549)", mx, (long long)n);
  return create_dense(plan, m, n, ldJ, mx < 0 ? 0 : (int64_t)mx, opts);
}

fdb_status fdb_plan_destroy(fdb_plan *plan) {
  free_plan(plan);
  return FDB_OK;
}

fdb_status fdb_plan_info(const fdb_plan *P, fdb_plan_info_t *info) {
  if (!P || !info) return fail(FDB_ERR_INVALID, "NULL argument");
  memset(info, 0, sizeof *info);
  info->m = P->m;
  info->n = P->n;
  info->n_entries = P->E;
  info->j_len = P->j_len;
  info->n_colors = P->C;
  const int64_t n_local = P->sp_kind == SP_NONE ? P->col_end - P->col_begin
                          : P->sp_kind == SP_HESS ? P->n : (int64_t)P->local_colors.size();
  info->n_local_colors = n_local;
  info->n_groups = P->n_groups;
  info->slabs = P->slabs;
  info->fcalls_per_jacobian = P->fdtype == FDB_CENTRAL ? 2 * n_local : (P->fdtype == FDB_COMPLEX ? n_local : 1 + n_local);
  if (P->sp_kind == SP_HESS) info->fcalls_per_jacobian = P->hess_points;   // 2n^2+1 (hessians.jl:209,233,269)
  info->device_bytes = (int64_t)P->device_bytes;
  info->fdtype = P->fdtype;
  info->jkind = P->jkind;
  info->sp_kind = P->sp_kind;
  info->color_bits = P->color_bits;
  info->alg_bytes_scatter = P->alg_bytes;
  info->strategy = P->strategy;
  info->lanes = P->lanes;
  info->mean_row_jump = P->mean_row_jump;
  info->staged = P->staged ? 1 : 0;
  info->lists_resident = P->lists_resident ? 1 : 0;
  {
    // compulsory bytes of the formulation that runs (see the header); slabs read per entry: 1 (forward / complex), 2 (central)
    const int64_t ct = P->color_bits / 8;
    const int64_t slabs_read = P->fdtype == FDB_CENTRAL ? 2 : 1;
    const int64_t fx_once = P->fdtype == FDB_FORWARD ? 8 * P->m : 0;
    if (P->sp_kind == SP_CSC || P->sp_kind == SP_COO) {
      if (P->sp_kind == SP_CSC && P->strategy == 1) {
        const int64_t e_local = P->cm_start_h.empty() ? 0 : P->cm_start_h.back();
        info->moved_bytes_scatter = e_local * (4 + (P->dest ? 8 : 4) + 8 * slabs_read + 8) + fx_once + (P->fx_cm ? e_local * (4 + 8 + 8) : 0);
      } else {
        const int64_t C = std::max<int32_t>(P->C, 1);
        const int64_t owned = P->world > 1 ? P->E * (int64_t)P->local_colors.size() / C : P->E;   // approx. share
        info->moved_bytes_scatter = P->E * (4 + ct) * std::max<int64_t>(P->n_groups, 1) + owned * (8 * slabs_read + 8 + (P->dest ? 8 : 0)) + fx_once;
        if (P->staged)   // 16-bit row offsets; every slab row and f(x) row staged once
          info->moved_bytes_scatter = P->E * (2 + (P->stage_packed ? 0 : ct) + 8) + 8 * P->m * (int64_t)(P->fdtype == FDB_CENTRAL ? 2 * P->C : P->C + 1);
      }
    } else {
      info->moved_bytes_scatter = P->alg_bytes;
    }
  }
  return FDB_OK;
}

fdb_status fdb_plan_counters(const fdb_plan *P, fdb_counters_t *out) {
  if (!P || !out) return fail(FDB_ERR_INVALID, "NULL argument");
  *out = P->cnt;
  return FDB_OK;
}

fdb_status fdb_plan_dense_range(const fdb_plan *P, int64_t *b, int64_t *e) {
  if (!P || !b || !e) return fail(FDB_ERR_INVALID, "NULL argument");
  *b = P->col_begin;
  *e = P->col_end;
  return FDB_OK;
}

fdb_status fdb_plan_color_owner(const fdb_plan *P, int32_t *owner_out, int64_t cap) {
  if (!P || !owner_out) return fail(FDB_ERR_INVALID, "NULL argument");
  if (P->sp_kind == SP_NONE) return fail(FDB_ERR_INVALID, "dense plans partition columns by range");
  if (cap < (int64_t)P->owner.size()) return fail(FDB_ERR_INVALID, "owner_out too small");
  std::copy(P->owner.begin(), P->owner.end(), owner_out);
  return FDB_OK;
}

fdb_status fdb_plan_get_eps(fdb_plan *P, double *h_eps, int64_t cap, void *stream) {
  if (!P || !h_eps) return fail(FDB_ERR_INVALID, "NULL argument");
  DeviceGuard g(P->device);
  const int64_t count = P->sp_kind == SP_NONE ? P->col_end - P->col_begin : P->C;   // JVP plans: C == 1; Hessian plans: C == n
  if (cap < count) return fail(FDB_ERR_INVALID, "h_eps too small (%lld < %lld)", (long long)cap, (long long)count);
  const double *src = P->sp_kind == SP_NONE ? P->eps_cols : P->eps;
  if (count > 0) {
    CU(cudaMemcpyAsync(h_eps, src, (size_t)count * 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
  }
  return FDB_OK;
}

fdb_status fdb_plan_enable_timing(fdb_plan *P, int enable) {
  if (!P) return fail(FDB_ERR_INVALID, "NULL plan");
  P->timing = enable != 0;
  return FDB_OK;
}

fdb_status fdb_plan_read_timing(fdb_plan *P, double *scatter_ms, int64_t *scatter_launches) {
  if (!P || !scatter_ms || !scatter_launches) return fail(FDB_ERR_INVALID, "NULL argument");
  DeviceGuard g(P->device);
  double total = 0.0;
  int64_t count = 0;
  for (auto &ev : P->ev_pending) {
    CU(cudaEventSynchronize(ev.second));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, ev.first, ev.second));
    total += ms;
    count += 1;
    P->ev_pool.push_back(ev);
  }
  P->ev_pending.clear();
  *scatter_ms = total;
  *scatter_launches = count;
  return FDB_OK;
}

fdb_status fdb_plan_set_peers(fdb_plan *P, int n_peers, double *const *peer_J) {
  if (!P) return fail(FDB_ERR_INVALID, "NULL plan");
  if (n_peers < 0 || n_peers > 64) return fail(FDB_ERR_INVALID, "n_peers out of range");
  if (P->sp_kind == SP_NONE || P->sp_kind == SP_BANDED || P->sp_kind == SP_HESS)
    return fail(FDB_ERR_UNSUPPORTED, "peer stores are implemented for the entry-driven (CSC / COO) scatters");
  DeviceGuard g(P->device);
  if (!P->d_peers) TRY(P->alloc_t(&P->d_peers, 64));
  if (n_peers > 0) CU(cudaMemcpy(P->d_peers, peer_J, (size_t)n_peers * sizeof(double *), cudaMemcpyHostToDevice));
  P->n_peers = n_peers;
  P->peer_generation += 1;
  P->peers_aligned = true;
  for (int i = 0; i < n_peers; ++i)
    if (reinterpret_cast<uintptr_t>(peer_J[i]) & 15) P->peers_aligned = false;
  return FDB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ the hot path
struct ScatterTimer {
  fdb_plan *P;
  cudaStream_t s;
  std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
  ScatterTimer(fdb_plan *p, cudaStream_t st) : P(p), s(st) {
    if (!P->timing) return;
    if (!P->ev_pool.empty()) { ev = P->ev_pool.back(); P->ev_pool.pop_back(); }
    else { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); }
    cudaEventRecord(ev.first, s);
  }
  ~ScatterTimer() {
    if (!P->timing || !ev.first) return;
    cudaEventRecord(ev.second, s);
    P->ev_pending.push_back(ev);
  }
};

// fill_matrix!(J, false) (jacobians.jl:530-532, :663).  A dense J may be a strided column-major view (ldJ > m): only
// rows [0, m) of every column belong to J — the padding rows between the columns are not touched.
static fdb_status zero_J(const fdb_plan *P, double *J, cudaStream_t s) {
  if (P->jkind == FDB_J_DENSE && P->ldJ > P->m) {
    const int64_t ncols = P->sp_kind == SP_NONE ? P->col_end - P->col_begin : P->n;
    if (P->m > 0 && ncols > 0)
      CU(cudaMemset2DAsync(J, (size_t)P->ldJ * 8, 0, (size_t)P->m * 8, (size_t)ncols, s));
    return FDB_OK;
  }
  CU(cudaMemsetAsync(J, 0, (size_t)P->j_len * 8, s));
  return FDB_OK;
}

static fdb_status call_f(fdb_plan *P, fdb_fn f, void *ctx, double *fx, const double *x, int64_t batch, cudaStream_t s) {
  const int rc = f(ctx, fx, x, batch, P->ldF, P->ldx, (void *)s);
  P->cnt.f_invocations += 1;
  P->cnt.f_points += batch;
  if (rc != 0) return fail(FDB_ERR_CALLBACK, "user f! returned %d", rc);
  return FDB_OK;
}

// Persistent-grid sizing: exactly the number of blocks that are resident at once (SMs x blocks/SM from the occupancy
// calculator), capped by the work — a single full wave, no partial-wave tail (the r1 ncu capture showed 1184 blocks on
// 888 resident slots costing a half-empty second wave).
template <typename K>
static int resident_grid(const fdb_plan *P, K kernel, size_t dyn_smem, int64_t work_blocks) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, dyn_smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    per_sm = 4;
  }
  int64_t g = (int64_t)P->sm_count * per_sm;
  if (g > work_blocks) g = work_blocks;
  if (g < 1) g = 1;
  return (int)g;
}

template <typename CT>
static fdb_status run_eps(fdb_plan *P, const double *x, double relstep, double absstep, double dir, cudaStream_t s) {
  const int32_t C = P->C;
  if (C <= 0) return FDB_OK;
  if (P->fdtype == FDB_COMPLEX) {   // epsilon = eps(eltype(x))  jacobians.jl:624 — the same for every colour
    fill_value<<<(C + kThreads - 1) / kThreads, kThreads, 0, s>>>(P->eps, C, DBL_EPSILON);
    P->cnt.kernel_launches += 1;
    CU(cudaGetLastError());
    return FDB_OK;
  }
  EpsParams prm{P->fdtype == FDB_CENTRAL ? 1 : 0, relstep, absstep, dir};
  if (P->eps_lists) {
    if (!P->tune.no_eps_lists) {
      dim3 grid((unsigned)std::min<int64_t>(P->eps_list_max_chunks, 1024), (unsigned)std::min<int32_t>(C, 65535));
      color_sumsq_lists<<<grid, kThreads, 0, s>>>(x, P->cols_by_color, P->bucket_start_d, P->chunk_base_d, C, P->eps_list_partial);
      finalize_eps_lists<<<(int)std::min<int64_t>(((int64_t)C * 32 + kThreads - 1) / kThreads, (int64_t)P->sm_count * 8), kThreads, 0, s>>>(
          P->eps_list_partial, P->chunk_base_d, C, prm, P->eps, P->sumsq);
      P->cnt.kernel_launches += 2;
      CU(cudaGetLastError());
      return FDB_OK;
    }
  }
  if (C <= kEpsRegColors) {
    const int64_t ntiles = (P->n + kTile - 1) / kTile;
    const int aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    auto go = [&](auto kern) {
      const int grid = std::min(resident_grid(P, kern, 0, ntiles), P->eps_blocks);  // partial capacity
      kern<<<grid, kThreads, 0, s>>>(x, (const CT *)P->jcolor, P->n, aligned, C, prm, P->partial, P->ticket, P->eps, P->sumsq);
    };
    if (C <= 4) { if (P->tune.eps_depth == 2) go(color_sumsq_reg<CT, 4, 2>); else go(color_sumsq_reg<CT, 4, 1>); }
    else { if (P->tune.eps_depth == 2) go(color_sumsq_reg<CT, 8, 2>); else go(color_sumsq_reg<CT, 8, 1>); }
    P->cnt.kernel_launches += 1;
  } else {
    for (int32_t k0 = 0; k0 < C; k0 += kEpsWindow) {
      const int32_t W = std::min<int32_t>(kEpsWindow, C - k0);
      color_sumsq_win<CT><<<P->eps_blocks, kThreads, (size_t)kEpsWarps * W * sizeof(double), s>>>(
          x, (const CT *)P->jcolor, P->n, P->eps_chunk, k0, W, P->eps_group, P->partial);
      // partial rows are W wide for this pass
      finalize_eps<<<(W * 32 + kThreads - 1) / kThreads, kThreads, 0, s>>>(P->partial, P->eps_blocks, W, k0, W, prm,
                                                                        P->eps, P->sumsq);
      P->cnt.kernel_launches += 2;
    }
  }
  CU(cudaGetLastError());
  return FDB_OK;
}

template <typename CT, int MODE>
static fdb_status run_colored(fdb_plan *P, fdb_fn f, void *ctx, const double *x, double *J, double *fx,
                              const double *f_in, double relstep, double absstep, double dir, cudaStream_t s) {
  constexpr bool CENTRAL = MODE == kCentral;
  constexpr bool COMPLEX = MODE == kComplex;
  // strides, in doubles, of one f! output slab / one perturbed point (complex128 in complex-step mode)
  const int64_t sF = COMPLEX ? 2 * P->ldF : P->ldF, sX = COMPLEX ? 2 * P->ldx : P->ldx;
  const int64_t n_local = (int64_t)P->local_colors.size();
  // fill_matrix!(J, false)  jacobians.jl:530-532 — needed where the scatter does not define every slot itself
  const bool ident = P->dest == nullptr && P->sp_kind != SP_BANDED;
  const bool band_data = P->sp_kind == SP_BANDED && P->jkind == FDB_J_BAND;
  // (identity / band-data launches define every slot this rank is responsible for, including zeros for columns without
  //  a valid colour).  With peer buffers set the caller zero-fills J and synchronises the ranks BEFORE the call: a memset
  //  here would race with the peers' stores.
  const bool self_defining = (ident || band_data) && n_local > 0;
  if (!self_defining && P->n_peers == 0 && !P->shared_J && P->j_len > 0) TRY(zero_J(P, J, s));
  // forward mode without f_in: f(x) (jacobians.jl:541) and the step-size pass are independent — the eps kernels run on the
  // side stream beside the user's f(x) and are joined before the first perturbation (a parallel branch of the CUDA graph)
  bool eps_beside_fx = MODE == kForward && !f_in && !P->ext_eps && P->side && P->ev_fork && P->C > 0;
  if (P->tune.no_eps_overlap) eps_beside_fx = false;
  if (P->ext_eps) {
    // sharded runs: the step sizes of the FULL x come from outside (fdb_color_eps on the full vector)
    if (P->C > 0) CU(cudaMemcpyAsync(P->eps, P->ext_eps, (size_t)P->C * 8, cudaMemcpyDeviceToDevice, s));
  } else if (eps_beside_fx) {
    CU(cudaEventRecord(P->ev_fork, s));
    CU(cudaStreamWaitEvent(P->side, P->ev_fork, 0));
    TRY(run_eps<CT>(P, x, relstep, absstep, dir, P->side));
    CU(cudaEventRecord(P->ev_eps, P->side));
  } else {
    TRY(run_eps<CT>(P, x, relstep, absstep, dir, s));
  }
  const double *vfx = nullptr;
  if (MODE == kForward) {
    if (f_in) vfx = f_in;                                  // jacobians.jl:543-544
    else { TRY(call_f(P, f, ctx, fx, x, 1, s)); vfx = fx; } // :541-542
  }
  if (eps_beside_fx) CU(cudaStreamWaitEvent(s, P->ev_eps, 0));
  // colour-major lists, forward: f(x) once into list order (read as a coalesced stream by every colour's launch)
  if (MODE == kForward && P->sp_kind == SP_CSC && P->strategy == 1 && P->fx_cm && n_local > 0) {
    const int64_t cnt = P->cm_start_h[(size_t)n_local];
    if (cnt > 0) {
      const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((cnt + kThreads * 4 - 1) / (kThreads * 4), (int64_t)P->sm_count * 16));
      ScatterTimer tm(P, s);            // part of the diff+scatter formulation: timed with it
      gather_fx_cm<<<grid, kThreads, 0, s>>>(P->cm_row, vfx, cnt, P->fx_cm);
      P->cnt.kernel_launches += 1;
    }
  }
  // build the perturbed points of local colours [li0, li0+kc) into the point buffers (one pass over x per 4 colours)
  auto perturb_window = [&](int64_t li0, int64_t kc) -> fdb_status {
      for (int64_t q0 = 0; q0 < kc; q0 += kPerturbMaxPoints) {
        PerturbArgs pa{};
        pa.x = x; pa.jcolor = P->jcolor; pa.eps = P->eps;
        pa.xp = P->xp + q0 * sX; pa.xm = CENTRAL ? P->xm + q0 * sX : nullptr;
        pa.n = P->n; pa.ldx = sX; pa.C = P->C; pa.drift = P->no_drift ? 0 : 1;
        pa.reverse = (P->tune.reverse >> 1) & 1;
        pa.kcount = (int32_t)std::min<int64_t>(kPerturbMaxPoints, kc - q0);
        for (int32_t q = 0; q < pa.kcount; ++q) pa.k[q] = P->local_colors[(size_t)(li0 + q0 + q)];
        pa.aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(P->xp) |
                       reinterpret_cast<uintptr_t>(P->xm)) & 15) == 0 && (P->ldx & 1) == 0;
        const size_t sm = P->C <= kPerturbSmemColors ? (size_t)P->C * sizeof(double) : 0;
        const int64_t tiles = (P->n + kTile - 1) / kTile;
        if (COMPLEX) {
          if (pa.kcount == 1) perturb_complex<CT, 1><<<P->grid(P->n), kThreads, 0, s>>>(pa);
          else perturb_complex<CT, kPerturbMaxPoints><<<P->grid(P->n), kThreads, 0, s>>>(pa);
        } else {
          // store-heavy (NP points written per element read): an oversubscribed grid, like the band and dense-column
          // kernels (C2 step, 1x -> 16x the resident wave: forward 0.299 -> 0.291 ms, central 0.424 -> 0.408 ms)
          constexpr int kPerturbGridOver = 16;
          auto over = [&](int g) { return (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)g * kPerturbGridOver, tiles)); };
          if (pa.kcount == 1)
            perturb_colors<CT, CENTRAL, 1><<<over(resident_grid(P, perturb_colors<CT, CENTRAL, 1>, sm, tiles)), kThreads, sm, s>>>(pa);
          else
            perturb_colors<CT, CENTRAL, kPerturbMaxPoints><<<over(resident_grid(P, perturb_colors<CT, CENTRAL, kPerturbMaxPoints>, sm, tiles)), kThreads, sm, s>>>(pa);
        }
        P->cnt.kernel_launches += 1;
      }
      return FDB_OK;
  };

  // per-colour column-list scatter of local colours [l0, l0+G): <= kMaxSegs colours per launch
  // Double-buffered overlap (multi-GPU, column lists): group g's f! outputs live in buffer (g & 1); its scatter — the
  // kernel that also pushes the values to the peers over NVLink — runs on a side stream while the main stream already
  // evaluates group g+1 into the other buffer.  Events order buffer reuse; everything joins the caller's stream at the end.
  const bool overlap = P->double_buffer && P->side != nullptr;
  const double *Fp_g = P->Fp, *Fm_g = P->Fm;
  cudaStream_t ss = s;
  auto scatter_lists = [&](int64_t g, int64_t l0, int64_t G) -> fdb_status {
    const bool wide = P->dest != nullptr;
    // columns without a valid colour (rank 0, with the first group): their entries are 0
    if (g == 0 && P->rank == 0 && P->cm_invalid_end > P->cm_start_h[(size_t)n_local]) {
      const int64_t z0 = P->cm_start_h[(size_t)n_local], z1 = P->cm_invalid_end;
      const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((z1 - z0 + kThreads - 1) / kThreads, (int64_t)P->sm_count * 8));
      if (wide) zero_slots<int64_t><<<grid, kThreads, 0, ss>>>(P->cm_slot, z0, z1, J, P->d_peers, P->n_peers);
      else zero_slots<int32_t><<<grid, kThreads, 0, ss>>>(P->cm_slot, z0, z1, J, P->d_peers, P->n_peers);
      P->cnt.kernel_launches += 1;
    }
    if (G <= 0) return FDB_OK;
    const int64_t total = P->cm_start_h[(size_t)(l0 + G)] - P->cm_start_h[(size_t)l0];
    if (total == 0) return FDB_OK;
    CmArgs a{};
    a.row = P->cm_row; a.slot = P->cm_slot; a.seg_start = P->cm_start; a.local_colors = P->d_local_colors;
    a.fx = vfx; a.Fp = Fp_g; a.Fm = Fm_g; a.eps = P->eps; a.J = J; a.peers = P->d_peers; a.n_peers = P->n_peers;
    a.fx_cm = MODE == kForward ? P->fx_cm : nullptr;
    a.l0 = (int32_t)l0; a.G = (int32_t)G; a.ldF = sF;
    a.m = COMPLEX ? 2 * P->m : P->m;
    // (software L2 prefetch of the next colour's slab: measured SLOWER on C4 — 1.255 vs 0.962 ms — the 40 MB slab, the next
    //  one and f(x) do not fit the L2 together; off unless FDB_CM_PREFETCH=1)
    a.prefetch_next = (G > 1 && P->tune.cm_prefetch) ? 1 : 0;
    a.slab_stream = P->tune.cm_slab_stream;
    const int64_t tiles = (total + kCmTile - 1) / kCmTile;
    ScatterTimer tm(P, ss);
    if (wide) {
      const int grid = resident_grid(P, diff_scatter_cm<MODE, int64_t>, 0, tiles);
      diff_scatter_cm<MODE, int64_t><<<grid, kThreads, 0, ss>>>(a);
    } else {
      const int grid = resident_grid(P, diff_scatter_cm<MODE, int32_t>, 0, tiles);
      diff_scatter_cm<MODE, int32_t><<<grid, kThreads, 0, ss>>>(a);
    }
    P->cnt.kernel_launches += 1;
    P->cnt.scatter_launches += 1;
    return FDB_OK;
  };

  auto scatter_group = [&](int64_t g, int64_t l0, int64_t G) -> fdb_status {
    if (P->sp_kind == SP_CSC && P->strategy == 1) return scatter_lists(g, l0, G);
    if (P->sp_kind == SP_BANDED) {
      BandArgs a{};
      ScatterTimer tm(P, s);   // one timed region per group: the pre-division pass (when used) + the band kernel
      a.jcolor = P->jcolor; a.fx = vfx; a.Fp = P->Fp; a.Fm = P->Fm; a.eps = P->eps; a.local_of = P->local_of;
      a.J = J; a.C = P->C; a.l0 = (int32_t)l0; a.G = (int32_t)G;
      a.write_other = (g == 0 && P->rank == 0) ? 1 : 0;
      a.to_dense = P->jkind == FDB_J_DENSE ? 1 : 0;
      a.ldF = sF; a.ldJ = P->ldJ; a.m = P->m; a.n = P->n; a.l = P->l; a.u = P->u;
      const int64_t w = P->l + P->u + 1;
      int64_t ntiles;
      a.cols_per_tile = std::max<int64_t>(1, 4096 / w);
      ntiles = (P->n + a.cols_per_tile - 1) / a.cols_per_tile;
      // every (colour, row) quotient lands in about (l+u+1)/C columns of the whole-band fill: when that reuse is >= 2,
      // divide once per (colour, row) in place (the reference's own `vfx1 = (vfx1 - vfx)/eps` pass) and let the band
      // kernel copy; otherwise divide at gather time.
      // r1 measurements on C3 (16 GB band, 5 colours; scatter ms per Jacobian): warp-per-column 3.60, flat stream
      // dividing at gather time 4.76, flat stream over pre-divided slabs 3.19, the same with 4-deep batched loads 3.04
      // (kept); row-stationary 3.58, colour-grouped columns 3.46 and block-per-column 4.06 were tried and dropped.
      const bool prediv = !COMPLEX && w >= 64 && P->n > 0 && P->C > 0 && G > 0 && w >= 2 * (int64_t)P->C;
      if (prediv) {
        dim3 grid((unsigned)std::max(1, std::min(P->grid(P->m), std::max(1, P->sm_count * 8 / (int)G))), (unsigned)G);
        diff_slabs<MODE><<<grid, kThreads, 0, s>>>(P->Fp, CENTRAL ? P->Fm : vfx, P->eps, P->d_local_colors + l0, P->m, sF);
        P->cnt.kernel_launches += 1;
      }
      if (w >= 64 && P->n > 0) {
        // wide band: one warp per column
        const size_t sm = P->C <= kSmemTable ? (size_t)P->C * (sizeof(double) + sizeof(int32_t)) : 0;
        if (!a.to_dense && (reinterpret_cast<uintptr_t>(J) & 15) == 0) {
          // band-data target: aligned flat stream, 16-byte stores
          const int32_t CH = (int32_t)std::min<int64_t>(2048, w & ~(int64_t)1);
          const int64_t nchunks = (w * P->n + CH - 1) / CH;
          if (prediv) {
            // unlike the read-modify kernels (C2: no gain), this store-dominated stream gains from an oversubscribed grid:
            // C3 3.03 ms with exactly one resident wave, 2.72 (x4), 2.48 (x16), 2.38 (x64), 2.40 (one chunk per warp);
            // a bare store-only probe shows the same trend (6.0 -> 6.7 TB/s, profiles/write_bw_probe.py)
            constexpr int kBandGridOver = 64;
            int grid = resident_grid(P, diff_scatter_band_flat<CT, kCopy>, sm, (nchunks + 7) / 8);
            grid = (int)std::max<int64_t>(1, std::min<int64_t>((int64_t)grid * kBandGridOver, (nchunks + 7) / 8));
            diff_scatter_band_flat<CT, kCopy><<<grid, kThreads, sm, s>>>(a, CH);
          } else {
            const int grid = resident_grid(P, diff_scatter_band_flat<CT, MODE>, sm, (nchunks + 7) / 8);
            diff_scatter_band_flat<CT, MODE><<<grid, kThreads, sm, s>>>(a, CH);
          }
        } else if (prediv) {
          const int grid = resident_grid(P, diff_scatter_band_wide<CT, kCopy>, sm, (P->n + 7) / 8);
          diff_scatter_band_wide<CT, kCopy><<<grid, kThreads, sm, s>>>(a);
        } else {
          const int grid = resident_grid(P, diff_scatter_band_wide<CT, MODE>, sm, (P->n + 7) / 8);
          diff_scatter_band_wide<CT, MODE><<<grid, kThreads, sm, s>>>(a);
        }
        P->cnt.kernel_launches += 1;
        P->cnt.scatter_launches += 1;
      } else if (ntiles > 0) {
        const int blocks = (int)std::min<int64_t>(ntiles, (int64_t)P->sm_count * 16);
        diff_scatter_band<CT, MODE><<<blocks, kThreads, 0, s>>>(a);
        P->cnt.kernel_launches += 1;
        P->cnt.scatter_launches += 1;
      }
    } else if (P->E > 0) {
      ScatterArgs a{};
      a.row = P->row32; a.ecolor = P->ecolor; a.dest = P->dest; a.fx = vfx; a.Fp = P->Fp; a.Fm = P->Fm; a.eps = P->eps;
      a.local_of = P->local_of; a.J = J; a.peers = P->d_peers; a.n_peers = P->n_peers; a.C = P->C;
      a.l0 = (int32_t)l0; a.G = (int32_t)G;
      a.write_invalid_zero = (g == 0 && P->rank == 0 && P->has_invalid) ? 1 : 0;
      a.ldF = sF; a.E = P->E;
      a.j_aligned = (reinterpret_cast<uintptr_t>(J) & 15) == 0 && P->peers_aligned;
      {
        // random patterns (mean row jump beyond a few cache lines): slab gathers are read-once
        a.hi_stream = P->tune.hi_stream >= 0 ? P->tune.hi_stream : (P->mean_row_jump > 4096.0 ? 1 : 0);
      }
      const size_t sm = P->C <= kSmemTable ? (size_t)P->C * (sizeof(double) + sizeof(int32_t)) : 0;
      ScatterTimer tm(P, s);
      if (ident) {
        const int64_t tiles = (P->E + kTile - 1) / kTile;
        // single group on a single rank: every valid colour is resident -> the FULL variant (no ownership tests)
        const bool full = P->n_groups == 1 && P->world == 1 && P->n_peers == 0;
        // staged form: needs 16-byte aligned sources and (forward) ldF readable doubles behind f(x)
        bool staged = full && P->staged && MODE != kComplex;
        if (staged && MODE == kForward)
          staged = (reinterpret_cast<uintptr_t>(vfx) & 15) == 0 && ((P->m & 1) == 0 || vfx == P->fx_own);
        if (staged) {
          if constexpr (MODE != kComplex) {
            StagedArgs sa{};
            sa.row16 = P->row16; sa.ecolor = P->ecolor; sa.tile_w0 = P->tile_w0; sa.row32 = P->row32;
            sa.fx = vfx; sa.Fp = P->Fp; sa.Fm = P->Fm; sa.eps = P->eps; sa.J = J; sa.C = P->C; sa.W = P->stage_W;
            sa.ldF = sF; sa.src_len = P->ldF; sa.E = P->E; sa.j_aligned = a.j_aligned;
            sa.reverse = P->tune.reverse & 1;
            const int nwin = CENTRAL ? 2 * P->C : P->C + 1;
            int stages = P->tune.stages;
            if ((size_t)stages * nwin * P->stage_W * 8 + 2 * kStagesMax * 8 + (size_t)P->C * 8 > (size_t)kStageMaxSmem) stages = 2;
            sa.stages = stages;
            const size_t ssm = (size_t)stages * nwin * P->stage_W * 8 + 2 * kStagesMax * 8 + (size_t)P->C * 8;
            // variants (profiles/ A/B; FDB_STAGED_VARIANT = 8n | 6p | 6n): resident blocks per SM x index prefetch
            const char v0 = P->tune.staged_variant[0], v1 = P->tune.staged_variant[1];
            auto go = [&](auto kern) {
              const int grid = resident_grid(P, kern, ssm, tiles);
              kern<<<grid, kThreads, ssm, s>>>(sa);
            };
            if (P->stage_packed && v1 == 'e') go(diff_scatter_staged<CT, MODE, 6, false, true, true>);
            else if (P->stage_packed) go(diff_scatter_staged<CT, MODE, 6, false, true>);
            else if (v0 == '8') go(diff_scatter_staged<CT, MODE, 8, false, false>);
            else if (v1 == 'n') go(diff_scatter_staged<CT, MODE, 6, false, false>);
            else go(diff_scatter_staged<CT, MODE, 6, true, false>);
          }
        } else if (full) {
          const int grid = resident_grid(P, diff_scatter_ident<CT, MODE, true, kScatterMinBlocks>, sm, tiles);
          diff_scatter_ident<CT, MODE, true, kScatterMinBlocks><<<grid, kThreads, sm, s>>>(a);
        } else {
          const int grid = resident_grid(P, diff_scatter_ident<CT, MODE, false, kScatterMinBlocks>, sm, tiles);
          diff_scatter_ident<CT, MODE, false, kScatterMinBlocks><<<grid, kThreads, sm, s>>>(a);
        }
      } else {
        const int grid = resident_grid(P, diff_scatter_dest<CT, MODE>, sm, (P->E + kThreads - 1) / kThreads);
        diff_scatter_dest<CT, MODE><<<grid, kThreads, sm, s>>>(a);
      }
      P->cnt.kernel_launches += 1;
      P->cnt.scatter_launches += 1;
    }
    return FDB_OK;
  };

  // colours ascending (jacobians.jl:547).  Points are built in windows of `pbatch` colours, f! is called once per point
  // (reference order f(fx1,x1) then f(fx,x) per colour, :563 / :605-606) or once per `batch` points for batch-capable
  // callbacks; a group's scatter is launched as soon as its `slabs` outputs are complete.
  int64_t li = 0;
  while (li < n_local) {
    const int64_t g = li / P->slabs, g0 = g * P->slabs, gend = std::min<int64_t>(g0 + P->slabs, n_local);
    if (li % P->pbatch == 0) TRY(perturb_window(li, std::min<int64_t>(P->pbatch, n_local - li)));
    const int64_t wend = std::min<int64_t>((li / P->pbatch + 1) * P->pbatch, n_local);
    const int64_t fc = std::min<int64_t>(P->batch, std::min<int64_t>(wend - li, gend - li));
    const int64_t gb = overlap ? (g & 1) * P->slabs * sF : 0;           // this group's output buffer
    if (overlap && li == g0 && g >= 2) CU(cudaStreamWaitEvent(s, P->ev_scat[g & 1], 0));   // buffer free again?
    TRY(call_f(P, f, ctx, P->Fp + gb + (li - g0) * sF, P->xp + (li % P->pbatch) * sX, fc, s));
    if (CENTRAL) TRY(call_f(P, f, ctx, P->Fm + gb + (li - g0) * sF, P->xm + (li % P->pbatch) * sX, fc, s));
    li += fc;
    if (li == gend) {
      Fp_g = P->Fp + gb;
      Fm_g = CENTRAL ? P->Fm + gb : nullptr;
      if (overlap) {
        CU(cudaEventRecord(P->ev_f[g & 1], s));
        CU(cudaStreamWaitEvent(P->side, P->ev_f[g & 1], 0));
        ss = P->side;
        TRY(scatter_group(g, g0, gend - g0));
        CU(cudaEventRecord(P->ev_scat[g & 1], P->side));
        ss = s;
      } else {
        TRY(scatter_group(g, g0, gend - g0));
      }
    }
  }
  if (overlap) {   // join the side stream back into the caller's stream
    const int64_t ng = (n_local + P->slabs - 1) / P->slabs;
    for (int64_t b = 0; b < std::min<int64_t>(ng, 2); ++b) CU(cudaStreamWaitEvent(s, P->ev_scat[b], 0));
  }
  // columns without a valid colour when this rank evaluates no colour at all
  if (n_local == 0 && P->sp_kind == SP_CSC && P->strategy == 1 && (P->n_peers > 0 || P->shared_J)) TRY(scatter_group(0, 0, 0));
  CU(cudaGetLastError());
  return FDB_OK;
}

template <int MODE>
static fdb_status run_dense(fdb_plan *P, fdb_fn f, void *ctx, const double *x, double *J, double *fx, const double *f_in,
                            double relstep, double absstep, double dir, cudaStream_t s) {
  constexpr bool CENTRAL = MODE == kCentral;
  constexpr bool COMPLEX = MODE == kComplex;
  const int64_t sF = COMPLEX ? 2 * P->ldF : P->ldF, sX = COMPLEX ? 2 * P->ldx : P->ldx;
  const int64_t ncl = P->col_end - P->col_begin;
  const double *vfx = nullptr;
  if (MODE == kForward) {
    if (f_in) vfx = f_in;
    else { TRY(call_f(P, f, ctx, fx, x, 1, s)); vfx = fx; }
  }
  if (ncl == 0) return FDB_OK;
  const int32_t B = (int32_t)P->batch;
  if (COMPLEX) {
    // epsilon = eps(eltype(x)) for every column (jacobians.jl:624); X[b] = complex(x)
    fill_value<<<(int)((ncl + kThreads - 1) / kThreads), kThreads, 0, s>>>(P->eps_cols, ncl, DBL_EPSILON);
    replicate_x_complex<<<P->grid(P->n), kThreads, 0, s>>>(x, P->n, sX, B, P->xp);
  } else {
    component_eps<<<(int)((ncl + kThreads - 1) / kThreads), kThreads, 0, s>>>(x, P->col_begin, ncl, CENTRAL ? 1 : 0, relstep,
                                                                            absstep, dir, P->eps_cols);
    replicate_x<<<P->grid(P->n), kThreads, 0, s>>>(x, P->n, P->ldx, B, P->xp);
  }
  P->cnt.kernel_launches += 2;
  int64_t prev_c0 = 0;
  int32_t prevB = 0;
  for (int64_t c0l = 0; c0l < ncl; c0l += B) {
    const int32_t kc = (int32_t)std::min<int64_t>(B, ncl - c0l);
    const int64_t c0 = P->col_begin + c0l;
    const int sb = (std::max(kc, prevB) + kThreads - 1) / kThreads;
    if (COMPLEX) set_components_complex<<<sb, kThreads, 0, s>>>(P->eps_cols, c0l, c0, prev_c0, kc, prevB, sX, P->xp);
    else set_components<<<sb, kThreads, 0, s>>>(x, P->eps_cols, c0l, c0, prev_c0, kc, prevB, P->ldx, 1.0, P->xp);
    TRY(call_f(P, f, ctx, P->Fp, P->xp, kc, s));                         // f(fx1, x1)   jacobians.jl:553 / :594 / :629
    if (CENTRAL) {
      set_components<<<sb, kThreads, 0, s>>>(x, P->eps_cols, c0l, c0, 0, kc, 0, P->ldx, -1.0, P->xp);
      TRY(call_f(P, f, ctx, P->Fm, P->xp, kc, s));                       // f(fx, x1)    :596
      P->cnt.kernel_launches += 1;
    }
    // a store-heavy stream (24 bytes moved per 8 written): many small blocks rather than one resident wave — each thread
    // handles about four row pairs (see the band kernel's grid note)
    const int gx = (int)std::max<int64_t>(1, std::min<int64_t>((P->m / 2 + kThreads * 4 - 1) / (kThreads * 4), P->tune.cols_gx));
    dim3 grid((unsigned)gx, (unsigned)kc);
    {
      const double *lo_ptr = CENTRAL ? P->Fm : vfx;
      const int pairs_ok = ((reinterpret_cast<uintptr_t>(J + c0l * P->ldJ) | reinterpret_cast<uintptr_t>(lo_ptr) |
                             reinterpret_cast<uintptr_t>(P->Fp)) & 15) == 0 && (P->ldJ & 1) == 0 && (sF & 1) == 0;
      ScatterTimer tm(P, s);
      auto go = [&](auto kern) { kern<<<grid, kThreads, 0, s>>>(P->Fp, lo_ptr, P->eps_cols, c0l, kc, P->m, sF, P->ldJ, J + c0l * P->ldJ, pairs_ok); };
      // independent 16-byte loads in flight per thread before the first quotient (same box, C5 shape, us per 256-column
      // launch, depth 1 / 2 / 4: central 112.1 / 95.6 / 94.8, forward 88.1 / 74.3 / 76.2; profiles/r2_ab7.txt)
      const int depth = P->tune.cols_depth ? P->tune.cols_depth : (CENTRAL ? 4 : 2);
      if (depth == 4) go(diff_columns<MODE, 4>);
      else if (depth == 2) go(diff_columns<MODE, 2>);
      else go(diff_columns<MODE, 1>);
    }
    P->cnt.kernel_launches += 2;
    P->cnt.scatter_launches += 1;
    prev_c0 = c0;
    prevB = kc;
  }
  CU(cudaGetLastError());
  return FDB_OK;
}

extern "C" {

static fdb_status jacobian_eager(fdb_plan *P, fdb_fn f, void *ctx, const double *d_x, double *d_J, double *fx,
                                 const double *d_f_in, double relstep, double absstep, double dir, cudaStream_t s) {
  if (P->sp_kind == SP_NONE) {
    if (P->fdtype == FDB_CENTRAL) return run_dense<kCentral>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
    if (P->fdtype == FDB_COMPLEX) return run_dense<kComplex>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
    return run_dense<kForward>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
  }
  return dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
    using CT = decltype(tag);
    if (P->fdtype == FDB_CENTRAL) return run_colored<CT, kCentral>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
    if (P->fdtype == FDB_COMPLEX) return run_colored<CT, kComplex>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
    return run_colored<CT, kForward>(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
  });
}

fdb_status fdb_jacobian(fdb_plan *P, fdb_fn f, void *ctx, const double *d_x, double *d_J, double *d_fx,
                        const double *d_f_in, double relstep, double absstep, double dir, void *stream) {
  if (!P || !f) return fail(FDB_ERR_INVALID, "NULL plan or f");
  if ((P->n > 0 && !d_x) || (P->j_len > 0 && !d_J)) return fail(FDB_ERR_INVALID, "NULL x or J");
  if (P->sp_kind == SP_JVP) return fail(FDB_ERR_INVALID, "this is a JVP plan: call fdb_jvp");
  if (P->sp_kind == SP_HESS) return fail(FDB_ERR_INVALID, "this is a Hessian plan: call fdb_hessian");
  if (P->sp_kind == SP_EPS) return fail(FDB_ERR_INVALID, "this is a step-size plan: call fdb_color_eps");
  if (P->fdtype == FDB_COMPLEX && !P->complex_entry)
    return fail(FDB_ERR_INVALID, "this plan is a complex-step plan: call fdb_jacobian_complex with a complex128 callback");
  DeviceGuard g(P->device);
  if (!g.ok) return fail(FDB_ERR_CUDA, "cannot select device %d", P->device);
  cudaStream_t s = (cudaStream_t)stream;
  // jacobians.jl:508-509 defaults
  resolve_steps(P->fdtype, relstep, absstep);
  double *fx = d_fx ? d_fx : P->fx_own;
  fdb_status st;
  if (P->use_graph && !P->timing) {
    // CUDA-graph replay of the whole call: the launch sequence depends only on the plan and on these arguments
    // (the step sizes are computed on the device inside the graph), so it is captured once and re-launched.
    const GraphKey key{(void *)f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, P->n_peers, P->peer_generation, P->ext_eps};
    if (!P->graph_exec || !(key == P->graph_key)) {
      if (P->graph_exec) { cudaGraphExecDestroy(P->graph_exec); P->graph_exec = nullptr; }
      if (!P->cstream) CU(cudaStreamCreateWithFlags(&P->cstream, cudaStreamNonBlocking));
      const fdb_counters_t before = P->cnt;
      CU(cudaStreamBeginCapture(P->cstream, cudaStreamCaptureModeThreadLocal));
      st = jacobian_eager(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, P->cstream);
      cudaGraph_t graph = nullptr;
      cudaError_t e = cudaStreamEndCapture(P->cstream, &graph);
      if (st != FDB_OK) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); return st; }
      if (e != cudaSuccess || !graph) {
        cudaGetLastError();
        return fail(FDB_ERR_CUDA, "stream capture of the Jacobian failed (%s): the f! callback must be capture-safe "
                                  "(enqueue-only, no allocation) when use_graph is set", cudaGetErrorString(e));
      }
      e = cudaGraphInstantiate(&P->graph_exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { P->graph_exec = nullptr; return fail(FDB_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
      P->graph_key = key;
      // what one replay amounts to (the capture pass itself launched nothing)
      P->graph_delta.f_points = P->cnt.f_points - before.f_points;
      P->graph_delta.f_invocations = P->cnt.f_invocations - before.f_invocations;
      P->graph_delta.kernel_launches = P->cnt.kernel_launches - before.kernel_launches;
      P->graph_delta.scatter_launches = P->cnt.scatter_launches - before.scatter_launches;
      P->cnt = before;
    }
    CU(cudaGraphLaunch(P->graph_exec, s));
    P->cnt.f_points += P->graph_delta.f_points;
    P->cnt.f_invocations += P->graph_delta.f_invocations;
    P->cnt.kernel_launches += P->graph_delta.kernel_launches;
    P->cnt.scatter_launches += P->graph_delta.scatter_launches;
    st = FDB_OK;
  } else {
    st = jacobian_eager(P, f, ctx, d_x, d_J, fx, d_f_in, relstep, absstep, dir, s);
  }
  if (st == FDB_OK) P->cnt.jacobians += 1;
  return st;
}

fdb_status fdb_jacobian_complex(fdb_plan *P, fdb_fn_c f, void *ctx, const double *d_x, double *d_J, void *stream) {
  if (!P || !f) return fail(FDB_ERR_INVALID, "NULL plan or f");
  if (P->fdtype != FDB_COMPLEX) return fail(FDB_ERR_INVALID, "fdb_jacobian_complex needs a plan created with fdtype = FDB_COMPLEX");
  // same C signature up to the element type of the buffers: the complex128 slabs are handed over as raw pointers
  P->complex_entry = true;
  const fdb_status st = fdb_jacobian(P, reinterpret_cast<fdb_fn>(f), ctx, d_x, d_J, nullptr, nullptr, FDB_STEP_DEFAULT, FDB_STEP_DEFAULT, 1.0, stream);
  P->complex_entry = false;
  return st;
}

// ------------------------------------------------------------------------------------------------ step sizes on their own
// (column-block sharded runs: every shard perturbs with the step sizes of the FULL x — jacobians.jl:559-561 takes the
//  norm over all colour-k components)
fdb_status fdb_eps_plan_create(fdb_plan **plan, int64_t n, const int64_t *colorvec, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, 0, n));
  P = *plan;
  DeviceGuard g(P->device);
  P->sp_kind = SP_EPS;
  I64View cv;
  PLAN_TRY(setup_colors(P, colorvec, cv));
  PLAN_TRY(alloc_eps_buffers(P));
  // the same list-based eps pass as the Jacobian plans: a column block's external step sizes are then bit-identical to
  // the ones the unsharded plan computes for itself
  if (P->C > kEpsRegColors && n > 0) {
    unsigned long long *d_bucket = nullptr;
    PLAN_TRY(P->alloc_t(&d_bucket, (size_t)P->C + 2));
    cudaMemset(d_bucket, 0, ((size_t)P->C + 2) * 8);
    PLAN_TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
      using CT = decltype(tag);
      count_color_buckets<CT><<<P->grid(n), kThreads>>>((const CT *)P->jcolor, n, P->C, d_bucket);
      CU(cudaGetLastError());
      return FDB_OK;
    }));
    PLAN_TRY(bucket_offsets(P, d_bucket));
    PLAN_TRY(build_color_lists(P));
  }
  return FDB_OK;
}

fdb_status fdb_color_eps(fdb_plan *P, const double *d_x, double relstep, double absstep, double dir, double *d_eps_out,
                         void *stream) {
  if (!P) return fail(FDB_ERR_INVALID, "NULL plan");
  if (P->sp_kind == SP_NONE || P->sp_kind == SP_JVP || P->sp_kind == SP_HESS)
    return fail(FDB_ERR_INVALID, "fdb_color_eps needs a coloured plan");
  if (P->n > 0 && !d_x) return fail(FDB_ERR_INVALID, "NULL x");
  DeviceGuard g(P->device);
  if (!g.ok) return fail(FDB_ERR_CUDA, "cannot select device %d", P->device);
  cudaStream_t s = (cudaStream_t)stream;
  resolve_steps(P->fdtype, relstep, absstep);
  TRY(dispatch_ct(P->color_bits, [&](auto tag) -> fdb_status {
    using CT = decltype(tag);
    return run_eps<CT>(P, d_x, relstep, absstep, dir, s);
  }));
  if (d_eps_out && P->C > 0) CU(cudaMemcpyAsync(d_eps_out, P->eps, (size_t)P->C * 8, cudaMemcpyDeviceToDevice, s));
  return FDB_OK;
}

fdb_status fdb_plan_set_external_eps(fdb_plan *P, const double *d_eps) {
  if (!P) return fail(FDB_ERR_INVALID, "NULL plan");
  if (P->sp_kind == SP_NONE || P->sp_kind == SP_JVP || P->sp_kind == SP_EPS || P->sp_kind == SP_HESS)
    return fail(FDB_ERR_INVALID, "external step sizes apply to coloured Jacobian plans");
  P->ext_eps = d_eps;
  return FDB_OK;
}

// ------------------------------------------------------------------------------------------------ JVP (src/jvp.jl:238-274)
fdb_status fdb_jvp_plan_create(fdb_plan **plan, int64_t m, int64_t n, const fdb_plan_opts *opts) {
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, opts, m, n));
  P = *plan;
  DeviceGuard g(P->device);
  if (P->fdtype == FDB_COMPLEX) {
    free_plan(P); *plan = nullptr;
    return fail(FDB_ERR_UNSUPPORTED, "finite_difference_jvp doesn't support :complex-mode finite diff");   // jvp.jl:248-250
  }
  P->sp_kind = SP_JVP;
  P->C = 1;
  P->ldF = std::max<int64_t>(2, (m + 1) & ~(int64_t)1);
  P->ldx = std::max<int64_t>(2, (n + 1) & ~(int64_t)1);
  int64_t nb = std::max<int64_t>(1, std::min<int64_t>((n + kTile - 1) / kTile, (int64_t)P->sm_count * 8));
  P->eps_blocks = (int)nb;
  PLAN_TRY(P->alloc_t(&P->partial, (size_t)nb));
  PLAN_TRY(P->alloc_t(&P->ticket, 4));
  cudaMemset(P->ticket, 0, 16);
  PLAN_TRY(P->alloc_t(&P->eps, 2));
  PLAN_TRY(P->alloc_t(&P->sumsq, 2));
  PLAN_TRY(P->alloc_t(&P->fx_own, (size_t)P->ldF));
  PLAN_TRY(P->alloc_t(&P->xp, (size_t)P->ldx));
  P->alg_bytes = 24 * n + 24 * m;   // dot: 16n; point: 16n read + 8n write; quotient: 16m read + 8m write
  return FDB_OK;
}

fdb_status fdb_jvp(fdb_plan *P, fdb_fn f, void *ctx, double *d_jvp, const double *d_x, const double *d_v, double *d_x1,
                   double *d_fx1, const double *d_f_in, double relstep, double absstep, double dir, void *stream) {
  if (!P || !f) return fail(FDB_ERR_INVALID, "NULL plan or f");
  if (P->sp_kind != SP_JVP) return fail(FDB_ERR_INVALID, "not a JVP plan (fdb_jvp_plan_create)");
  if ((P->n > 0 && (!d_x || !d_v)) || (P->m > 0 && !d_jvp)) return fail(FDB_ERR_INVALID, "NULL jvp, x or v");
  DeviceGuard g(P->device);
  if (!g.ok) return fail(FDB_ERR_CUDA, "cannot select device %d", P->device);
  cudaStream_t s = (cudaStream_t)stream;
  resolve_steps(P->fdtype, relstep, absstep);                       // jvp.jl:245-246
  double *x1 = d_x1 ? d_x1 : P->xp;
  double *fx1 = d_fx1 ? d_fx1 : P->fx_own;
  const bool central = P->fdtype == FDB_CENTRAL;
  const int64_t n = P->n, m = P->m;
  const int al_xv = ((reinterpret_cast<uintptr_t>(d_x) | reinterpret_cast<uintptr_t>(d_v)) & 15) == 0;
  const int al_x1 = al_xv && (reinterpret_cast<uintptr_t>(x1) & 15) == 0;
  EpsParams prm{central ? 1 : 0, relstep, absstep, dir};
  const int64_t tiles = (n + kTile - 1) / kTile;
  const int grid_n = std::min(resident_grid(P, jvp_dot_eps, 0, tiles), P->eps_blocks);
  jvp_dot_eps<<<grid_n, kThreads, 0, s>>>(d_x, d_v, n, al_xv, prm, P->partial, P->ticket, P->eps, P->sumsq);   // :252-253
  P->cnt.kernel_launches += 1;
  const double *base = fx1;
  if (!central) {
    if (d_f_in) base = d_f_in;                                      // fx1 = f_in        :257-258
    else TRY(call_f(P, f, ctx, fx1, d_x, 1, s));                    // f(fx1, x)         :255
  } else {
    jvp_point<<<resident_grid(P, jvp_point, 0, tiles), kThreads, 0, s>>>(d_x, d_v, P->eps, 1, x1, n, al_x1);   // x1 = x - eps v :264
    P->cnt.kernel_launches += 1;
    TRY(call_f(P, f, ctx, fx1, x1, 1, s));                          // f(fx1, x1)        :265
  }
  jvp_point<<<resident_grid(P, jvp_point, 0, tiles), kThreads, 0, s>>>(d_x, d_v, P->eps, 0, x1, n, al_x1);     // x1 = x + eps v :260/:266
  TRY(call_f(P, f, ctx, d_jvp, x1, 1, s));                          // f(jvp, x1)        :261/:267
  jvp_quotient<<<P->grid(m), kThreads, 0, s>>>(d_jvp, base, P->eps, central ? 1 : 0, m);                        // :262/:268
  P->cnt.kernel_launches += 2;
  CU(cudaGetLastError());
  P->cnt.jacobians += 1;
  return FDB_OK;
}

// ------------------------------------------------------------------------------------------------ Hessian (src/hessians.jl:202-292)
fdb_status fdb_hessian_plan_create(fdb_plan **plan, int64_t n, const fdb_plan_opts *opts) {
  if (!plan) return fail(FDB_ERR_INVALID, "plan output pointer is NULL");
  *plan = nullptr;
  if (!opts || opts->fdtype != FDB_HCENTRAL)   // @assert fdtype == Val(:hcentral)   hessians.jl:206
    return fail(FDB_ERR_UNSUPPORTED, "finite_difference_hessian supports only the hcentral fdtype (%d)", FDB_HCENTRAL);
  if (opts->world > 1) return fail(FDB_ERR_UNSUPPORTED, "Hessian plans run on one GPU (world > 1 given)");
  if (opts->use_graph) return fail(FDB_ERR_UNSUPPORTED, "Hessian plans do not capture CUDA graphs (use_graph = 1 given)");
  if (n > ((int64_t)1 << 26))
    return fail(FDB_ERR_NOMEM, "n = %lld: the 2n^2+1 point values would not fit in device memory", (long long)n);
  // the Jacobian plans' common set-up validates forward / central / complex; the Hessian's own type is set afterwards
  fdb_plan_opts o = *opts;
  o.fdtype = FDB_CENTRAL;
  fdb_plan *P = nullptr;
  TRY(new_plan(plan, &o, 1, n));
  P = *plan;
  DeviceGuard g(P->device);
  P->fdtype = FDB_HCENTRAL;
  P->sp_kind = SP_HESS;
  P->jkind = FDB_J_DENSE;
  P->C = (int32_t)n;
  P->ldF = 1;
  P->ldx = std::max<int64_t>(2, (n + 1) & ~(int64_t)1);
  P->hess_points = 2 * n * n + 1;
  int64_t batch = opts->max_batch > 1 ? opts->max_batch : 1;
  const int64_t budget = opts->scratch_bytes > 0 ? opts->scratch_bytes : (int64_t)8 << 30;
  batch = std::max<int64_t>(1, std::min<int64_t>(batch, budget / (8 * P->ldx)));
  batch = std::min<int64_t>(batch, P->hess_points);
  P->batch = batch;
  P->slabs = batch;
  P->n_groups = (P->hess_points + batch - 1) / batch;
  P->j_len = n * n;
  P->E = n * n;
  PLAN_TRY(P->alloc_t(&P->hess_F, (size_t)P->hess_points + 1));
  PLAN_TRY(P->alloc_t(&P->xp, (size_t)batch * P->ldx));
  PLAN_TRY(P->alloc_t(&P->eps, (size_t)std::max<int64_t>(n, 1)));
  // combine pass: F read once, the n steps, H written once
  P->alg_bytes = 8 * P->hess_points + 8 * n + 8 * n * n;
  return FDB_OK;
}

fdb_status fdb_hessian(fdb_plan *P, fdb_fn f, void *ctx, const double *d_x, double *d_H, int64_t ldH, double relstep,
                       double absstep, void *stream) {
  if (!P || !f) return fail(FDB_ERR_INVALID, "NULL plan or f");
  if (P->sp_kind != SP_HESS) return fail(FDB_ERR_INVALID, "not a Hessian plan (fdb_hessian_plan_create)");
  const int64_t n = P->n;
  if (n > 0 && (!d_x || !d_H)) return fail(FDB_ERR_INVALID, "NULL x or H");
  if (ldH < n) return fail(FDB_ERR_INVALID, "ldH = %lld < n = %lld", (long long)ldH, (long long)n);
  DeviceGuard g(P->device);
  if (!g.ok) return fail(FDB_ERR_CUDA, "cannot select device %d", P->device);
  cudaStream_t s = (cudaStream_t)stream;
  resolve_steps(FDB_HCENTRAL, relstep, absstep);                    // hessians.jl:204-205
  double *F = P->hess_F + 1;                                        // F + 1 is 16-byte aligned (hess_combine)
  if (n == 0) {                                                     // fx = f(x); the loops are empty     :209
    TRY(call_f(P, f, ctx, F, P->xp, 1, s));
    P->cnt.jacobians += 1;
    return FDB_OK;
  }
  // e_k = compute_epsilon(Val(:hcentral) / Val(:central), x_k, relstep, absstep): one formula    :223, :234, :252
  component_eps<<<(int)((n + kThreads - 1) / kThreads), kThreads, 0, s>>>(d_x, 0, n, 1, relstep, absstep, 1.0, P->eps);
  hess_replicate<<<P->grid(n * P->batch), kThreads, 0, s>>>(d_x, n, P->ldx, P->batch, P->xp);
  P->cnt.kernel_launches += 2;
  const int64_t total = P->hess_points, B = P->batch;
  int64_t prev_p0 = 0, prevB = 0;
  for (int64_t p0 = 0; p0 < total; p0 += B) {
    const int64_t kc = std::min<int64_t>(B, total - p0);
    const int64_t slots = std::max(kc, prevB);
    hess_points<<<(unsigned)((slots + kThreads - 1) / kThreads), kThreads, 0, s>>>(d_x, P->eps, n, p0, kc, prev_p0, prevB,
                                                                                P->ldx, P->xp);
    P->cnt.kernel_launches += 1;
    TRY(call_f(P, f, ctx, F + p0, P->xp, kc, s));                  // f(x), f(_xpp), f(_xmm), f(_xpm), ...
    prev_p0 = p0;
    prevB = kc;
  }
  {
    const int64_t nt = (n + kHessTile - 1) / kHessTile;
    ScatterTimer tm(P, s);
    hess_combine<<<dim3((unsigned)nt, (unsigned)nt), kThreads, 0, s>>>(F, P->eps, n, d_H, ldH);   // :233, :269, :291
  }
  P->cnt.kernel_launches += 1;
  P->cnt.scatter_launches += 1;
  CU(cudaGetLastError());
  P->cnt.jacobians += 1;
  return FDB_OK;
}

fdb_status fdb_jacobian_host(fdb_plan *P, fdb_fn f, void *ctx, const double *h_x, double *h_J, double *h_fx,
                             const double *h_f_in, double relstep, double absstep, double dir) {
  if (!P || !f) return fail(FDB_ERR_INVALID, "NULL plan or f");
  if ((P->n > 0 && !h_x) || (P->j_len > 0 && !h_J)) return fail(FDB_ERR_INVALID, "NULL x or J");
  if (P->sp_kind == SP_HESS) return fail(FDB_ERR_INVALID, "this is a Hessian plan: call fdb_hessian");
  DeviceGuard g(P->device);
  if (!g.ok) return fail(FDB_ERR_CUDA, "cannot select device %d", P->device);
  if (!P->hstream) {
    CU(cudaStreamCreateWithFlags(&P->hstream, cudaStreamNonBlocking));
    TRY(P->alloc_t(&P->h_dx, (size_t)std::max<int64_t>(P->n, 1)));
    TRY(P->alloc_t(&P->h_dJ, (size_t)std::max<int64_t>(P->j_len, 1)));
    TRY(P->alloc_t(&P->h_dfx, (size_t)P->ldF));
    TRY(P->alloc_t(&P->h_dfin, (size_t)P->ldF));
  }
  cudaStream_t s = P->hstream;
  if (P->n > 0) CU(cudaMemcpyAsync(P->h_dx, h_x, (size_t)P->n * 8, cudaMemcpyHostToDevice, s));
  const double *fin = nullptr;
  if (h_f_in && P->fdtype == FDB_FORWARD) {
    CU(cudaMemcpyAsync(P->h_dfin, h_f_in, (size_t)P->m * 8, cudaMemcpyHostToDevice, s));
    fin = P->h_dfin;
  }
  fdb_status st = fdb_jacobian(P, f, ctx, P->h_dx, P->h_dJ, P->h_dfx, fin, relstep, absstep, dir, (void *)s);
  if (st != FDB_OK) { cudaStreamSynchronize(s); return st; }
  if (P->j_len > 0) {
    if (P->jkind == FDB_J_DENSE && P->ldJ > P->m) {
      // strided dense view: only rows [0, m) of each column are J's (the host padding rows stay untouched)
      const int64_t ncols = P->sp_kind == SP_NONE ? P->col_end - P->col_begin : P->n;
      if (P->m > 0 && ncols > 0)
        CU(cudaMemcpy2DAsync(h_J, (size_t)P->ldJ * 8, P->h_dJ, (size_t)P->ldJ * 8, (size_t)P->m * 8, (size_t)ncols,
                             cudaMemcpyDeviceToHost, s));
    } else {
      CU(cudaMemcpyAsync(h_J, P->h_dJ, (size_t)P->j_len * 8, cudaMemcpyDeviceToHost, s));
    }
  }
  if (h_fx && P->fdtype == FDB_FORWARD && !fin && P->m > 0)
    CU(cudaMemcpyAsync(h_fx, P->h_dfx, (size_t)P->m * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  return FDB_OK;
}

// ------------------------------------------------------------------------------------------------ helpers
fdb_status fdb_host_alloc(void **p, size_t bytes) {
  if (!p) return fail(FDB_ERR_INVALID, "NULL argument");
  CU(cudaHostAlloc(p, bytes ? bytes : 16, cudaHostAllocDefault));
  return FDB_OK;
}
fdb_status fdb_host_free(void *p) { if (p) CU(cudaFreeHost(p)); return FDB_OK; }
fdb_status fdb_device_alloc(void **p, size_t bytes) {
  if (!p) return fail(FDB_ERR_INVALID, "NULL argument");
  CU(cudaMalloc(p, bytes ? bytes : 16));
  return FDB_OK;
}
fdb_status fdb_device_free(void *p) { if (p) CU(cudaFree(p)); return FDB_OK; }
fdb_status fdb_memcpy_h2d(void *d, const void *h, size_t bytes, void *stream) {
  CU(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return FDB_OK;
}
fdb_status fdb_memcpy_d2h(void *h, const void *d, size_t bytes, void *stream) {
  CU(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return FDB_OK;
}
fdb_status fdb_stream_sync(void *stream) { CU(cudaStreamSynchronize((cudaStream_t)stream)); return FDB_OK; }

fdb_status fdb_ipc_get_handle(void *d_ptr, unsigned char handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, d_ptr));
  memcpy(handle, &h, 64);
  return FDB_OK;
}
fdb_status fdb_ipc_open(const unsigned char handle[64], void **d_ptr) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CU(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return FDB_OK;
}
fdb_status fdb_ipc_close(void *d_ptr) { CU(cudaIpcCloseMemHandle(d_ptr)); return FDB_OK; }

}  // extern "C"

#include "fdjac_group.cuh"
