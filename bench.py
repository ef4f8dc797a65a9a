#!/usr/bin/env python
"""bench.py — the coloured sparse-Jacobian hot path on B200, measured per the driver contract.

A "step" = ONE full finite_difference_jacobian! call (eps pass, f!(x), per-colour perturb + f!, fused diff+scatter)
over one synthetic problem.  Workloads (BASELINE.json configs; SURVEY.md §8d):
    c2  N=10^7 tridiagonal f!, 3 colours, CSC J, forward — THE headline at --gpus 1 (`--fdtype central` for the central leg)
    c4  N=5*10^6 random sparse f! (8 nnz/row), 64 colours, CSC J — colours sharded over the ranks (default at --gpus>1,
        strong scaling: the problem is fixed; each rank's scatter kernel stores its entries straight into rank 0's
        nzval over NVLink; ranks ordered by the C ABI's device-side barrier — no NCCL call per Jacobian)
    c3 (banded 16 GB), c5 (dense 80 GB), c1: selectable; at --gpus 1 the default run also measures c2 central, c3, c4 and
    c5 and reports them under "workloads" of the ONE JSON line (`--no-extras` skips them).

JSON line: metric/value = whole-job Jacobian nnz/s with inputs resident in HBM; e2e = the same metric through host
buffers (N=1: fdb_jacobian_host, H2D of x + D2H of nzval inside the timed region; N>1: pinned x -> every rank, nzval ->
host from rank 0); roofline = the diff+scatter kernel: COMPULSORY bytes of the shipped formulation
(fdb_plan_info.moved_bytes_scatter) / CUDA-event launch time vs MEASURED_PEAKS.json hbm_gbs, SURVEY §8(d)'s
reference-shaped byte count beside it; parity = in-run correctness records (bit-compare with the oracle inside the
cpu_baseline leg, analytic sampled checks at full size, sharded-vs-unsharded bit-compare at N>1); cpu_baseline = the CPU
oracle (port of the reference; no Julia in this image) timed on the host cores in the same run.

`--impl reference` times the reference's own CPU algorithm (the oracle port, all host threads) on the same workload,
same instance (the C4 instance comes from one counter-based generator implemented for numpy and torch).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

SEED = 0x5EED
C4_N, C4_K, C4_C = 5_000_000, 8, 64


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------ workloads
def tridiag_pattern_torch(n, device):
    """colptr/rowval (Int64, 1-based) of the n x n tridiagonal CSC pattern, built on `device`."""
    import torch
    c = torch.arange(n + 1, dtype=torch.int64, device=device)
    colptr = 3 * c
    colptr[0] = 1
    colptr[n] = 3 * n - 1
    p = torch.arange(3 * n - 2, dtype=torch.int64, device=device)
    # slot p belongs to column col = (p+1)//3, offset k = (p+1)%3 ; row (1-based) = col + k
    q = p + 1
    rowval = q // 3 + q % 3
    return colptr, rowval


def tridiag_pattern_numpy(n):
    c = np.arange(n + 1, dtype=np.int64)
    colptr = 3 * c
    colptr[0] = 1
    colptr[n] = 3 * n - 1
    q = np.arange(1, 3 * n - 1, dtype=np.int64)
    return colptr, q // 3 + q % 3


# ---- C4 instance: ONE counter-based generator (splitmix64 of (row, slot, stream)), written for numpy (CPU arm) and
# torch (GPU arm, on the device) so both arms differentiate the SAME problem.  Row i takes K distinct colours
# (base + j*odd_stride mod 64) and one column of each; ELL layout [K][n]; CSC = transpose with sorted rows.
_SM_A, _SM_B, _SM_C = 0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9, 0x94D049BB133111EB


def _signed(v):
    return v - (1 << 64) if v >= (1 << 63) else v


def _splitmix_np(key):
    z = key + np.uint64(_SM_A)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(_SM_B)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(_SM_C)
    return z ^ (z >> np.uint64(31))


def _splitmix_torch(key):
    def lsr(v, s):
        return (v >> s) & ((1 << (64 - s)) - 1)
    z = key + _signed(_SM_A)
    z = (z ^ lsr(z, 30)) * _signed(_SM_B)
    z = (z ^ lsr(z, 27)) * _signed(_SM_C)
    return z ^ lsr(z, 31)


def c4_instance_numpy(n=C4_N, K=C4_K, Cc=C4_C, seed=11):
    """(cols[K][n] int32, coef[K][n] f64)"""
    with np.errstate(over="ignore"):
        i = np.arange(n, dtype=np.uint64)
        s = np.uint64(seed)
        base = _splitmix_np(i * np.uint64(16) + (np.uint64(1) << np.uint64(40)) + s) & np.uint64(Cc - 1)
        stride = ((_splitmix_np(i * np.uint64(16) + (np.uint64(2) << np.uint64(40)) + s) & np.uint64(Cc // 2 - 1)) << np.uint64(1)) | np.uint64(1)
        cols = np.empty((K, n), np.int32)
        coef = np.empty((K, n), np.float64)
        per = np.uint64(n // Cc)
        for j in range(K):
            color = (base + np.uint64(j) * stride) & np.uint64(Cc - 1)
            hw = _splitmix_np(i * np.uint64(16) + np.uint64(j) + (np.uint64(3) << np.uint64(40)) + s)
            which = (hw >> np.uint64(1)) % per
            cols[j] = (which * np.uint64(Cc) + color).astype(np.int32)
            hc = _splitmix_np(i * np.uint64(16) + np.uint64(j) + (np.uint64(4) << np.uint64(40)) + s)
            coef[j] = (hc >> np.uint64(11)).astype(np.float64) * (2.0 ** -52) - 1.0
    return cols, coef


def c4_instance_torch(device, n=C4_N, K=C4_K, Cc=C4_C, seed=11):
    import torch
    i = torch.arange(n, dtype=torch.int64, device=device)
    base = _splitmix_torch(i * 16 + (1 << 40) + seed) & (Cc - 1)
    stride = ((_splitmix_torch(i * 16 + (2 << 40) + seed) & (Cc // 2 - 1)) << 1) | 1
    cols = torch.empty((K, n), dtype=torch.int32, device=device)
    coef = torch.empty((K, n), dtype=torch.float64, device=device)
    per = n // Cc
    for j in range(K):
        color = (base + j * stride) & (Cc - 1)
        hw = _splitmix_torch(i * 16 + j + (3 << 40) + seed)
        which = ((hw >> 1) & ((1 << 63) - 1)) % per
        cols[j] = (which * Cc + color).to(torch.int32)
        hc = _splitmix_torch(i * 16 + j + (4 << 40) + seed)
        coef[j] = ((hc >> 11) & ((1 << 53) - 1)).to(torch.float64) * (2.0 ** -52) - 1.0
    return cols, coef


def ell_csc_numpy(n, K, cols):
    """CSC (1-based Int64 colptr / rowval, rows sorted) of the transpose of the ELL row structure cols[K][n]"""
    import scipy.sparse as sps
    rows = np.tile(np.arange(n, dtype=np.int32), K)
    A = sps.csc_matrix((np.ones(n * K, np.int8), (rows, cols.reshape(-1))), shape=(n, n))
    A.sort_indices()
    assert A.nnz == n * K
    return A.indptr.astype(np.int64) + 1, A.indices.astype(np.int64) + 1


class Clocks:
    """Samples nvidia-smi clocks / throttle reasons during the measurement phase (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(", ") for r in Path(self.f.name).read_text().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower() == "active":
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------ CPU arm
def usable_cores() -> int:
    """Host threads this process can really use: scheduler affinity capped by the cgroup CPU quota (the GPU boxes report
    128 CPUs but run the container under a 16-CPU quota: 128 OpenMP threads there are ~300x SLOWER than 16)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        try:
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            p = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return max(1, n)


def cpu_jacobian_runner(workload, fdtype, nthreads, scale=1.0):
    """Returns (run(eps_override=None) -> (fcalls, nzval), nnz, n_fcalls, description) for the oracle on `workload`
    (scale < 1 shrinks n: a bounded sample)."""
    from oracle import fd_oracle as orc
    fd = 0 if fdtype == "forward" else 1
    if workload in ("c1", "c2"):
        n = 1000 if workload == "c1" else int(10_000_000 * scale)
        colptr, rowval = tridiag_pattern_numpy(n)
        cv = (np.arange(n, dtype=np.int64) % 3) + 1
        P = orc.Problem.csc_same(n, n, colptr, rowval)
        x = orc.fill_x(n, SEED + 2, nthreads)
        nz = np.zeros(len(rowval))
        ctx = orc.SynthTridiagCtx(n, nthreads)
        cache = dict(x1=np.zeros(n), x2=np.zeros(n), fx=np.zeros(n), fx1=np.zeros(n))
        fn = orc.native_fn("synth_tridiag")
        if fdtype == "complex":
            fnc = orc.native_fn("synth_tridiag_c")

            def run_c(eps_override=None):
                return orc.jacobian_complex(P, nz, fnc, x, colorvec=cv, nthreads=nthreads, ctx=ctx)["fcalls"], nz
            return run_c, len(rowval), 3, f"N={n} tridiagonal, 3 colours, complex step"

        def run(eps_override=None):
            return orc.jacobian(P, nz, fn, x, fdtype=fd, colorvec=cv, nthreads=nthreads, ctx=ctx, cache=cache,
                                eps_override=eps_override)["fcalls"], nz
        run.x, run.cv, run.fd = x, cv, fd
        return run, len(rowval), (4 if fd == 0 else 6), f"N={n} tridiagonal, 3 colours, {fdtype}"
    if workload == "c4":
        n = int(C4_N * scale) // C4_C * C4_C
        cols, coef = c4_instance_numpy(n)
        colptr, rowval = ell_csc_numpy(n, C4_K, cols)
        cv = (np.arange(n, dtype=np.int64) % C4_C) + 1
        P = orc.Problem.csc_same(n, n, colptr, rowval)
        x = orc.fill_x(n, SEED + 4, nthreads)
        nz = np.zeros(len(rowval))
        ctx = orc.SynthEllCtx(n, C4_K, cols.ctypes.data_as(C.POINTER(C.c_int32)), coef.ctypes.data_as(C.POINTER(C.c_double)), nthreads)
        cache = dict(x1=np.zeros(n), x2=np.zeros(n), fx=np.zeros(n), fx1=np.zeros(n))
        fn = orc.native_fn("synth_ellrows")
        keep = (cols, coef)

        def run(eps_override=None, _keep=keep):
            return orc.jacobian(P, nz, fn, x, fdtype=fd, colorvec=cv, nthreads=nthreads, ctx=ctx, cache=cache,
                                eps_override=eps_override)["fcalls"], nz
        return run, len(rowval), (65 if fd == 0 else 128), f"N={n} random sparse 8 nnz/row, 64 colours, {fdtype}"
    raise SystemExit(f"no CPU runner for workload {workload}")


def time_cpu(run, budget_s=12.0, max_reps=5):
    t0 = time.perf_counter()
    run()
    first = time.perf_counter() - t0
    ts = [first]
    while len(ts) < max_reps and sum(ts) + first < budget_s:
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), len(ts)


L2_NOTE = ("inputs larger than L2 (no flush needed): x, the stacked f! outputs and J's value storage total far more than "
           "126 MB per step")


def workload_config(w, fdtype):
    """`config` of the JSON line — identical in both arms (ours / --impl reference) for the same workload."""
    name = {
        "c1": f"C1: N=1000 tridiagonal f!, 3 colours, CSC J, {fdtype}",
        "c2": f"C2: N=10^7 tridiagonal f!, colorvec=((j-1) mod 3)+1, SparseMatrixCSC J, {fdtype} fdtype, 1xB200",
        "c3": f"C3: N=10^6 2-D 5-point stencil, 5 colours, BandedMatrix l=u=1000, {fdtype}",
        "c4": f"C4: N=5*10^6 random sparse f! (8 nnz/row), 64-colour colorvec, CSC J, {fdtype}, colours sharded across ranks",
        "c5": f"C5: N=10^5 dense Jacobian (no colorvec), {fdtype}, columns partitioned across ranks",
    }[w]
    return {"workload": name, "l2": L2_NOTE if w != "c1" else "C1 is L2-resident (latency config)"}


def reference_arm(args):
    """`--impl reference`: the reference's own CPU algorithm (oracle port; the reference is Julia and cannot run here)
    with all host threads, on the same workload / instance / metric.  Each step = one Jacobian."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import fd_oracle as orc
    cores = usable_cores()
    scale = args.cpu_scale
    run, nnz, fcalls, desc = cpu_jacobian_runner(args.workload, args.fdtype, cores, scale)
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = time.perf_counter() - t0
    value = nnz * args.steps / dt
    # the reference itself is single-threaded Julia: also report the port run the way the reference actually runs
    run1, nnz1, _, desc1 = cpu_jacobian_runner(args.workload, args.fdtype, 1, min(scale, 0.2) if args.workload == "c4" else scale)
    med1, reps1 = time_cpu(run1, budget_s=6.0, max_reps=3)
    line = {
        "impl": "reference", "metric": "jacobian_nnz_per_s", "value": value, "unit": "nnz/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, args.fdtype),
        "f_evals_per_s": fcalls * args.steps / dt,
        "cpu_baseline": {"value": value, "unit": "nnz/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full Jacobian(s) of {desc}" + ("" if scale == 1.0 else f" (problem scaled by {scale})")
                                   + f"; OpenMP over the reference's full-length passes ({cores} threads; the reference itself is single-threaded)"},
        "e2e": {"value": value, "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "single_thread": {"value": nnz1 / med1, "unit": "nnz/s", "cores": 1, "reps": reps1, "sample": desc1,
                          "note": "the reference's own execution model (serial broadcast loops)"},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def build_gpu_problem(pkg, workload, fdtype, dev, rank, world, max_batch, use_graph=True, strategy=0):
    """Returns dict(J, f, x, cache, nnz, n, ctx, keep)."""
    import torch
    L = pkg._lib
    synth = L.synth()

    def native(name, ctx, mb=1):
        return pkg.NativeFn(C.cast(getattr(synth, name), C.c_void_p).value, ctx, max_batch=mb)

    if workload in ("c1", "c2"):
        n = 1000 if workload == "c1" else 10_000_000
        colptr, rowval = tridiag_pattern_torch(n, dev)
        cv = (torch.arange(n, dtype=torch.int64, device=dev) % 3) + 1
        x = torch.empty(n, dtype=torch.float64, device=dev)
        synth.fdbs_fill_x(x.data_ptr(), n, SEED + 2, None)
        J = pkg.SparseMatrixCSC(n, n, colptr, rowval, torch.full((3 * n - 2,), float("nan"), dtype=torch.float64, device=dev))
        ctx = L.TridiagCtx(n, 0)
        f = native("fdbs_tridiag_c" if fdtype == "complex" else "fdbs_tridiag", ctx, max_batch)
        cache = pkg.JacobianCache(x, fdtype, colorvec=cv, sparsity=J, max_batch=max_batch, rank=rank, world=world,
                                  use_graph=use_graph, strategy=strategy)
        return dict(J=J, f=f, x=x, cache=cache, nnz=3 * n - 2, n=n, ctx=ctx, keep=(colptr, rowval, cv))
    if workload == "c4":
        n, K, Cc = C4_N, C4_K, C4_C
        d_cols, d_coef = c4_instance_torch(dev, n, K, Cc)         # same instance on every rank and in the CPU arm
        cols64 = d_cols.to(torch.int64)
        rows = torch.arange(n, device=dev, dtype=torch.int64).repeat(K)
        order = torch.argsort(cols64.reshape(-1) * n + rows)
        rowval = (rows[order] + 1).contiguous()
        colptr = torch.cat([torch.ones(1, dtype=torch.int64, device=dev),
                            1 + torch.cumsum(torch.bincount(cols64.reshape(-1), minlength=n), 0)])
        del cols64, rows, order
        cv = (torch.arange(n, dtype=torch.int64, device=dev) % Cc) + 1
        x = torch.empty(n, dtype=torch.float64, device=dev)
        synth.fdbs_fill_x(x.data_ptr(), n, SEED + 4, None)
        J = pkg.SparseMatrixCSC(n, n, colptr, rowval,
                                torch.full((n * K,), float("nan"), dtype=torch.float64, device=dev))
        ctx = L.EllCtx(n, K, d_cols.data_ptr(), d_coef.data_ptr(), 0)
        f = native("fdbs_ellrows", ctx, max_batch)
        cache = pkg.JacobianCache(x, fdtype, colorvec=cv, sparsity=J, max_batch=max_batch, rank=rank, world=world,
                                  partition=0, use_graph=use_graph, strategy=strategy)
        return dict(J=J, f=f, x=x, cache=cache, nnz=n * K, n=n, ctx=ctx, keep=(d_cols, d_coef, cv))
    if workload == "c3":
        g = 1000
        n = g * g
        idx = torch.arange(n, dtype=torch.int64, device=dev)
        cv = ((idx % g) + 2 * (idx // g)) % 5 + 1
        x = torch.empty(n, dtype=torch.float64, device=dev)
        synth.fdbs_fill_x(x.data_ptr(), n, SEED + 3, None)
        J = pkg.BandedMatrix(n, n, g, g, device=dev)
        ctx = L.Lap5Ctx(g, 0)
        f = native("fdbs_lap5", ctx, max_batch)
        cache = pkg.JacobianCache(x, fdtype, colorvec=cv, sparsity=J, max_batch=max_batch, use_graph=use_graph)
        return dict(J=J, f=f, x=x, cache=cache, nnz=None, n=n, ctx=ctx, keep=(cv,), g=g)
    if workload == "c5":
        n = 100_000
        mb = max(max_batch, 256)
        w = torch.rand(n, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
        nblk = (n + 1023) // 1024
        bs = torch.zeros(nblk * mb, dtype=torch.float64, device=dev)
        ctx = L.Rank1Ctx(n, w.data_ptr(), bs.data_ptr(), mb, 0)
        x = torch.empty(n, dtype=torch.float64, device=dev)
        synth.fdbs_fill_x(x.data_ptr(), n, SEED + 5, None)
        f = native("fdbs_rank1", ctx, mb)
        if world > 1:
            # column blocks per rank (north_star config 5): this rank's J is its own (m x ncols_local) slab
            cache = pkg.JacobianCache(x, fdtype, max_batch=mb, use_graph=use_graph, rank=rank, world=world)
            per = (n + world - 1) // world
            col0 = min(n, per * rank)
            ncl = max(0, min(n, col0 + per) - col0)
            J = pkg.DenseColumnBlock(n, n, col0, ncl, dev)
            return dict(J=J, f=f, x=x, cache=cache, nnz=n * n, n=n, ctx=ctx, keep=(w, bs), col0=col0, ncl=ncl)
        cache = pkg.JacobianCache(x, fdtype, max_batch=mb, use_graph=use_graph)
        J = pkg.zeros_colmajor(n, n, dev)
        return dict(J=J, f=f, x=x, cache=cache, nnz=n * n, n=n, ctx=ctx, keep=(w, bs), col0=0, ncl=n)
    raise SystemExit(f"unknown workload {workload}")


DUMP_ELEMENTS = 4 << 20          # at most this many float64 values written by --dump-outputs: 32 MiB
DUMP_SEED = 20261017


def j_values_flat(pkg, J):
    """J's values as the caller holds them after a call, flat in storage order: nzval (CSC), the band storage (banded),
    or the dense matrix column by column (zeros_colmajor)."""
    if isinstance(J, pkg.SparseMatrixCSC):
        return J.nzval
    if isinstance(J, pkg.BandedMatrix):
        return J.data
    return J.t().reshape(-1)


def output_dumper(out_dir, name, a):
    """Returns a function that writes the flat device array `a`, as it is when called, to out_dir/<name>.npy in float64.
    An array longer than DUMP_ELEMENTS is sampled at sorted positions drawn from DUMP_SEED and its length alone (drawn
    here, not when the function runs), so runs with the same arguments write files that compare entry for entry."""
    import torch
    pos = None
    if a.numel() > DUMP_ELEMENTS:
        pos = np.unique(np.random.default_rng(DUMP_SEED).integers(0, a.numel(), size=DUMP_ELEMENTS))
        pos = torch.from_numpy(pos).to(a.device)

    def dump():
        out = Path(out_dir)
        out.mkdir(parents=True, exist_ok=True)
        np.save(out / f"{name}.npy", (a if pos is None else a[pos]).to(torch.float64).cpu().numpy())
    return dump


def analytic_parity(pkg, workload, fdtype, prob, samples=4096):
    """Size-independent correctness property at FULL size, evaluated on the device: sampled entries of the computed J
    against the closed-form derivative of the synthetic f! (the reference's own bounds: 1e-6 forward, 1e-8 central/complex,
    test/finitedifftests.jl:455-462).  Returns the `parity` record."""
    import torch
    tol = 1e-6 if fdtype == "forward" else 1e-8
    J, x, n = prob["J"], prob["x"], prob["n"]
    dev = x.device
    g = torch.Generator(device=dev).manual_seed(123)
    if workload in ("c1", "c2"):
        nz = J.nzval
        q = torch.arange(1, nz.numel() + 1, device=dev, dtype=torch.int64)
        want = torch.where(q % 3 == 1, -2.0, 1.0).to(torch.float64)
        err = float((nz - want).abs().max())
        return {"kind": "analytic (exact stencil -2/1), every entry", "checked": int(nz.numel()), "max_abs_err": err, "tol": tol,
                "ok": bool(err <= tol and torch.isfinite(nz).all())}
    if workload == "c3":
        gg = prob["g"]
        w = 2 * gg + 1
        c = torch.randint(0, n, (samples,), device=dev, generator=g)
        d = torch.randint(0, w, (samples,), device=dev, generator=g)
        r = c - gg + d
        inb = (r >= 0) & (r < n)
        got = J.data[c * w + d]
        # whole-band fill (ext/FiniteDiffBandedMatricesExt.jl:13-27): slot (r,c) holds the colour-k(c) quotient of row r
        # = the number of stencil points of row r whose column has colour k(c) (f is linear with unit coefficients)
        rr = r.clamp(0, n - 1)
        i, j = rr % gg, rr // gg
        kc = ((c % gg) + 2 * (c // gg)) % 5
        cnt = torch.zeros(samples, dtype=torch.float64, device=dev)
        for (ii, jj) in ((i, j), ((i - 1).clamp(min=0), j), ((i + 1).clamp(max=gg - 1), j), (i, (j - 1).clamp(min=0)),
                         (i, (j + 1).clamp(max=gg - 1))):
            cnt += ((ii + 2 * jj) % 5 == kc).to(torch.float64)
        want = torch.where(inb, cnt, torch.zeros_like(cnt))
        err = float((got - want).abs().max())
        return {"kind": "analytic (colour-k stencil count per band slot, corner slots 0), sampled", "checked": samples,
                "max_abs_err": err, "tol": tol, "ok": bool(err <= tol)}
    if workload == "c4":
        d_cols, d_coef, _cv = prob["keep"]
        K = d_cols.shape[0]
        p = torch.randint(0, J.nzval.numel(), (samples,), device=dev, generator=g)
        r = J.rowval[p] - 1
        c = torch.searchsorted(J.colptr, p + 1, right=True) - 1
        want = torch.zeros(samples, dtype=torch.float64, device=dev)
        for qk in range(K):
            hit = d_cols[qk][r].to(torch.int64) == c
            term = d_coef[qk][r] + (0.2 * x[c] if qk == 0 else 0.0)
            want += torch.where(hit, term, torch.zeros_like(term))
        err = float((J.nzval[p] - want).abs().max())
        return {"kind": "analytic (a_ip + 0.2 x_c [p=1]), sampled", "checked": samples, "max_abs_err": err, "tol": tol,
                "ok": bool(err <= tol and bool(torch.isfinite(J.nzval).all()))}
    if workload == "c5":
        w = prob["keep"][0]
        ncl, col0 = prob["ncl"], prob["col0"]
        if ncl == 0:
            return {"kind": "analytic", "checked": 0, "ok": True}
        slab = J.slab if isinstance(J, pkg.DenseColumnBlock) else J
        jl = torch.randint(0, ncl, (samples,), device=dev, generator=g)
        i = torch.randint(0, n, (samples,), device=dev, generator=g)
        i[: samples // 4] = (jl[: samples // 4] + col0).clamp(max=n - 1)            # a quarter of the samples on the diagonal
        jg = jl + col0
        got = slab[i, jl]
        want = w[i] / n + torch.where(i == jg, 2.0 * x[i], torch.zeros_like(x[i]))
        err = float((got - want).abs().max())
        return {"kind": "analytic (diag(2x) + w 1^T/n), sampled", "checked": samples, "max_abs_err": err, "tol": tol,
                "ok": bool(err <= tol)}
    return None


def known_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the scatter kernel from the committed ncu capture
    (profiles/traffic.json names the capture file), or None when no capture exists for this configuration."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        d = json.loads(p.read_text())
        v = d.get(key)
        if isinstance(v, dict):
            return v.get("bytes"), v.get("source"), bool(v.get("per_jacobian", False))
        if v is not None:
            return v, "profiles/ (round-1 capture)", False
    return None, None, False


def traffic_key(workload, fdtype, info):
    """key into profiles/traffic.json: which ncu capture describes the scatter launches of this plan"""
    key = f"{workload}_{fdtype}"
    if info["sp_kind"] == 1 and info["strategy"] == 1:
        key += "_lists" if info["n_groups"] == 1 else "_lists_per_group"
    elif info["sp_kind"] == 1 and not info.get("staged"):
        key += "_gather"
    return key


def scatter_kernel_name(info, fdtype):
    if info["sp_kind"] == 1:
        if info["strategy"] == 1:
            return "diff_scatter_cm<%s>" % fdtype
        if info.get("staged"):
            return "diff_scatter_staged<u%d,%s> (TMA-staged fused pass)" % (info["color_bits"], fdtype)
        return "diff_scatter_ident<u%d,%s%s>" % (info["color_bits"], fdtype, ",FULL" if info["n_groups"] == 1 else "")
    return {4: "diff_slabs + diff_scatter_band_flat", 0: "diff_columns", 3: "diff_scatter_dest"}.get(info["sp_kind"], "diff_scatter")


def roofline_record(info, fdtype, scat_ms, scat_n, tsteps, traffic_key):
    peak, peak_src = peaks()
    per_jac_ms = scat_ms / tsteps if tsteps else 0.0
    launches = scat_n / tsteps if tsteps else 0
    moved = info["moved_bytes_scatter"]
    survey = info["alg_bytes_scatter"]
    achieved = moved / (per_jac_ms * 1e-3) / 1e9 if per_jac_ms > 0 else None
    traffic, tsrc, per_jac = known_traffic(traffic_key)
    traffic_per_jac = (traffic if per_jac else traffic * launches) if traffic else None
    return {"bound": "hbm", "kernel": scatter_kernel_name(info, fdtype), "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": tsrc, "peak_source": peak_src,
            "bytes_per_launch": moved / launches if launches else None, "launch_ms": per_jac_ms / launches if launches else None,
            "bytes_per_jacobian": moved, "scatter_ms_per_jacobian": per_jac_ms, "scatter_launches_per_jacobian": launches,
            "survey_bytes_per_jacobian": survey,
            "achieved_vs_reference_shape": (survey / (per_jac_ms * 1e-3) / 1e9 / peak) if per_jac_ms > 0 else None,
            "traffic_per_jacobian": traffic_per_jac,
            "frac_traffic": (traffic_per_jac / (per_jac_ms * 1e-3) / 1e9 / peak) if (traffic_per_jac and per_jac_ms > 0) else None,
            "note": "achieved = compulsory bytes of the shipped formulation (fdb_plan_info.moved_bytes_scatter: int32 rows, narrow "
                    "colours / slots, each slab value and J slot once, fx once) / CUDA-event time of the scatter launches; "
                    "achieved_vs_reference_shape uses SURVEY.md §8(d)'s reference-shaped count (Int64 indices, fx re-read per "
                    "nonzero) and may exceed 1; traffic = ncu dram bytes per launch from the named capture"}


def measure(pkg, step, plan, steps, warmup, barrier, dist_max=None, spin_s=0.0, after_timed=None):
    """first call already done by the caller; warm-up (>= 3 steps, optionally at least spin_s seconds so the clock sampler
    sees the load), K timed steps between CUDA events, after_timed() (sees the last timed step's results), then an eager
    pass with the library's own events around the scatter launches."""
    import torch
    for _ in range(max(warmup, 3)):
        step()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < spin_s:
        for _ in range(10):
            step()
        torch.cuda.synchronize()
    barrier()
    c0 = plan.counters()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    if dist_max is not None:
        ms_total = dist_max(ms_total)
    c1 = plan.counters()
    if after_timed is not None:
        after_timed()
    tsteps = min(steps, 20)
    plan.enable_timing(True)
    plan.read_timing()
    for _ in range(tsteps):
        step()
    barrier()
    scat_ms, scat_n = plan.read_timing()
    plan.enable_timing(False)
    return dict(ms_total=ms_total, ms_step=ms_total / steps, c0=c0, c1=c1, scat_ms=scat_ms, scat_n=scat_n, tsteps=tsteps)


def run_single(pkg, workload, fdtype, dev, args, steps, spin_s=0.0, strategy=0, sample_clocks=False, dump_dir=None):
    """One workload on one GPU: build, measure, parity record; with dump_dir, J's values after the last timed step go
    to dump_dir/J.npy (output_dumper).  Returns (record, prob, plan, nnz)."""
    import torch
    prob = build_gpu_problem(pkg, workload, fdtype, dev, 0, 1, args.max_batch, args.graph, strategy=strategy)
    J, f, x, cache = prob["J"], prob["f"], prob["x"], prob["cache"]

    def step():
        pkg.finite_difference_jacobian_(J, f, x, cache)

    def barrier():
        torch.cuda.synchronize()

    barrier()
    t_first = time.perf_counter()
    step()        # builds the plan (index compression, colour buckets, scratch) and captures the graph: one-off cost
    barrier()
    first_call_ms = (time.perf_counter() - t_first) * 1e3
    plan = cache._last_plan
    # nvidia-smi samples every 100 ms: the sampler runs over warm-up (>= spin_s of the same step), the timed region and the
    # kernel-timing pass — all the same kernel sequence under load — and not over problem construction
    after = output_dumper(dump_dir, "J", j_values_flat(pkg, J)) if dump_dir else None
    clocks = Clocks(dev.index if dev.index is not None else 0) if sample_clocks else None
    try:
        m = measure(pkg, step, plan, steps, args.warmup, barrier, spin_s=spin_s, after_timed=after)
    finally:
        clk = clocks.stop() if clocks else None          # never leave the nvidia-smi sampler running
    info = plan.info()
    nnz = prob["nnz"] if prob["nnz"] is not None else info["n_entries"]
    f_points = m["c1"]["f_points"] - m["c0"]["f_points"]
    lib_launches = m["c1"]["kernel_launches"] - m["c0"]["kernel_launches"]
    f_inv = m["c1"]["f_invocations"] - m["c0"]["f_invocations"]
    f_launch_per_point = {"c5": 3}.get(workload, 1)
    key = traffic_key(workload, fdtype, info)
    roof_kernel = scatter_kernel_name(info, fdtype)
    rec = {
        "workload": workload_config(workload, fdtype)["workload"], "ms_per_step": m["ms_step"], "value": nnz / (m["ms_step"] * 1e-3),
        "unit": "nnz/s", "steps": steps, "f_evals_per_s": f_points / (m["ms_total"] * 1e-3), "first_call_ms": first_call_ms,
        "roofline": roofline_record(info, fdtype, m["scat_ms"], m["scat_n"], m["tsteps"], key),
        "parity": analytic_parity(pkg, workload, fdtype, prob),
        "gpu_launches": int(lib_launches + f_inv * f_launch_per_point),
        "gpu_launches_detail": {"library_kernels": int(lib_launches), "f_callback_invocations": int(f_inv)},
        "scatter_strategy": ({0: "fused storage-order pass" + (" (TMA-staged)" if "staged" in roof_kernel else ""),
                              1: "colour-major lists, one launch" if info["n_groups"] == 1 else "colour-major lists per group"}[info["strategy"]]
                             if info["sp_kind"] == 1 else None),
        "scatter_groups": info["n_groups"], "clocks": clk,
    }
    return rec, prob, plan, nnz


def gpu_arm(args):
    import torch
    import torch.distributed as dist
    import _bootstrap
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pkg = _bootstrap.load_package()
    L = pkg._lib
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        return gpu_arm_multi(args, pkg, dev, rank, world)
    workload, fdtype = args.workload, args.fdtype
    if args.group > 1:
        return gpu_arm_group(args, pkg, dev)
    rec, prob, plan, nnz = run_single(pkg, workload, fdtype, dev, args, args.steps, spin_s=args.spin, strategy=args.strategy,
                                      sample_clocks=True, dump_dir=args.dump_outputs)
    clk = rec.pop("clocks")
    J, f, x = prob["J"], prob["f"], prob["x"]
    info = plan.info()

    # ---- e2e: host buffers through the C ABI (fdb_jacobian_host), H2D x + D2H J values inside the timed region
    e2e = None
    if workload in ("c1", "c2", "c4") and not args.no_e2e and fdtype != "complex":
        n = prob["n"]
        hx = pkg.pinned_empty(n)
        hx[:] = x.cpu().numpy()
        hJ = pkg.pinned_empty(info["j_len"])
        fptr, cptr = C.c_void_p(f.address), f.ctx_ptr
        for _ in range(2):
            L.check(L.lib().fdb_jacobian_host(plan.handle, fptr, cptr, hx.ctypes.data, hJ.ctypes.data, None, None, L.STEP_DEFAULT, L.STEP_DEFAULT, 1.0))
        ts = []
        reps = max(3, min(args.steps, 10))
        for _ in range(reps):
            t0 = time.perf_counter()
            L.check(L.lib().fdb_jacobian_host(plan.handle, fptr, cptr, hx.ctypes.data, hJ.ctypes.data, None, None, L.STEP_DEFAULT, L.STEP_DEFAULT, 1.0))
            ts.append(time.perf_counter() - t0)
        te = statistics.median(ts)
        same = bool(np.array_equal(hJ, J.nzval.cpu().numpy()))
        e2e = {"value": nnz / te, "unit": "nnz/s", "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8 * info["j_len"],
               "ms_per_step": te * 1e3, "api": "fdb_jacobian_host (C ABI, pinned host x and nzval)", "reps": reps,
               "result_equals_device_resident_run": same,
               "note": "PCIe-bound: %.0f MB per call over the host link = %.1f GB/s" % ((8 * n + 8 * info["j_len"]) / 1e6,
                                                                                  (8 * n + 8 * info["j_len"]) / te / 1e9)}

    # ---- cpu_baseline: the oracle, 1 thread (the reference is single-threaded), bounded sample; a final untimed run is fed
    #      the device-computed step sizes and its nzval is bit-compared with the GPU's (parity inside the run the driver sees)
    cpu = None
    if not args.no_cpu and workload in ("c1", "c2", "c4"):
        from oracle import fd_oracle as orc
        scale = 1.0 if workload != "c4" else 0.2
        run, cnnz, cf, desc = cpu_jacobian_runner(workload, fdtype, 1, scale)
        med, reps = time_cpu(run, budget_s=14.0, max_reps=5)
        cpu = {"value": cnnz / med, "unit": "nnz/s", "cores": 1, "kind": "port",
               "sample": f"{reps} full Jacobian(s) of {desc} (median {med:.3f} s); host offers {usable_cores()} usable cores",
               "f_evals_per_s": cf / med}
        if scale == 1.0 and fdtype != "complex":
            _, ref_nz = run(eps_override=plan.eps())
            got = J.nzval.cpu().numpy()
            equal = bool(np.array_equal(got, ref_nz))
            rec["parity"]["oracle_bitwise"] = {"against": "CPU oracle fed the device-computed step sizes, every nzval entry",
                                               "entries": int(got.size), "equal": equal,
                                               "mismatches": int((got != ref_nz).sum()) if not equal else 0}
            rec["parity"]["ok"] = bool(rec["parity"]["ok"] and equal)
            try:
                # the device's step sizes against the ones the reference's own `norm` gives (oracle: OpenBLAS dnrm2 restated
                # in x87 extended precision, pinned bit for bit by tests/test_oracle_norm.py) — reported, in ulps
                dev_eps = np.asarray(plan.eps(), dtype=np.float64)
                ref_eps = np.array([orc.color_eps(run.x, run.cv, k + 1, run.fd) for k in range(dev_eps.size)])
                ulps = (dev_eps - ref_eps) / np.spacing(np.abs(ref_eps))
                rec["parity"]["eps_vs_reference_norm"] = {
                    "against": "eps from LinearAlgebra.norm as the reference evaluates it (oracle fdo_norm2 = OpenBLAS dnrm2 for n >= 32)",
                    "max_abs_ulps": float(np.max(np.abs(ulps))), "max_rel_err": float(np.max(np.abs(dev_eps / ref_eps - 1.0))),
                    "bit_equal": int((dev_eps == ref_eps).sum()), "colors": int(dev_eps.size)}
                if equal and bool((dev_eps == ref_eps).all()):
                    # same step sizes => the oracle run above is also what the oracle computes entirely on its own
                    rec["parity"]["oracle_bitwise"]["holds_with_the_oracles_own_step_sizes"] = True
            except Exception as e:  # a diagnostic must never cost the headline line
                rec["parity"]["eps_vs_reference_norm"] = {"error": repr(e)[:200]}

    # ---- the other BASELINE configs at full size on this GPU (sub-records of the one line)
    others = {}
    if args.extras:
        del prob, J, f, x, plan
        torch.cuda.empty_cache()
        todo = [("c2_central", "c2", "central", 100, 0), ("c3_forward", "c3", "forward", 30, 0),
                ("c4_forward_fused", "c4", "forward", 20, 1), ("c4_forward_lists", "c4", "forward", 20, 3),
                ("c5_central", "c5", "central", 3, 0)]
        for key, w, fd, st, strat in todo:
            try:
                r2, p2, pl2, _ = run_single(pkg, w, fd, dev, args, st, strategy=strat, sample_clocks=True)
                others[key] = r2
                del p2, pl2
            except Exception as e:  # an extra must never cost the headline line
                others[key] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
        c4s = [others[k] for k in ("c4_forward_fused", "c4_forward_lists") if "ms_per_step" in others.get(k, {})]
        if c4s:
            best = min(c4s, key=lambda r: r["ms_per_step"])
            others["scale_base"] = {"workload": best["workload"], "t1_ms": best["ms_per_step"], "strategy": best["scatter_strategy"],
                                    "note": "single-GPU time of the workload `--gpus N` (N>1) strong-scales; every N>1 line "
                                            "re-measures it on rank 0 in the same run (strong_scaling.t1_ms)"}

    line = {
        "metric": "jacobian_nnz_per_s", "value": rec["value"], "unit": "nnz/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(workload, fdtype),
        "details": {"cuda_graph": bool(args.graph), "max_batch": args.max_batch, "scatter_groups": rec["scatter_groups"],
                    "scatter_strategy": rec["scatter_strategy"], "first_call_ms": rec["first_call_ms"],
                    "warmup_note": "warm-up = max(W,3) steps + 0.6 s of the same step so the 100 ms clock sampler sees the load"},
        "f_evals_per_s": rec["f_evals_per_s"],
        "roofline": rec["roofline"], "parity": rec["parity"], "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": rec["gpu_launches"], "gpu_launches_detail": rec["gpu_launches_detail"],
        "clocks": clk, "workloads": others,
    }
    print(json.dumps(line))


def gpu_arm_group(args, pkg, dev):
    """`--group N`: ONE process drives N GPUs through the C ABI's fdb_group_* (what a Julia host calling
    finite_difference_jacobian! once would use) — no torch.distributed, no NCCL, no second process.  C4, colours sharded over
    the devices, every member's scatter stores straight into device 0's nzval; bit-compared with the 1-GPU Jacobian."""
    import torch
    from finitediff_jl_b200 import distributed as fdist
    L = pkg._lib
    n_dev = args.group
    if torch.cuda.device_count() < n_dev:
        raise SystemExit(f"--group {n_dev} needs {n_dev} visible GPUs")
    fdtype = args.fdtype
    r1, p1, pl1, nnz = run_single(pkg, "c4", fdtype, dev, args, max(5, min(args.steps, 20)))
    J1, eps1 = p1["J"].nzval.clone(), pl1.eps().copy()
    J, x, cv = p1["J"], p1["x"], p1["keep"][2]
    d_cols, d_coef = p1["keep"][0], p1["keep"][1]
    devices = list(range(n_dev))
    keep, fs = [], []
    for d in devices:
        dd = torch.device("cuda", d)
        c_d, a_d = (d_cols, d_coef) if d == dev.index else (d_cols.to(dd), d_coef.to(dd))
        ctx = L.EllCtx(p1["n"], C4_K, c_d.data_ptr(), a_d.data_ptr(), 0)
        keep.append((c_d, a_d, ctx))
        fs.append(pkg.NativeFn(C.cast(L.synth().fdbs_ellrows, C.c_void_p).value, ctx))
    del pl1
    J.nzval.fill_(float("nan"))
    g = fdist.GroupJacobian(J, cv, fdtype, devices, use_graph=args.graph)

    def step():
        g.run(fs, x)

    step()
    g.synchronize()
    for _ in range(max(args.warmup, 3)):
        step()
    g.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()          # the root stream waits on every member's completion event inside fdb_group_jacobian
    g.synchronize()
    ms_step = ev0.elapsed_time(ev1) / args.steps
    equal = bool(torch.equal(J.nzval, J1))
    line = {"metric": "jacobian_nnz_per_s", "value": nnz / (ms_step * 1e-3), "unit": "nnz/s", "n_gpus": n_dev, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config("c4", fdtype),
            "details": {"driver": "one process, fdb_group_create_csc / fdb_group_jacobian (C ABI), CUDA graph per member" if args.graph else "one process, fdb_group_*",
                        "devices": devices},
            "strong_scaling": {"t1_ms": r1["ms_per_step"], "tN_ms": ms_step, "speedup": r1["ms_per_step"] / ms_step, "n_gpus": n_dev},
            "parity": {"sharded_equals_unsharded": {"equal": equal, "eps_equal": bool(np.array_equal(g.plans[0].eps(), eps1))}, "ok": equal},
            "cpu_baseline": None, "e2e": None, "gpu_launches": None}
    print(json.dumps(line))
    g.close()


def gpu_arm_multi(args, pkg, dev, rank, world):
    """N > 1, one process per GPU.  c4: colours sharded (strong scaling; rank 0 first times the same problem alone and
    keeps that J for the bit-compare).  c5: column blocks, J left column-sharded (north_star config 5)."""
    import torch
    import torch.distributed as dist
    from finitediff_jl_b200 import distributed as fdist
    workload, fdtype = args.workload, args.fdtype

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def dist_max(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def dist_sum(v):
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return float(t.item())

    if workload == "c2" and args.shard == "columns":
        return gpu_arm_columns(args, pkg, dev, rank, world)
    if workload not in ("c4", "c5"):
        raise SystemExit("--gpus N>1 runs c4 (colour shards), c5 (column blocks) or c2 with --shard columns")

    strong = None
    J1 = eps1 = None
    if workload == "c4":
        # ---- same-workload 1-GPU reference, rank 0 alone, same run: t1 for the strong-scaling record, J1 for parity
        if rank == 0:
            best = None
            for strat in (1, 3):
                r1, p1, pl1, _ = run_single(pkg, "c4", fdtype, dev, args, max(5, min(args.steps, 20)), strategy=strat)
                if best is None or r1["ms_per_step"] < best[0]["ms_per_step"]:
                    best = (r1, p1["J"].nzval.clone(), pl1.eps().copy())
                del p1, pl1
                torch.cuda.empty_cache()
            strong = {"t1_ms": best[0]["ms_per_step"], "t1_strategy": best[0]["scatter_strategy"], "t1_roofline_frac": best[0]["roofline"]["frac"]}
            J1, eps1 = best[1], best[2]
        barrier()

    prob = build_gpu_problem(pkg, workload, fdtype, dev, rank, world, args.max_batch, args.graph, strategy=args.strategy)
    J, f, x, cache = prob["J"], prob["f"], prob["x"], prob["cache"]
    sharded = None
    if workload == "c4":
        sharded = fdist.ShardedJacobian(J, cache, x.numel(), dev, gather=args.gather, barrier=args.barrier)

    def step():
        if sharded is not None:
            sharded.run(f, x)
        else:
            pkg.finite_difference_jacobian_(J, f, x, cache)

    barrier()
    t_first = time.perf_counter()
    step()
    barrier()
    first_call_ms = (time.perf_counter() - t_first) * 1e3
    plan = cache._last_plan
    clocks = Clocks(dev.index) if rank == 0 else None
    try:
        m = measure(pkg, step, plan, args.steps, args.warmup, barrier, dist_max=dist_max, spin_s=args.spin)
    finally:
        clk = clocks.stop() if clocks else None
    info = plan.info()
    nnz = prob["nnz"]
    ms_step = m["ms_step"]
    value = nnz / (ms_step * 1e-3)
    f_points_all = dist_sum(m["c1"]["f_points"] - m["c0"]["f_points"])
    lib_launches = m["c1"]["kernel_launches"] - m["c0"]["kernel_launches"]
    f_inv = m["c1"]["f_invocations"] - m["c0"]["f_invocations"]
    gpu_launches = lib_launches + f_inv * {"c5": 3}.get(workload, 1)
    key = traffic_key(workload, fdtype, info)
    roofline = roofline_record(info, fdtype, m["scat_ms"], m["scat_n"], m["tsteps"], key)

    # ---- parity inside the run: analytic sampled check on every rank's result + (c4) sharded == unsharded, bit for bit
    check_here = workload == "c5" or rank == 0 or args.gather != "root"
    par = analytic_parity(pkg, workload, fdtype, prob) if check_here else {"ok": True, "checked": 0}
    ok_all = dist_sum(0.0 if par["ok"] else 1.0) == 0.0
    if workload == "c4" and rank == 0:
        got = J.nzval
        equal = bool(torch.equal(got, J1))
        par["sharded_equals_unsharded"] = {"against": "the 1-GPU Jacobian of the same problem computed by rank 0 in this run "
                                           "(bit-compare of all %d nzval entries)" % got.numel(), "equal": equal,
                                           "eps_equal": bool(np.array_equal(plan.eps(), eps1)),
                                           "checksum": float(got.sum()), "mismatches": int((got != J1).sum()) if not equal else 0}
        par["ok"] = bool(par["ok"] and equal)
        strong.update(tN_ms=ms_step, speedup=strong["t1_ms"] / ms_step, n_gpus=world)
    if rank == 0:
        par["all_ranks_ok"] = bool(ok_all)
    del J1

    # ---- e2e at N GPUs: pinned host x -> every rank's device x, sharded run, rank 0's nzval -> pinned host
    e2e = None
    if workload == "c4" and not args.no_e2e:
        n = prob["n"]
        hx = torch.empty(n, dtype=torch.float64).pin_memory()
        hx.copy_(x.cpu())
        hJ = torch.empty(J.nzval.numel(), dtype=torch.float64).pin_memory() if rank == 0 else None
        xd = torch.empty_like(x)
        ts = []
        for it in range(5):
            barrier()
            t0 = time.perf_counter()
            xd.copy_(hx, non_blocking=True)
            sharded.run(f, xd)
            if rank == 0:
                hJ.copy_(J.nzval, non_blocking=True)
            torch.cuda.synchronize()
            dist.barrier()
            if it >= 2:
                ts.append(time.perf_counter() - t0)
        te = dist_max(statistics.median(ts))
        e2e = {"value": nnz / te, "unit": "nnz/s", "h2d_bytes_per_step": 8 * n * world, "d2h_bytes_per_step": 8 * nnz,
               "ms_per_step": te * 1e3, "api": "ShardedJacobian.run (pinned host x -> every rank; rank 0's nzval -> pinned host)"}
    elif workload == "c5":
        e2e = {"value": None, "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
               "note": "the 80 GB dense J stays column-sharded on the devices (no host copy measured)"}

    # ---- cpu_baseline on rank 0: the oracle, 1 thread, a bounded sample of the same workload
    cpu = None
    if rank == 0 and not args.no_cpu and workload == "c4":
        from oracle import fd_oracle as orc
        run, cnnz, cf, desc = cpu_jacobian_runner("c4", fdtype, 1, 0.2)
        med, reps = time_cpu(run, budget_s=10.0, max_reps=3)
        cpu = {"value": cnnz / med, "unit": "nnz/s", "cores": 1, "kind": "port",
               "sample": f"{reps} full Jacobian(s) of {desc} (median {med:.3f} s; problem scaled by 0.2)", "f_evals_per_s": cf / med}
    if rank == 0:
        line = {
            "metric": "jacobian_nnz_per_s", "value": value, "unit": "nnz/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(workload, fdtype),
            "details": {"cuda_graph": bool(args.graph), "max_batch": args.max_batch, "gather": args.gather if workload == "c4" else "none (column-sharded J)",
                        "rank_barrier": (args.barrier + (" (fdb_sync: device-side flags in peer memory)" if args.barrier == "device" else " all_reduce")) if workload == "c4" else None,
                        "colors_local": info["n_local_colors"], "scatter_groups": info["n_groups"], "first_call_ms": first_call_ms},
            "f_evals_per_s": f_points_all / (m["ms_total"] * 1e-3),
            "strong_scaling": strong, "roofline": roofline, "parity": par, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(gpu_launches),
            "gpu_launches_detail": {"library_kernels": int(lib_launches), "f_callback_invocations": int(f_inv), "scope": "rank 0"},
            "clocks": clk,
        }
        print(json.dumps(line))
    if sharded is not None:
        sharded.close()
    dist.barrier()
    dist.destroy_process_group()


def gpu_arm_columns(args, pkg, dev, rank, world):
    """c2 over contiguous column blocks with a slice-aware f! (3 colours cannot be spread by colour over > 3 GPUs)."""
    import torch
    import torch.distributed as dist
    from finitediff_jl_b200 import distributed as fdist
    L = pkg._lib
    fdtype = args.fdtype
    if fdtype == "complex":
        raise SystemExit("--shard columns: forward / central")
    prob = build_gpu_problem(pkg, "c2", fdtype, dev, 0, 1, args.max_batch, args.graph)
    J, x = prob["J"], prob["x"]
    n_glob = prob["n"]
    keep_ctx = []

    def factory(r0, r1, x0, x1):
        c = L.TridiagRowsCtx(n_glob, r0, r1 - r0, x0, 0)
        keep_ctx.append(c)
        return pkg.NativeFn(C.cast(L.synth().fdbs_tridiag_rows, C.c_void_p).value, c, max_batch=args.max_batch)

    cs = fdist.ColumnShardedJacobian(J, prob["keep"][2], fdtype, dev, factory, gather=None if args.gather == "none" else "root",
                                     max_batch=args.max_batch, use_graph=args.graph)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def dist_max(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step():
        cs.run(x)

    step()
    barrier()
    plan = cs.block.plan
    m = measure(pkg, step, plan, args.steps, args.warmup, barrier, dist_max=dist_max)
    info = plan.info()
    if rank == 0:
        line = {"metric": "jacobian_nnz_per_s", "value": prob["nnz"] / (m["ms_step"] * 1e-3), "unit": "nnz/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": m["ms_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config("c2", fdtype),
                "details": {"shard": "columns", "gather": args.gather, "cuda_graph": bool(args.graph)},
                "roofline": roofline_record(info, fdtype, m["scat_ms"], m["scat_n"], m["tsteps"], f"c2_{fdtype}_block"),
                "cpu_baseline": None, "e2e": None, "gpu_launches": int(m["c1"]["kernel_launches"] - m["c0"]["kernel_launches"])}
        print(json.dumps(line))
    cs.close()
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: per workload, a few seconds in total)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["c1", "c2", "c3", "c4", "c5"])
    ap.add_argument("--fdtype", default=None, choices=["forward", "central", "complex"])
    ap.add_argument("--max-batch", type=int, default=1, dest="max_batch")
    ap.add_argument("--strategy", type=int, default=0, choices=[0, 1, 2, 3],
                    help="CSC scatter: 0 auto, 1 fused storage-order pass, 2 colour-major lists per group, 3 colour-major lists, one launch")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch eagerly instead of replaying the captured CUDA graph of the call")
    ap.add_argument("--gather", default="root", choices=["all", "root", "all_p2p", "none"],
                    help="N>1 (c4): rank 0 ends with the full Jacobian (root: every rank's scatter stores straight into rank "
                         "0's nzval over NVLink), or every rank does (all: + NCCL broadcast; all_p2p: stores to every peer)")
    ap.add_argument("--barrier", default="device", choices=["device", "nccl"],
                    help="N>1: how the ranks are ordered around a Jacobian — fdb_sync (device-side flags, default) or an NCCL all_reduce")
    ap.add_argument("--shard", default="colors", choices=["colors", "columns"],
                    help="N>1: colour set (c4) or contiguous column blocks with a slice-aware f! (c2)")
    ap.add_argument("--spin", type=float, default=0.6, help="seconds of extra warm-up of the same step (lets the 100 ms clock sampler see the load; 0 under ncu)")
    ap.add_argument("--group", type=int, default=1,
                    help="run C4 over N GPUs from ONE process through fdb_group_* (no torchrun); ad-hoc, not the driver contract")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="--gpus 1 default run: skip the c2-central / c3 / c4 / c5 sub-records")
    ap.add_argument("--cpu-scale", type=float, default=1.0, dest="cpu_scale",
                    help="--impl reference: problem-size fraction per step (1.0 = the full configuration)")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="single-GPU run: after the timed steps write J's values from the last one to DIR/J.npy (float64; "
                         "a fixed, seeded sample of at most 4 Mi entries) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    explicit = args.workload is not None or args.fdtype is not None
    if args.workload is None:
        args.workload = "c2" if max(args.gpus, world) == 1 else "c4"
    if args.fdtype is None:
        args.fdtype = "central" if args.workload == "c5" else "forward"
    if explicit or args.workload != "c2":
        args.extras = False
    if args.fdtype == "complex" and args.workload not in ("c1", "c2"):
        raise SystemExit("--fdtype complex is benchmarked on the tridiagonal workloads (c1, c2)")
    if args.group > 1:
        args.workload, args.extras = "c4", False
        args.fdtype = args.fdtype or "forward"
    if args.dump_outputs and (args.impl != "ours" or max(args.gpus, world) > 1 or args.group > 1):
        ap.error("--dump-outputs applies to the single-GPU run of this implementation (--impl ours, --gpus 1)")
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else {"c1": 500, "c2": 200, "c3": 50, "c4": 30, "c5": 5}[args.workload]
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
