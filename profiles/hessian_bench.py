"""Hessian benchmark: fdb_hessian on the synthetic scalar function fdbs_hess_poly
(f(x) = sum w_i x_i^3 + sum x_i x_{i+1} + (sum x_i)^2/(2n)), n in {256, 1024, 4096}, with a sweep of the batch size B
(points per callback).

Per (n, B): median step time over >= 20 CUDA-event-timed Hessians after warm-up; Hessians/s and f-points/s; the combine
kernel's time (fdb_plan_enable_timing) and its compulsory bytes (fdb_plan_info.moved_bytes_scatter: F read once, the n
steps, H written once) over the measured copy bandwidth of the card; and, from one torch.profiler step of its own, the
device time of each library kernel, the point-update kernels' share of the step included.  The CPU oracle (1 thread)
runs at n = 256 and 1024 on the same seeded inputs: its time is reported and H must be bit-identical to it.  The card's
name and power limit are read (read-only nvidia-smi query) in the same run.

Loads what build() left (finitediff.jl_b200/*.so, oracle_hessian/libfd_hessian_oracle.so); writes only --out.
    python profiles/hessian_bench.py --out hessian_bench.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

SWEEP = {256: [256, 2048, 16384, 131073], 1024: [512, 2048, 8192, 32768], 4096: [1024, 4096, 16384, 65536]}
ORACLE_N = (256, 1024)
LIB_KERNELS = ("component_eps", "hess_replicate", "hess_points", "hess_combine")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001 — reported, not fatal
        return {"name": None, "power_limit": None, "error": repr(e)}


def copy_bandwidth_gbs(torch):
    """Measured device-to-device copy rate (read + write bytes / time) of a 4 GiB buffer, median of 10."""
    n = (4 << 30) // 8
    a = torch.empty(n, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(10):
        s.record()
        b.copy_(a)
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e) * 1e-3)
    del a, b
    return 2 * n * 8 / statistics.median(ts) / 1e9


def inputs(n):
    rng = np.random.default_rng(1000 + n)
    return rng.uniform(0.5, 1.5, n), rng.uniform(-1.0, 1.0, n)


def run_config(torch, L, n, B, steps, warmup, profile):
    dev = torch.device("cuda:0")
    x, w = inputs(n)
    dx, dw = torch.from_numpy(x).to(dev), torch.from_numpy(w).to(dev)
    H = torch.zeros((n, n), dtype=torch.float64, device=dev)
    ctx = L.HessPolyCtx(n, dw.data_ptr(), 0)
    fptr, cptr = C.cast(L.synth().fdbs_hess_poly, C.c_void_p), C.cast(C.pointer(ctx), C.c_void_p)
    h = C.c_void_p()
    L.check(L.lib().fdb_hessian_plan_create(C.byref(h), n, C.byref(L.PlanOpts(fdtype=L.FDB_HCENTRAL, max_batch=B))))
    stream = torch.cuda.current_stream(dev).cuda_stream
    try:
        info = L.PlanInfo()
        L.check(L.lib().fdb_plan_info(h, C.byref(info)))

        def step():
            L.check(L.lib().fdb_hessian(h, fptr, cptr, dx.data_ptr(), H.data_ptr(), n, L.STEP_DEFAULT, L.STEP_DEFAULT,
                                        C.c_void_p(stream)))
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        c0 = L.Counters()
        L.check(L.lib().fdb_plan_counters(h, C.byref(c0)))
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        L.check(L.lib().fdb_plan_enable_timing(h, 1))
        for s, e in evs:
            s.record()
            step()
            e.record()
        torch.cuda.synchronize()
        times = [s.elapsed_time(e) for s, e in evs]
        comb_ms, comb_n = C.c_double(), C.c_int64()
        L.check(L.lib().fdb_plan_read_timing(h, C.byref(comb_ms), C.byref(comb_n)))
        L.check(L.lib().fdb_plan_enable_timing(h, 0))
        c1 = L.Counters()
        L.check(L.lib().fdb_plan_counters(h, C.byref(c1)))
        kernels = None
        if profile:
            from torch.profiler import ProfilerActivity, profile as tprof
            with tprof(activities=[ProfilerActivity.CUDA]) as prof:
                step()
                torch.cuda.synchronize()
            kernels = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA:
                    key = next((k for k in LIB_KERNELS + ("k_hess_poly",) if k in ev.name), "other")
                    kernels[key] = kernels.get(key, 0.0) + ev.device_time_total / 1e3   # ms
        med = statistics.median(times)
        pts = 2 * n * n + 1
        return {
            "n": n, "max_batch": B, "batch": int(info.slabs), "callbacks_per_hessian": int(info.n_groups),
            "point_buffer_bytes": int(info.slabs) * (n + (n & 1)) * 8,
            "steps": steps, "median_ms": med, "min_ms": min(times), "max_ms": max(times),
            "hessians_per_s": 1e3 / med, "f_points_per_s": pts * 1e3 / med,
            "f_points_per_hessian": (c1.f_points - c0.f_points) // steps, "expected_f_points": pts,
            "combine_ms": comb_ms.value / max(comb_n.value, 1), "combine_launches": comb_n.value,
            "combine_compulsory_bytes": int(info.moved_bytes_scatter),
            "profiled_kernel_ms": kernels,
        }, H, x, w
    finally:
        L.lib().fdb_plan_destroy(h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sizes", default="256,1024,4096")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hessian_bench.py needs a GPU: no CPU timings are reported")
    import _bootstrap
    pkg = _bootstrap.load_package()
    L = pkg._lib
    from oracle_hessian import hessian_oracle as horc
    res = {"card": card(), "torch": torch.__version__, "device": torch.cuda.get_device_name(0)}
    res["copy_gbs"] = copy_bandwidth_gbs(torch)
    res["runs"] = []
    res["oracle"] = {}
    for n in [int(s) for s in a.sizes.split(",")]:
        oracle = None
        if n in ORACLE_N:
            x, w = inputs(n)
            t0 = time.perf_counter()
            oracle = horc.hess_poly(x, w)
            res["oracle"][str(n)] = {"threads": 1, "seconds": time.perf_counter() - t0, "fcalls": oracle["fcalls"]}
        for B in SWEEP.get(n, [1024, 8192]):
            r, H, x, w = run_config(torch, L, n, B, a.steps, a.warmup, profile=True)
            Hh = H.cpu().numpy()
            r["symmetric_bitwise"] = bool(np.array_equal(Hh.view(np.uint64), Hh.T.view(np.uint64)))
            if oracle is not None:
                # H is symmetric bit for bit, so the row-major tensor compares with the column-major oracle as is
                r["bit_identical_to_oracle"] = bool(np.array_equal(Hh.view(np.uint64), oracle["H"].view(np.uint64)))
                r["speedup_vs_oracle_1thread"] = res["oracle"][str(n)]["seconds"] * 1e3 / r["median_ms"]
            if r["combine_ms"] > 0:
                r["combine_gbs"] = r["combine_compulsory_bytes"] / (r["combine_ms"] * 1e-3) / 1e9
                r["combine_frac_of_copy_bw"] = r["combine_gbs"] / res["copy_gbs"]
            k = r["profiled_kernel_ms"] or {}
            if k:
                step_ms = r["median_ms"]
                r["point_update_share_of_step"] = k.get("hess_points", 0.0) / step_ms
                r["library_kernels_share_of_step"] = sum(k.get(s, 0.0) for s in LIB_KERNELS) / step_ms
                r["f_share_of_step"] = k.get("k_hess_poly", 0.0) / step_ms
            print(json.dumps(r), flush=True)
            res["runs"].append(r)
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text)
    print(json.dumps({k: res[k] for k in ("card", "copy_gbs", "oracle")}))


if __name__ == "__main__":
    main()
