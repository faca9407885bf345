#!/usr/bin/env python
"""Measures ppp_mls_smooth (the reference's smooth(): MLS, order 3, radius 15) on noisy panels and writes one JSON
file: per configuration the kernel device time (ppp_kernel_profile, CUDA events around each launch, >= 20 calls
after warm-up), the host-API call's wall time, the double-precision operations the algorithm needs (from the exact
neighbour counts of a counts-only ppp_radius call) and the achieved rate, and the CPU oracle's time with 16 threads
on the same machine.  The GPU's name and power limit are read (nvidia-smi --query-gpu, read only) in the same run.

    python tools/mls_perf.py [--out mls_perf.json] [--calls 20] [--warmup 3] [--quick]

DP operations per neighbour (an FMA counts as two), order 3:
  visit 1 (count, centroid, covariance): 3 subtractions, 3 additions, 6 FMAs                      = 18
  visit 2 (weights, frame coordinates, moments): d = p - mean 3, d.d 5, scale 1, u/v/f 15, powers of
  v 5, w u^a 6, 28 moment FMAs 56, w f u^a 4, 10 right-hand-side FMAs 20                        = 115
  plus one double exp per neighbour, not counted.
Candidates outside the ball cost a float32 distance each and no DP work."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from polishpathplanning_b200 import api, synth  # noqa: E402

DP_VISIT1 = 18
DP_VISIT2 = 115


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return dict(gpu_name=name, power_limit=power, max_sm_clock=clock)


def measure(ctx, cloud, calls, warmup, oracle_threads):
    n = cloud.shape[0]
    gc = api.Cloud(ctx, cloud)
    counts = np.empty(n, np.int32)
    api.check(gc.lib.ppp_radius(gc._h, None, 0, 0, 15.0, counts.ctypes.data_as(C.c_void_p), None, None, None))
    nb = counts.astype(np.int64)
    emitted = nb >= 3
    fitted = nb >= 10
    dp_ops = int(DP_VISIT1 * nb[emitted].sum() + DP_VISIT2 * nb[fitted].sum())
    out = ctx.pinned_empty((n, 8), np.float32)
    src = ctx.pinned_empty((n,), np.int32)
    m = C.c_int64(0)

    def call():
        api.check(gc.lib.ppp_mls_smooth(gc._h, 15.0, 3, out.ctypes.data_as(C.c_void_p), 32, None,
                                        src.ctypes.data_as(C.c_void_p), C.byref(m)))

    for _ in range(warmup):
        call()
    ctx.kernel_profile(True)
    ctx.kernel_profile_read(reset=True)
    for _ in range(calls):
        call()
    prof = ctx.kernel_profile_read(reset=True)
    ctx.kernel_profile(False)
    kern_ms = prof["mls_order3"][0] / prof["mls_order3"][1]
    all_ms = sum(ms for ms, _ in prof.values()) / calls
    walls = []
    for _ in range(calls):
        t0 = time.perf_counter()
        call()
        walls.append((time.perf_counter() - t0) * 1e3)
    rows = m.value
    gc.close()
    res = dict(
        points=n, rows=rows, neighbours_mean=float(nb.mean()), neighbours_max=int(nb.max()),
        dp_ops=dp_ops, mls_kernel_ms=kern_ms, all_kernels_ms=all_ms,
        kernels={k: dict(ms_per_call=v[0] / calls, launches_per_call=v[1] / calls) for k, v in prof.items()},
        call_ms_median=float(np.median(walls)), call_ms_min=float(np.min(walls)),
        dp_rate_tflops=dp_ops / (kern_ms * 1e-3) / 1e12,
    )
    if oracle_threads:
        sys.path.insert(0, ROOT)
        from oracle_mls import ppp_oracle_mls as pom
        pom.build()
        t0 = time.perf_counter()
        _, _, osrc, _ = pom.mls_smooth(cloud, 15.0, 3, threads=oracle_threads)
        res["cpu_oracle_s"] = time.perf_counter() - t0
        res["cpu_oracle_threads"] = oracle_threads
        res["rows_match_oracle"] = bool(np.array_equal(osrc, src[:rows]))
        res["speedup_vs_cpu_oracle_call"] = res["cpu_oracle_s"] * 1e3 / res["call_ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="mls_perf.json")
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--oracle-threads", type=int, default=16)
    ap.add_argument("--quick", action="store_true", help="small clouds (a rehearsal, not a measurement)")
    a = ap.parse_args()
    configs = [("panel_1M_density1", 1_000_000, 1.0), ("panel_1M_density4", 1_000_000, 4.0),
               ("panel_5M_density1", 5_000_000, 1.0)]
    if a.quick:
        configs = [(name, n // 100, d) for name, n, d in configs]
    info = gpu_info()
    ctx = api.Context(0)
    result = dict(info, radius=15.0, order=3, noise_sigma_mm=0.05, calls=a.calls, warmup=a.warmup,
                  dp_ops_per_neighbour=dict(visit1=DP_VISIT1, visit2=DP_VISIT2), configs={})
    for name, n, density in configs:
        cloud = synth.panel(n, seed=21, density=density, noise_sigma=0.05)
        result["configs"][name] = r = measure(ctx, cloud, a.calls, a.warmup, a.oracle_threads)
        print(name, json.dumps(r), flush=True)
    ctx.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
