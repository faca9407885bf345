#!/usr/bin/env python
"""Measures ppp_voxel_grid (the reference's voxel_down(): pcl::VoxelGrid) on panels of 1M, 5M and 20M points at
densities 16 and 64 points/mm^2 with leaves of 0.5 and 1.0 mm, and writes one JSON file: per configuration the
kernel device time (ppp_kernel_profile, CUDA events around each launch, after warm-up), the host-API call's wall time
(ppp_voxel_grid into pinned buffers: rows of 32 bytes, row offsets and members), the row count, and the single-thread
CPU oracle's time in PCL's order (PCL's VoxelGrid is single-threaded).  Every configuration is checked against the
oracle's stable order (rows, offsets, members and x, y, z bit-identical), and the fraction of rows bit-identical to
PCL's order is recorded.  The GPU's name and power limit are read (nvidia-smi --query-gpu, read only) in the same run.

    python tools/voxel_perf.py [--out profiles/voxel_perf_b200.json] [--calls 10] [--warmup 2] [--quick]"""
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

from oracle_voxel import ppp_oracle_voxel as ov  # noqa: E402
from polishpathplanning_b200 import _lib, api, synth  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return dict(gpu_name=name, power_limit=power, max_sm_clock=clock)


def measure(ctx, gc, cloud, leaf, calls, warmup):
    n = cloud.shape[0]
    out = ctx.pinned_empty((n, 8), np.float32)
    off = ctx.pinned_empty((n + 1,), np.int64)
    mem = ctx.pinned_empty((n,), np.int32)
    lf = np.full(3, leaf, np.float32)
    m = C.c_int64(0)

    def call():
        api.check(gc.lib.ppp_voxel_grid(gc._h, lf.ctypes.data_as(_lib._f32p), out.ctypes.data_as(C.c_void_p), 32,
                                        off.ctypes.data_as(C.c_void_p), mem.ctypes.data_as(C.c_void_p), C.byref(m)))

    for _ in range(warmup):
        call()
    ctx.kernel_profile(True)
    ctx.kernel_profile_read(reset=True)
    for _ in range(calls):
        call()
    prof = ctx.kernel_profile_read(reset=True)
    ctx.kernel_profile(False)
    walls = []
    for _ in range(calls):
        t0 = time.perf_counter()
        call()
        walls.append((time.perf_counter() - t0) * 1e3)
    rows = m.value
    res = dict(
        points=n, leaf=leaf, rows=rows,
        all_kernels_ms=sum(ms for ms, _ in prof.values()) / calls,
        kernels={k: dict(ms_per_call=v[0] / calls, launches_per_call=v[1] / calls) for k, v in prof.items()},
        call_ms_median=float(np.median(walls)), call_ms_min=float(np.min(walls)),
    )
    got_xyz = np.array(out[:rows, :3])
    got_off = np.array(off[:rows + 1])
    got_mem = np.array(mem[:int(got_off[-1])])
    srec, soff, smem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    res["bit_identical_to_stable_oracle"] = bool(
        np.array_equal(got_off, soff) and np.array_equal(got_mem, smem)
        and np.array_equal(got_xyz.view(np.uint32), srec[:, :3].view(np.uint32)))
    t0 = time.perf_counter()
    prec, poff, _ = ov.voxel_grid(cloud, leaf, ov.PCL_ORDER)
    res["cpu_oracle_pcl_order_s"] = time.perf_counter() - t0
    res["cpu_oracle_threads"] = 1
    res["rows_match_pcl_order"] = bool(np.array_equal(got_off, poff))
    res["rows_bit_identical_to_pcl_order"] = float(np.mean(np.all(got_xyz == prec[:, :3], axis=1))) if rows else 1.0
    res["speedup_call_vs_cpu_oracle"] = res["cpu_oracle_pcl_order_s"] * 1e3 / res["call_ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "voxel_perf_b200.json"))
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--quick", action="store_true", help="small clouds (a rehearsal, not a measurement)")
    a = ap.parse_args()
    sizes = [1_000_000, 5_000_000, 20_000_000]
    if a.quick:
        sizes = [s // 100 for s in sizes]
    info = gpu_info()
    ctx = api.Context(0)
    result = dict(info, calls=a.calls, warmup=a.warmup, configs={})
    for n in sizes:
        for density in (16.0, 64.0):
            cloud = synth.panel(n, seed=31, density=density)
            gc = api.Cloud(ctx, cloud)
            for leaf in (0.5, 1.0):
                name = "panel_%dk_density%d_leaf%g" % (n // 1000, density, leaf)
                result["configs"][name] = r = measure(ctx, gc, cloud, leaf, a.calls, a.warmup)
                print(name, json.dumps(r), flush=True)
            gc.close()
    ctx.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
