#!/usr/bin/env python
"""Times ppp_knn with a query array (queries that are not the cloud's own points in cell order) and compares two
builds of libppp_gpu.so on it.  Per cloud, query set and k it records the device time of the search kernels per
call (ppp_kernel_profile, CUDA events around each launch: the fixed-block "knn" kernel plus the one-warp-per-query
"knn_redo" hand-over kernel, after warm-up) and a hash of the index and d2 bits of the result.

Clouds: 1M-point panel, closed cylinder and box with walls (synth.py).  Query sets: 100k points of the cloud in
random order, and 10k drawpath-like slice samples (ten planes x = const across the cloud, each sampled at 1000 y
positions with z interpolated along the band |x - plane| < 2).  k = 1, 10, 16, 32, 50, 64.

Each library runs in a worker process of its own (PPP_GPU_LIB), the libraries alternate over the rounds, and the
parent process asserts that every library returned the same bits for every case.  The GPU's name and power limit
are read (nvidia-smi --query-gpu, read only) in the same run.

    python tools/knn_query_perf.py --lib A.so [--lib B.so ...] [--rounds 3] [--calls 20] [--warmup 3] [--out F.json]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KS = [1, 10, 16, 32, 50, 64]
N_POINTS = 1_000_000
N_RANDOM = 100_000
N_PLANES, N_PER_PLANE = 10, 1000


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return dict(gpu_name=name, power_limit=power, max_sm_clock=clock)


def clouds(n):
    from polishpathplanning_b200 import synth
    return {"panel": synth.panel(n, seed=41), "cylinder": synth.cylinder(n, seed=42),
            "box_with_walls": synth.box_with_walls(n, seed=43)}


def slice_samples(p, planes, per_plane):
    """drawpath-like way-points: per plane x = xc, the band |x - xc| < 2 sorted by y, z interpolated at even y steps."""
    lo, hi = p[:, 0].min(), p[:, 0].max()
    out = []
    for xc in np.linspace(lo, hi, planes + 2)[1:-1]:
        band = p[np.abs(p[:, 0] - xc) < 2]
        band = band[np.argsort(band[:, 1], kind="stable")]
        y = np.linspace(band[0, 1], band[-1, 1], per_plane)
        out.append(np.stack([np.full(per_plane, xc), y, np.interp(y, band[:, 1], band[:, 2])], axis=1))
    return np.concatenate(out).astype(np.float32)


def query_sets(cloud, n_random, planes, per_plane, seed=44):
    p = cloud[:, :3]
    rng = np.random.default_rng(seed)
    return {"random_on_surface": np.ascontiguousarray(p[rng.choice(p.shape[0], n_random, replace=False)]),
            "slice_samples": slice_samples(p, planes, per_plane)}


def worker(a):
    """One library (PPP_GPU_LIB): every case, timings and result hashes as one JSON line on stdout."""
    from polishpathplanning_b200 import api
    ctx = api.Context(0)
    res = {}
    n_random, per_plane = (N_RANDOM // 100, N_PER_PLANE // 100) if a.quick else (N_RANDOM, N_PER_PLANE)
    for cname, cloud in clouds(N_POINTS // 100 if a.quick else N_POINTS).items():
        gc = api.Cloud(ctx, cloud)
        for qname, q in query_sets(cloud, n_random, N_PLANES, per_plane).items():
            for k in KS:
                for _ in range(a.warmup):
                    gc.knn(k, q)
                ctx.kernel_profile(True)
                ctx.kernel_profile_read(reset=True)
                for _ in range(a.calls):
                    idx, d2 = gc.knn(k, q)
                prof = ctx.kernel_profile_read(reset=True)
                ctx.kernel_profile(False)
                h = hashlib.sha256(idx.tobytes())
                h.update(d2.view(np.uint32).tobytes())
                ms = {name: prof.get(name, (0.0, 0))[0] / a.calls for name in ("knn", "knn_redo")}
                res["%s/%s/k%d" % (cname, qname, k)] = dict(
                    queries=int(q.shape[0]), knn_ms=ms["knn"], knn_redo_ms=ms["knn_redo"],
                    search_ms=ms["knn"] + ms["knn_redo"], sha256=h.hexdigest())
        gc.close()
    ctx.close()
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="a libppp_gpu.so to measure (repeat to compare)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="knn_query_perf.json")
    ap.add_argument("--quick", action="store_true", help="clouds and query sets 100x smaller (a rehearsal)")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    libs = [os.path.abspath(p) for p in a.lib]
    if not libs:
        ap.error("--lib is required")
    info = gpu_info()
    runs = {lib: [] for lib in libs}
    for r in range(a.rounds):
        for lib in (libs if r % 2 == 0 else libs[::-1]):   # alternate which library goes first
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--calls", str(a.calls), "--warmup", str(a.warmup)]
            out = subprocess.run(cmd + (["--quick"] if a.quick else []), env=dict(os.environ, PPP_GPU_LIB=lib),
                                 capture_output=True, text=True, check=True).stdout
            runs[lib].append(json.loads(out.strip().splitlines()[-1]))
            print("round %d %s done" % (r, lib), flush=True)
    cases = sorted(runs[libs[0]][0])
    mismatches = [c for c in cases if len({run[c]["sha256"] for lib in libs for run in runs[lib]}) != 1]
    table = {}
    for c in cases:
        row = table[c] = {"queries": runs[libs[0]][0][c]["queries"]}
        for i, lib in enumerate(libs):
            t = [run[c]["search_ms"] for run in runs[lib]]
            row["lib%d" % i] = dict(search_ms=t, search_ms_min=min(t),
                                    knn_ms=[run[c]["knn_ms"] for run in runs[lib]],
                                    knn_redo_ms=[run[c]["knn_redo_ms"] for run in runs[lib]])
        if len(libs) > 1:
            row["ratio_min_lib1_over_lib0"] = row["lib1"]["search_ms_min"] / row["lib0"]["search_ms_min"]
        print("%-40s %s" % (c, "  ".join("%.4f" % row["lib%d" % i]["search_ms_min"] for i in range(len(libs)))), flush=True)
    result = dict(info, libs={"lib%d" % i: os.path.relpath(lib, ROOT) for i, lib in enumerate(libs)},
                  rounds=a.rounds, calls=a.calls, warmup=a.warmup, ks=KS, quick=a.quick,
                  identical_bits=not mismatches, mismatches=mismatches, cases=table, gpu_after=gpu_info())
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)
    if mismatches:
        sys.exit("results differ between the libraries: %s" % mismatches)


if __name__ == "__main__":
    main()
