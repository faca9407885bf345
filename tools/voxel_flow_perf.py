#!/usr/bin/env python
"""Measures what keeping voxel_down()'s rows in device memory saves: for panels of 5M and 20M points at densities 16
and 64 points/mm^2 with leaves of 0.5 and 1.0 mm (PointXYZRGB records, 32 bytes, random colours), the wall time of

  host flow:    Cloud.voxel_grid on a host-uploaded cloud (ppp_voxel_grid into host records, colours averaged on the
                host) + ppp_cloud_upload of the rows -> the next cloud;
  device flow:  ppp_dev_voxel_grid on the same records attached from device memory (whole records, colours included,
                written into a device buffer) + ppp_dev_cloud_attach of the rows -> the next cloud;

each ending in a synchronise, alternated call by call, medians over --calls after --warmup.  The device flow's kernel
time (ppp_kernel_profile) is recorded too.  Both flows' records are compared bit for bit in the same run, and the bytes
the host flow moves over PCIe are counted from the shapes (rows, offsets and members down, rows up).  The GPU's name and
power limit are read (nvidia-smi --query-gpu, read only) in the same run.

    python tools/voxel_flow_perf.py [--out profiles/voxel_flow_b200.json] [--calls 10] [--warmup 2] [--quick]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from polishpathplanning_b200 import api, synth  # noqa: E402
from voxel_perf import gpu_info  # noqa: E402


def measure(ctx, cloud, leaf, calls, warmup):
    import torch
    n, sf = cloud.shape
    stride = sf * 4
    hc = api.Cloud(ctx, cloud)
    src = torch.from_numpy(cloud).to("cuda:0")
    rows = torch.empty((n, sf), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    dc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=n, stride_bytes=stride)

    def host_flow():
        t0 = time.perf_counter()
        rec, off, mem = hc.voxel_grid(leaf)
        nxt = api.Cloud(ctx, rec)
        ctx.sync()
        t = (time.perf_counter() - t0) * 1e3
        nxt.close()
        return t, rec, off, mem

    def device_flow():
        t0 = time.perf_counter()
        m = dc.dev_voxel_grid(leaf, rows.data_ptr(), stride)
        nxt = api.Cloud(ctx, device_ptr=rows.data_ptr(), n=m, stride_bytes=stride)
        ctx.sync()
        t = (time.perf_counter() - t0) * 1e3
        nxt.close()
        return t, m

    for _ in range(warmup):
        host_flow()
        device_flow()
    host_ms, dev_ms = [], []
    for _ in range(calls):
        t, rec, off, mem = host_flow()
        host_ms.append(t)
        t, m = device_flow()
        dev_ms.append(t)
    ctx.kernel_profile(True)
    ctx.kernel_profile_read(reset=True)
    for _ in range(calls):
        dc.dev_voxel_grid(leaf, rows.data_ptr(), stride)
    prof = ctx.kernel_profile_read(reset=True)
    ctx.kernel_profile(False)
    got = rows[:m].cpu().numpy()
    hc.close()
    dc.close()
    res = dict(
        points=n, leaf=leaf, rows=m, stride_bytes=stride,
        host_flow_ms_median=float(np.median(host_ms)), host_flow_ms_min=float(np.min(host_ms)),
        device_flow_ms_median=float(np.median(dev_ms)), device_flow_ms_min=float(np.min(dev_ms)),
        device_kernels_ms=sum(ms for ms, _ in prof.values()) / calls,
        kernels={k: dict(ms_per_call=v[0] / calls, launches_per_call=v[1] / calls) for k, v in prof.items()},
        host_flow_pcie_bytes=int(m * stride * 2 + (m + 1) * 8 + int(off[-1]) * 4),
        records_bit_identical=bool(m == rec.shape[0] and np.array_equal(got.view(np.uint32), rec.view(np.uint32))),
    )
    res["speedup_device_vs_host_flow"] = res["host_flow_ms_median"] / res["device_flow_ms_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "voxel_flow_b200.json"))
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--quick", action="store_true", help="small clouds (a rehearsal, not a measurement)")
    a = ap.parse_args()
    sizes = [5_000_000, 20_000_000]
    if a.quick:
        sizes = [s // 100 for s in sizes]
    info = gpu_info()
    ctx = api.Context(0)
    result = dict(info, calls=a.calls, warmup=a.warmup, configs={})
    ok = True
    for n in sizes:
        for density in (16.0, 64.0):
            cloud = synth.panel(n, seed=31, density=density)
            cloud[:, 4] = np.random.default_rng(32).integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32).view(np.float32)
            for leaf in (0.5, 1.0):
                name = "panel_%dk_density%d_leaf%g" % (n // 1000, density, leaf)
                result["configs"][name] = r = measure(ctx, cloud, leaf, a.calls, a.warmup)
                ok &= r["records_bit_identical"]
                print(name, json.dumps({k: v for k, v in r.items() if k != "kernels"}), flush=True)
    ctx.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", a.out)
    if not ok:
        sys.exit("device and host flows differ")


if __name__ == "__main__":
    main()
