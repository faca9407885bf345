#!/usr/bin/env python
"""MLS smooth() of one cloud over several GPUs (run under torchrun, one rank per GPU), against one GPU in the same run.

The cloud starts in ONE host buffer every rank has mapped (parallel.SharedHost, as bench.py --gpus N does).  Per step:
exchange into x-slabs with the MLS halo (parallel.mls_halo) -> every rank smooths the points it owns and stores each
record into its home rank over NVLink -> the home ranks compact their index ranges (parallel.mls_smooth_sharded).
Two modes:
  device  the chunks are already in HBM, every rank's rows end in a device buffer of its own;
  e2e     every rank copies its chunk from the shared host buffer, the rows of all ranks end in ONE shared host buffer.
Rank 0 also times the one-GPU form of each mode on the whole cloud: device = ppp_dev_cloud_attach + ppp_dev_mls_smooth
+ ppp_dev_mls_compact; e2e = ppp_cloud_upload + ppp_mls_smooth.  Both include the index build, as the sharded step does.
Step times are host clocks around a step that ends in a device synchronise and a barrier (median over --steps after
--warmup).  A separate set of steps with ppp_kernel_profile on gives every rank's kernel time and its exchange share.
--check compares the assembled result of each mode with one GPU's ppp_mls_smooth of the whole cloud on rank 0 (rows
identical, x, y, z within 2 float32 ulps with >= 99 % bit-identical, normals within 1e-5) and prints one line each.

    torchrun --nproc-per-node 8 tools/mls_multi.py [--sizes 1000000,5000000,10000000] [--steps 10] [--warmup 2]
             [--check] [--out profiles/mls_multi_8gpu.json]   (--out "": no file)

Without torchrun, --ranks-on-one-gpu W puts W ranks on GPU 0 (Exchange.connect_local) and runs each rank's
ppp_dev_mls_smooth alone on the whole GPU (a synchronise between ranks): its kernel time is what that rank's kernel
takes on a GPU of its own.  The NVLink stores of the records and the exchange are not in it.

    python tools/mls_multi.py --ranks-on-one-gpu 8 [--sizes ...] [--out profiles/mls_multi_ranks8_on_1gpu.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from polishpathplanning_b200 import api, parallel, synth  # noqa: E402

R, ORDER, REC = 15.0, 3, 32


def gpu_info():
    from mls_perf import gpu_info as info
    return info()


def contract(pts, src, nrm, ref):
    """(ok, fraction of rows with bit-identical x, y, z) against Cloud.mls_smooth's (points, src_index, normals)."""
    rpts, rsrc, rnrm = ref
    if not (np.array_equal(src, rsrc) and np.array_equal(pts[:, 3:].view(np.uint32), rpts[:, 3:].view(np.uint32))):
        return False, 0.0
    if src.shape[0] == 0:
        return True, 1.0
    ulps = np.abs(pts[:, 0:3].astype(np.float64) - rpts[:, 0:3]) / np.spacing(np.maximum(np.abs(pts[:, 0:3]), np.abs(rpts[:, 0:3])))
    same = float(np.mean(np.all(pts[:, 0:3] == rpts[:, 0:3], axis=1)))
    return bool(ulps.max() <= 2.0 and same >= 0.99 and np.abs(nrm - rnrm).max() <= 1e-5), same


def timed(fn, steps, warmup, barrier):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        barrier()
        t0 = time.perf_counter()
        fn()
        barrier()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def one_gpu(ctx, cloud, dev, steps, warmup):
    """Rank 0: the one-GPU form of both modes on the whole cloud."""
    n = cloud.shape[0]
    chunk = torch.from_numpy(cloud).to(dev)
    recs = torch.empty((n, 8), dtype=torch.float32, device=dev)
    pts = torch.empty((n, 8), dtype=torch.float32, device=dev)
    nrm = torch.empty((n, 4), dtype=torch.float32, device=dev)
    src = torch.empty(n, dtype=torch.int32, device=dev)

    def device_step():
        gc = api.Cloud(ctx, device_ptr=chunk.data_ptr(), n=n, stride_bytes=REC)
        gc.dev_mls_smooth(R, ORDER, recs.data_ptr())
        ctx.dev_mls_compact(recs.data_ptr(), n, chunk.data_ptr(), REC, 0, 0, pts.data_ptr(), REC, nrm.data_ptr(), src.data_ptr(), n)
        gc.close()
        ctx.sync()

    hpts = ctx.pinned_empty((n, 8), np.float32)
    hnrm = ctx.pinned_empty((n, 4), np.float32)
    hsrc = ctx.pinned_empty((n,), np.int32)
    m = C.c_int64(0)

    def e2e_step():
        gc = api.Cloud(ctx, cloud)
        api.check(ctx.lib.ppp_mls_smooth(gc._h, R, ORDER, hpts.ctypes.data, REC, hnrm.ctypes.data, hsrc.ctypes.data, C.byref(m)))
        gc.close()

    nobar = lambda: None  # noqa: E731
    res = {"device": timed(device_step, steps, warmup, nobar), "e2e": timed(e2e_step, steps, warmup, nobar)}
    ctx.kernel_profile(True)
    ctx.kernel_profile_read(reset=True)
    device_step()
    res["device_kernels"] = ctx.kernel_profile_read(reset=True)
    ctx.kernel_profile(False)
    gc = api.Cloud(ctx, cloud)
    ref = gc.mls_smooth(R, ORDER, normals=True)
    gc.close()
    del chunk, recs, pts, nrm, src
    return res, ref


def ranks_on_one_gpu(world, sizes, calls, out_path):
    out = dict(gpu_info(), radius=R, order=ORDER, ranks=world, calls=calls, sizes={})
    for n in sizes:
        cloud = synth.panel(n, seed=51, noise_sigma=0.05)
        starts = parallel.index_ranges(n, world)
        halo = parallel.mls_halo(R, float(np.abs(cloud[:, 0]).max()))
        ctxs = [api.Context(0) for _ in range(world)]
        exs = [parallel.Exchange(ctxs[r], r, world, starts, int(n / world * 1.5) + 65536, 1, 1024, REC) for r in range(world)]
        parallel.Exchange.connect_local(exs)
        chunks = [torch.from_numpy(cloud[starts[r]:starts[r + 1]]).to("cuda:0") for r in range(world)]
        torch.cuda.synchronize()
        for p in range(4):
            for ex, ch in zip(exs, chunks):
                ex.phase(p, ch.data_ptr(), ch.shape[0], REC, halo)
        both = [ex.finish_attach(to_rank0=False) for ex in exs]
        per_rank = []
        for r in range(world):
            c = both[r][1]
            c.dev_mls_smooth(R, ORDER)              # warm-up (index build)
            ctxs[r].sync()
            ctxs[r].kernel_profile(True)
            ctxs[r].kernel_profile_read(reset=True)
            for _ in range(calls):
                c.dev_mls_smooth(R, ORDER)
            ctxs[r].sync()
            prof = ctxs[r].kernel_profile_read(reset=True)
            ctxs[r].kernel_profile(False)
            per_rank.append(dict(n_local=both[r][0]["n_local"], n_owned=both[r][0]["n_owned"],
                                 mls_kernel_ms=sum(ms for k, (ms, _) in prof.items() if k.startswith("mls_")) / calls))
        for ex in exs:
            ex.results_signal(ex.NORMALS)
        for ex in exs:
            ex.results_wait(ex.NORMALS)
        for c in ctxs:
            c.sync()
        gc = api.Cloud(ctxs[0], cloud)
        gc.dev_index(radius_hint=R)
        recs = torch.empty((n, 8), dtype=torch.float32, device="cuda:0")
        gc.dev_mls_smooth(R, ORDER, recs.data_ptr())
        ctxs[0].sync()
        ctxs[0].kernel_profile(True)
        ctxs[0].kernel_profile_read(reset=True)
        for _ in range(calls):
            gc.dev_mls_smooth(R, ORDER, recs.data_ptr())
        ctxs[0].sync()
        prof = ctxs[0].kernel_profile_read(reset=True)
        ctxs[0].kernel_profile(False)
        one = sum(ms for k, (ms, _) in prof.items() if k.startswith("mls_")) / calls
        slowest = max(p["mls_kernel_ms"] for p in per_rank)
        out["sizes"][str(n)] = dict(one_gpu_mls_kernel_ms=one, per_rank=per_rank, slowest_rank_mls_kernel_ms=slowest,
                                    kernel_ratio=slowest / one)
        print("MLS_RANKS_ON_ONE_GPU ranks=%d n=%d one_gpu %.2f ms slowest rank %.2f ms (%.3f of one GPU) halo rows %d" % (
            world, n, one, slowest, slowest / one, sum(p["n_local"] - p["n_owned"] for p in per_rank)), flush=True)
        gc.close()
        for b in both:
            b[1].close()
        for ex in exs:
            ex.close()
        for c in ctxs:
            c.close()
        del chunks, recs
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(out, f, indent=1)
        print("wrote", out_path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,5000000,10000000")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--out", default=None)
    ap.add_argument("--ranks-on-one-gpu", type=int, default=0)
    a = ap.parse_args()
    if a.ranks_on_one_gpu:
        ranks_on_one_gpu(a.ranks_on_one_gpu, [int(v) for v in a.sizes.split(",")], a.steps,
                         a.out if a.out is not None else os.path.join(ROOT, "profiles", "mls_multi_ranks%d_on_1gpu.json" % a.ranks_on_one_gpu))
        return
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dev = torch.device("cuda", lr)
    dist.init_process_group("nccl", device_id=dev)
    barrier = dist.barrier
    ctx = api.Context(lr)
    out = dict(radius=R, order=ORDER, world=world, steps=a.steps, warmup=a.warmup, noise_sigma_mm=0.05, sizes={})
    if rank == 0:
        out.update(gpu_info())
    ok_all = True
    for n in (int(s) for s in a.sizes.split(",")):
        sh_in = parallel.SharedHost(dist, rank, world, n * REC, "mls_in_%d" % n, ctx=ctx)
        if rank == 0:
            sh_in.array(np.float32, (n, 8))[:] = synth.panel(n, seed=51, noise_sigma=0.05)
        barrier()
        cloud = sh_in.array(np.float32, (n, 8))
        fin = np.isfinite(cloud[:, :3]).all(axis=1)
        halo = parallel.mls_halo(R, float(np.abs(cloud[fin, 0]).max()))
        starts = parallel.index_ranges(n, world)
        lo, hi = int(starts[rank]), int(starts[rank + 1])
        ex = parallel.Exchange.over_dist(ctx, dist, dev, rank, world, n, int((hi - lo) * 1.5) + 65536, 1, 1024, REC)
        chunk = torch.from_numpy(cloud[lo:hi]).to(dev)
        d_pts = torch.empty((hi - lo, 8), dtype=torch.float32, device=dev)
        d_nrm = torch.empty((hi - lo, 4), dtype=torch.float32, device=dev)
        d_src = torch.empty(hi - lo, dtype=torch.int32, device=dev)
        dev_out = (d_pts.data_ptr(), d_nrm.data_ptr(), d_src.data_ptr(), hi - lo, False)
        lay = [n * REC, n * 16, n * 4]
        sh_out = parallel.SharedHost(dist, rank, world, sum(lay), "mls_out_%d" % n, ctx=ctx)
        host_out = (sh_out.dev_base, sh_out.dev_base + lay[0], sh_out.dev_base + lay[0] + lay[1], n, True)
        last = {}

        def device_step():
            last["counts"], last["bases"] = parallel.mls_smooth_sharded([ex], [chunk.data_ptr()], REC, R, ORDER, halo, [dev_out], dist, dev)
            ctx.sync()

        def e2e_step():
            ctx.upload(chunk.data_ptr(), sh_in.host_base + lo * REC, (hi - lo) * REC)
            last["counts"], last["bases"] = parallel.mls_smooth_sharded([ex], [chunk.data_ptr()], REC, R, ORDER, halo, [host_out], dist, dev)
            ctx.sync()

        cell = dict(points=n, halo=halo)
        for mode, fn in (("device", device_step), ("e2e", e2e_step)):
            med, mn, mx = timed(fn, a.steps, a.warmup, barrier)
            ctx.kernel_profile(True)
            ctx.kernel_profile_read(reset=True)
            fn()
            prof = ctx.kernel_profile_read(reset=True)
            ctx.kernel_profile(False)
            ex.check()
            profs = [None] * world
            dist.all_gather_object(profs, prof)
            per_rank = []
            for p in profs:
                k_ms = sum(ms for ms, _ in p.values())
                ex_ms = sum(ms for name, (ms, _) in p.items() if name.startswith("ex_"))
                mls_ms = sum(ms for name, (ms, _) in p.items() if name.startswith("mls_"))
                per_rank.append(dict(kernel_ms=k_ms, exchange_ms=ex_ms, exchange_share=ex_ms / k_ms if k_ms else 0.0,
                                     mls_ms=mls_ms, kernels=p))
            cell[mode] = dict(step_ms_median=med, step_ms_min=mn, step_ms_max=mx, rows=int(sum(last["counts"])),
                              rank_rows=[int(c) for c in last["counts"]], per_rank=per_rank)
            if mode == "device" and a.check:   # the rows of every rank into the shared host buffer, for the check below
                c = int(last["counts"][rank])
                b = int(last["bases"][rank])
                sh_out.array(np.float32, (n, 8))[b:b + c] = d_pts[:c].cpu().numpy()
                sh_out.array(np.float32, (n, 4), lay[0])[b:b + c] = d_nrm[:c].cpu().numpy()
                sh_out.array(np.int32, (n,), lay[0] + lay[1])[b:b + c] = d_src[:c].cpu().numpy()
                barrier()
            if a.check and mode == "device":
                cell["_device_rows"] = [x.copy() for x in (sh_out.array(np.float32, (n, 8)), sh_out.array(np.float32, (n, 4), lay[0]),
                                                            sh_out.array(np.int32, (n,), lay[0] + lay[1]))] if rank == 0 else None
        barrier()
        if rank == 0:
            single, ref = one_gpu(ctx, np.ascontiguousarray(cloud), dev, a.steps, a.warmup)
            cell["one_gpu"] = dict(device_step_ms_median=single["device"][0], e2e_step_ms_median=single["e2e"][0],
                                   device_kernels=single["device_kernels"],
                                   mls_kernel_ms=sum(ms for k, (ms, _) in single["device_kernels"].items() if k.startswith("mls_")))
            for mode in ("device", "e2e"):
                cell[mode]["speedup_vs_one_gpu"] = single[mode][0] / cell[mode]["step_ms_median"]
            if a.check:
                m = ref[1].shape[0]
                for mode in ("device", "e2e"):
                    if mode == "device":
                        p, nr, s = cell["_device_rows"]
                    else:
                        p, nr, s = (sh_out.array(np.float32, (n, 8)), sh_out.array(np.float32, (n, 4), lay[0]),
                                    sh_out.array(np.int32, (n,), lay[0] + lay[1]))
                    ok = cell[mode]["rows"] == m
                    same = 0.0
                    if ok:
                        ok, same = contract(p[:m], s[:m], nr[:m], ref)
                    cell[mode].update(check=bool(ok), bit_identical=same)
                    ok_all = ok_all and ok
                    print("MLS_MULTI_CHECK world=%d n=%d mode=%s rows=%d check=%s bit_identical=%.6f" % (world, n, mode, m, ok, same),
                          flush=True)
            cell.pop("_device_rows", None)
            out["sizes"][str(n)] = cell
            print("MLS_MULTI world=%d n=%d one_gpu device %.2f ms e2e %.2f ms | sharded device %.2f ms e2e %.2f ms" % (
                world, n, single["device"][0], single["e2e"][0], cell["device"]["step_ms_median"], cell["e2e"]["step_ms_median"]),
                flush=True)
        barrier()
        del chunk, d_pts, d_nrm, d_src
        ex.close(dist)
        sh_out.close()
        sh_in.close()
    flag = torch.tensor([1 if ok_all else 0], device=dev)
    dist.broadcast(flag, 0)
    if rank == 0:
        out["gpu_after"] = gpu_info()
        path = a.out if a.out is not None else os.path.join(ROOT, "profiles", "mls_multi_%dgpu.json" % world)
        if path:
            os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
            with open(path, "w") as f:
                json.dump(out, f, indent=1)
            print("wrote", path)
    barrier()
    dist.destroy_process_group()
    ctx.close()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
