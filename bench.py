#!/usr/bin/env python
"""bench.py — points/sec through kNN(k=16) + PCA normals + plane slicing + ordered contours.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg3] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 1M-point synthetic freeform panel per GPU, k=16 normals +
200*sqrt(N) slices (5 mm apart, band +-2 mm, SectPath pairing); weak scaling: the ONE cloud has N x 1M
points.  One "step" = one pass of the hot path over that cloud, starting from the raw
pcl::PointXYZRGB records.

  N = 1   pack + bounding box, grid index, fused kNN + normals (neighbour ids and normals written),
          bands of all planes, per-slice pairing + interpolation + ordering.
  N > 1   (torchrun, one rank per GPU) the cloud starts split by ORIGINAL INDEX; inside the step:
          partition + halo exchange (csrc/exchange.cu: NVLink stores, no NCCL on the data path), the N = 1
          path on every slab, every normal record delivered to the rank that holds its original index
          range, contour nodes to rank 0.

  value : device-resident (records already in HBM, results left in HBM), CUDA-event timed on the
          library's stream, max over ranks.
  e2e   : the same step from ONE host buffer to ONE host result: the cloud lives in a host buffer every
          rank has mapped (shared memory, page-locked), rank r moves the records of its index range over
          its own PCIe link, and the normals (original order) + contour nodes end up in one host buffer
          that a Spline consumer on rank 0 reads.  H2D and D2H inside the timed region; wall clock
          between barriers, max over ranks.  The neighbour-id lists (64 B / point) stay in HBM in both
          arms: estimate_normal() returns normals only.
  roofline : dominant kernel's algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json.
  cpu_baseline / --impl reference : the CPU oracle (port of the reference's PCL/FLANN path; the
          reference itself cannot be built here, see DESIGN.md) on the box's host cores.
  --dump-outputs DIR (one GPU) : after the timed steps, what the last of them computed, as DIR/<name>.npy
          (float32 / float64, integers stored exactly): normals (pcl::Normal records), neighbour_ids,
          contour_offsets (per plane) and contour_y / _x / _z.  An output with more rows than DUMP_ROWS allows
          is written as a fixed seeded sample of rows, their indices in <name>_rows.npy.  The inputs depend on
          the arguments only, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # the tree bench.py runs from may be read-only: nothing is written there
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "points/sec kNN(k=16)+normals+slicing"
UNIT = "points/s"
HALF_WIDTH = 2.0
HALO_MM = 12.0
SETTLE_STEPS = 10         # untimed steps in front of the W warm-up steps (see timed_device_steps)
PAIRING = "B"             # SectPath::insert_point (src/contour_alg.cpp:165-237)
CPU_SAMPLE_MAX = 2_000_000   # --impl reference: points of the workload one CPU step processes
# --dump-outputs: rows written per output before it is sampled, so that every configuration stays under
# DUMP_MAX_BYTES (cfg2 on one GPU is written whole except for the neighbour ids)
DUMP_ROWS = {"normals": 1 << 20, "neighbour_ids": 1 << 15, "contour": 1 << 18}
DUMP_MAX_BYTES = 64_000_000


def make_cfg(name, gpus):
    """The workload as a function of the configuration name and the GPU count only (both arms print it)."""
    gpus = max(int(gpus), 1)
    if name == "cfg3":   # SURVEY 8d / BASELINE configs[2]: 10M points in TOTAL, k = 32, 1000 planes
        n_total, k, S = 10_000_000, 32, 1000
        text = ("cfg3: %d-point synthetic freeform panel in total (seed 0, 1 pt/mm^2), k=%d normals + %d evenly spaced "
                "slices (+-2 mm bands, SectPath pairing)" % (n_total, k, S))
        scaling = "strong"
    else:
        n_total, k = 1_000_000 * gpus, 16
        S = int(round(200 * np.sqrt(gpus)))
        text = ("cfg2: %d-point synthetic freeform panel per GPU (one cloud of %d points, seed 0, 1 pt/mm^2), k=%d normals + "
                "%d slices (5 mm spacing, +-2 mm bands, SectPath pairing)" % (1_000_000, n_total, k, S))
        scaling = "weak"
    return {"name": name, "n_total": n_total, "k": k, "S": S, "text": text, "scaling": scaling, "gpus": gpus}


def workload_config(cfg):
    g = cfg["gpus"]
    return {"workload": cfg["text"], "points_total": cfg["n_total"], "points_per_gpu": cfg["n_total"] // g, "k": cfg["k"],
            "slices_total": cfg["S"], "pairing": "B(SectPath)",
            "partition": ("single GPU" if g == 1 else
                          "cloud split by original index; x-slabs + %g mm halo exchanged inside the step (NVLink stores); "
                          "normals to their index-range owner, contours to rank 0" % HALO_MM),
            "result": "normals in original order + contour nodes per plane; neighbour-id lists stay in HBM",
            "l2": "flushed between timed steps (256 MiB write + 256 MiB read)"}


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self.proc = None
        self.thr = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 8:
                self.samples.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for p in self.samples:
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_planes(x_min, x_max, S):
    step = (float(x_max) - float(x_min)) / S
    return (float(x_min) + step * (np.arange(S) + 0.5)).astype(np.float32)


def host_threads():
    """Host cores this process may use, whatever OMP_NUM_THREADS says (torchrun exports 1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference's CPU path)
# ------------------------------------------------------------------------------------------------
def cpu_step(po, cloud, planes, k, threads):
    oc = po.OracleCloud(cloud)                      # kd-tree build  (Set_kdtree)
    oc.normals(k=k, threads=threads)                # estimate_normal (k-search variant)
    oc.slice_contours(planes, PAIRING, HALF_WIDTH, True, threads=threads)  # rangedX_index + insert_point + ordering
    oc.close()


def cpu_sample(cfg):
    """A bounded sample of the workload: the x-slab holding the first CPU_SAMPLE_MAX points (all of them if
    the cloud is smaller) with the planes whose bands lie inside it."""
    from polishpathplanning_b200 import synth
    cloud = synth.panel(cfg["n_total"], seed=0)
    planes = make_planes(cloud[:, 0].min(), cloud[:, 0].max(), cfg["S"])
    if cfg["n_total"] > CPU_SAMPLE_MAX:
        x_cut = float(np.partition(cloud[:, 0], CPU_SAMPLE_MAX)[CPU_SAMPLE_MAX])
        cloud = np.ascontiguousarray(cloud[cloud[:, 0] < x_cut])
        planes = planes[planes < x_cut - HALO_MM]
        what = ("the x < %.1f mm slab of the %d-point cloud: %d points, %d of the %d slices" %
                (x_cut, cfg["n_total"], cloud.shape[0], len(planes), cfg["S"]))
    else:
        what = "the full workload: %d points, %d slices" % (cloud.shape[0], len(planes))
    return cloud, planes, what


def cpu_baseline(cfg, threads):
    from oracle import ppp_oracle as po
    cloud, planes, what = cpu_sample(cfg)
    t0 = time.perf_counter()
    cpu_step(po, cloud, planes, cfg["k"], threads)
    dt = time.perf_counter() - t0
    return cloud.shape[0] / dt, dt, what


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ppp_oracle as po
    cfg = make_cfg(args.config, args.gpus)
    cloud, planes, what = cpu_sample(cfg)
    cores = host_threads()
    for _ in range(args.warmup):
        cpu_step(po, cloud, planes, cfg["k"], cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(po, cloud, planes, cfg["k"], cores)
    dt = time.perf_counter() - t0
    v = cloud.shape[0] * args.steps / dt
    sample = ("oracle port of the reference CPU path (kd-tree build, k=%d normals, slicing pairing %s); each step processes %s; "
              "OpenMP over points / slices with %d threads (the kd-tree build is single-threaded)" % (cfg["k"], PAIRING, what, cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Env:
    """Process-wide handles shared by the measurements."""

    def __init__(self, args):
        import torch
        from polishpathplanning_b200 import api
        self.torch = torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun with %d ranks (python -m torch.distributed.run ...)" % (args.gpus, args.gpus))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group(backend="nccl", device_id=self.dev)
            self.dist = dist
        self.ctx = api.Context(self.local_rank)
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)
        with torch.cuda.stream(self.stream):
            self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)
            self.flush_rd = torch.zeros(64 << 20, dtype=torch.int32, device=self.dev)
        self.stream.synchronize()

    def sync_all(self):
        self.stream.synchronize()
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def flush_l2(self):
        # write 256 MiB (evicts everything), then read another 256 MiB so that the lines left in
        # L2 are clean: otherwise the first timed kernel pays for writing the flush buffer back
        with self.torch.cuda.stream(self.stream):
            self.flush.zero_()
            self.flush_rd.sum()

    def max_over_ranks(self, v):
        if self.dist is None:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()
        self.ctx.close()


def timed_device_steps(env, step, steps, warmup, last_step=None):
    """W warm-up + K timed steps, each behind an L2 flush; CUDA events on the library's stream.
    last_step: run in place of step for the last timed step (one that keeps its outputs readable)."""
    ctx = env.ctx
    # settle first: the first steps of a process see one-off costs (memory pools growing to their working size, lazy
    # module loads, clocks leaving idle) that have shown up as single steps of tens of milliseconds; then the W warm-ups
    for _ in range(SETTLE_STEPS):
        step()
    for _ in range(warmup):
        env.flush_l2(); step()
    env.sync_all()
    ctx.timer_read(0, reset=True)
    ctx.timer_read(1, reset=True)
    l0 = ctx.launch_count()
    env.sync_all()
    t_wall0 = time.perf_counter()
    for i in range(steps):
        env.flush_l2()
        env.stream.synchronize()
        ctx.timer_begin(0)
        (last_step if last_step is not None and i == steps - 1 else step)()
        ctx.timer_end(0)
    env.sync_all()
    t_wall = time.perf_counter() - t_wall0
    total_ms, regions = ctx.timer_read(0, reset=True)
    assert regions == steps
    launches = ctx.launch_count() - l0
    return env.max_over_ranks(total_ms), total_ms, launches, t_wall


def kernel_profile(env, step, steps):
    ctx = env.ctx
    ctx.kernel_profile(True)
    ctx.kernel_profile_read(reset=True)
    for _ in range(steps):
        env.flush_l2()
        step()
    env.sync_all()
    prof = ctx.kernel_profile_read(reset=True)
    ctx.kernel_profile(False)
    return prof


def roofline_of(prof, steps, n_local, k, members, nodes):
    peak, peak_src = read_peaks()
    work = {kk: v for kk, v in prof.items() if not kk.startswith("ex_wait")}
    if not work:
        return None
    dom_name, (dom_ms, dom_launches) = max(work.items(), key=lambda kv: kv[1][0])
    alg_bytes = {
        "knn_normals": n_local * (32 + 4 * k),   # 16 B point in + 4k B ids + 16 B normal out (SURVEY §8d)
        "knn": n_local * (16 + 4 * k),
        "pair_nodes": 16 * members + 16 * nodes,
        "contour": 16 * members + 24 * nodes,
        "band_count": 16 * n_local, "band_fill": 16 * n_local + 4 * members,
        "pack_bbox": 12 * n_local + 16 * n_local,
        "cell_count": 16 * n_local, "cell_scatter": 16 * n_local + 20 * n_local,
    }.get(dom_name)
    if not alg_bytes or not dom_launches:
        return None
    achieved = alg_bytes / (dom_ms * 1e-3 / dom_launches) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get(dom_name)
        except Exception:
            traffic = None
    return {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": dom_ms / dom_launches,
            "kernel_ms_per_step": {kk: v[0] / steps for kk, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}


# ---- one GPU ------------------------------------------------------------------------------------
def normals_call(c, cfg, normals_ptr, stride, idx_ptr):
    """estimate_normal: k-nearest (the benchmark's configuration) or the reference's own radius 2.5 mode."""
    if cfg.get("radius"):
        c.dev_normals_radius(cfg["radius"], normals_ptr, stride)
    else:
        c.dev_normals_knn(cfg["k"], normals_ptr, stride, idx_ptr=idx_ptr)


def dump_rows(n, cap):
    """The rows of an n-row output that --dump-outputs writes: all of them, or a fixed seeded sample of cap."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def last_step_outputs(env, cfg, contours, normals_d, idx_d):
    """The outputs of the last timed step as host arrays, for --dump-outputs (read after the timed window)."""
    torch, ctx = env.torch, env.ctx
    out = {}
    for name, t, dtype in (("normals", normals_d, np.float32), ("neighbour_ids", idx_d, np.float64)):
        rows = dump_rows(t.shape[0], DUMP_ROWS[name])
        out[name] = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy().astype(dtype)
        if len(rows) < t.shape[0]:
            out[name + "_rows"] = rows.astype(np.float64)
    nodes = int(contours["total_nodes"])
    out["contour_offsets"] = ctx.download(contours["node_offsets"], (cfg["S"] + 1,), np.int64).astype(np.float64)
    rows = dump_rows(nodes, DUMP_ROWS["contour"])
    for axis in "yxz":
        out["contour_" + axis] = ctx.download(contours[axis], (nodes,), np.float64)[rows]
    if len(rows) < nodes:
        out["contour_rows"] = rows.astype(np.float64)
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    return out


def write_outputs(path, outputs):
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a)


def measure_single(env, cfg, steps, warmup, e2e=True, dump=False):
    from polishpathplanning_b200 import api, synth
    torch, ctx, dev = env.torch, env.ctx, env.dev
    n, k, S = cfg["n_total"], cfg["k"], cfg["S"]
    cloud = synth.panel(n, seed=0)
    planes = make_planes(cloud[:, 0].min(), cloud[:, 0].max(), S)
    with torch.cuda.stream(env.stream):
        raw_d = torch.from_numpy(cloud).to(dev)
        normals_d = torch.empty((n, 8), dtype=torch.float32, device=dev)
        idx_d = torch.empty((n, k), dtype=torch.int32, device=dev)
    env.stream.synchronize()
    last = {}

    def dev_step(keep=False):
        c = api.Cloud(ctx, device_ptr=raw_d.data_ptr(), n=n, stride_bytes=32)
        normals_call(c, cfg, normals_d.data_ptr(), 32, idx_d.data_ptr())
        res = c.dev_slice_contours(planes, PAIRING, HALF_WIDTH, True)
        last["nodes"], last["members"] = res["total_nodes"], res["total_members"]
        if keep:        # the cloud owns the contour buffers: read back after the timed window, then closed
            last["cloud"], last["contours"] = c, res
        else:
            c.close()

    total_ms, _, launches, t_wall = timed_device_steps(env, dev_step, steps, warmup,
                                                       last_step=(lambda: dev_step(keep=True)) if dump else None)
    outputs = None
    if dump:
        outputs = last_step_outputs(env, cfg, last["contours"], normals_d, idx_d)
        last.pop("cloud").close()
    prof = kernel_profile(env, dev_step, steps)
    if not e2e:
        del raw_d, normals_d, idx_d
        return {"units": n, "total_ms": total_ms, "launches": launches, "t_wall": t_wall, "prof": prof, "e2e_s": float("nan"),
                "h2d": 0, "d2h": 0, "n_local": n, "members": last.get("members", 0), "nodes": last.get("nodes", 0),
                "exchange_ms": None, "parity": None, "outputs": outputs}

    # ---- end to end through the host-pointer C ABI (pinned buffers) ----
    pin_cloud = ctx.pinned_empty(cloud.shape, np.float32)
    pin_cloud[...] = cloud
    pin_normals = ctx.pinned_empty((n, 8), np.float32)
    node_cap = int(max(last.get("nodes", 0), 1024) * 1.25)
    pin_nodes = tuple(ctx.pinned_empty((node_cap,), np.float64) for _ in range(3))
    e2e_bytes = {}

    def host_step():
        # the reference's call sequence: constructor/Set_kdtree (upload + index), getMinMax3D + plane
        # positions on the host, then estimate_normal + the sweep (one combined C-ABI call)
        c = api.Cloud(ctx, pin_cloud)
        mn, mx = c.bbox()
        pl = make_planes(mn[0], mx[0], S)
        _, off, y, x, z = c.normals_and_contours(pl, PAIRING, k=k, half_width=HALF_WIDTH, truncate_center=True,
                                                 normals_out=pin_normals, nodes_out=pin_nodes)
        e2e_bytes["h2d"] = pin_cloud.nbytes + pl.nbytes * 5 + 4 * len(pl)
        e2e_bytes["d2h"] = pin_normals.nbytes + off.nbytes + 3 * y.nbytes
        c.close()

    for _ in range(SETTLE_STEPS // 2 + min(warmup, 3)):
        host_step()
    env.sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        host_step()
    env.sync_all()
    e2e_s = time.perf_counter() - t0
    del raw_d, normals_d, idx_d
    return {"units": n, "total_ms": total_ms, "launches": launches, "t_wall": t_wall, "prof": prof, "e2e_s": e2e_s,
            "h2d": e2e_bytes.get("h2d", 0), "d2h": e2e_bytes.get("d2h", 0), "n_local": n, "members": last.get("members", 0),
            "nodes": last.get("nodes", 0), "exchange_ms": None, "parity": None, "outputs": outputs}


# ---- N GPUs, one rank each ----------------------------------------------------------------------
def measure_multi(env, cfg, steps, warmup, verify=True, e2e=True):
    from polishpathplanning_b200 import api, parallel, synth
    torch, ctx, dev, dist, rank, world = env.torch, env.ctx, env.dev, env.dist, env.rank, env.world
    n_total, k, S = cfg["n_total"], cfg["k"], cfg["S"]
    starts = parallel.index_ranges(n_total, world)
    a, b = int(starts[rank]), int(starts[rank + 1])
    n_r = b - a
    tag = "%s_%s" % (os.environ.get("MASTER_PORT", "0"), cfg["name"])
    # ONE host buffer holds the cloud (it stands for the loaded PCD); every rank maps and page-locks it
    src = parallel.SharedHost(dist, rank, world, n_total * 32, "cloud_" + tag, ctx)
    cloud_h = src.array(np.float32, (n_total, 8))
    if rank == 0:
        cloud_h[...] = synth.panel(n_total, seed=0)
    dist.barrier()
    cap_recv = int(n_r * 1.25) + 65536
    node_cap = max(262144, n_r // 3, int(0.25 * 4 * np.sqrt(n_total) * S / world) + 65536)   # ~14 % of the band members become nodes
    ex = parallel.Exchange.over_dist(ctx, dist, dev, rank, world, n_total, cap_recv, S, node_cap, 32)
    cap_recv, node_cap = ex.cap_recv, ex.node_cap
    lay = parallel.host_region_layout(world, n_total, 32, S, node_cap)
    ctl_bytes = 4096                                   # barrier slots in front of the result sections
    dst = parallel.SharedHost(dist, rank, world, ctl_bytes + lay["total_bytes"], "result_" + tag, ctx)
    arrive = dst.array(np.int64, (world, 8), 0)       # one 64-byte line per rank
    if rank == 0:
        arrive[...] = 0
    dist.barrier()
    bar = {"n": 0}

    def host_barrier():
        """All ranks, through the shared result buffer (no GPU work, a few microseconds)."""
        bar["n"] += 1
        arrive[rank, 0] = bar["n"]
        t_end = time.perf_counter() + 120.0
        while int(arrive[:, 0].min()) < bar["n"]:
            if time.perf_counter() > t_end:
                raise SystemExit("bench.py: rank %d waited 120 s for the other ranks at a host barrier" % rank)

    with torch.cuda.stream(env.stream):
        chunk_d = torch.empty((n_r, 8), dtype=torch.float32, device=dev)
        idx_d = torch.empty((cap_recv, k), dtype=torch.int32, device=dev)
    ctx.upload(chunk_d.data_ptr(), src.host_base + a * 32, n_r * 32)
    ctx.sync()
    last = {}
    region_host = ctl_bytes + lay["normals_bytes"] + rank * lay["region_bytes"]

    stage = {}

    def mark(name, t0):
        """PPP_BENCH_VERBOSE: synchronise and book the wall time since t0 under `name` (breakdown pass only)."""
        if not stage.get("on"):
            return t0
        ctx.sync()
        t1 = time.perf_counter()
        stage[name] = stage.get(name, 0.0) + (t1 - t0)
        return t1

    def slab_work(to_host):
        """Everything after the records are on this GPU: exchange, the single-GPU path on the slab, results."""
        t_s = time.perf_counter()
        ctx.timer_begin(1)
        ex.exchange(chunk_d.data_ptr(), n_r, 32, HALO_MM)
        # ONE synchronisation for the exchange AND the ingest of the received slab: slab size, cuts, x-range, bounding box
        info, c = ex.finish_attach(to_rank0=not to_host)
        ctx.timer_end(1)
        t_s = mark("exchange+attach", t_s)
        planes = make_planes(np.float32(info["x_range"][0]), np.float32(info["x_range"][1]), S)   # getMinMax3D -> sweep
        pos = parallel.owned_planes(planes, info["cuts"], rank)
        if to_host:     # contour nodes + per-slice offsets straight into this rank's region of the host result
            base = dst.dev_base + region_host
            c.dev_set_contour_offsets_buffer(base, S + 1)
            c.dev_set_contour_buffers(base + lay["off_bytes"], base + lay["off_bytes"] + lay["arr_bytes"],
                                      base + lay["off_bytes"] + 2 * lay["arr_bytes"], node_cap)
            want_y = base + lay["off_bytes"]
        else:
            want_y = ex.nodes_region(rank)["y"] if rank == 0 else None
        normals_call(c, cfg, ex.home_normals_ptr, 32, idx_d.data_ptr())
        t_s = mark("index+knn", t_s)
        ex.results_signal(ex.NORMALS)
        if to_host:
            # the normals of MY index range are complete once every rank has signalled: their copy to the host
            # (copy engine, my PCIe link) then runs under the slicing kernels, which use the auxiliary stream
            ex.results_wait(ex.NORMALS)
            ctx.download_async(dst.host_base + ctl_bytes + a * 32, ex.home_normals_ptr, n_r * 32)
            t_s = mark("normals wait + d2h", t_s)
        res = c.dev_slice_contours(planes[pos], PAIRING, HALF_WIDTH, True)
        t_s = mark("slicing", t_s)
        if res["total_nodes"] > node_cap or (want_y is not None and res["total_nodes"] and res["y"] != want_y):
            raise SystemExit("bench.py: %d contour nodes exceed the result region (%d)" % (res["total_nodes"], node_cap))
        if not to_host:
            ex.results_signal(ex.CONTOURS)
            ex.results_wait(ex.NORMALS)
            ex.results_wait(ex.CONTOURS)                               # rank 0's regions hold every rank's contours
        last.update(nodes=res["total_nodes"], members=res["total_members"], n_local=info["n_local"], n_owned=info["n_owned"],
                    planes=planes, cuts=info["cuts"], pos=pos)
        return c

    def dev_step():
        slab_work(False).close()

    total_ms, own_ms, launches, t_wall = timed_device_steps(env, dev_step, steps, warmup)
    ex_ms, ex_regions = ctx.timer_read(1, reset=True)
    exchange_ms = env.max_over_ranks(ex_ms / max(ex_regions, 1))
    prof = kernel_profile(env, dev_step, steps)
    if os.environ.get("PPP_BENCH_VERBOSE"):
        sys.stderr.write("[rank %d] own step %.4f ms; exchange %.4f ms; n_local %d; kernels %s\n" % (
            rank, own_ms / steps, ex_ms / max(ex_regions, 1), last["n_local"],
            {kk: round(v[0] / steps, 4) for kk, v in sorted(prof.items(), key=lambda kv: -kv[1][0])[:5]}))

    if not e2e:
        out = {"units": n_total, "total_ms": total_ms, "launches": launches, "t_wall": t_wall, "prof": prof, "e2e_s": float("nan"),
               "h2d": 0, "d2h": 0, "n_local": last["n_local"], "members": last["members"], "nodes": last["nodes"],
               "exchange_ms": exchange_ms, "parity": None}
        del cloud_h, arrive
        ex.close(dist)
        src.close()
        dst.close()
        del chunk_d, idx_d
        return out

    # ---- end to end: ONE host buffer in, ONE host buffer out ----
    normals_h = dst.array(np.float32, (n_total, 8), ctl_bytes)
    table = {}

    def host_step():
        t_s = time.perf_counter()
        ctx.upload(chunk_d.data_ptr(), src.host_base + a * 32, n_r * 32)          # my index range, my PCIe link
        t_s = mark("h2d", t_s)
        c = slab_work(True)
        ctx.sync()
        c.close()
        t_s = time.perf_counter()
        host_barrier()
        stage["barrier+table"] = stage.get("barrier+table", 0.0) - t_s
        if rank == 0:
            # per-plane table into the one result buffer: where each plane's y / x / z arrays start and how many
            # nodes it has -- the (n, y, x, z) a Spline is constructed from (include/Spline.h:10-20)
            planes, cuts = last["planes"], last["cuts"]
            at_y = np.zeros(S, np.int64)
            cnt = np.zeros(S, np.int64)
            for r in range(world):
                pos = parallel.owned_planes(planes, cuts, r)
                reg = ctl_bytes + lay["normals_bytes"] + r * lay["region_bytes"]
                off = dst.array(np.int64, (len(pos) + 1,), reg)
                cnt[pos] = np.diff(off)
                at_y[pos] = reg + lay["off_bytes"] + 8 * off[:-1]
            table.update(at_y=at_y, count=cnt)
        host_barrier()
        stage["barrier+table"] += time.perf_counter()

    for _ in range(min(warmup, 3)):
        host_step()
    env.sync_all()
    host_barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        host_step()
    e2e_s = env.max_over_ranks(time.perf_counter() - t0)
    env.sync_all()
    if os.environ.get("PPP_BENCH_VERBOSE"):      # untimed: the same step with a synchronise after every stage
        stage.clear()
        stage["on"] = True
        for _ in range(5):
            host_step()
        stage.pop("on")
        sys.stderr.write("[rank %d] e2e stages (ms, serialised): %s\n" % (rank, {kk: round(1e3 * v / 5, 3) for kk, v in stage.items()}))
        stage.clear()
    nodes_all = int(table["count"].sum()) if rank == 0 else 0
    h2d = n_total * 32 + world * (S * 5 * 4 + 4 * S)
    d2h = n_total * 32 + (S + world) * 8 + 3 * 8 * nodes_all

    # ---- untimed: the one host result against the single-GPU run of the whole cloud, bit for bit ----
    parity = None
    if verify:
        bad = torch.zeros(3, dtype=torch.int64, device=dev)
        if rank == 0:
            full = api.Cloud(ctx, np.ascontiguousarray(cloud_h))
            ref_n = full.normals_knn(k, stride_floats=8)
            mn, mx = full.bbox()
            ro, ry, rx, rz = full.slice_contours(make_planes(mn[0], mx[0], S), PAIRING, HALF_WIDTH, True)
            full.close()
            got_n = np.concatenate([normals_h[:, 0:3], normals_h[:, 4:5]], axis=1).view(np.uint32)
            bad[0] = int((got_n != np.concatenate([ref_n[:, 0:3], ref_n[:, 4:5]], axis=1).view(np.uint32)).any(axis=1).sum())
            raw = dst.array(np.uint8, (dst.nbytes,), 0)
            ok_c = np.array_equal(table["count"], np.diff(ro))
            if ok_c:
                for j, ref in enumerate((ry, rx, rz)):
                    for s in np.nonzero(table["count"])[0]:
                        at = int(table["at_y"][s]) + j * lay["arr_bytes"]
                        seg = raw[at:at + 8 * int(table["count"][s])].view(np.float64)
                        if not np.array_equal(seg.view(np.uint64), ref[ro[s]:ro[s + 1]].view(np.uint64)):
                            ok_c = False
                            break
            bad[1] = 0 if ok_c else 1
            del raw
        dist.all_reduce(bad)
        parity = {"normal_rows_differing": int(bad[0].item()), "contours_differ": int(bad[1].item()),
                  "against": "single-GPU run of the whole %d-point cloud on rank 0" % n_total}
    out = {"units": n_total, "total_ms": total_ms, "launches": launches, "t_wall": t_wall, "prof": prof, "e2e_s": e2e_s,
           "h2d": h2d, "d2h": d2h, "n_local": last["n_local"], "members": last["members"], "nodes": last["nodes"],
           "exchange_ms": exchange_ms, "parity": parity}
    del cloud_h, normals_h, arrive
    ex.close(dist)
    src.close()
    dst.close()
    del chunk_d, idx_d
    return out


def run_ours(args):
    env = Env(args)
    cfg = make_cfg(args.config, env.world)
    sampler = ClockSampler(env.local_rank)
    if env.rank == 0:
        sampler.start()
    if env.world == 1:
        m = measure_single(env, cfg, args.steps, args.warmup, dump=args.dump_outputs is not None)
    else:
        m = measure_multi(env, cfg, args.steps, args.warmup)
    clocks = sampler.stop() if env.rank == 0 else None
    if args.dump_outputs is not None:
        write_outputs(args.dump_outputs, m.pop("outputs"))
    extra = None
    if args.config == "cfg2" and not args.no_cfg3:
        # the north-star configuration (BASELINE.json configs[2]: 10M points, k = 32, 1000 slices) on the same GPUs,
        # a few steps, so that the driver's record carries the "< 50 ms on 8 GPUs" figure next to the headline
        cfg3 = make_cfg("cfg3", env.world)
        m3 = measure_single(env, cfg3, 5, 3) if env.world == 1 else measure_multi(env, cfg3, 5, 3, verify=False)
        extra = {"workload": cfg3["text"], "n_gpus": env.world, "steps": 5, "warmup": 3,
                 "device_ms_per_step": m3["total_ms"] / 5, "e2e_ms_per_step": 1e3 * m3["e2e_s"] / 5,
                 "exchange_ms_per_step": m3["exchange_ms"], "target_ms": 50.0}
    if env.rank == 0:
        value = m["units"] * args.steps / (m["total_ms"] * 1e-3)
        roof = roofline_of(m["prof"], args.steps, m["n_local"], cfg["k"], m["members"], m["nodes"])
        cpu = None
        if env.world == 1 and args.config == "cfg2":
            cores = host_threads()
            v_all, secs, what = cpu_baseline(cfg, cores)
            v_one, secs1, _ = cpu_baseline(cfg, 1)
            cpu = {"value": v_all, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "oracle port of the reference CPU path on %s (k=%d normals, pairing %s); %.2f s with %d threads, "
                             "%.2f s single-thread" % (what, cfg["k"], PAIRING, secs, cores, secs1),
                   "single_thread_value": v_one}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["total_ms"] / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(cfg),
            "clocks": clocks,
            "e2e": {"value": m["units"] * args.steps / m["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": int(m["h2d"]),
                    "d2h_bytes_per_step": int(m["d2h"]), "ms_per_step": 1e3 * m["e2e_s"] / args.steps},
            "gpu_launches": int(m["launches"]),
            "roofline": roof, "cpu_baseline": cpu,
            "wall_ms_per_step_incl_flush": 1e3 * m["t_wall"] / args.steps,
            "points_local": m["n_local"], "band_members": m["members"], "contour_nodes": m["nodes"],
        }
        if m["exchange_ms"] is not None:
            line["exchange_ms_per_step"] = m["exchange_ms"]
        if m["parity"] is not None:
            line["multi_gpu_parity"] = m["parity"]
        if extra is not None:
            line["north_star_cfg3"] = extra
        print(json.dumps(line))
    env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3"],
                    help="cfg2 (default, the driver's contract): 1M points per GPU, k=16, 200*sqrt(N) planes, weak scaling. "
                         "cfg3 (SURVEY 8d): 10M points in TOTAL split over the GPUs, k=32, 1000 planes.")
    ap.add_argument("--no-cfg3", action="store_true", help="skip the extra north-star (cfg3) measurement of a cfg2 run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (one GPU, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.gpus != 1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the one-GPU path: use it with --gpus 1 --impl ours")
    if args.impl != "reference" and args.warmup < 3:
        args.warmup = 3       # timing rule: at least three warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
