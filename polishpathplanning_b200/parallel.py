"""Multi-GPU sharding of the hot path: one process per GPU, x-slab decomposition with halo.

The reference is single-process (SURVEY.md §5); its path shards naturally because every query
point and every slice is independent given read access to its neighbourhood (§8e).  Each rank
owns the points (and the slicing planes) of one x-interval and additionally holds a halo of
`halo` mm on both sides, so that
  * the k nearest / radius neighbours of every OWNED point, and
  * the +-half_width band of every OWNED plane plus the nearest-neighbour reach of its pairing
are all inside the rank's local cloud.

Data path of one step (bench.py --gpus N, tools/multi_gpu_check.py):
  1. the cloud starts in ONE host buffer that every rank's process has mapped (SharedHost); rank r
     copies the records of its ORIGINAL INDEX range to its GPU over its own PCIe link;
  2. Exchange (csrc/exchange.cu): hand-written kernels redistribute the records into x-slabs + halo by
     storing straight into the owner GPU's memory over NVLink (no NCCL collective on the data path);
  3. every rank runs the single-GPU path on its slab; each normal record goes from the search kernel to
     its HOME rank (the rank that holds that original index range), contour nodes go to rank 0's region
     or straight into the shared host buffer;
  4. every rank copies the normals of its index range into the ONE host result array over its own PCIe
     link; rank 0 orders the contour nodes by plane (assemble_contours): the arrays a Spline consumer
     (include/Spline.h:10-20) and path connection read are complete on one host.

Exactness guard: `halo_violations` reports owned points whose k-th neighbour distance reaches the
edge of the local x-extent (they would need a wider halo); callers re-run those with a wider halo
(the synthetic panels never trigger it with the default 12 mm).

The slab helpers are backend-agnostic (numpy in / numpy out) so the world_size-2 gloo tests can
drive them on CPU; Exchange / SharedHost take the context object as an argument, which lets those tests
exercise the rank protocol with a stand-in.
"""
import ctypes as C
import mmap
import os

import numpy as np


def slab_cuts(x, world):
    """world+1 cut positions (float64) splitting the finite x values into equal-count intervals.
    cuts[0] = -inf, cuts[-1] = +inf."""
    xs = np.sort(x[np.isfinite(x)].astype(np.float64))
    cuts = [-np.inf]
    for r in range(1, world):
        cuts.append(float(xs[min(len(xs) - 1, (len(xs) * r) // world)]) if len(xs) else 0.0)
    cuts.append(np.inf)
    return np.asarray(cuts, np.float64)


def slab_select(cloud, cuts, rank, halo):
    """Indices (ascending, global numbering) of the rank's local points and the owned mask among them."""
    x = cloud[:, 0].astype(np.float64)
    lo, hi = cuts[rank], cuts[rank + 1]
    local = np.nonzero((x >= lo - halo) & (x < hi + halo))[0]
    xl = x[local]
    owned = (xl >= lo) & (xl < hi)
    return local.astype(np.int64), owned


def owned_planes(planes, cuts, rank):
    """Positions (into `planes`) of the planes this rank owns: cut[rank] <= x < cut[rank+1]."""
    p = np.asarray(planes, np.float64)
    return np.nonzero((p >= cuts[rank]) & (p < cuts[rank + 1]))[0]


def halo_violations(local_cloud, owned, kth_d2, cuts, rank, halo):
    """Owned points whose k-th neighbour distance reaches beyond the halo (local numbering)."""
    x = local_cloud[:, 0].astype(np.float64)
    lo, hi = cuts[rank] - halo, cuts[rank + 1] + halo
    reach = np.sqrt(np.maximum(kth_d2.astype(np.float64), 0.0)) * (1.0 + 1e-6)
    bad = owned & np.isfinite(reach) & np.isfinite(x)   # non-finite points have no neighbours at all
    bad &= ((x - reach) < lo) & np.isfinite(lo) | ((x + reach) >= hi) & np.isfinite(hi)
    return np.nonzero(bad)[0]


def gather_to_rank0(dist, arrays, rank, world, device=None):
    """Variable-length gather of a list of equally-long 1-D/2-D numpy arrays (or torch tensors on
    `device`) from every rank to rank 0 with torch.distributed.  Returns on rank 0 a list (per
    rank) of lists of numpy arrays; None elsewhere."""
    import torch
    n = int(arrays[0].shape[0])
    sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([n], dtype=torch.int64, device=device))
    sizes = [int(s.item()) for s in sizes]
    mx = max(max(sizes), 1)
    out = [[] for _ in range(world)] if rank == 0 else None
    for a in arrays:
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        if device is not None:
            t = t.to(device)
        pad_shape = (mx,) + tuple(t.shape[1:])
        buf = torch.zeros(pad_shape, dtype=t.dtype, device=device)
        buf[:n] = t
        recv = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
        dist.gather(buf, recv, dst=0)
        if rank == 0:
            for r in range(world):
                out[r].append(recv[r][:sizes[r]].cpu().numpy())
    return out


def assemble_normals(n_total, stride_floats, per_rank):
    """per_rank: list of (global_idx, normals_rows). Rows not covered stay NaN."""
    full = np.full((n_total, stride_floats), np.nan, np.float32)
    for gidx, rows in per_rank:
        full[gidx] = rows
    return full


def assemble_contours(S, per_rank):
    """per_rank: list of (plane_positions, node_offsets, y, x, z) for the planes each rank owns.
    Returns global (node_offsets, y, x, z) ordered by plane position."""
    counts = np.zeros(S, np.int64)
    for pos, off, _, _, _ in per_rank:
        counts[pos] = np.diff(off)
    goff = np.zeros(S + 1, np.int64)
    np.cumsum(counts, out=goff[1:])
    y = np.empty(int(goff[-1]), np.float64)
    x = np.empty_like(y)
    z = np.empty_like(y)
    for pos, off, yy, xx, zz in per_rank:
        for j, s in enumerate(pos):
            a, b = int(off[j]), int(off[j + 1])
            y[goff[s]:goff[s + 1]] = yy[a:b]
            x[goff[s]:goff[s + 1]] = xx[a:b]
            z[goff[s]:goff[s + 1]] = zz[a:b]
    return goff, y, x, z



def index_ranges(n_total, world):
    """starts[world + 1]: rank r holds the records [starts[r], starts[r+1]) of the file."""
    return np.asarray([(int(n_total) * r) // int(world) for r in range(int(world) + 1)], np.int64)


# -------------------------------------------------------------------------------------------------
# Exchange: the device-side redistribution + result delivery (csrc/exchange.cu, include/ppp_gpu.h).
# -------------------------------------------------------------------------------------------------
class Exchange:
    """One rank's end of the multi-GPU exchange.  `ctx` is an api.Context.

    exchange(chunk_ptr, n, stride, halo) enqueues the four phases; finish() waits for every rank's
    records and reports the slab; attach() wraps the slab as a Cloud whose normal estimators deliver
    every owned row's record to its home rank; results_signal() / results_wait() close the step."""

    def __init__(self, ctx, rank, world, starts, cap_recv, S_cap, node_cap, normal_stride_bytes=32):
        from . import api
        self._api = api
        self.ctx, self.lib = ctx, ctx.lib
        self.rank, self.world = int(rank), int(world)
        self.starts = np.ascontiguousarray(starts, np.int64)
        assert self.starts.shape[0] == self.world + 1
        self.cap_recv, self.S_cap, self.node_cap = int(cap_recv), int(S_cap), int(node_cap)
        self.normal_stride_bytes = int(normal_stride_bytes)
        h = C.c_void_p()
        api.check(self.lib.ppp_exch_create(ctx._h, self.rank, self.world, self.starts.ctypes.data_as(C.POINTER(C.c_int64)),
                                           self.cap_recv, self.S_cap, self.node_cap, self.normal_stride_bytes, C.byref(h)))
        self._h = h

    # -- wiring -------------------------------------------------------------------------------------
    def handle(self):
        buf = (C.c_ubyte * 64)()
        self._api.check(self.lib.ppp_exch_ipc_handle(self._h, buf))
        return bytes(buf)

    def connect_ipc(self, handles):
        """handles: one 64-byte handle per rank (the own entry is ignored)."""
        blob = b"".join(bytes(h) for h in handles)
        assert len(blob) == 64 * self.world
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self._api.check(self.lib.ppp_exch_connect_ipc(self._h, buf))

    @staticmethod
    def connect_local(exchanges):
        """All ranks live in this process (loop-back on one GPU, or one process driving several GPUs)."""
        arr = (C.c_void_p * len(exchanges))(*[e._h for e in exchanges])
        for e in exchanges:
            e._api.check(e.lib.ppp_exch_connect_local(e._h, arr))

    @classmethod
    def over_dist(cls, ctx, dist, device, rank, world, n_total, cap_recv, S_cap, node_cap, normal_stride_bytes=32, factory=None):
        """One exchange per torch.distributed rank: agrees on the capacities (maxima over the ranks),
        creates the arenas, all-gathers the IPC handles and connects.  A failure on any rank is raised on
        EVERY rank, with nothing left allocated, so that callers can react together."""
        import torch
        caps = torch.tensor([int(cap_recv), int(S_cap), int(node_cap)], dtype=torch.int64, device=device)
        dist.all_reduce(caps, op=dist.ReduceOp.MAX)
        cap_recv, S_cap, node_cap = (int(v) for v in caps.tolist())
        ex, ok, why = None, 1, ""
        hbuf = torch.zeros(64, dtype=torch.uint8, device=device)
        try:
            ex = (factory or cls)(ctx, rank, world, index_ranges(n_total, world), cap_recv, S_cap, node_cap, normal_stride_bytes)
            hbuf.copy_(torch.frombuffer(bytearray(ex.handle()), dtype=torch.uint8))
        except Exception as e:                                         # noqa: BLE001 - reported to every rank below
            ok, why = 0, str(e)
        all_h = [torch.zeros_like(hbuf) for _ in range(world)]
        dist.all_gather(all_h, hbuf)
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            try:
                ex.connect_ipc([t.cpu().numpy().tobytes() for t in all_h])
            except Exception as e:                                     # noqa: BLE001
                ok, why = 0, str(e)
            flag = torch.tensor([ok], dtype=torch.int32, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if ex is not None:
                ex.close(dist)
            else:
                dist.barrier()       # the barrier inside the others' close()
            raise RuntimeError("the exchange could not be set up on every rank" + (": " + why if why else ""))
        return ex

    # -- one step -----------------------------------------------------------------------------------
    def phase(self, p, chunk_ptr, n, stride_bytes, halo):
        self._api.check(self.lib.ppp_exch_phase(self._h, int(p), C.c_void_p(chunk_ptr), int(n), int(stride_bytes), float(halo)))

    def exchange(self, chunk_ptr, n, stride_bytes, halo):
        for p in range(4):
            self.phase(p, chunk_ptr, n, stride_bytes, halo)

    def finish(self):
        nl, no = C.c_int64(0), C.c_int64(0)
        cuts = np.zeros(self.world + 1, np.float64)
        xr = np.zeros(2, np.float64)
        self._api.check(self.lib.ppp_exch_finish(self._h, C.byref(nl), C.byref(no), cuts.ctypes.data_as(C.POINTER(C.c_double)),
                                                 xr.ctypes.data_as(C.POINTER(C.c_double))))
        return {"n_local": nl.value, "n_owned": no.value, "cuts": cuts, "x_range": xr}

    def attach(self, to_rank0=True):
        h = C.c_void_p()
        self._api.check(self.lib.ppp_exch_attach(self._h, int(bool(to_rank0)), C.byref(h)))
        return self._api.Cloud(self.ctx, handle=h)

    def finish_attach(self, to_rank0=True):
        """finish() + attach() with one host synchronisation; returns (info, cloud)."""
        nl, no = C.c_int64(0), C.c_int64(0)
        cuts = np.zeros(self.world + 1, np.float64)
        xr = np.zeros(2, np.float64)
        h = C.c_void_p()
        self._api.check(self.lib.ppp_exch_finish_attach(self._h, int(bool(to_rank0)), C.byref(nl), C.byref(no),
                                                        cuts.ctypes.data_as(C.POINTER(C.c_double)),
                                                        xr.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h)))
        return ({"n_local": nl.value, "n_owned": no.value, "cuts": cuts, "x_range": xr}, self._api.Cloud(self.ctx, handle=h))

    NORMALS, CONTOURS = 0, 1

    def results_signal(self, what):
        """what: Exchange.NORMALS / Exchange.CONTOURS -- this rank's results of that kind are delivered."""
        self._api.check(self.lib.ppp_exch_results_signal(self._h, int(what)))

    def results_wait(self, what):
        """Later work of the stream sees every rank's results of that kind."""
        self._api.check(self.lib.ppp_exch_results_wait(self._h, int(what)))

    def check(self):
        self._api.check(self.lib.ppp_exch_check(self._h))

    @property
    def slab_ptr(self):
        return self.lib.ppp_exch_slab(self._h)

    @property
    def row_map_ptr(self):
        return self.lib.ppp_exch_row_map(self._h)

    @property
    def home_normals_ptr(self):
        return self.lib.ppp_exch_home_normals(self._h)

    @property
    def home_rows(self):
        return int(self.starts[self.rank + 1] - self.starts[self.rank])

    def nodes_region(self, r):
        """Rank 0: device pointers of rank r's contour region."""
        po, py, px, pz = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._api.check(self.lib.ppp_exch_nodes_region(self._h, int(r), C.byref(po), C.byref(py), C.byref(px), C.byref(pz)))
        return {"off": po.value, "y": py.value, "x": px.value, "z": pz.value}

    def read_home_normals(self):
        """After results_wait + a sync: the normal records of the own index range (rows, stride/4)."""
        return self.ctx.download(self.home_normals_ptr, (self.home_rows, self.normal_stride_bytes // 4), np.float32)

    def read_nodes(self, S_per_rank):
        """Rank 0, after results_wait + a sync: [(offsets, y, x, z) per rank]."""
        assert self.rank == 0
        out = []
        for r in range(self.world):
            g = self.nodes_region(r)
            off = self.ctx.download(g["off"], (int(S_per_rank[r]) + 1,), np.int64)
            n = int(off[-1])
            out.append((off, self.ctx.download(g["y"], (n,), np.float64), self.ctx.download(g["x"], (n,), np.float64),
                        self.ctx.download(g["z"], (n,), np.float64)))
        return out

    def close(self, dist=None):
        """With `dist` (ranks in different processes) this is collective: everybody unmaps the peers' arenas,
        then, after a barrier, frees its own."""
        if getattr(self, "_h", None):
            if dist is not None:
                self.lib.ppp_exch_disconnect(self._h)
                dist.barrier()
            self.lib.ppp_exch_destroy(self._h)
            self._h = None


# -------------------------------------------------------------------------------------------------
# MLS smooth() over the exchange: halo = the MLS radius (mls_halo), every rank smooths the points it owns, each record
# travels to its home rank, and the home ranks compact their index ranges into one result in source order.
# -------------------------------------------------------------------------------------------------
MLS_RECORD_BYTES = 32   # {x, y, z, flag, nx, ny, nz, curvature}: the exchange must be created with normal_stride_bytes=32


def mls_halo(radius, x_abs_max):
    """The exchange halo an MLS call of `radius` needs on a cloud whose finite x lie within +-x_abs_max (ppp_mls_halo:
    the float32 reach of the radius plus the double rounding of the cut positions; derivation in csrc/mls.cu).  The
    library refuses an MLS call on a slab cut with a narrower halo."""
    from . import _lib
    return float(_lib.load().ppp_mls_halo(float(radius), float(x_abs_max)))


def mls_smooth_sharded(exs, chunk_ptrs, stride_bytes, radius, order, halo, outputs, dist=None, device=None):
    """One MLS step for the ranks this process drives (exs: their Exchange objects, one under torchrun, every rank with
    Exchange.connect_local; chunk_ptrs: each rank's chunk, device records of stride_bytes, its index range).

    exchange -> attach -> ppp_dev_mls_smooth (records to the home ranks) -> results signal / wait -> count -> share the
    counts (dist.all_gather across processes, the list itself when every rank lives here) -> compact.
    outputs[i] = (points_ptr, normals_ptr or None, src_index_ptr, cap_rows, shared) for exs[i]: shared=True: one
    buffer every rank writes (device or mapped host memory, e.g. SharedHost.dev_base sections), the rank's rows start at
    the rows of the lower ranks; shared=False: a buffer of this rank's own, its rows from row 0.  Points are records of
    stride_bytes: x, y, z smoothed, every other field from the source record.  Nothing is synchronised at the end:
    call ctx.sync() (and meet the other processes) before reading.

    Returns (counts, row_bases): rows of every rank and where each rank's rows start in the whole result.  The rows
    themselves are what Cloud.mls_smooth returns for the whole cloud -- (points, src_index, normals) in ascending
    source order -- written into the caller's buffers rather than returned: under torchrun the result is one shared
    host buffer (or one device buffer per rank) that a returned copy would have to duplicate; mls_rows() views it."""
    for p in range(4):                                   # phase by phase over the ranks of this process
        for ex, ptr in zip(exs, chunk_ptrs):
            ex.phase(p, ptr, ex.home_rows, stride_bytes, halo)
    clouds = []
    for ex in exs:
        assert ex.normal_stride_bytes == MLS_RECORD_BYTES
        clouds.append(ex.finish_attach(to_rank0=False)[1])
        clouds[-1].dev_mls_smooth(radius, order)
        ex.results_signal(ex.NORMALS)
    for ex in exs:
        ex.results_wait(ex.NORMALS)
    mine = [ex.ctx.dev_mls_compact(ex.home_normals_ptr, ex.home_rows) for ex in exs]
    world = exs[0].world
    if dist is not None and len(exs) < world:
        import torch
        t = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
        dist.all_gather(t, torch.tensor(mine, dtype=torch.int64, device=device))
        counts = [int(v.item()) for v in t]
    else:
        assert len(exs) == world
        counts = mine
    bases = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    for ex, ptr, (pts, nrm, src, cap, shared) in zip(exs, chunk_ptrs, outputs):
        ex.ctx.dev_mls_compact(ex.home_normals_ptr, ex.home_rows, ptr, stride_bytes, int(ex.starts[ex.rank]),
                               int(bases[ex.rank]) if shared else 0, pts, stride_bytes, nrm, src, cap)
    for c in clouds:
        c.close()
    return counts, bases[:-1]


def mls_rows(points, src_index, normals, counts):
    """The (points, src_index, normals) tuple of Cloud.mls_smooth as views of shared output buffers (numpy arrays of
    n_total rows that mls_smooth_sharded filled with shared=True); normals may be None."""
    m = int(sum(int(c) for c in counts))
    return points[:m], src_index[:m], (normals[:m] if normals is not None else None)


def host_region_layout(world, n_total, normal_stride_bytes, S_cap, node_cap):
    """Byte layout of the ONE host result buffer (every section 256-byte aligned):
    [normals n_total x stride][rank 0: offsets (S_cap + 1) int64 | y | x | z (node_cap doubles each)] ... [rank world-1]."""
    a256 = lambda v: (int(v) + 255) // 256 * 256
    normals_bytes = a256(int(n_total) * int(normal_stride_bytes))
    off_bytes = a256((int(S_cap) + 1) * 8)
    arr_bytes = a256(max(int(node_cap), 1) * 8)
    region_bytes = off_bytes + 3 * arr_bytes
    return {"normals_bytes": normals_bytes, "off_bytes": off_bytes, "arr_bytes": arr_bytes, "region_bytes": region_bytes,
            "total_bytes": normals_bytes + int(world) * region_bytes}


class SharedHost:
    """A host buffer that EVERY rank's process maps (POSIX shared memory) and page-locks, so that each
    GPU moves its share over its own PCIe link and the result is one array on one host.

    Rank 0 creates the backing object (a file under /dev/shm; an anonymous memfd reached through
    /proc/<pid>/fd when /dev/shm is too small), the path travels by broadcast, the others open it.
    `ctx` (optional): page-lock the mapping through ctx.host_register; `dev_base` is then the address
    kernels use for byte 0."""

    def __init__(self, dist, rank, world, nbytes, tag, ctx=None):
        self.rank, self.world, self.nbytes, self.ctx, self._dist = int(rank), int(world), int(nbytes), ctx, dist
        self._fd, self._unlink, self.dev_base, self._registered = -1, None, None, False
        path = [None]
        if self.rank == 0:
            p = "/dev/shm/ppp_%s_%d" % (tag, os.getpid())
            try:
                if os.environ.get("PPP_SHM_MEMFD"):               # test aid: take the memfd route
                    raise OSError("memfd requested")
                fd = os.open(p, os.O_CREAT | os.O_EXCL | os.O_RDWR, 0o600)
                try:
                    os.posix_fallocate(fd, 0, self.nbytes)          # fails now (not at first touch) if tmpfs is too small
                    self._unlink = p
                except OSError:
                    os.close(fd)
                    os.unlink(p)
                    raise
            except OSError:
                fd = os.memfd_create("ppp_" + tag)
                os.ftruncate(fd, self.nbytes)
                p = "/proc/%d/fd/%d" % (os.getpid(), fd)
            self._fd = fd
            path[0] = p
        if dist is not None and self.world > 1:
            dist.broadcast_object_list(path, src=0)
        if self.rank != 0:
            self._fd = os.open(path[0], os.O_RDWR)
        self.mm = mmap.mmap(self._fd, self.nbytes, mmap.MAP_SHARED, mmap.PROT_READ | mmap.PROT_WRITE)
        self._view = (C.c_char * self.nbytes).from_buffer(self.mm)
        self.host_base = C.addressof(self._view)
        if ctx is not None:
            self.dev_base = ctx.host_register(self.host_base, self.nbytes)
            self._registered = True

    def array(self, dtype, shape, offset=0):
        """numpy view of a section (no copy)."""
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        assert offset + count * dtype.itemsize <= self.nbytes
        return np.frombuffer(self._view, dtype=dtype, count=count, offset=int(offset)).reshape(shape)

    def close(self):
        """Collective: everybody unmaps, then rank 0 removes the backing object."""
        if self._registered:
            self.ctx.host_unregister(self.host_base)
            self._registered = False
        self._view = None
        try:
            self.mm.close()
        except BufferError:           # a numpy view is still alive somewhere: the mapping goes with the process
            pass
        if self._dist is not None and self.world > 1:
            self._dist.barrier()
        if self._fd >= 0:
            os.close(self._fd)
            self._fd = -1
        if self._unlink:
            try:
                os.unlink(self._unlink)
            except OSError:
                pass
            self._unlink = None
