"""Host-side objects over the C ABI (include/ppp_gpu.h): Context (one per GPU) and Cloud
(device-resident copy + column-grid index).  numpy in / numpy out through the host API; the
`dev_*` methods take raw device pointers (e.g. torch tensors' data_ptr()) for the device-resident
pipeline used by bench.py and the multi-GPU sharding.
"""
import ctypes as C
import weakref

import numpy as np

from . import _lib
from ._lib import PPP_COV_PCL110, PPP_COV_SHIFTED, PPP_PAIR_GEN2, PPP_PAIR_SECT, PPPError, check  # noqa: F401

_vp = C.c_void_p


def _ptr(a):
    return a.ctypes.data_as(_vp) if a is not None else None


class Context:
    def __init__(self, device=0):
        self.lib = _lib.load()
        h = _vp()
        check(self.lib.ppp_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        self._clouds = weakref.WeakSet()

    def close(self):
        if getattr(self, "_h", None):
            for c in list(self._clouds):  # cloud handles hold device memory of this context
                c.close()
            self.lib.ppp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return self.lib.ppp_stream(self._h)

    def sync(self):
        check(self.lib.ppp_sync(self._h))

    def launch_count(self):
        return int(self.lib.ppp_launch_count(self._h))

    def timer_begin(self, tag=0):
        check(self.lib.ppp_timer_begin(self._h, tag))

    def timer_end(self, tag=0):
        check(self.lib.ppp_timer_end(self._h, tag))

    def timer_read(self, tag=0, reset=True):
        ms = C.c_double(0)
        n = C.c_int64(0)
        check(self.lib.ppp_timer_read(self._h, tag, C.byref(ms), C.byref(n), int(reset)))
        return ms.value, n.value

    def kernel_profile(self, enable):
        check(self.lib.ppp_kernel_profile(self._h, int(bool(enable))))

    def kernel_profile_read(self, reset=True):
        buf = C.create_string_buffer(1 << 16)
        check(self.lib.ppp_kernel_profile_read(self._h, buf, len(buf), int(reset)))
        out = {}
        for item in buf.value.decode().split(";"):
            if not item:
                continue
            name, _, rest = item.partition("=")
            ms, _, cnt = rest.partition(":")
            out[name] = (float(ms), int(cnt))
        return out

    def kernel_trace(self, enable):
        check(self.lib.ppp_kernel_trace(self._h, int(bool(enable))))

    def kernel_trace_read(self):
        """[(name, stream 0 main / 1 auxiliary, start_ms, end_ms)] in launch order; clears the trace."""
        buf = C.create_string_buffer(1 << 20)
        check(self.lib.ppp_kernel_trace_read(self._h, buf, len(buf)))
        out = []
        for item in buf.value.decode().split(";"):
            if item:
                name, _, rest = item.partition("=")
                aux, t0, t1 = rest.split(":")
                out.append((name, int(aux), float(t0), float(t1)))
        return out

    # -- buffers the GPUs of other processes can write (CUDA IPC over NVLink / NVSwitch) ------------
    def peer_buffer_alloc(self, nbytes):
        """Owner side: returns (device pointer, 64-byte handle as bytes)."""
        p = C.c_void_p(0)
        h = (C.c_ubyte * 64)()
        check(self.lib.ppp_peer_buffer_alloc(self._h, int(nbytes), C.byref(p), h))
        return p.value, bytes(h)

    def peer_buffer_open(self, handle):
        p = C.c_void_p(0)
        h = (C.c_ubyte * 64).from_buffer_copy(bytes(handle))
        check(self.lib.ppp_peer_buffer_open(self._h, h, C.byref(p)))
        return p.value

    def peer_buffer_close(self, ptr):
        check(self.lib.ppp_peer_buffer_close(self._h, _vp(ptr)))

    def peer_buffer_free(self, ptr):
        check(self.lib.ppp_peer_buffer_free(self._h, _vp(ptr)))

    def signal(self, flag_ptr, value):
        """*flag = value after all earlier work of the context's stream (no kernel launch)."""
        check(self.lib.ppp_dev_signal(self._h, _vp(flag_ptr), int(value)))

    def wait(self, flag_ptr, value):
        """Later work of the context's stream waits until *flag >= value."""
        check(self.lib.ppp_dev_wait(self._h, _vp(flag_ptr), int(value)))

    def download(self, dev_ptr, shape, dtype):
        """Device range -> new numpy array (synchronises)."""
        out = np.empty(shape, dtype)
        check(self.lib.ppp_dev_download(self._h, _ptr(out), _vp(dev_ptr), out.nbytes))
        return out

    def upload(self, dev_ptr, host_ptr, nbytes):
        """Stream-ordered host -> device copy (host memory should be page-locked); does not synchronise."""
        check(self.lib.ppp_dev_upload(self._h, _vp(dev_ptr), _vp(host_ptr), int(nbytes)))

    def download_async(self, host_ptr, dev_ptr, nbytes):
        """Stream-ordered device -> host copy; does not synchronise."""
        check(self.lib.ppp_dev_download_async(self._h, _vp(host_ptr), _vp(dev_ptr), int(nbytes)))

    def host_register(self, host_ptr, nbytes):
        """Page-lock an existing host range; returns the address kernels use for its first byte."""
        d = C.c_void_p(0)
        check(self.lib.ppp_host_register(_vp(host_ptr), int(nbytes), C.byref(d)))
        return d.value

    def host_unregister(self, host_ptr):
        check(self.lib.ppp_host_unregister(_vp(host_ptr)))

    def dev_mls_compact(self, rows_ptr, n, src_ptr=None, src_stride_bytes=0, src_index_base=0, row_base=0, points_ptr=None,
                        out_stride_bytes=32, normals_ptr=None, src_index_ptr=None, cap_rows=0):
        """ppp_dev_mls_compact: MLS records [0, n) at rows_ptr -> output rows in source order from row_base on.
        Without points_ptr / src_index_ptr only counts.  Returns the number of rows of the range (raises PPPError with
        status PPP_ERR_CAPACITY when row_base + that number exceeds cap_rows)."""
        m = C.c_int64(0)
        check(self.lib.ppp_dev_mls_compact(self._h, _vp(rows_ptr) if rows_ptr else None, int(n), _vp(src_ptr) if src_ptr else None,
                                           int(src_stride_bytes), int(src_index_base), int(row_base),
                                           _vp(points_ptr) if points_ptr else None, int(out_stride_bytes),
                                           _vp(normals_ptr) if normals_ptr else None,
                                           _vp(src_index_ptr) if src_index_ptr else None, int(cap_rows), C.byref(m)))
        return m.value

    def pinned_empty(self, shape, dtype):
        """numpy array over pinned host memory from ppp_host_alloc (freed with the array)."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = self.lib.ppp_host_alloc(max(n, 1))
        if not p:
            raise MemoryError("ppp_host_alloc(%d) failed" % n)
        buf = (C.c_char * max(n, 1)).from_address(p)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        _PINNED[id(buf)] = (buf, p, self.lib)
        return arr


_PINNED = {}


class Cloud:
    """points: float32 (N, stride_floats) host array (stride 8 = pcl::PointXYZRGB) or, with
    device_ptr=..., a device buffer of n records of stride_bytes."""

    def __init__(self, ctx, points=None, device_ptr=None, n=None, stride_bytes=None, handle=None):
        self.ctx = ctx
        self.lib = ctx.lib
        h = _vp()
        self._records = None   # where mls_smooth copies the fields other than x, y, z from
        if handle is not None:         # an existing ppp_cloud* (e.g. from ppp_exch_attach); owned from here on
            h = handle
            self.n = int(self.lib.ppp_cloud_size(h))
        elif device_ptr is not None:
            check(self.lib.ppp_dev_cloud_attach(ctx._h, _vp(device_ptr), int(n), int(stride_bytes), C.byref(h)))
            self.n = int(n)
            self._records = (int(device_ptr), int(stride_bytes))
        else:
            pts = np.asarray(points)
            if pts.dtype != np.float32 or pts.ndim != 2 or pts.shape[1] < 3 or not pts.flags.c_contiguous:
                raise ValueError("points must be a C-contiguous float32 array of shape (N, >=3)")
            check(self.lib.ppp_cloud_upload(ctx._h, _ptr(pts), pts.shape[0], pts.shape[1] * 4, C.byref(h)))
            self.n = pts.shape[0]
            self._records = pts
        self._h = h
        ctx._clouds.add(self)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ppp_cloud_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_cell_hint(self, h):
        check(self.lib.ppp_cloud_set_cell_hint(self._h, float(h)))

    def bbox(self):
        mn = np.zeros(3, np.float32)
        mx = np.zeros(3, np.float32)
        check(self.lib.ppp_cloud_bbox(self._h, mn.ctypes.data_as(_lib._f32p), mx.ctypes.data_as(_lib._f32p)))
        return mn, mx

    # ---- neighbour searches -------------------------------------------------------------------
    def knn(self, k, queries=None, want_d2=True):
        if queries is None:
            rows, q, nq, qs = self.n, None, 0, 0
        else:
            queries = np.ascontiguousarray(queries, np.float32)
            rows, q, nq, qs = queries.shape[0], _ptr(queries), queries.shape[0], queries.shape[1] * 4
        idx = np.empty((rows, k), np.int32)
        d2 = np.empty((rows, k), np.float32) if want_d2 else None
        check(self.lib.ppp_knn(self._h, q, nq, qs, int(k), _ptr(idx), _ptr(d2)))
        return idx, d2

    def radius(self, r, queries=None):
        if queries is None:
            rows, q, nq, qs = self.n, None, 0, 0
        else:
            queries = np.ascontiguousarray(queries, np.float32)
            rows, q, nq, qs = queries.shape[0], _ptr(queries), queries.shape[0], queries.shape[1] * 4
        counts = np.empty(rows, np.int32)
        check(self.lib.ppp_radius(self._h, q, nq, qs, float(r), _ptr(counts), None, None, None))
        offsets = np.zeros(rows + 1, np.int64)
        np.cumsum(counts, out=offsets[1:])
        idx = np.empty(int(offsets[-1]), np.int32)
        d2 = np.empty(int(offsets[-1]), np.float32)
        check(self.lib.ppp_radius(self._h, q, nq, qs, float(r), _ptr(counts), _ptr(offsets), _ptr(idx), _ptr(d2)))
        return counts, offsets, idx, d2

    # ---- normals ------------------------------------------------------------------------------
    def normals_knn(self, k, viewpoint=(0.0, 0.0, 0.0), flags=PPP_COV_PCL110, stride_floats=8, return_idx=False,
                    out=None):
        vp = np.asarray(viewpoint, np.float32)
        nrm = out if out is not None else np.empty((self.n, stride_floats), np.float32)
        idx = np.empty((self.n, k), np.int32) if return_idx else None
        check(self.lib.ppp_normals_knn(self._h, int(k), vp.ctypes.data_as(_lib._f32p), flags, _ptr(nrm),
                                       nrm.shape[1] * 4, _ptr(idx)))
        return (nrm, idx) if return_idx else nrm

    def normals_radius(self, r, viewpoint=(0.0, 0.0, 0.0), flags=PPP_COV_PCL110, stride_floats=8, out=None):
        vp = np.asarray(viewpoint, np.float32)
        nrm = out if out is not None else np.empty((self.n, stride_floats), np.float32)
        check(self.lib.ppp_normals_radius(self._h, float(r), vp.ctypes.data_as(_lib._f32p), flags, _ptr(nrm),
                                          nrm.shape[1] * 4))
        return nrm

    # ---- slicing ------------------------------------------------------------------------------
    def slice_bands(self, planes, half_width=2.0, truncate_center=True):
        planes = np.ascontiguousarray(planes, np.float32)
        S = planes.shape[0]
        off = np.zeros(S + 1, np.int64)
        check(self.lib.ppp_slice_bands(self._h, _ptr(planes), S, half_width, int(truncate_center), _ptr(off), None, 0))
        idx = np.empty(int(off[-1]), np.int32)
        check(self.lib.ppp_slice_bands(self._h, _ptr(planes), S, half_width, int(truncate_center), _ptr(off), _ptr(idx),
                                       idx.shape[0]))
        return off, idx

    def slice_contours(self, planes, mode, half_width=2.0, truncate_center=True, node_cap=None, out=None):
        """mode: PPP_PAIR_GEN2 ('A') or PPP_PAIR_SECT ('B'). Returns (node_offsets, y, x, z).
        out: optional (y, x, z) float64 buffers (e.g. pinned) to write into."""
        if isinstance(mode, str):
            mode = PPP_PAIR_GEN2 if mode.upper() == "A" else PPP_PAIR_SECT
        planes = np.ascontiguousarray(planes, np.float32)
        S = planes.shape[0]
        off = np.zeros(S + 1, np.int64)
        cap = int(node_cap) if node_cap else max(self.n // 4, 1024)
        while True:
            if out is not None and (node_cap is None or out[0].shape[0] >= cap):
                y, x, z = out                      # caller's buffers (e.g. pinned): filled in place if large enough
                cap = y.shape[0]
            else:
                y = np.empty(cap, np.float64)
                x = np.empty(cap, np.float64)
                z = np.empty(cap, np.float64)
            st = self.lib.ppp_slice_contours(self._h, _ptr(planes), S, half_width, int(truncate_center), mode, _ptr(off),
                                             _ptr(y), _ptr(x), _ptr(z), cap)
            if st == _lib.PPP_ERR_CAPACITY:
                cap = int(off[-1])
                out = None
                continue
            check(st)
            t = int(off[-1])
            return off, y[:t], x[:t], z[:t]

    def insert_point(self, indices, plane_x, mode):
        """insert_point with an explicit (strictly ascending) index list. Returns (y, x, z)."""
        if isinstance(mode, str):
            mode = PPP_PAIR_GEN2 if mode.upper() == "A" else PPP_PAIR_SECT
        indices = np.ascontiguousarray(indices, np.int32)
        cap = max(indices.shape[0], 1)
        y, x, z = (np.empty(cap, np.float64) for _ in range(3))
        n = C.c_int64(0)
        check(self.lib.ppp_insert_point(self._h, _ptr(indices), indices.shape[0], float(plane_x), mode, _ptr(y), _ptr(x),
                                        _ptr(z), cap, C.byref(n)))
        return y[:n.value], x[:n.value], z[:n.value]

    def normals_and_contours(self, planes, mode, k=0, radius=0.0, viewpoint=(0.0, 0.0, 0.0), flags=PPP_COV_PCL110,
                             half_width=2.0, truncate_center=True, normals_out=None, nodes_out=None, stride_floats=8):
        """estimate_normal + plane sweep in one call (normals D2H overlaps the slicing kernels).
        Returns (normals, node_offsets, y, x, z)."""
        if isinstance(mode, str):
            mode = PPP_PAIR_GEN2 if mode.upper() == "A" else PPP_PAIR_SECT
        planes = np.ascontiguousarray(planes, np.float32)
        S = planes.shape[0]
        vp = np.asarray(viewpoint, np.float32)
        nrm = normals_out if normals_out is not None else np.empty((self.n, stride_floats), np.float32)
        off = np.zeros(S + 1, np.int64)
        if nodes_out is not None:
            y, x, z = nodes_out
        else:
            cap = max(self.n // 4, 1024)
            y, x, z = (np.empty(cap, np.float64) for _ in range(3))
        st = self.lib.ppp_normals_and_contours(self._h, int(k), float(radius), vp.ctypes.data_as(_lib._f32p), flags,
                                               _ptr(nrm), nrm.shape[1] * 4, _ptr(planes), S, half_width,
                                               int(truncate_center), mode, _ptr(off), _ptr(y), _ptr(x), _ptr(z), y.shape[0])
        if st == _lib.PPP_ERR_CAPACITY:   # normals are valid; fetch the contours again with enough room
            off, y, x, z = self.slice_contours(planes, mode, half_width, truncate_center, node_cap=int(off[-1]))
            return nrm, off, y, x, z
        check(st)
        t = int(off[-1])
        return nrm, off, y[:t], x[:t], z[:t]

    def principal_curvatures(self, normals, queries, k):
        """compute_transform's device part: returns (out[nq,5] = pcx,pcy,pcz,pc1,pc2, nn0[nq])."""
        normals = np.ascontiguousarray(normals, np.float32)
        queries = np.ascontiguousarray(queries, np.float32)
        out = np.empty((queries.shape[0], 5), np.float32)
        nn0 = np.empty(queries.shape[0], np.int32)
        check(self.lib.ppp_principal_curvatures(self._h, _ptr(normals), normals.shape[1] * 4, _ptr(queries),
                                                queries.shape[0], queries.shape[1] * 4, int(k), _ptr(out), _ptr(nn0)))
        return out, nn0

    def sor_mean_distances(self, mean_k=50, sqrt_float=False):
        """First pass of StatisticalOutlierRemoval: (mean neighbour distance float32[N], n_valid)."""
        dist = np.empty(self.n, np.float32)
        nv = C.c_int64(0)
        check(self.lib.ppp_sor_mean_distances(self._h, int(mean_k), 1 if sqrt_float else 0, _ptr(dist), C.byref(nv)))
        return dist, nv.value

    def coverage_mark(self, queries, radius, flags=None):
        """compute_coverage for a batch of nodes; flags (uint8, N) is updated in place and returned."""
        queries = np.ascontiguousarray(queries, np.float32)
        if flags is None:
            flags = np.zeros(self.n, np.uint8)
        check(self.lib.ppp_coverage_mark(self._h, _ptr(queries), queries.shape[0], queries.shape[1] * 4, float(radius),
                                         _ptr(flags)))
        return flags

    def coverage_mark_radii(self, queries, radii, flags=None):
        """compute_coverage for nodes with one radius each (Area2Cloud); flags updated in place and returned."""
        queries = np.ascontiguousarray(queries, np.float32)
        radii = np.ascontiguousarray(radii, np.float64)
        assert radii.shape[0] == queries.shape[0]
        if flags is None:
            flags = np.zeros(self.n, np.uint8)
        check(self.lib.ppp_coverage_mark_radii(self._h, _ptr(queries), queries.shape[0], queries.shape[1] * 4, _ptr(radii),
                                               _ptr(flags)))
        return flags

    def mls_smooth(self, radius=15.0, order=3, normals=False):
        """smooth(): MovingLeastSquares (no upsampling, SIMPLE projection).  Returns (points, src_index, normals):
        points (m, stride) float32 records -- x, y, z smoothed, every other field copied from source row
        src_index[i] --, normals (m, 4) {nx, ny, nz, curvature} or None.  Points with fewer than 3 neighbours
        within the radius, and non-finite points, have no row."""
        recs = self._records
        if recs is None:
            raise ValueError("mls_smooth needs the cloud's records (not available for a cloud built from a handle)")
        if not isinstance(recs, np.ndarray):   # device-attached cloud: fetch the records once
            ptr, stride = recs
            recs = self.ctx.download(ptr, (self.n, stride // 4), np.float32)
        pts = np.empty((self.n, recs.shape[1]), np.float32)
        src = np.empty(self.n, np.int32)
        nrm = np.empty((self.n, 4), np.float32) if normals else None
        m = C.c_int64(0)
        check(self.lib.ppp_mls_smooth(self._h, float(radius), int(order), _ptr(pts), pts.shape[1] * 4, _ptr(nrm),
                                      _ptr(src), C.byref(m)))
        m = m.value
        src = src[:m].copy()
        out = recs[src].copy()
        out[:, 0:3] = pts[:m, 0:3]
        return out, src, (nrm[:m].copy() if normals else None)

    # ---- device-resident pipeline ---------------------------------------------------------------
    def dev_index(self, k_hint=16, radius_hint=0.0):
        check(self.lib.ppp_dev_index(self._h, int(k_hint), float(radius_hint)))

    def dev_normals_knn(self, k, normals_ptr, normal_stride_bytes, idx_ptr=None, d2_ptr=None, first=0, count=-1,
                        viewpoint=(0.0, 0.0, 0.0), flags=PPP_COV_PCL110):
        vp = np.asarray(viewpoint, np.float32)
        check(self.lib.ppp_dev_normals_knn(self._h, int(k), vp.ctypes.data_as(_lib._f32p), flags, int(first), int(count),
                                           _vp(normals_ptr) if normals_ptr else None, int(normal_stride_bytes),
                                           _vp(idx_ptr) if idx_ptr else None, _vp(d2_ptr) if d2_ptr else None))

    def dev_normals_radius(self, r, normals_ptr, normal_stride_bytes, first=0, count=-1, viewpoint=(0.0, 0.0, 0.0),
                           flags=PPP_COV_PCL110):
        vp = np.asarray(viewpoint, np.float32)
        check(self.lib.ppp_dev_normals_radius(self._h, float(r), vp.ctypes.data_as(_lib._f32p), flags, int(first),
                                              int(count), _vp(normals_ptr), int(normal_stride_bytes)))

    def dev_mls_smooth(self, radius=15.0, order=3, rows_ptr=None, row_stride_bytes=32):
        """ppp_dev_mls_smooth: one 32-byte record {x, y, z, flag, nx, ny, nz, curvature} per point into the device buffer
        rows_ptr (plain cloud) or, on a slab from Exchange.attach, into the home ranks' buffers.  Does not synchronise."""
        check(self.lib.ppp_dev_mls_smooth(self._h, float(radius), int(order), _vp(rows_ptr) if rows_ptr else None,
                                          int(row_stride_bytes)))

    def dev_set_normal_row_map(self, map_ptr):
        """Device int32 map row -> record of the normals buffer (negative: skip); None = identity."""
        check(self.lib.ppp_dev_set_normal_row_map(self._h, _vp(map_ptr) if map_ptr else None))

    def dev_set_contour_offsets_buffer(self, off_ptr, cap_entries):
        check(self.lib.ppp_dev_set_contour_offsets_buffer(self._h, _vp(off_ptr) if off_ptr else None, int(cap_entries)))

    def dev_set_contour_buffers(self, y_ptr, x_ptr, z_ptr, cap):
        check(self.lib.ppp_dev_set_contour_buffers(self._h, _vp(y_ptr) if y_ptr else None, _vp(x_ptr) if x_ptr else None,
                                                   _vp(z_ptr) if z_ptr else None, int(cap)))

    def dev_slice_contours(self, planes, mode, half_width=2.0, truncate_center=True):
        """Returns dict(node_offsets=ptr, y=ptr, x=ptr, z=ptr, total_nodes, total_members); buffers are
        owned by the cloud and valid until the next call."""
        if isinstance(mode, str):
            mode = PPP_PAIR_GEN2 if mode.upper() == "A" else PPP_PAIR_SECT
        planes = np.ascontiguousarray(planes, np.float32)
        po, py, px, pz = _vp(), _vp(), _vp(), _vp()
        tn, tm = C.c_int64(0), C.c_int64(0)
        check(self.lib.ppp_dev_slice_contours(self._h, _ptr(planes), planes.shape[0], half_width, int(truncate_center),
                                              mode, C.byref(po), C.byref(py), C.byref(px), C.byref(pz), C.byref(tn),
                                              C.byref(tm)))
        return dict(node_offsets=po.value, y=py.value, x=px.value, z=pz.value, total_nodes=tn.value,
                    total_members=tm.value)
