"""Python mirror of the reference's operator interface for the hot path (same names, argument
meaning and error behaviour), backed by libppp_gpu.so.  The C++ mirror that a reference
maintainer links is polishpathplanning_b200/host/ (Path_Generate_gpu.h, contour_alg_gpu.h).

  path_generater  : include/Path_Generate.h:35-76  + src/Path_Generation.cpp   (gen-2, ./main)
  SectPath        : include/contour_alg.h:50-91    + src/contour_alg.cpp       (config.txt flow)

The hot-path members (estimate_normal, Set_kdtree, rangedX_index, insert_point, slicing_method,
path_track / OnePath, the GenPath plane sweep) and their direct consumers (SURVEY.md §8f: compute_transform /
Area2Cloud / compute_boundary / bisection / dynamic_adjust_path, drawpath, getPath's way-point sampling and
normal lookup, compute_coverage, remove_outlier) are mirrored; every one of them issues its neighbour queries
for ALL nodes of a path in one device call where the reference loops node by node.  Visualisation, the
hand-eye / flange transforms and file export stay with the reference's own host code.
Plane positions are generated here exactly as each reference loop does, in float32.
"""
import os

import numpy as np

from . import api, synth

_f32 = np.float32


# -------------------------------------------------------------------------------------------------
# plane sweeps (host logic; SURVEY.md Appendix D).  All arithmetic in float32 like the reference.
# -------------------------------------------------------------------------------------------------
def planes_gen2_contact(min_x, max_x, tool_radius):
    """Contact_Path_Generation: float locateX = min.x + toolRadius (double add, then float);
    locateX += int(2R) while locateX < max.x.  src/Path_Generation.cpp:711-723"""
    step = int(tool_radius * 2)
    out = []
    loc = _f32(float(_f32(min_x)) + float(tool_radius))
    while loc < _f32(max_x) and step > 0:
        out.append(loc)
        loc = _f32(loc + _f32(step))
    return np.asarray(out, _f32)


def planes_gen2_slicing(min_x, max_x, tool_radius):
    """slicing_method: min.x += step/2 (INTEGER division), += step.  src/Path_Generation.cpp:295-303"""
    step = int(tool_radius * 2)
    out = []
    m = _f32(_f32(min_x) + _f32(step // 2))
    while m < _f32(max_x) and step > 0:
        out.append(m)
        m = _f32(m + _f32(step))
    return np.asarray(out, _f32)


def planes_gen1_slicing(min_x, max_x):
    """free slicing_method: first plane min.x + 40, step 40.  src/slicing_method.cpp:617-626"""
    out = []
    m = _f32(_f32(min_x) + _f32(40))
    while m < _f32(max_x):
        out.append(m)
        m = _f32(m + _f32(40))
    return np.asarray(out, _f32)


def planes_sectpath(min_x, max_x, tool_radius):
    """SectPath::GenPath: backward from centre - step while > min.x (inserted at the front), then
    forward from the centre while < max.x.  Returned in Path_set order.  src/contour_alg.cpp:305-327"""
    step = int(tool_radius * 2)
    centre = _f32(_f32(_f32(min_x) + _f32(max_x)) / _f32(2))
    front, back = [], []
    loc = _f32(centre - _f32(step))
    while loc > _f32(min_x) and step > 0:
        front.insert(0, loc)
        loc = _f32(loc - _f32(step))
    loc = centre
    while loc < _f32(max_x) and step > 0:
        back.append(loc)
        loc = _f32(loc + _f32(step))
    return np.asarray(front + back, _f32)


def planes_gen3_two_thread(min_x, max_x, tool_radius):
    """gen-3 path_generater::GenPath + thread_worker (src/Path_Alg/path_dynamic_alg.cpp:308-366): the centre path at
    the FLOAT centre (min.x + max.x) / 2; the two workers walk outwards in INT steps from the centre of the
    int-TRUNCATED bounding box (include/Path_Generate_Algorithm.h:110-117), while max > loc && loc > min.
    Returned in Path_set order (ascending x)."""
    step = int(tool_radius * 2)
    mn, mx = int(_f32(min_x)), int(_f32(max_x))
    mid = int((mx + mn) / 2)                      # C int division; both truncate toward zero
    front, back = [], []
    loc = mid - step
    while mx > loc > mn and step > 0:
        front.insert(0, _f32(loc))
        loc -= step
    loc = mid + step
    while mx > loc > mn and step > 0:
        back.append(_f32(loc))
        loc += step
    centre = _f32(_f32(_f32(min_x) + _f32(max_x)) / _f32(2))
    return np.asarray(front + [centre] + back, _f32)


def planes_gen3_sdir(min_x, max_x, tool_radius):
    """gen-3 single-direction sweep (src/Path_Alg/dynamic_alg_sdir.cpp:349-374): int loc = min_pt.x + toolRadius
    (float + double, truncated), first path there, then loc += int(2R) while loc < max_pt.x: planes at integer x."""
    step = int(tool_radius * 2)
    loc = int(float(_f32(min_x)) + float(tool_radius))
    out = [_f32(loc)]
    loc += step
    while _f32(loc) < _f32(max_x) and step > 0:
        out.append(_f32(loc))
        loc += step
    return np.asarray(out, _f32)


class Spline:
    """include/Spline.h:7-51 — two GSL Steffen splines x(y), z(y) over the ordered contour nodes.
    gsl_interp_steffen [upstream, recalled: GSL is not in the image]: monotone cubic Hermite of
    Steffen (1990); same arithmetic order as the oracle restatement, in float64."""

    def __init__(self, point_y, point_x, point_z):
        y = np.ascontiguousarray(point_y, np.float64)
        if y.shape[0] < 3 or not np.all(np.diff(y) > 0):
            raise ValueError("Spline needs >= 3 strictly increasing y (GSL would abort)")
        self.y = y
        self._cx = self._coeffs(y, np.ascontiguousarray(point_x, np.float64))
        self._cz = self._coeffs(y, np.ascontiguousarray(point_z, np.float64))
        self.small_y, self.big_y = float(y[0]), float(y[-1])

    @staticmethod
    def _coeffs(xa, ya):
        n = xa.shape[0]
        h = xa[1:] - xa[:-1]
        s = (ya[1:] - ya[:-1]) / h
        yp = np.empty(n, np.float64)
        yp[0] = s[0]
        hi, him1, si, sim1 = h[1:], h[:-1], s[1:], s[:-1]
        pi = (sim1 * hi + si * him1) / (him1 + hi)
        yp[1:-1] = (np.copysign(1.0, sim1) + np.copysign(1.0, si)) * np.minimum(np.abs(sim1), np.minimum(np.abs(si), 0.5 * np.abs(pi)))
        yp[-1] = s[-1]
        a = (yp[:-1] + yp[1:] - 2 * s) / h / h
        b = (3 * s - 2 * yp[:-1] - yp[1:]) / h
        return a, b, yp[:-1].copy(), ya[:-1].copy()

    def _eval(self, c, yq):
        a, b, cc, d = c
        yq = np.asarray(yq, np.float64)
        i = np.clip(np.searchsorted(self.y, yq, side="right") - 1, 0, self.y.shape[0] - 2)
        dx = yq - self.y[i]
        out = d[i] + dx * (cc[i] + dx * (b[i] + dx * a[i]))
        return np.where((yq >= self.y[0]) & (yq <= self.y[-1]), out, np.nan)

    def point(self, y):
        """Eigen::Vector3d point(double y): (x(y), y, z(y)); vectorised over y."""
        y = np.atleast_1d(np.asarray(y, np.float64))
        return np.stack([self._eval(self._cx, y), y, self._eval(self._cz, y)], axis=1)

    def miny(self):
        return self.small_y

    def bigy(self):
        return self.big_y


class _Base:
    NORMAL_RADIUS = 2.5   # normal_estimation.setRadiusSearch(2.5): src/Path_Generation.cpp:329
    BAND_HALF_WIDTH = 2.0  # setFilterLimits(-2 + position, 2 + position): src/Path_Generation.cpp:100
    SMOOTH_RADIUS = 15.0   # mls.setSearchRadius(15): src/Path_Generation.cpp:340-360
    SMOOTH_ORDER = 3       # mls.setPolynomialOrder(3)

    def __init__(self, ctx=None, device=0, backend=None):
        # backend: callable(cloud) -> an object with api.Cloud's methods; the CPU tests pass an oracle-backed
        # stand-in so that the host logic here can be checked without a GPU (the product path never does)
        self._backend = backend
        self._ctx = None if backend is not None else (ctx or api.Context(device))
        self._gpu = None
        self.cloud = None
        self.cloud_with_normals = None
        self.Path_set = []

    def _load(self, cloud_name, change_range=True):
        self.cloud_name = cloud_name if isinstance(cloud_name, str) else "cloud.pcd"
        if isinstance(cloud_name, str):
            try:
                cloud = synth.read_pcd(cloud_name)
            except (OSError, ValueError) as e:
                # the reference prints PCL_ERROR and carries on with an empty cloud
                print("Cloudn't read file! (%s)" % e)
                cloud = np.zeros((0, synth.POINT_STRIDE_FLOATS), np.float32)
        else:
            cloud = np.ascontiguousarray(cloud_name, np.float32).copy()
        if change_range:
            synth.reference_ctor_scale(cloud)
        self.cloud = cloud
        self._invalidate()

    def _invalidate(self):
        """xyz changed (voxel_down / trans2center / smooth / remove_outlier in the reference):
        drop the device copy and its index."""
        if self._gpu is not None:
            self._gpu.close()
        self._gpu = None

    def _dev(self):
        if self._gpu is None:
            self._gpu = self._backend(self.cloud) if self._backend is not None else api.Cloud(self._ctx, self.cloud)
        return self._gpu

    # -- mirrored members ---------------------------------------------------------------------------
    def Set_kdtree(self):
        """kdtree.setInputCloud(cloud): builds the device index."""
        self._dev().dev_index(16, 0.0)

    def estimate_normal(self):
        """NormalEstimation, radius 2.5, viewpoint (0,0,0) -> (N, 8) pcl::Normal records."""
        self.cloud_with_normals = self._dev().normals_radius(self.NORMAL_RADIUS)
        return self.cloud_with_normals

    def smooth(self):
        """smooth() (src/Path_Generation.cpp:340-360): MovingLeastSquares, order 3, radius 15, no upsampling,
        SIMPLE projection.  The cloud becomes the smoothed records (points with fewer than 3 neighbours are
        dropped; fields other than x, y, z come from the source point), is written to smooth_<file name>.pcd in
        the working directory, and the device copy is rebuilt on next use.  Returns the source index per row."""
        pts, src, _ = self._dev().mls_smooth(self.SMOOTH_RADIUS, self.SMOOTH_ORDER)
        self.cloud = np.ascontiguousarray(pts)
        self._invalidate()
        synth.write_pcd("smooth_" + os.path.basename(self.cloud_name), self.cloud)
        return src

    def rangedX_index(self, position):
        """std::vector<int> rangedX_index(int position): the argument is truncated to int."""
        position = int(position)
        off, idx = self._dev().slice_bands(np.asarray([position], _f32), self.BAND_HALF_WIDTH, True)
        return idx

    def getMinMax3D(self):
        return self._dev().bbox()

    def _contours(self, planes, mode):
        return self._dev().slice_contours(np.asarray(planes, _f32), mode, self.BAND_HALF_WIDTH, True)

    # -- "next" rows (SURVEY.md §8f): consumers of the ordered contours --------------------------------
    def splines(self):
        """Spline objects of Path_set (paths with < 3 nodes are skipped, GSL would abort on them)."""
        return [Spline(y, x, z) for (y, x, z) in self.Path_set if len(y) >= 3]

    def drawpath_samples(self, path, gen2=True):
        """The sample points drawpath snaps to the cloud: gen-2 takes 200 samples
        dy = (maxy-miny)/200*i + miny (src/Path_Generation.cpp:644-646); SectPath steps dy += 1
        while dy < maxy (src/contour_alg.cpp:273-283)."""
        miny, maxy = path.miny(), path.bigy()
        if gen2:
            dy = (maxy - miny) / 200 * np.arange(200) + miny
        else:
            dy = miny + np.arange(int(np.ceil(maxy - miny)) + 1, dtype=np.float64)
            dy = dy[dy < maxy]
        return path.point(dy)

    def drawpath(self, path, gen2=True):
        """Indices of the cloud points drawpath recolours: nearestKSearch(point, k)[0] per sample
        (k = 3 in gen-2, 1 in SectPath: only element [0] is used)."""
        pts = self.drawpath_samples(path, gen2).astype(np.float32)   # PCLp.x = pathPoint[0] (double -> float)
        idx, _ = self._dev().knn(1, queries=np.ascontiguousarray(pts), want_d2=False)
        return idx[:, 0]

    def compute_transform(self, points, k=10):
        """Batched compute_transform (src/Path_Generation.cpp:362-400; k = 50 in the gen-3 planner):
        returns (pt2Base matrices (n,4,4) float32, principle_curvature (n,2))."""
        pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
        out, nn0 = self._dev().principal_curvatures(self.cloud_with_normals, pts, k)
        nrm = self.cloud_with_normals[nn0, 0:3]
        cur = out[:, 0:3]
        # Eigen cross: normalVector.cross(curvatureVector), float32
        cr = np.stack([nrm[:, 1] * cur[:, 2] - nrm[:, 2] * cur[:, 1], nrm[:, 2] * cur[:, 0] - nrm[:, 0] * cur[:, 2],
                       nrm[:, 0] * cur[:, 1] - nrm[:, 1] * cur[:, 0]], axis=1).astype(np.float32)
        Y = np.zeros((pts.shape[0], 4, 4), np.float32)
        Y[:, :3, 0], Y[:, :3, 1], Y[:, :3, 2], Y[:, :3, 3], Y[:, 3, 3] = cr, cur, nrm, pts, 1.0
        return Y, out[:, 3:5]

    # -- Area2Cloud / compute_boundary / bisection (src/Path_Generation.cpp:403-585), batched over nodes -----------
    DEPTH = 0.005            # double depth = 0.005            include/Path_Generate.h:70
    ADJUST_THRESHOLD = 1.0   # Adjust_Threshold = 1
    TOOLTHICKNESS = 10.0     # toolthickness = 10

    def _ellipse_axes(self, pc):
        """longAxis / shortAxis of Area2Cloud (src/Path_Generation.cpp:415-436) from principle_curvature[0..1]
        (float32): 1 / pc is a float division, everything after it double."""
        pc = np.asarray(pc, np.float32)
        with np.errstate(divide="ignore", invalid="ignore"):
            inv1 = (_f32(1) / pc[:, 1]).astype(np.float64)
            inv0 = (_f32(1) / pc[:, 0]).astype(np.float64)
            R, depth, thick = float(self.toolRadius), self.DEPTH, self.TOOLTHICKNESS
            la_pos = np.sqrt(inv1 * inv1 - (np.abs(inv1) - depth) ** 2)
            sa_pos = np.sqrt(inv0 * inv0 - (np.abs(inv0) - depth) ** 2)
            la_pos = np.where(la_pos > R, R, la_pos)
            sa_pos = np.where(sa_pos > R, R, sa_pos)
            la_neg = np.abs(inv1) - np.sqrt(inv1 * inv1 - R * R)
            sa_neg = np.abs(inv0) - np.sqrt(inv0 * inv0 - R * R)
            la_neg = np.where(la_neg > thick, thick, la_neg)
            sa_neg = np.where(sa_neg > thick, thick, sa_neg)
        both = (pc[:, 0] >= 0) & (pc[:, 1] >= 0)
        return np.where(both, la_pos, la_neg), np.where(both, sa_pos, sa_neg)

    _ELLIPSE_ANGLE = np.arange(721, dtype=np.float32) * _f32(0.5)            # for (float angle(0.0); angle <= 360.0; angle += 0.5)
    _ELLIPSE_COS = np.cos(_ELLIPSE_ANGLE * _f32(0.017453293))                # std::cos(pcl::deg2rad(angle)), float
    _ELLIPSE_SIN = np.sin(_ELLIPSE_ANGLE * _f32(0.017453293))

    def Area2Cloud(self, points, flag=False, key=False, k=10):
        """Eigen::Vector3f Area2Cloud(PathNode, flag, key) for a BATCH of path nodes: one device call for the
        k-nearest-neighbour + principal-curvature part of every node, the 721-point contact ellipse of each node
        transformed to the node (float32, as pcl::transformPointCloud) and its extreme-x point picked
        (key = 0: max x, the "up" boundary, + compute_coverage with the ellipse half-width; key = 1: min x).
        Returns (n, 3) float32 boundary points.  flag (draw the ellipse into other_cloud) is visual only."""
        pts = np.asarray(points, np.float64).reshape(-1, 3)
        sp = pts.astype(np.float32)                               # SearchPoint.x = point[0] ...
        T, pc = self.compute_transform(sp, k)
        la, sa = self._ellipse_axes(pc)
        ex = (la[:, None] * self._ELLIPSE_COS[None, :].astype(np.float64)).astype(np.float32)   # double * float -> float
        ey = (sa[:, None] * self._ELLIPSE_SIN[None, :].astype(np.float64)).astype(np.float32)
        # pcl::transformPointCloud [upstream, recalled: PCL 1.10 detail::Transformer, SSE form]:
        # out = x * c0 + (y * c1 + (z * c2 + c3)) with z = 0, all float32
        out = []
        for r in range(3):
            c0, c1, c2, c3 = T[:, r, 0][:, None], T[:, r, 1][:, None], T[:, r, 2][:, None], T[:, r, 3][:, None]
            with np.errstate(invalid="ignore"):
                out.append(ex * c0 + (ey * c1 + (_f32(0) * c2 + c3)))
        tx, ty, tz = out
        with np.errstate(invalid="ignore"):
            hi = np.argmax(np.where(np.isnan(tx), -np.inf, tx), axis=1)      # first largest / first smallest element
            lo = np.argmin(np.where(np.isnan(tx), np.inf, tx), axis=1)
        rows = np.arange(pts.shape[0])
        pick = lo if key else hi
        bound = np.stack([tx[rows, pick], ty[rows, pick], tz[rows, pick]], axis=1).astype(np.float32)
        bound[np.isnan(tx).any(axis=1)] = np.nan
        if not key:
            comput_lan = ((tx[rows, lo] - tx[rows, hi]) / _f32(2)).astype(np.float64)       # float arithmetic, then double
            self.compute_coverage_radii(pts, comput_lan)
        return bound

    def compute_coverage_radii(self, nodes, radii):
        if not hasattr(self, "coverage_flag") or self.coverage_flag.shape[0] != self.cloud.shape[0]:
            self.coverage_flag = np.zeros(self.cloud.shape[0], np.uint8)
        q = np.ascontiguousarray(np.asarray(nodes, np.float64).astype(np.float32).reshape(-1, 3))
        self._dev().coverage_mark_radii(q, np.asarray(radii, np.float64), self.coverage_flag)
        return self.coverage_flag

    def compute_boundary(self, path):
        """int compute_boundary(Spline path, Spline* boundary) (src/Path_Generation.cpp:499-553): the "up" boundary
        points of the nodes dy = miny + 2, += toolRadius / 4 while dy < maxy - 2, keyed by their y in a std::map
        (ascending, last insertion wins), extended by 20 at both ends.  The reference's extra "last point" call
        re-uses the last node (its dy is never applied), so it only repeats an insertion.  Returns a Spline, or
        None where the reference returns 0 (fewer than 3 distinct boundary nodes)."""
        miny, maxy = path.miny(), path.bigy()
        dys = []
        dy = miny + 2
        while dy < maxy - 2:
            dys.append(dy)
            dy += self.toolRadius / 4
        if not dys:
            return None
        bp = self.Area2Cloud(path.point(np.asarray(dys)), True, False)
        node = {}
        for b in bp:
            if np.isnan(b[0]):
                continue                                          # "Area Estimatin is NAN"
            node[float(b[1])] = (float(b[0]), float(b[2]))
        last = bp[-1]
        node[float(last[1])] = (float(last[0]), float(last[2]))  # the unconditional insertion after the loop
        keys = sorted(kk for kk in node if not np.isnan(kk))
        if np.isnan(last[1]):
            keys.append(float("nan"))                             # a NaN key would sit somewhere in the map; GSL then aborts
        if len(keys) <= 2:
            return None
        y = np.empty(len(keys) + 2)
        x = np.empty_like(y)
        z = np.empty_like(y)
        y[1:-1] = keys
        x[1:-1] = [node[kk][0] for kk in keys]
        z[1:-1] = [node[kk][1] for kk in keys]
        x[0], y[0], z[0] = x[1], y[1] - 20, z[1]
        x[-1], y[-1], z[-1] = x[-2], y[-2] + 20, z[-2]
        return Spline(y, x, z)

    def bisection(self, nodes, boundary):
        """Eigen::Vector3d bisection(PathNode, boundary, itr = 0) for a batch of nodes: up to six rounds of
        "down" boundary point -> offset against the boundary spline -> shift the node in x; every round is ONE
        batched Area2Cloud over the nodes still moving (src/Path_Generation.cpp:555-585)."""
        nodes = np.array(nodes, np.float64).reshape(-1, 3)
        active = np.ones(nodes.shape[0], bool)
        for _ in range(6):                                        # itr = 0..5; itr > 5 returns
            ids = np.nonzero(active)[0]
            if not len(ids):
                break
            ab = self.Area2Cloud(nodes[ids], False, True)
            aby = ab[:, 1].astype(np.float64)
            with np.errstate(invalid="ignore"):
                overflow = (aby < boundary.miny()) | (aby > boundary.bigy())
            bpt = boundary.point(np.where(overflow | np.isnan(aby), boundary.miny(), aby))
            norm0 = ab[:, 0].astype(np.float64) - bpt[:, 0]
            with np.errstate(invalid="ignore"):
                stop = overflow | (np.abs(norm0) < self.ADJUST_THRESHOLD)
            move = ids[~stop]
            nodes[move, 0] = nodes[move, 0] - norm0[~stop]
            active[ids[stop]] = False
            active[move[np.isnan(nodes[move, 0])]] = False        # "adjust path node NAN"
        return nodes

    def dynamic_adjust_path(self, origin_path, pre_path):
        """void dynamic_adjust_path(Spline* origin_path, Spline pre_path) (src/Path_Generation.cpp:587-634): returns
        the re-started origin path (None where the reference prints "generate boundary fail" and leaves it)."""
        boundary = self.compute_boundary(pre_path)
        if boundary is None:
            return None
        miny, maxy = origin_path.miny(), origin_path.bigy()
        num = int((maxy - miny) / 5)
        if num <= 1:
            raise ValueError("dynamic_adjust_path: path shorter than 10: the reference re-starts a spline without nodes (GSL aborts)")
        i = np.arange(1, num, dtype=np.float64)
        dy = ((maxy - miny) / num * i) + miny
        nodes = self.bisection(origin_path.point(dy), boundary)
        snap = self._snap(nodes)                                  # kdtree.nearestKSearch(point, 3)[0]
        new_path = {}
        for j in snap:
            p = self.cloud[j]
            new_path[float(p[1])] = (float(p[0]), float(p[2]))
        keys = sorted(new_path)
        return Spline(np.asarray(keys), np.asarray([new_path[kk][0] for kk in keys]), np.asarray([new_path[kk][1] for kk in keys]))

    def _snap(self, nodes):
        """Index of the nearest cloud point of every node (one device call)."""
        q = np.ascontiguousarray(np.asarray(nodes, np.float64).astype(np.float32).reshape(-1, 3))
        idx, _ = self._dev().knn(1, queries=q, want_d2=False)
        return idx[:, 0]

    def compute_coverage(self, nodes, radius):
        """compute_coverage for a batch of nodes (src/Path_Generation.cpp:483-496)."""
        if not hasattr(self, "coverage_flag") or self.coverage_flag.shape[0] != self.cloud.shape[0]:
            self.coverage_flag = np.zeros(self.cloud.shape[0], np.uint8)
        q = np.ascontiguousarray(np.asarray(nodes, np.float64).astype(np.float32).reshape(-1, 3))
        self._dev().coverage_mark(q, radius, self.coverage_flag)
        return self.coverage_flag

    def get_coverage(self):
        """get_coverage (src/Path_Generation.cpp:757-771): rate = yes / (yes + no), float arithmetic."""
        yes = _f32(int(self.coverage_flag.sum()))
        no = _f32(int(self.coverage_flag.shape[0] - self.coverage_flag.sum()))
        return float(yes / (yes + no))


class path_generater(_Base):
    """gen-2 planner (what ./main builds): brute-force pairing with greedy flags (variant A)."""

    def __init__(self, cloud_name, Radius, ctx=None, device=0, backend=None):
        super().__init__(ctx, device, backend)
        self.toolRadius = float(Radius)
        self._load(cloud_name, change_range=True)

    def voxel_down(self, leaf):
        """voxel_down() (src/Path_Generation.cpp:53-59): pcl::VoxelGrid, filter(*cloud).  The reference's leaf size
        is not part of this repository, so it is an argument (one float or three).  The cloud becomes one record per
        occupied voxel (Cloud.voxel_grid) and the device copy is rebuilt on next use.  Where PCL warns that the leaf
        is too small and keeps the input, so does this (and prints PCL's warning).  Returns the row offsets and
        members of the voxels, or None when the cloud was kept."""
        try:
            recs, off, mem = self._dev().voxel_grid(leaf)
        except api.PPPError as e:
            if e.status != api._lib.PPP_ERR_UNSUPPORTED:
                raise
            print("[pcl::VoxelGrid::applyFilter] %s" % api._lib.load().ppp_last_error().decode())
            return None
        self.cloud = np.ascontiguousarray(recs)
        self._invalidate()
        return off, mem

    def insert_point(self, indices, PlanePoint):
        """std::map<double, std::vector<double>> insert_point(indices, PlanePoint): returns the map
        as (y, x, z) arrays in ascending y.  `indices`: strictly ascending point indices (every reference
        call site passes rangedX_index(PlanePoint[0]), src/Path_Generation.cpp:300-301,665)."""
        return self._dev().insert_point(np.asarray(indices, np.int32), _f32(PlanePoint[0]), api.PPP_PAIR_GEN2)

    def path_track(self, plane_point):
        y, x, z = self.insert_point(self.rangedX_index(plane_point[0]), plane_point)
        self.Path_set.append((y, x, z))  # Spline(node_number, point_y, point_x, point_z)

    def slicing_method(self):
        """All planes of the sweep in one device pass; returns (planes, node_offsets, y, x, z)."""
        mn, mx = self.getMinMax3D()
        planes = planes_gen2_slicing(mn[0], mx[0], self.toolRadius)
        off, y, x, z = self._contours(planes, api.PPP_PAIR_GEN2)
        print("number of paths: %d" % len(planes))
        return planes, off, y, x, z

    def Contact_Path_Generation(self, adjust=False):
        """void Contact_Path_Generation() (src/Path_Generation.cpp:689-755).  The contours of ALL planes come from
        one device pass (they depend on the cloud only).  adjust = False stops there (Path_set = the raw contours).
        adjust = True replays the reference's sweep: for every plane compute_boundary of the fresh path (coverage
        flags), then, from the second plane on, dynamic_adjust_path against the previous (already adjusted) path --
        sequential from plane to plane as in the reference, batched over the nodes inside each call."""
        if self.cloud_with_normals is None and adjust:
            self.estimate_normal()
        self.coverage_flag = np.zeros(self.cloud.shape[0], np.uint8)
        mn, mx = self.getMinMax3D()
        planes = planes_gen2_contact(mn[0], mx[0], self.toolRadius)
        off, y, x, z = self._contours(planes, api.PPP_PAIR_GEN2)
        self.Path_set = [(y[off[s]:off[s + 1]], x[off[s]:off[s + 1]], z[off[s]:off[s + 1]]) for s in range(len(planes))]
        if adjust:
            paths = []
            for s, (py, px, pz) in enumerate(self.Path_set):
                path = Spline(py, px, pz)                         # path_track: GSL aborts on < 3 nodes, so does this
                self.compute_boundary(path)
                if s > 0:
                    path = self.dynamic_adjust_path(path, paths[s - 1]) or path
                paths.append(path)
            self.Path_splines = paths
        print("Number of paths: %d" % len(planes))
        return planes


def sor_select(distances, n_valid, stddev_mul=1.0, negative=False):
    """Second pass of pcl::StatisticalOutlierRemoval::applyFilterIndices: running double sums in index
    order over all distances (np.cumsum accumulates sequentially), variance over n_valid - 1, inliers
    distance <= mean + stddev_mul * stddev.  Returns (kept indices ascending, threshold)."""
    d = np.ascontiguousarray(distances, np.float32)
    if d.shape[0] == 0 or n_valid < 1:
        return np.zeros(0, np.int32), float("nan")
    total = float(np.cumsum(d.astype(np.float64))[-1])
    sq_total = float(np.cumsum((d * d).astype(np.float64))[-1])        # float32 products, widened when added
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = np.float64(total) / np.float64(n_valid)
        variance = (np.float64(sq_total) - np.float64(total) * np.float64(total) / np.float64(n_valid)) / (np.float64(n_valid) - 1.0)
        thr = float(mean + np.float64(stddev_mul) * np.sqrt(variance))
    outlier = (d <= thr) if negative else (d > thr)
    return np.flatnonzero(~outlier).astype(np.int32), thr


class SectPath(_Base):
    """SectPath (contour_alg.h): kd-tree pairing without flags (variant B), centre-out sweep."""

    def __init__(self, cloud_name, Tool_Radius, ChangeRange=True, RemoveOutlier=False, Smooth=False, ctx=None, device=0,
                 backend=None):
        super().__init__(ctx, device, backend)
        self.toolRadius = float(Tool_Radius)
        self._load(cloud_name, change_range=ChangeRange)
        if Smooth:                                          # src/contour_alg.cpp:27, before remove_outlier
            self.smooth()
        if RemoveOutlier and self.cloud.shape[0] > 50:      # src/contour_alg.cpp:29
            self.remove_outlier()

    def insert_point(self, indices, PlanePoint):
        return self._dev().insert_point(np.asarray(indices, np.int32), _f32(PlanePoint[0]), api.PPP_PAIR_SECT)

    def remove_outlier(self, mean_k=50, stddev_mul=1.0):
        """SectPath::remove_outlier (src/contour_alg.cpp:101-108): StatisticalOutlierRemoval with
        setMeanK(50), setStddevMulThresh(1.0), filtered in place.  The kNN pass runs on the device; the
        mean / stddev / threshold pass is the reference's sequential double arithmetic."""
        dist, n_valid = self._dev().sor_mean_distances(mean_k)
        keep, _ = sor_select(dist, n_valid, stddev_mul)
        self.cloud = np.ascontiguousarray(self.cloud[keep])
        self._invalidate()
        return keep

    def OnePath(self, plane_point):
        return self.insert_point(self.rangedX_index(plane_point[0]), plane_point)

    def getPath_waypoints(self, PathResolution, TransAlign=None):
        """The device-backed part of SectPath::getPath (src/contour_alg.cpp:483-540): drop the first and the last
        path, sample every path at dy = miny + 5, += PathResolution while dy < bigy - 5, map the samples through
        inverse(TransAlign) (float32 4x4), reverse every second path (boustrophedon), then for ALL way-points in one
        device call the nearest cloud point (kdtree.nearestKSearch(SPoint, 1)) whose normal gives the tool frame:
        Approach = -N, Orientation = Approach x UnitX, Normal = Orientation x Approach (float32 cross products).
        Returns (xyz (m, 3) float32, nearest index (m,), rotation matrices (m, 3, 3) float32 with columns
        Normal | Orientation | Approach, TailIndex: last way-point of every path).  The cloud is expected in the
        frame the way-points end up in (the reference transforms cloud and way-points by the same inverse);
        eulerAngles / HandEyeTransform / smoothing / file export stay host code of the reference."""
        inv = np.linalg.inv(np.asarray(TransAlign, np.float32)).astype(np.float32) if TransAlign is not None else np.eye(4, dtype=np.float32)
        paths = self.splines()[1:-1] if len(self.Path_set) >= 2 else []
        chunks, tails, flag, total = [], [], 1, 0
        for path in paths:
            dys = []
            dy = path.miny() + 5
            while dy < path.bigy() - 5:
                dys.append(dy)
                dy += PathResolution
            p = path.point(np.asarray(dys)) if dys else np.zeros((0, 3))
            px, py, pz = (p[:, j].astype(np.float32)[:, None] for j in range(3))                    # Vector4f(x, y, z, 1)
            w = (((inv[None, :, 0] * px + inv[None, :, 1] * py) + inv[None, :, 2] * pz) + inv[None, :, 3]).astype(np.float32)  # column by column
            if flag == -1:
                w = w[::-1]
            chunks.append(w[:, :3])
            total += w.shape[0]
            tails.append(total - 1)
            flag *= -1
        xyz = np.ascontiguousarray(np.concatenate(chunks, axis=0) if chunks else np.zeros((0, 3), np.float32))
        if self.cloud_with_normals is None:
            self.estimate_normal()
        idx = self._snap(xyz) if xyz.shape[0] else np.zeros(0, np.int32)
        N = self.cloud_with_normals[idx, 0:3]
        A = (-N).astype(np.float32)
        ux = np.asarray([1, 0, 0], np.float32)
        cross = lambda a, b: np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                                       a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1).astype(np.float32)
        O = cross(A, np.broadcast_to(ux, A.shape))
        Nn = cross(O, A)
        rot = np.stack([Nn, O, A], axis=2).astype(np.float32)      # columns Normal | Orientation | Approach
        return xyz, idx, rot, np.asarray(tails, np.int64)

    def GenPath(self):
        mn, mx = self.getMinMax3D()
        planes = planes_sectpath(mn[0], mx[0], self.toolRadius)
        off, y, x, z = self._contours(planes, api.PPP_PAIR_SECT)
        self.Path_set = [(y[off[s]:off[s + 1]], x[off[s]:off[s + 1]], z[off[s]:off[s + 1]]) for s in range(len(planes))]
        print("Number of paths: %d" % len(planes))
        print("Number of Point Cloud: %d" % self.cloud.shape[0])
        return planes
