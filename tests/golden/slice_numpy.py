"""Brute-force numpy restatement of the slicing chain (DESIGN §1, A4-A9): PassThrough bands, left/right
classification, gen-2 pairing (variant A), SectPath pairing (variant B), interpolation onto the plane and the
std::map<double, ...> node order.  Plain numpy float32 / float64; nothing is shared with oracle/ or the product.

Reference lines restated:
  A4 rangedX_index     src/Path_Generation.cpp:94-104, src/contour_alg.cpp:153-163 (pcl::PassThrough on x)
  A5 classify          src/Path_Generation.cpp:110-128: (p - PlanePoint).dot((1, 0, 0)) > 0 left, < 0 right
  A6 pairing A         src/Path_Generation.cpp:129-179: std::map<float, int> of Eigen norms (equal keys keep the last
                       j), then the greedy flag pass (right pushed before the left flag is tested)
  A7 pairing B         src/contour_alg.cpp:185-211: kd-trees over El and Er, nearestKSearch(., 1), every winner
                       replaced by kdtree.nearestKSearch(winner, 1) over the whole cloud
  A8 interpolate + map src/Path_Generation.cpp:181-205: node[(double)y] = {x, z}; the loop runs over left_pair.size()
  A9 flatten           src/Path_Generation.cpp:659-676: the map in ascending key order as (y, x, z) arrays

Rules that are this library's contract rather than the reference's text:
  - a plane that is not finite or has |x| >= 2e9 has an empty band (the truncating limits would overflow int);
  - nearest-neighbour ties in variant B go to the lowest index (FLANN keeps the first point its tree visits);
  - a point that is not finite is on neither side.  The reference's dot product is NaN for an infinite or NaN y or z;
    for x = +-inf with finite y and z the reference would hand an infinite point to FLANN, and this library drops it.
"""
import numpy as np

F32 = np.float32
_CHUNK = 1 << 22   # matrix elements per block of the brute-force searches


def band_limits(plane, half_width=2.0, truncate_center=True):
    """(lo, hi) as float32, or None for a plane that gets an empty band."""
    p, hw = F32(plane), F32(half_width)
    if not np.isfinite(p) or abs(p) >= F32(2.0e9):
        return None
    if truncate_center:   # rangedX_index(int position): (float)(-hw + position), (float)(hw + position)
        pos, h = int(p), int(hw)
        return F32(float(-h + pos)), F32(float(h + pos))
    return F32(p - hw), F32(p + hw)


def finite3(pts):
    return np.isfinite(pts[:, :3]).all(axis=1)


def band(pts, plane, half_width=2.0, truncate_center=True):
    """PassThrough("x"): finite points with !(x < lo || x > hi), ascending index."""
    lim = band_limits(plane, half_width, truncate_center)
    if lim is None:
        return np.zeros(0, np.int32)
    lo, hi = lim
    x = pts[:, 0]
    with np.errstate(invalid="ignore"):
        keep = finite3(pts) & ~((x < lo) | (x > hi))
    return np.flatnonzero(keep).astype(np.int32)


def slice_bands(pts, planes, half_width=2.0, truncate_center=True):
    bands = [band(pts, p, half_width, truncate_center) for p in np.asarray(planes, F32)]
    off = np.zeros(len(bands) + 1, np.int64)
    off[1:] = np.cumsum([b.shape[0] for b in bands])
    return off, (np.concatenate(bands) if bands else np.zeros(0, np.int32)).astype(np.int32)


def classify(pts, ind, plane):
    """(El, Er) in list order: dx * 1 + (dy * 0 + dz * 0) in float32, > 0 left, < 0 right."""
    ind = np.asarray(ind, np.int32)
    q = pts[ind, :3].astype(F32)
    P = F32(plane)
    with np.errstate(invalid="ignore", over="ignore"):
        d = (q[:, 0] - P) * F32(1.0) + ((q[:, 1] - F32(0.0)) * F32(0.0) + (q[:, 2] - F32(0.0)) * F32(0.0))
    fin = np.isfinite(q).all(axis=1)
    return ind[(d > 0) & fin], ind[(d < 0) & fin]


def _nearest(pts, queries, cand, metric):
    """Position in `cand` (ascending indices) of each query's nearest candidate.
    metric 0: FLANN d2 ((dx² + dy²) + dz²), ties -> first (lowest index).
    metric 1: Eigen norm sqrt(dx² + (dy² + dz²)), ties -> last (highest index)."""
    C = pts[cand, :3].astype(F32)
    Q = pts[queries, :3].astype(F32)
    out = np.empty(Q.shape[0], np.int64)
    step = max(1, _CHUNK // max(C.shape[0], 1))
    for a in range(0, Q.shape[0], step):
        q = Q[a:a + step]
        dx = q[:, None, 0] - C[None, :, 0]
        dy = q[:, None, 1] - C[None, :, 1]
        dz = q[:, None, 2] - C[None, :, 2]
        if metric == 0:
            d = (dx * dx + dy * dy) + dz * dz
            out[a:a + step] = np.argmin(d, axis=1)
        else:
            d = np.sqrt(dx * dx + (dy * dy + dz * dz))
            out[a:a + step] = C.shape[0] - 1 - np.argmin(d[:, ::-1], axis=1)
    return out


def pair_a(pts, El, Er):
    """gen-2: nearest right of every left and nearest left of every right, then the greedy flag pass."""
    lp, rp = [], []
    if El.shape[0] == 0 or Er.shape[0] == 0:
        return np.array(lp, np.int32), np.array(rp, np.int32)
    posR = _nearest(pts, El, Er, 1)
    posL = _nearest(pts, Er, El, 1)
    fl = np.zeros(El.shape[0], bool)
    fr = np.zeros(Er.shape[0], bool)
    for i in range(El.shape[0]):
        if fl[i]:
            continue
        j = posR[i]
        if fr[j]:
            continue
        rp.append(Er[j])
        fr[j] = True
        i2 = posL[j]
        if not fl[i2]:
            lp.append(El[i2])
            fl[i2] = True
    return np.array(lp, np.int32), np.array(rp, np.int32)


class Cloud:
    """The cloud plus what NN_full needs: kdtree.nearestKSearch(p, 1) for a cloud point p is the lowest index among the
    finite points at float32 d² == 0 from p.  Such points differ from p by less than 2^-75 in every coordinate, so the
    candidates come from a sort on x and are confirmed with the float32 d²."""

    def __init__(self, pts):
        self.pts = np.ascontiguousarray(pts, F32)
        fin = np.flatnonzero(finite3(self.pts))
        order = np.argsort(self.pts[fin, 0].astype(np.float64), kind="stable")
        self.fin = fin[order]
        self.xs = self.pts[self.fin, 0].astype(np.float64)

    def nn_full(self, ind):
        ind = np.asarray(ind, np.int64)
        out = ind.copy()
        q = self.pts[ind, :3]
        lo = np.searchsorted(self.xs, q[:, 0].astype(np.float64) - 1e-20, "left")
        hi = np.searchsorted(self.xs, q[:, 0].astype(np.float64) + 1e-20, "right")
        for t in np.flatnonzero(hi - lo > 1):
            c = self.fin[lo[t]:hi[t]]
            C = self.pts[c, :3]
            d = q[t] - C
            d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
            out[t] = min(int(c[d2 == 0].min()), int(ind[t]))
        return out.astype(np.int32)

    def pair_b(self, El, Er):
        """SectPath: pr = NN_Er(pl); right = NN_full(pr); pl' = NN_El(pr); left = NN_full(pl'), for every left in order."""
        if El.shape[0] == 0 or Er.shape[0] == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32)
        pr = Er[_nearest(self.pts, El, Er, 0)]
        pl2 = El[_nearest(self.pts, pr, El, 0)]
        return self.nn_full(pl2), self.nn_full(pr)

    def insert_point(self, ind, plane, mode):
        """insert_point + flattening for one slice: (y, x, z, left_pair, right_pair)."""
        El, Er = classify(self.pts, ind, plane)
        lp, rp = pair_a(self.pts, El, Er) if mode == "A" else self.pair_b(El, Er)
        y, x, z = nodes(self.pts, lp, rp, plane)
        return y, x, z, lp, rp

    def slice_contours(self, planes, mode, half_width=2.0, truncate_center=True):
        ys, xs, zs = [], [], []
        off = [0]
        for p in np.asarray(planes, F32):
            y, x, z, _, _ = self.insert_point(band(self.pts, p, half_width, truncate_center), p, mode)
            ys.append(y), xs.append(x), zs.append(z)
            off.append(off[-1] + y.shape[0])
        cat = lambda a: np.concatenate(a) if a else np.zeros(0, np.float64)  # noqa: E731
        return np.array(off, np.int64), cat(ys), cat(xs), cat(zs)


def nodes(pts, lp, rp, plane):
    """Interpolation of the pairs (right_pair[i], left_pair[i]), i < left_pair.size(), onto the plane in float32 without
    fused operations, inserted into a map keyed by (double)y: a key keeps the y of its first insertion (-0.0 and +0.0
    are one key) and the z of its last.  Returns (y, x, z) in ascending key order, x = (double)plane."""
    n = lp.shape[0]
    P = F32(plane)
    r = pts[rp[:n], :3].astype(F32)
    l = pts[lp[:n], :3].astype(F32)
    t = (P - r[:, 0]) / (l[:, 0] - r[:, 0])
    y = r[:, 1] + t * (l[:, 1] - r[:, 1])
    z = r[:, 2] + t * (l[:, 2] - r[:, 2])
    node = {}
    for yv, zv in zip(y.tolist(), z.tolist()):
        node[yv] = zv               # a dict, like std::map, keeps the first key object of equal keys
    keys = sorted(node)
    return (np.array(keys, np.float64), np.full(len(keys), float(P), np.float64),
            np.array([node[k] for k in keys], np.float64))
