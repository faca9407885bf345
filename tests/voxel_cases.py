"""Edge-case clouds of the VoxelGrid pre-filter (voxel_down) and an independent numpy restatement of
pcl::VoxelGrid::applyFilter with the members of each voxel summed in ascending source order.  Used by the CPU test of
the oracle and by the device tests."""
import numpy as np

from polishpathplanning_b200 import synth


def _recs(xyz, seed=0):
    """(n, 3) -> (n, 8) PointXYZRGB records with varied r, g, b, a bytes."""
    out = synth.to_pointxyzrgb(np.asarray(xyz, np.float32))
    rng = np.random.default_rng(seed)
    out[:, 4] = rng.integers(0, 2 ** 32, out.shape[0], dtype=np.uint64).astype(np.uint32).view(np.float32)
    return out


def edge_cases():
    """[(name, records, leaf)]"""
    rng = np.random.default_rng(11)
    cases = []
    # negative coordinates, and a bounding box that straddles zero
    cases.append(("negative", _recs(rng.uniform(-60.0, -5.0, (4000, 3)), 1), 2.5))
    cases.append(("straddle_zero", _recs(rng.uniform(-7.3, 9.1, (4000, 3)), 2), 1.0))
    # points exactly on leaf multiples (floorf edge), on both sides of zero, plus their float neighbours
    k = rng.integers(-40, 40, (3000, 3)).astype(np.float32) * np.float32(0.5)
    nb = np.concatenate([k, np.nextafter(k, np.float32(-np.inf)), np.nextafter(k, np.float32(np.inf))])
    cases.append(("leaf_multiples", _recs(nb, 3), 0.5))
    # anisotropic leaf
    cases.append(("anisotropic", _recs(rng.uniform(-20.0, 30.0, (5000, 3)), 4), (0.3, 1.7, 4.0)))
    # duplicate points (whole voxels of copies, and copies spread over the cloud)
    base = rng.uniform(0.0, 10.0, (500, 3)).astype(np.float32)
    dup = np.concatenate([base, base, base[::-1], np.repeat(base[:20], 30, axis=0)])
    cases.append(("duplicates", _recs(dup[rng.permutation(dup.shape[0])], 5), 1.0))
    # non-finite points (NaN / inf in any coordinate, including the first and last record)
    nf = rng.uniform(-10.0, 10.0, (3000, 3)).astype(np.float32)
    nf[0, 0] = np.nan
    nf[-1, 2] = np.inf
    nf[rng.choice(3000, 200, replace=False), rng.integers(0, 3, 200)] = np.nan
    nf[rng.choice(3000, 50, replace=False), 1] = -np.inf
    cases.append(("non_finite", _recs(nf, 6), 1.5))
    # one crowded voxel: every point in the same voxel
    cases.append(("crowded", _recs(rng.uniform(100.0, 100.9, (6000, 3)), 7), 1.0))
    # a few voxels far apart (keys need many bits, most voxels empty)
    far = np.concatenate([rng.uniform(0, 1, (300, 3)), rng.uniform(0, 1, (300, 3)) + np.array([1500.0, 200.0, 0.0])])
    cases.append(("far_apart", _recs(far, 8), 1.0))
    # a single point
    cases.append(("single", _recs(np.array([[1.25, -2.5, 3.75]], np.float32), 9), 0.5))
    return cases


def overflow_cloud():
    """A cloud whose leaf is too small for int32 voxel indices (dx * dy * dz > INT32_MAX): PCL keeps it."""
    xyz = np.array([[0.0, 0.0, 0.0], [2000.0, 2000.0, 2000.0], [10.0, 20.0, 30.0]], np.float32)
    return _recs(xyz, 10), 1.0


def voxel_numpy(pts, leaf):
    """VoxelGrid::applyFilter restated in numpy, members summed in ascending source order.  Returns (records (m, sf),
    row_offsets, members) like the oracle; raises OverflowError where PCL keeps the input."""
    pts = np.ascontiguousarray(pts, np.float32)
    sf = pts.shape[1]
    inv = np.float32(1.0) / np.broadcast_to(np.asarray(leaf, np.float32), (3,))
    xyz = pts[:, :3]
    fin = np.isfinite(xyz).all(axis=1)
    src = np.flatnonzero(fin).astype(np.int32)
    p = xyz[fin]
    if p.shape[0] == 0:
        return np.zeros((0, sf), np.float32), np.zeros(1, np.int64), np.zeros(0, np.int32)
    mn, mx = p.min(axis=0), p.max(axis=0)
    ext = (mx - mn) * inv
    if not np.all(ext < np.float32(2 ** 31)):
        raise OverflowError("leaf too small")
    d = ext.astype(np.int64) + 1
    if int(d[0]) * int(d[1]) * int(d[2]) > 2 ** 31 - 1:
        raise OverflowError("leaf too small")
    min_b = np.floor(mn * inv).astype(np.int64)
    max_b = np.floor(mx * inv).astype(np.int64)
    div = max_b - min_b + 1
    ijk = (np.floor(p * inv) - min_b.astype(np.float32)).astype(np.int64)
    key = (ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * (div[0] * div[1])) & 0xFFFFFFFF
    order = np.argsort(key, kind="stable")
    k = key[order]
    starts = np.flatnonzero(np.r_[True, k[1:] != k[:-1]])
    off = np.r_[starts, k.shape[0]].astype(np.int64)
    cnt = np.diff(off)
    members = src[order]
    vals = pts[members]
    rows = cnt.shape[0]
    sums = np.zeros((rows, 3), np.float32)
    chan = vals[:, 4].view(np.uint32)[:, None] >> np.arange(0, 32, 8, dtype=np.uint32) & np.uint32(0xFF) if sf >= 5 else None
    csum = np.zeros((rows, 4), np.float32)
    for j in range(int(cnt.max())):   # one member of every row per step: float32 sums in member order
        live = np.flatnonzero(cnt > j)
        at = off[live] + j
        sums[live] = sums[live] + vals[at, :3]
        if chan is not None:
            csum[live] = csum[live] + chan[at].astype(np.float32)
    out = np.zeros((rows, sf), np.float32)
    cf = cnt.astype(np.float32)
    out[:, :3] = sums / cf[:, None]
    if sf >= 4:
        out[:, 3] = 1.0
    if chan is not None:
        q = (csum / cf[:, None]).astype(np.uint32) & np.uint32(0xFF)
        out[:, 4] = (q << np.arange(0, 32, 8, dtype=np.uint32)).sum(axis=1, dtype=np.uint32).view(np.float32)
    return out, off, members


def pcl_order_bound(pts, off, members):
    """Per row and axis, the most a centroid summed in another member order can differ: (2n + 1) * 2^-24 * M, n the
    member count and M the largest |coordinate| among the members."""
    xyz = np.abs(np.asarray(pts, np.float32)[members, :3]).astype(np.float64)
    cnt = np.diff(off)
    M = np.maximum.reduceat(xyz, off[:-1], axis=0)
    return (2.0 * cnt[:, None] + 1.0) * 2.0 ** -24 * M
