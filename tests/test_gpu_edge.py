"""GPU edge cases the domain has: empty / tiny clouds, k > N, duplicate points, non-finite points,
points exactly on a plane, empty sides, external query points, strides, error codes; plus the
committed golden fixtures and the Python mirror of the reference interface."""
import os

import numpy as np
import pytest

from oracle import ppp_oracle as po
from pinned_golden import assert_pinned
from polishpathplanning_b200 import api, reference_api as ra, synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _n4(g):
    return np.concatenate([g[:, 0:3], g[:, 4:5]], axis=1)


def _same_normals(g, o, tol=1e-5):
    gn = _n4(g) if g.shape[1] == 8 else g
    assert np.array_equal(np.isnan(gn[:, 0]), np.isnan(o[:, 0]))
    ok = ~np.isnan(o[:, 0])
    if ok.any():
        assert np.abs(gn[ok] - o[ok]).max() <= tol


def test_golden_independent_vectors(ctx):
    """GPU against the cv2.flann / scipy goldens directly (no oracle in the loop)."""
    g = np.load(os.path.join(GOLD, "independent.npz"))
    for n, seed, ks in ((4000, 1, (8, 16, 32, 64)), (20000, 4, (16,))):
        gc = api.Cloud(ctx, synth.panel(n, seed))
        for k in ks:
            idx, d2 = gc.knn(k)
            assert_pinned(g, "knn_idx_n%d_s%d_k%d" % (n, seed, k), idx)
            assert_pinned(g, "knn_d2_n%d_s%d_k%d" % (n, seed, k), d2)
        gc.close()
    gc = api.Cloud(ctx, synth.panel(4000, 1))
    counts, off, idx, d2 = gc.radius(2.5)
    boundary = set(g["radius_boundary_rows_n4000_s1"].tolist())
    gcnt = g["radius_counts_n4000_s1"]
    keep = np.array([i not in boundary for i in range(4000)])
    assert np.array_equal(counts[keep], gcnt[keep])
    gc.close()


def test_golden_regression_vectors(ctx):
    r = np.load(os.path.join(GOLD, "oracle_regression.npz"))
    gc = api.Cloud(ctx, synth.panel(4000, 1))
    _same_normals(gc.normals_radius(2.5), r["normals_r2p5_n4000_s1"])
    _same_normals(gc.normals_knn(16), r["normals_k16_n4000_s1"])
    mn, mx = gc.bbox()
    assert np.array_equal(np.stack([mn, mx]), r["bbox_n4000_s1"])
    planes = r["planes_gen2_contact_n4000_s1_R6"]
    off, idx = gc.slice_bands(planes)
    assert np.array_equal(off, r["bands_off_n4000_s1"]) and np.array_equal(idx, r["bands_idx_n4000_s1"])
    for mode in "AB":
        o, y, x, z = gc.slice_contours(planes, mode)
        assert np.array_equal(o, r["contour_off_%s_n4000_s1" % mode])
        assert np.array_equal(y, r["contour_y_%s_n4000_s1" % mode])
        assert np.array_equal(x, r["contour_x_%s_n4000_s1" % mode])
        assert np.array_equal(z, r["contour_z_%s_n4000_s1" % mode])
    gc.close()


def test_empty_and_tiny_clouds(ctx):
    e = np.zeros((0, 8), np.float32)
    gc = api.Cloud(ctx, e)
    assert gc.knn(4)[0].shape == (0, 4)
    assert gc.normals_radius(2.5).shape == (0, 8)
    off, idx = gc.slice_bands(np.asarray([1.0, 2.0], np.float32))
    assert off.tolist() == [0, 0, 0] and idx.size == 0
    off, y, x, z = gc.slice_contours(np.asarray([1.0], np.float32), "B")
    assert off.tolist() == [0, 0]
    gc.close()
    # N < k: k is clamped to N (pcl::KdTreeFLANN::nearestKSearch), rows padded with -1
    c = synth.panel(5, 1)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    gi, gd = gc.knn(16)
    oi, od = oc.knn(16)
    assert np.array_equal(gi, oi) and np.all(gi[:, 5:] == -1)
    _same_normals(gc.normals_knn(16), oc.normals(k=16)[0])
    # two points: fewer than 3 neighbours -> NaN normals
    c2 = synth.panel(2, 1)
    g2 = api.Cloud(ctx, c2)
    assert np.all(np.isnan(_n4(g2.normals_radius(2.5))))
    g2.close()
    gc.close()


def test_k_sweep_and_large_k(ctx):
    c = synth.panel(30000, 12)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    for k in (1, 2, 3, 5, 10, 33, 50, 100):   # 33+ takes the generic ring-expanding kernel
        gi, gd = gc.knn(k)
        oi, od = oc.knn(k)
        assert np.array_equal(gi, oi), k
        assert np.array_equal(gd.view(np.uint32), od.view(np.uint32)), k
    gc.close()


def test_duplicates_nonfinite_and_sparse(ctx):
    rng = np.random.default_rng(5)
    c = synth.panel(20000, 13)
    c[100:140] = c[60:100]            # exact duplicates: ties on d2 = 0 broken by index
    c[500, 0] = np.nan
    c[501, 2] = np.inf
    c[700:720, 0:3] += 4000.0         # a far-away clump (sparse region, many rings)
    c[800, 0:3] = (-900.0, -900.0, 50.0)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    for k in (8, 16):
        gi, gd = gc.knn(k)
        oi, od = oc.knn(k)
        assert np.array_equal(gi, oi)
        assert np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    assert np.all(gi[500] == -1) and np.all(gi[501] == -1)
    gcnt, goff, gidx, gd2 = gc.radius(2.5)
    ocnt, ooff, oidx, od2 = oc.radius(2.5)
    assert np.array_equal(gcnt, ocnt) and np.array_equal(gidx, oidx)
    _same_normals(gc.normals_radius(2.5), oc.normals(radius=2.5)[0])
    _same_normals(gc.normals_knn(16), oc.normals(k=16)[0])
    mn, mx = gc.bbox()
    omn, omx = oc.minmax()
    assert np.array_equal(mn, omn) and np.array_equal(mx, omx)
    # slicing with duplicates (variant B canonicalises pairs through the global nearest index)
    planes = np.asarray([30.2, 47.9, 60.0, 3990.0, -2000.0], np.float32)
    goff, gidx = gc.slice_bands(planes)
    ooff, oidx = oc.slice_bands(planes)
    assert np.array_equal(goff, ooff) and np.array_equal(gidx, oidx)
    for mode in "AB":
        g = gc.slice_contours(planes, mode)
        o = oc.slice_contours(planes, mode)
        assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_point_on_plane_and_empty_side(ctx):
    c = synth.panel(20000, 14)
    px = np.float32(55.25)
    band = po.OracleCloud(c).band(float(px))
    c[band[:5], 0] = px                       # exactly on the plane: neither left nor right
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    planes = np.asarray([px, c[:, 0].min() - 1.0, c[:, 0].max() + 1.5], np.float32)  # 2nd/3rd: one side empty
    for mode in "AB":
        g = gc.slice_contours(planes, mode)
        o = oc.slice_contours(planes, mode)
        assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_external_queries_and_strides(ctx):
    c = synth.panel(20000, 15)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    rng = np.random.default_rng(1)
    q = np.empty((500, 3), np.float32)
    q[:, 0:2] = rng.random((500, 2)) * 170 - 15        # some outside the cloud's rectangle
    q[:, 2] = rng.random(500) * 40 - 10
    q[7] = (1e4, -1e4, 0)                                # far outside the grid
    for k in (1, 3, 10):                                 # the reference's own k values (SURVEY §2.2)
        gi, gd = gc.knn(k, queries=q)
        oi, od = oc.knn(k, queries=q)
        assert np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    gcnt, goff, gidx, _ = gc.radius(7.5, queries=q)
    ocnt, ooff, oidx, _ = oc.radius(7.5, queries=q)
    assert np.array_equal(gcnt, ocnt) and np.array_equal(gidx, oidx)
    # packed xyz (stride 12) and xyz+pad (stride 16) clouds give the same answers as stride 32
    for cols in (3, 4):
        g2 = api.Cloud(ctx, np.ascontiguousarray(c[:, :cols]))
        assert np.array_equal(g2.knn(8)[0], gc.knn(8)[0])
        g2.close()
    # compact normal records (stride 16)
    n16 = gc.normals_knn(16, stride_floats=4)
    n32 = gc.normals_knn(16)
    assert np.array_equal(n16.view(np.uint32), _n4(n32).view(np.uint32))
    gc.close()


def test_grid_axes_follow_extents(ctx):
    """A cloud that is thin in y instead of z: the grid must pick (x, z)."""
    c = synth.panel(20000, 16)
    c2 = c.copy()
    c2[:, 1], c2[:, 2] = c[:, 2].copy(), c[:, 1].copy()
    gc = api.Cloud(ctx, c2)
    oc = po.OracleCloud(c2)
    assert np.array_equal(gc.knn(16)[0], oc.knn(16)[0])
    planes = synth.even_planes(c2, 6)
    g = gc.slice_contours(planes, "B")
    o = oc.slice_contours(planes, "B")
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_error_codes(ctx):
    gc = api.Cloud(ctx, synth.panel(100, 1))
    with pytest.raises(api.PPPError) as e:
        gc.knn(0)
    assert e.value.status == api._lib.PPP_ERR_INVALID
    with pytest.raises(api.PPPError):
        gc.normals_radius(-1.0)
    with pytest.raises(api.PPPError) as e:
        gc.knn(100000)
    assert e.value.status == api._lib.PPP_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        api.Cloud(ctx, np.zeros((4, 2), np.float32))
    gc.close()


def test_radius_lists_beyond_the_shared_memory_limit_fail_loudly(ctx):
    """The documented limit of the radius paths (include/ppp_gpu.h): a query with more than ~900 neighbours cannot be
    ordered in shared memory; the call says so (PPP_ERR_UNSUPPORTED) instead of truncating.  Counting still works."""
    rng = np.random.default_rng(3)
    pts = synth.to_pointxyzrgb((rng.random((6000, 3)) * 4.0).astype(np.float32))     # 6000 points within a 4 mm cube
    gc = api.Cloud(ctx, pts)
    cnt = np.empty(6000, np.int32)
    api.check(gc.lib.ppp_radius(gc._h, None, 0, 0, 2.5, cnt.ctypes.data_as(api._vp), None, None, None))
    assert cnt.max() > 1500
    with pytest.raises(api.PPPError) as e:
        gc.radius(2.5)
    assert e.value.status == api._lib.PPP_ERR_UNSUPPORTED and "shared-memory" in str(e.value)
    with pytest.raises(api.PPPError) as e:
        gc.normals_radius(2.5)
    assert e.value.status == api._lib.PPP_ERR_UNSUPPORTED
    nk = gc.normals_knn(16)                     # the k-nearest path has no such limit
    assert np.isfinite(nk[:, 0]).all()
    gc.close()


def test_reference_interface_mirror(ctx, tmp_path):
    """./main-shaped flow: PCD in metres -> ctor scaling -> estimate_normal -> plane sweep."""
    metres = synth.to_pointxyzrgb(synth.panel_metres(30000, 21))
    pcd = str(tmp_path / "workpiece.pcd")
    synth.write_pcd(pcd, metres)
    pg = ra.path_generater(pcd, 15, ctx=ctx)
    oc = po.OracleCloud(pg.cloud)
    assert np.array_equal(pg.cloud, synth.panel(30000, 21))
    _same_normals(pg.estimate_normal(), oc.normals(radius=2.5)[0])
    band = pg.rangedX_index(40.9)
    assert np.array_equal(band, oc.band(40.9))
    y, x, z = pg.insert_point(band, (np.float32(40.9), 0, 0))
    oy, ox, oz, _, _ = oc.insert_point(band, 40.9, "A")
    assert np.array_equal(y, oy) and np.array_equal(z, oz)
    planes = pg.Contact_Path_Generation()
    mn, mx = oc.minmax()
    assert np.array_equal(planes, po.planes("gen2_contact", mn[0], mx[0], 15))
    ooff, oy, ox, oz = oc.slice_contours(planes, "A")
    for s, (yy, xx, zz) in enumerate(pg.Path_set):
        assert np.array_equal(yy, oy[ooff[s]:ooff[s + 1]]) and np.array_equal(zz, oz[ooff[s]:ooff[s + 1]])
    sp = ra.SectPath(pcd, 12, ChangeRange=True, ctx=ctx)
    planes = sp.GenPath()
    assert np.array_equal(planes, po.planes("sectpath", mn[0], mx[0], 12))
    ooff, oy, ox, oz = oc.slice_contours(planes, "B")
    for s, (yy, xx, zz) in enumerate(sp.Path_set):
        assert np.array_equal(yy, oy[ooff[s]:ooff[s + 1]]) and np.array_equal(zz, oz[ooff[s]:ooff[s + 1]])
    # unreadable file: the reference prints an error and carries on with an empty cloud
    bad = ra.path_generater(str(tmp_path / "missing.pcd"), 15, ctx=ctx)
    assert bad.cloud.shape[0] == 0


def test_full_size_properties(ctx):
    """BASELINE cfg2 size (1M points, k=16, 200 slices): size-independent checks."""
    c = synth.panel(1_000_000, 0)
    gc = api.Cloud(ctx, c)
    nrm, idx = gc.normals_knn(16, return_idx=True)
    n4 = _n4(nrm)
    assert np.all(idx[:, 0] == np.arange(c.shape[0]))                   # nearest neighbour of a point is itself
    assert idx.min() >= 0 and idx.max() < c.shape[0]
    assert np.all(np.abs(np.linalg.norm(n4[:, :3], axis=1) - 1) < 1e-5)  # unit normals
    assert np.all((-(c[:, :3]) * n4[:, :3]).sum(1) >= -1e-2)              # flipped towards (0,0,0)
    # rows sorted by (d2, idx): recompute d2 exactly as FLANN does
    sub = np.arange(0, c.shape[0], 997)
    d = c[sub][:, None, :3] - c[idx[sub]][:, :, :3]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    di = idx[sub]
    assert np.all((d2[:, 1:] > d2[:, :-1]) | ((d2[:, 1:] == d2[:, :-1]) & (di[:, 1:] > di[:, :-1])))
    # oracle on a sample of queries (exact, external-query path)
    oc = po.OracleCloud(c)
    oi, _ = oc.knn(16, queries=c[sub][:, :3].copy())
    assert np.array_equal(idx[sub], oi)
    planes = synth.even_planes(c, 200)
    off, bidx = gc.slice_bands(planes)
    x = c[:, 0]
    pos = planes.astype(np.int32)
    for s in (0, 57, 199):
        m = bidx[off[s]:off[s + 1]]
        assert np.all(np.diff(m) > 0)
        assert np.all((x[m] >= np.float32(pos[s] - 2)) & (x[m] <= np.float32(pos[s] + 2)))
        assert len(m) == int(((x >= np.float32(pos[s] - 2)) & (x <= np.float32(pos[s] + 2))).sum())
    noff, y, xx, z = gc.slice_contours(planes, "B")
    for s in range(200):
        ys = y[noff[s]:noff[s + 1]]
        assert np.all(np.diff(ys) > 0) and np.all(xx[noff[s]:noff[s + 1]] == np.float64(planes[s]))
    # idempotence: a second call gives identical bytes
    noff2, y2, _, z2 = gc.slice_contours(planes, "B")
    assert np.array_equal(noff, noff2) and np.array_equal(y, y2) and np.array_equal(z, z2)
    # ... and the whole cfg2 workload against the oracle: every neighbour list, every normal, every node
    oi, _ = oc.knn(16, want_d2=False)
    assert np.array_equal(idx, oi)
    on, _ = oc.normals(k=16)
    assert np.array_equal(np.isnan(on[:, 0]), np.isnan(n4[:, 0]))
    okn = ~np.isnan(on[:, 0])
    dn = np.abs(n4[okn] - on[okn])
    print("1M normals: max|diff| = %.3g, bit-identical rows = %.4f" % (dn.max(), (n4[okn] == on[okn]).all(axis=1).mean()))
    assert dn.max() <= 1e-5
    ooff, oy, ox, oz = oc.slice_contours(planes, "B")
    assert np.array_equal(noff, ooff) and np.array_equal(y, oy) and np.array_equal(xx, ox) and np.array_equal(z, oz)
    gc.close()


def test_combined_call_equals_separate_calls(ctx):
    c = synth.panel(50000, 31)
    gc = api.Cloud(ctx, c)
    planes = synth.even_planes(c, 25)
    for kw in (dict(k=16), dict(radius=2.5)):
        nrm, off, y, x, z = gc.normals_and_contours(planes, "B", **kw)
        ref_n = gc.normals_knn(16) if "k" in kw else gc.normals_radius(2.5)
        ro, ry, rx, rz = gc.slice_contours(planes, "B")
        assert np.array_equal(nrm.view(np.uint32), ref_n.view(np.uint32))
        assert np.array_equal(off, ro) and np.array_equal(y, ry) and np.array_equal(x, rx) and np.array_equal(z, rz)
    # too small node buffers: normals still delivered, contours re-fetched
    small = tuple(np.empty(8, np.float64) for _ in range(3))
    nrm, off, y, x, z = gc.normals_and_contours(planes, "A", k=16, nodes_out=small)
    ro, ry, rx, rz = gc.slice_contours(planes, "A")
    assert np.array_equal(off, ro) and np.array_equal(y, ry) and np.array_equal(z, rz)
    gc.close()


@pytest.mark.parametrize("density,noise", [(4.0, 0.0), (0.25, 0.05), (1.0, 0.3)])
def test_density_and_noise_variants(ctx, density, noise):
    """Dense scans (78 radius neighbours: generic radius path), sparse scans, noisy surfaces."""
    c = synth.panel(40000, 41, density=density, noise_sigma=noise)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    gi, gd = gc.knn(16)
    oi, od = oc.knn(16)
    assert np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    _same_normals(gc.normals_radius(2.5), oc.normals(radius=2.5)[0])
    _same_normals(gc.normals_knn(32), oc.normals(k=32)[0])
    planes = synth.even_planes(c, 9)
    for mode in "AB":
        g = gc.slice_contours(planes, mode)
        o = oc.slice_contours(planes, mode)
        assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_large_offsets_and_clusters(ctx):
    """Coordinates far from the origin (float32 cancellation regime) and a strongly non-uniform cloud."""
    rng = np.random.default_rng(3)
    c = synth.panel(30000, 42)
    c[:, 0] += np.float32(3000.0)
    c[:, 1] -= np.float32(2500.0)
    c[:, 2] += np.float32(50.0)
    # a dense cluster (10x density) in one corner and a hole in the middle
    cl = c[:3000].copy()
    cl[:, 0:2] = c[0, 0:2] + (rng.random((3000, 2)).astype(np.float32) * 10)
    keep = ~((np.abs(c[:, 0] - 3090) < 15) & (np.abs(c[:, 1] + 2420) < 15))
    c2 = np.ascontiguousarray(np.concatenate([c[keep], cl]))
    gc = api.Cloud(ctx, c2)
    oc = po.OracleCloud(c2)
    for k in (10, 16, 50):
        gi, gd = gc.knn(k)
        oi, od = oc.knn(k)
        assert np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    _same_normals(gc.normals_radius(2.5), oc.normals(radius=2.5)[0])
    _same_normals(gc.normals_knn(16), oc.normals(k=16)[0])
    gcnt, _, gidx, _ = gc.radius(2.5)
    ocnt, _, oidx, _ = oc.radius(2.5)
    assert np.array_equal(gcnt, ocnt) and np.array_equal(gidx, oidx)
    mn, mx = gc.bbox()
    planes = po.planes("sectpath", mn[0], mx[0], 12.0)
    for mode in "AB":
        g = gc.slice_contours(planes, mode)
        o = oc.slice_contours(planes, mode)
        assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_many_overlapping_planes(ctx):
    """cfg4-style: plane spacing below the band width, every point in several bands; > 3072 planes
    takes the global-atomic band path."""
    c = synth.panel(60000, 43)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    for S in (300, 4000):
        planes = synth.even_planes(c, S)
        goff, gidx = gc.slice_bands(planes)
        ooff, oidx = oc.slice_bands(planes)
        assert np.array_equal(goff, ooff) and np.array_equal(gidx, oidx)
    planes = synth.even_planes(c, 300)
    g = gc.slice_contours(planes, "B")
    o = oc.slice_contours(planes, "B")
    assert np.array_equal(g[0], o[0]) and np.array_equal(g[1], o[1]) and np.array_equal(g[3], o[3])
    gc.close()


def test_next_rows_drawpath_and_coverage(ctx):
    """SURVEY §8f rows: spline sampling + nearest-point snaps (drawpath) and compute_coverage flags."""
    c = synth.panel(40000, 51)
    pg = ra.path_generater(c.copy() / np.float32(1000.0) * np.float32(1.0), 15, ctx=ctx)  # ctor rescales by 1000
    pg.cloud[:, :3] = c[:, :3]
    pg._invalidate()
    oc = po.OracleCloud(pg.cloud)
    pg.Contact_Path_Generation()
    paths = pg.splines()
    assert len(paths) >= 3
    sp = paths[1]
    # drawpath: 200 samples along the spline, each snapped to its nearest cloud point
    pts = pg.drawpath_samples(sp, gen2=True)
    assert pts.shape == (200, 3)
    assert np.array_equal(pts[:, 2].view(np.uint64), po.steffen_eval(sp.y, pg.Path_set[1][2], pts[:, 1]).view(np.uint64))
    got = pg.drawpath(sp, gen2=True)
    want, _ = oc.knn(3, queries=pts.astype(np.float32))
    assert np.array_equal(got, want[:, 0])
    # compute_coverage: union of radius neighbourhoods of a batch of nodes, accumulated over calls
    nodes = pts[::10]
    flags = pg.compute_coverage(nodes, 7.5).copy()
    oflags = oc.coverage_mark(nodes.astype(np.float32), 7.5)
    assert np.array_equal(flags, oflags)
    flags2 = pg.compute_coverage(pts[5::10], 3.0)
    oflags = oc.coverage_mark(pts[5::10].astype(np.float32), 3.0, oflags)
    assert np.array_equal(flags2, oflags)
    assert abs(pg.get_coverage() - float(oflags.mean())) < 1e-6


@pytest.mark.parametrize("k", [10, 50])
def test_next_row_principal_curvatures(ctx, k):
    """compute_transform's kNN + computePointPrincipalCurvatures for a batch of spline points."""
    c = synth.panel(40000, 52)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    nrm = gc.normals_radius(2.5)
    rng = np.random.default_rng(2)
    q = c[rng.integers(0, c.shape[0], 400), :3] + rng.normal(0, 0.3, (400, 3)).astype(np.float32)
    out, nn0 = gc.principal_curvatures(nrm, q, k)
    oout, onn0 = oc.principal_curvatures(nrm, q, k)   # same normals in: isolates the curvature arithmetic
    assert np.array_equal(nn0, onn0)
    ok = ~np.isnan(oout).any(axis=1) & ~np.isnan(nrm[onn0, 0])
    # eigenvector sign is a property of the cross products and identical; values agree to float rounding
    assert np.abs(out[ok, 3:5] - oout[ok, 3:5]).max() <= 1e-6
    well = ok & (oout[:, 3] > 1.5 * oout[:, 4])          # distinct principal curvatures: direction is well defined
    assert np.abs(out[well, 0:3] - oout[well, 0:3]).max() <= 1e-4
    assert np.array_equal(np.isnan(out).any(axis=1), np.isnan(oout).any(axis=1))
    gc.close()


def test_two_host_threads_share_a_cloud(ctx):
    """The reference's gen-3 sweep queries one kd-tree from two threads
    (src/Path_Alg/path_dynamic_alg.cpp:308-334): concurrent calls on one handle must be safe."""
    import threading
    c = synth.panel(30000, 61)
    gc = api.Cloud(ctx, c)
    rng = np.random.default_rng(4)
    qs = [c[rng.integers(0, c.shape[0], 300), :3] + np.float32(0.1) for _ in range(2)]
    want = [gc.knn(3, queries=q)[0] for q in qs]
    planes = synth.even_planes(c, 5)
    want_c = gc.slice_contours(planes, "B")
    errs = []

    def worker(i):
        try:
            for _ in range(15):
                assert np.array_equal(gc.knn(3, queries=qs[i])[0], want[i])
                o = gc.slice_contours(planes, "B")
                assert np.array_equal(o[1], want_c[1])
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs
    gc.close()


def test_cfg3_shape_10m_points_k32_1000_slices(ctx):
    """BASELINE.json configs[2] shape on one GPU: 10M points, k = 32 normals, 1000 slices.
    Sampled exactness against the oracle plus size-independent properties."""
    n = 10_000_000
    c = synth.panel(n, 0)
    gc = api.Cloud(ctx, c)
    nrm, idx = gc.normals_knn(32, return_idx=True, stride_floats=4)
    assert np.all(idx[:, 0] == np.arange(n))
    assert idx.min() >= 0 and idx.max() < n
    # At ~3000 mm PCL 1.10's single-pass float32 covariance is mostly rounding noise (SURVEY §7.3): a
    # few neighbourhoods come out exactly rank-deficient and PCL's eigen33 then yields NaN.  That is
    # the reference's behaviour; it must be reproduced, not "fixed".
    ok = ~np.isnan(nrm[:, 0])
    assert ok.mean() > 0.99
    assert np.all(np.abs(np.linalg.norm(nrm[ok, :3], axis=1) - 1) < 1e-5)
    oc = po.OracleCloud(c)
    sub = np.arange(0, n, 9973)
    oi, _ = oc.knn(32, queries=c[sub][:, :3].copy())
    assert np.array_equal(idx[sub], oi)
    # normals of sampled rows (and of every NaN row among the first million) from the oracle's formula
    rows = np.concatenate([sub[::50], np.nonzero(~ok[:1_000_000])[0][:200]])
    for i in rows:
        o = po.normal_from_list(c, idx[i], c[i, :3])
        assert np.array_equal(np.isnan(o), np.isnan(nrm[i]))
        if not np.isnan(o[0]):
            assert np.abs(o - nrm[i]).max() <= 1e-5
    planes = synth.even_planes(c, 1000)
    noff, y, x, z = gc.slice_contours(planes, "B")
    assert noff[-1] > 0 and np.all(np.diff(noff) > 100)
    for s in (0, 499, 999):
        ys = y[noff[s]:noff[s + 1]]
        assert np.all(np.diff(ys) > 0)
    o = oc.slice_contours(planes[[17, 640]], "B")
    for j, s in enumerate((17, 640)):
        assert np.array_equal(y[noff[s]:noff[s + 1]], o[1][o[0][j]:o[0][j + 1]])
        assert np.array_equal(z[noff[s]:noff[s + 1]], o[3][o[0][j]:o[0][j + 1]])
    gc.close()


@pytest.mark.parametrize("mode", ["A", "B"])
def test_insert_point_explicit_indices(ctx, mode):
    """insert_point with the caller's own index list: the band itself, thinned bands, an
    arbitrary ascending subset that ignores the band limits, one-sided and empty lists."""
    pts = synth.panel(60000, 31)
    oc = po.OracleCloud(pts)
    gc = api.Cloud(ctx, pts)
    rng = np.random.default_rng(5)
    mn, mx = oc.minmax()
    for px in (float(mn[0]) + 7.3, 0.5 * float(mn[0] + mx[0]), float(mx[0]) - 3.1):
        band = oc.band(px)
        wide = np.flatnonzero(np.abs(pts[:, 0] - np.float32(px)) < 6).astype(np.int32)   # wider than the band
        left_only = band[pts[band, 0] < np.float32(px)]
        cases = [band, band[::2], band[rng.random(band.shape[0]) < 0.3], wide, left_only, band[:1], band[:0]]
        for idx in cases:
            oy, ox, oz, _, _ = oc.insert_point(idx, px, mode)
            y, x, z = gc.insert_point(idx, px, mode)
            assert np.array_equal(y, oy) and np.array_equal(x, ox) and np.array_equal(z, oz)
        off, y, x, z = gc.slice_contours([px], mode)
        yb, xb, zb = gc.insert_point(band, px, mode)
        assert np.array_equal(y, yb) and np.array_equal(z, zb)
    with pytest.raises(api.PPPError):
        gc.insert_point(np.array([5, 3], np.int32), 0.0, mode)      # not ascending
    with pytest.raises(api.PPPError):
        gc.insert_point(np.array([0, pts.shape[0]], np.int32), 0.0, mode)
    gc.close()


def test_sor_mean_distances_and_remove_outlier(ctx, tmp_path):
    """StatisticalOutlierRemoval (SectPath::remove_outlier): device distances bit-exact with the
    oracle for both sqrt overloads and several mean_k (k > 64 takes the generic search), kept set equal."""
    pts = synth.panel(60000, 13)
    rng = np.random.default_rng(3)
    out_rows = rng.choice(pts.shape[0], 300, replace=False)
    pts[out_rows, 2] += rng.uniform(15, 80, 300).astype(np.float32)     # outliers above the surface
    pts[77, 1] = np.inf
    pts[5000] = pts[5001]                                               # duplicate point
    oc = po.OracleCloud(pts)
    gc = api.Cloud(ctx, pts)
    for mean_k in (50, 1, 8, 31, 63, 100):
        for fl in (False, True):
            od, onv = oc.sor_mean_distances(mean_k, fl)
            gd, gnv = gc.sor_mean_distances(mean_k, fl)
            assert gnv == onv
            assert np.array_equal(gd.view(np.uint32), od.view(np.uint32)), (mean_k, fl)
    gd, gnv = gc.sor_mean_distances(50)
    keep, thr = ra.sor_select(gd, gnv, 1.0)
    okeep, othr = po.OracleCloud.sor_select(*oc.sor_mean_distances(50), 1.0)
    assert thr == othr and np.array_equal(keep, okeep)
    assert not set(out_rows.tolist()) & set(keep.tolist())
    gc.close()
    # reference-shaped flow: SectPath with RemoveOutlier=true, then normals + sweep on the filtered cloud
    pcd = str(tmp_path / "w.pcd")
    synth.write_pcd(pcd, synth.to_pointxyzrgb(synth.panel_metres(60000, 13)))
    sp = ra.SectPath(pcd, 12, ChangeRange=True, RemoveOutlier=True, ctx=ctx)
    clean = synth.panel(60000, 13)
    ock = po.OracleCloud(clean)
    ok2, _ = po.OracleCloud.sor_select(*ock.sor_mean_distances(50), 1.0)
    assert np.array_equal(sp.cloud, clean[ok2])
    of = po.OracleCloud(sp.cloud)
    _same_normals(sp.estimate_normal(), of.normals(radius=2.5)[0])
    tiny = api.Cloud(ctx, synth.panel(40, 1))
    with pytest.raises(api.PPPError) as e:
        tiny.sor_mean_distances(50)
    assert e.value.status == api._lib.PPP_ERR_UNSUPPORTED
    tiny.close()


def test_sync_free_slicing_corner_cases(ctx):
    """SectPath slicing without mid-chain fetches: bands larger than the shared-memory sort (global
    scratch path), more planes than the offsets fetch buffer holds, planes outside the cloud and
    non-finite planes, caller buffers too small (capacity error, then retried), repeated calls."""
    c = synth.panel(200000, 47)
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    mn, mx = oc.minmax()
    # 1. very wide bands: ~36k members per slice > 24576 keys of shared memory
    planes = np.array([mn[0] + 100.0, 0.5 * (mn[0] + mx[0]), mx[0] - 90.5], np.float32)
    for _ in range(2):                                   # second call sizes from the first one's largest band
        g = gc.slice_contours(planes, "B", half_width=40.0)
        o = oc.slice_contours(planes, "B", half_width=40.0)
        assert int(np.diff(oc.slice_bands(planes, half_width=40.0)[0]).max()) > 24576
        assert all(np.array_equal(a, b) for a, b in zip(g, o))
    # 2. planes outside the cloud, NaN / inf planes, duplicates of one plane
    planes = np.array([mn[0] - 50.0, np.nan, mn[0] + 7.25, mn[0] + 7.25, np.inf, mx[0] + 3.0, mx[0] - 1.5], np.float32)
    g = gc.slice_contours(planes, "B")
    o = oc.slice_contours(planes, "B")
    assert all(np.array_equal(a, b) for a, b in zip(g, o))
    # 3. caller buffers too small -> PPP_ERR_CAPACITY inside, wrapper retries with its own arrays
    planes = synth.even_planes(c, 60)
    small = tuple(np.empty(16, np.float64) for _ in range(3))
    g = gc.slice_contours(planes, "B", out=small)
    o = oc.slice_contours(planes, "B")
    assert all(np.array_equal(a, b) for a, b in zip(g, o)) and g[1].shape[0] > 16
    gc.close()
    # 4. more than 8191 planes: the offsets no longer fit the mapped fetch buffer
    c2 = synth.panel(10000, 48)
    g2 = api.Cloud(ctx, c2)
    o2 = po.OracleCloud(c2)
    planes = synth.even_planes(c2, 8500)
    g = g2.slice_contours(planes, "B")
    o = o2.slice_contours(planes, "B")
    assert all(np.array_equal(a, b) for a, b in zip(g, o))
    g2.close()


@pytest.mark.parametrize("cluster", [2, 4, 8])
def test_slice_order_thread_block_clusters(ctx, cluster, monkeypatch):
    """The cluster variant of the per-slice ordering (k_slice_order_cl: the node keys of a slice spread over the
    shared memories of 2, 4 or 8 CTAs, cross-CTA compare-exchange steps through distributed shared memory):
    short bands (all keys land in CTA 0's chunk), medium ones, bands beyond one CTA's shared memory, bands beyond the
    cluster's capacity (CTA 0 alone, in global scratch), empty slices and equal-y runs -- identical to the oracle."""
    monkeypatch.setenv("PPP_SLICE_CLUSTER", str(cluster))
    c = synth.panel(200000, 51)
    c[::7, 1] = np.round(c[::7, 1])          # repeated y values -> equal-y runs in the node keys
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    mn, mx = oc.minmax()
    for planes, hw in ((synth.even_planes(c, 40), 2.0),                                               # ~1.8k members
                       (np.array([mn[0] - 30.0, mn[0] + 60.0, mx[0] - 45.0], np.float32), 12.0),      # ~11k members, one empty slice
                       (np.array([0.5 * (mn[0] + mx[0])], np.float32), 40.0),                         # ~36k members
                       (np.array([0.5 * (mn[0] + mx[0]), mn[0] + 150.0], np.float32), 150.0)):        # ~135k members
        for _ in range(2):                       # the second call sizes the launch from the first one's largest band
            g = gc.slice_contours(planes, "B", half_width=hw)
            o = oc.slice_contours(planes, "B", half_width=hw)
            assert all(np.array_equal(a, b) for a, b in zip(g, o)), (cluster, hw)
    gc.close()


@pytest.mark.parametrize("k", [8, 16, 24, 32, 48, 64])
def test_fixed_point_key_kernels_on_exact_ties_and_duplicates(ctx, k):
    """The self-query search kernels order candidates by a 22/23-bit fixed-point d2 and hand every query whose
    first k+1 candidates are not strictly separated by it to the exact kernel.  A lattice (every distance is tied
    many times over), exact duplicates and a jittered copy (near-ties far below the fixed-point resolution) must
    come out in the oracle's (d2, index) order, bit for bit -- lists and distances."""
    g = np.arange(70, dtype=np.float32)
    xx, yy = np.meshgrid(g, g, indexing="ij")
    lattice = np.stack([xx.ravel(), yy.ravel(), np.zeros(xx.size, np.float32)], axis=1)          # 4900 points, spacing 1
    rng = np.random.default_rng(17)
    jitter = lattice[:1500] + np.float32(100.0) + rng.normal(0.0, 1e-4, (1500, 3)).astype(np.float32)
    pts = np.concatenate([lattice, lattice[200:260], jitter], axis=0).astype(np.float32)          # + 60 exact duplicates
    pts = pts[rng.permutation(pts.shape[0])]
    c = synth.to_pointxyzrgb(pts) if hasattr(synth, "to_pointxyzrgb") else pts
    gc = api.Cloud(ctx, c)
    oc = po.OracleCloud(c)
    gi, gd = gc.knn(k)
    oi, od = oc.knn(k)
    assert np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    assert np.array_equal(gi, oi)
    gc.close()
