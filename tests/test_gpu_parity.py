"""GPU parity: libppp_gpu.so (through the C ABI) against the CPU oracle on the same seeded inputs.
Integer / index results bit-exact; normals within 1e-5 per component (BASELINE.json north_star)."""
import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import api, synth

pytestmark = pytest.mark.gpu

NORMAL_TOL = 1e-5  # north_star: "normals agree within 1e-5 per component after sign alignment"


def _cmp_normals(g, o):
    """g: (N, 8) pcl::Normal records from the GPU; o: (N, 4) oracle. Returns max abs diff over finite rows."""
    gn = np.concatenate([g[:, 0:3], g[:, 4:5]], axis=1)
    nan_g = np.isnan(gn[:, 0])
    nan_o = np.isnan(o[:, 0])
    assert np.array_equal(nan_g, nan_o), "NaN-normal rows differ"
    ok = ~nan_o
    d = np.abs(gn[ok] - o[ok])
    return float(d.max()) if d.size else 0.0, float((gn[ok] == o[ok]).all(axis=1).mean()) if d.size else 1.0


@pytest.mark.parametrize("n,seed", [(4000, 1), (100000, 2)])
@pytest.mark.parametrize("k", [8, 16, 32, 64])
def test_knn_sets_bit_exact(ctx, n, seed, k):
    cloud = synth.panel(n, seed)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    gi, gd = gc.knn(k)
    oi, od = oc.knn(k, threads=0)
    assert np.array_equal(gi, oi)
    assert np.array_equal(gd.view(np.uint32), od.view(np.uint32))
    gc.close()


@pytest.mark.parametrize("n,seed", [(4000, 1), (100000, 2)])
def test_radius_lists_bit_exact(ctx, n, seed):
    cloud = synth.panel(n, seed)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    gcnt, goff, gidx, gd2 = gc.radius(2.5)
    ocnt, ooff, oidx, od2 = oc.radius(2.5)
    assert np.array_equal(gcnt, ocnt)
    assert np.array_equal(gidx, oidx)
    assert np.array_equal(gd2.view(np.uint32), od2.view(np.uint32))
    gc.close()


def _viewpoint(cloud, where):
    """'origin': PCL's default (0, 0, 0), at a corner of the panels; 'above': the x/y centre of the cloud at z = +100,
    well off the surface."""
    if where == "origin":
        return (0.0, 0.0, 0.0)
    lo, hi = np.nanmin(cloud[:, :3], axis=0), np.nanmax(cloud[:, :3], axis=0)
    return (float(lo[0] + hi[0]) / 2, float(lo[1] + hi[1]) / 2, 100.0)


def _assert_flip_margin(cloud, o, vp, where):
    """Normals within the tolerance of each other must not fall on opposite sides of the viewpoint flip: every finite
    row's |(vp - q).n| clears 1e-3.  The origin lies close to the tangent planes of a few points of the 100000-point
    panel (|(vp - q).n| down to 1.1e-4 at |vp - q| ~ 160: a normal 7e-7 away, ten float ulps, can have the other
    sign), so there the comparison holds only while those normals come out as the oracle's; the margin is asserted
    where the viewpoint is off the surface."""
    if where == "origin":
        return
    ok = ~np.isnan(o[:, 0])
    w = np.asarray(vp, np.float64) - cloud[ok, :3].astype(np.float64)
    assert np.abs((w * o[ok, :3].astype(np.float64)).sum(axis=1)).min() > 1e-3


@pytest.mark.parametrize("n,seed", [(4000, 1), (100000, 3)])
@pytest.mark.parametrize("flags", [api.PPP_COV_PCL110, api.PPP_COV_SHIFTED])
@pytest.mark.parametrize("where", ["origin", "above"])
def test_normals_radius(ctx, n, seed, flags, where):
    cloud = synth.panel(n, seed)
    vp = _viewpoint(cloud, where)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    g = gc.normals_radius(2.5, viewpoint=vp, flags=flags)
    o, _ = oc.normals(radius=2.5, viewpoint=vp, cov_variant=flags)
    _assert_flip_margin(cloud, o, vp, where)
    mx, frac_exact = _cmp_normals(g, o)
    print("normals_radius n=%d flags=%d vp=%s max|diff|=%.3g bit-exact rows=%.4f" % (n, flags, where, mx, frac_exact))
    assert mx <= NORMAL_TOL
    assert np.all(g[:, 3] == 0) and np.all(g[:, 5:8] == 0)  # pcl::Normal padding
    gc.close()


@pytest.mark.parametrize("n,seed", [(4000, 1), (100000, 3)])
@pytest.mark.parametrize("k", [10, 16, 32])
@pytest.mark.parametrize("flags", [api.PPP_COV_PCL110, api.PPP_COV_SHIFTED])
@pytest.mark.parametrize("where", ["origin", "above"])
def test_normals_knn(ctx, n, seed, k, flags, where):
    cloud = synth.panel(n, seed)
    vp = _viewpoint(cloud, where)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    g, gi = gc.normals_knn(k, viewpoint=vp, flags=flags, return_idx=True)
    o, _ = oc.normals(k=k, viewpoint=vp, cov_variant=flags)
    _assert_flip_margin(cloud, o, vp, where)
    oi, _ = oc.knn(k, want_d2=False)
    assert np.array_equal(gi, oi)
    mx, frac_exact = _cmp_normals(g, o)
    print("normals_knn n=%d k=%d flags=%d vp=%s max|diff|=%.3g bit-exact rows=%.4f" % (n, k, flags, where, mx, frac_exact))
    assert mx <= NORMAL_TOL
    gc.close()


def test_bbox_and_bands(ctx):
    cloud = synth.panel(100000, 2)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    mn, mx = gc.bbox()
    omn, omx = oc.minmax()
    assert np.array_equal(mn, omn) and np.array_equal(mx, omx)
    planes = po.planes("gen2_contact", mn[0], mx[0], 15.0)
    goff, gidx = gc.slice_bands(planes)
    ooff, oidx = oc.slice_bands(planes)
    assert np.array_equal(goff, ooff)
    assert np.array_equal(gidx, oidx)
    # overlapping bands, non-truncated centres
    planes2 = synth.even_planes(cloud, 300)
    for trunc in (True, False):
        goff, gidx = gc.slice_bands(planes2, truncate_center=trunc)
        ooff, oidx = oc.slice_bands(planes2, truncate_center=trunc)
        assert np.array_equal(goff, ooff)
        assert np.array_equal(gidx, oidx)
    gc.close()


@pytest.mark.parametrize("mode", ["A", "B"])
@pytest.mark.parametrize("variant", ["gen2_contact", "sectpath"])
def test_contours_identical(ctx, mode, variant):
    cloud = synth.panel(100000, 2)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    mn, mx = gc.bbox()
    planes = po.planes(variant, mn[0], mx[0], 15.0)
    goff, gy, gx, gz = gc.slice_contours(planes, mode)
    ooff, oy, ox, oz = oc.slice_contours(planes, mode)
    assert np.array_equal(goff, ooff)
    assert np.array_equal(gy.view(np.uint64), oy.view(np.uint64))
    assert np.array_equal(gx.view(np.uint64), ox.view(np.uint64))
    assert np.array_equal(gz.view(np.uint64), oz.view(np.uint64))
    gc.close()


def test_contours_many_slices_variant_b(ctx):
    cloud = synth.panel(200000, 5)
    oc = po.OracleCloud(cloud)
    gc = api.Cloud(ctx, cloud)
    planes = synth.even_planes(cloud, 80)
    goff, gy, gx, gz = gc.slice_contours(planes, "B")
    ooff, oy, ox, oz = oc.slice_contours(planes, "B")
    assert np.array_equal(goff, ooff)
    assert np.array_equal(gy.view(np.uint64), oy.view(np.uint64))
    assert np.array_equal(gz.view(np.uint64), oz.view(np.uint64))
    gc.close()
