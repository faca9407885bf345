"""The brute-force numpy references of tests/golden/query_numpy.py against the oracle's kd-tree (CPU only).

kNN lists, radius lists and coverage flags must agree bit for bit (indices and d² bits) on a panel, on an integer
lattice with exact duplicates and a 1e-4 jittered copy, and on a cylinder, for queries on points, off the surface,
outside the bounding box and far away.  The float64 principal-curvature restatement must agree with the oracle's
float32 arithmetic within a float32 error bound.  Once these pass, the references can be trusted as the yardstick
of tests/test_gpu_queries.py."""
import os
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import query_numpy as qn  # noqa: E402

F32 = np.float32
EPS32 = float(np.finfo(np.float32).eps)


def lattice_cloud(side=60, seed=3):
    """Integer lattice (spacing 1, z = 0) + 300 exact duplicates + a copy of 1500 points jittered by ~1e-4."""
    g = np.arange(side, dtype=F32)
    xx, yy = np.meshgrid(g, g, indexing="ij")
    lat = np.stack([xx.ravel(), yy.ravel(), np.zeros(xx.size, F32)], axis=1)
    rng = np.random.default_rng(seed)
    jit = lat[rng.choice(lat.shape[0], 1500, replace=False)] + rng.normal(0, 1e-4, (1500, 3)).astype(F32)
    pts = np.concatenate([lat, lat[rng.choice(lat.shape[0], 300, replace=False)], jit]).astype(F32)
    return synth.to_pointxyzrgb(pts[rng.permutation(pts.shape[0])])


def clouds():
    return {
        "panel": synth.panel(20000, seed=21, noise_sigma=0.05),
        "lattice": lattice_cloud(),
        "cylinder": synth.cylinder(20000, seed=22),
    }


def queries(cloud, seed):
    rng = np.random.default_rng(seed)
    p = cloud[:, :3]
    n = p.shape[0]
    lo, hi = p.min(axis=0), p.max(axis=0)
    on = p[rng.integers(0, n, 150)]
    off = on + rng.normal(0, 1.0, on.shape).astype(F32)
    out = hi + rng.uniform(1, 100, (40, 3)).astype(F32)
    far = np.array([[1e4, 0, 0], [0, -1e6, 0], [1e8, 1e8, 0], [0, 0, 1e12], [-1e20, 0, 0]], F32) + lo
    lat = np.round(p[rng.integers(0, n, 40)]) + F32(0.5) * rng.integers(0, 2, (40, 3)).astype(F32)
    return np.ascontiguousarray(np.concatenate([on, off, out, far, lat]).astype(F32))


@pytest.mark.parametrize("name", ["panel", "lattice", "cylinder"])
def test_knn_radius_coverage_match_the_oracle(name):
    cloud = clouds()[name]
    q = queries(cloud, 5)
    oc = po.OracleCloud(cloud)
    for k in (1, 10, 33, 100):
        ri, rd = qn.knn(cloud, q, k)
        oi, od = oc.knn(k, queries=q)
        assert np.array_equal(rd.view(np.uint32), od.view(np.uint32)), (name, k)
        assert np.array_equal(ri, oi), (name, k)
    # all-infinite rows: the k lowest indices, each at d² = inf
    far = ~np.isfinite(rd).any(axis=1)
    assert far.sum() >= 1 and (ri[far] == np.arange(100)[None, :]).all()
    for r in (0.5, 2.5, 7.5):
        rc, ro, ridx, rdd = qn.radius(cloud, q, r)
        oc_, oo, oidx, odd = oc.radius(r, queries=q)
        assert np.array_equal(rc, oc_) and np.array_equal(ro, oo), (name, r)
        assert np.array_equal(ridx, oidx) and np.array_equal(rdd.view(np.uint32), odd.view(np.uint32)), (name, r)
        assert np.array_equal(qn.coverage(cloud, q, r), oc.coverage_mark(q, r)), (name, r)
    oc.close()


def test_lattice_radius_exactly_on_r2_is_excluded():
    """d² == r² exactly (integer lattice, r = 1, 2, sqrt(2)): membership is strict, as FLANN's RadiusResultSet."""
    cloud = lattice_cloud()
    q = np.array([[10, 10, 0], [20.5, 20, 0], [30, 30, 0]], F32)
    oc = po.OracleCloud(cloud)
    for r in (1.0, 2.0, float(np.sqrt(F32(2.0)))):
        rc, _, ridx, rdd = qn.radius(cloud, q, r)
        oc_, _, oidx, _ = oc.radius(r, queries=q)
        assert np.array_equal(rc, oc_) and np.array_equal(ridx, oidx)
        assert (rdd < F32(r * r)).all()
    oc.close()


def test_coverage_edge_radii():
    cloud = clouds()["panel"]
    q = queries(cloud, 6)[:200]
    rng = np.random.default_rng(7)
    radii = rng.uniform(0.3, 40, q.shape[0])
    radii[::7] *= -1
    radii[3::11] = np.nan
    radii[5::13] = 0.0
    radii[6::17] = 1e-30
    oc = po.OracleCloud(cloud)
    want = np.zeros(cloud.shape[0], np.uint8)
    for t in range(q.shape[0]):
        if not np.isnan(radii[t]):
            oc.coverage_mark(q[t:t + 1], abs(radii[t]), want)
    assert np.array_equal(qn.coverage(cloud, q, radii), want)
    assert not qn.coverage(cloud, q, np.full(q.shape[0], np.nan)).any()
    oc.close()


@pytest.mark.parametrize("name", ["panel", "cylinder"])
@pytest.mark.parametrize("k", [10, 50])
def test_principal_curvatures_f64_within_a_float32_bound(name, k):
    cloud = clouds()[name]
    q = queries(cloud, 8)[:300]
    oc = po.OracleCloud(cloud)
    nrm, _ = oc.normals(k=16)
    out, nn0 = oc.principal_curvatures(nrm, q, k)
    idx, _ = qn.knn(cloud, q, k)
    assert np.array_equal(nn0, np.where(idx[:, 0] >= 0, idx[:, 0], -1))
    ref, gap, scale = qn.principal_curvatures_f64(nrm, idx)
    ok = np.isfinite(ref).all(axis=1)
    assert np.array_equal(np.isnan(out).any(axis=1), ~ok)
    check_curvatures_f64(out[ok], ref[ok], gap[ok], scale[ok], k)
    oc.close()


def check_curvatures_f64(got, ref, gap, scale, m, c_val=16.0, c_dir=4096.0, min_well=0.5):
    """float32 result vs float64.  scale (per row, from principal_curvatures_f64) times the unit roundoff is the size of
    the float32 evaluation's error in C: eigenvalues must be within c_val * eps32 * scale / m, the direction (up to
    sign) within c_dir * eps32 * scale / (l2 - l1) -- checked where that is below 0.1; beyond it the direction is
    not determined by float32 data.  Measured: eigenvalues <= 0.45 (panel, cylinder) and <= 7.5 (box with walls,
    k = 50; the closed-form cubic loses more when eigenvalues cluster), directions <= 670 (panel, cylinder) and <= 1312
    (box with walls) of these units.  Returns the two ratios per row."""
    err_v = np.abs(got[:, 3:5].astype(np.float64) - ref[:, 3:5]).max(axis=1) / (EPS32 * scale / m)
    assert (err_v <= c_val).all(), err_v.max()
    dots = np.abs((got[:, 0:3].astype(np.float64) * ref[:, 0:3]).sum(axis=1))
    sin = np.sqrt(np.maximum(0.0, 1.0 - dots * dots))
    unit = EPS32 * scale / np.maximum(gap, 1e-300)
    well = c_dir * unit < 0.1
    assert well.size == 0 or well.mean() >= min_well
    err_d = sin[well] / unit[well]
    assert (err_d <= c_dir).all(), err_d.max()
    return err_v, err_d


def _i32(x):
    return (int(x) + 2**31) % 2**32 - 2**31


@pytest.mark.parametrize("clamped", [False, True])
def test_far_query_ring_arithmetic_in_int32(clamped):
    """The hand-over kernel's ring loop restated with int32 wraparound, for a query 1e20 mm from a grid of 100 x 100
    cells of 1.2 mm: its cell coordinate saturates at INT_MIN / INT_MAX.  Unclamped, -cu, cu + R or R itself wrap
    (the loop then runs ~2^31 rings or stops on a wrapped test); with the coordinate clamped to +-2^29 no sum
    wraps and the loop ends, its block covering the grid, after at most nu + nv rings."""
    nu = nv = 100
    lim = 2**29
    for cu0, cv0 in ((2**31 - 1, 50), (-2**31, 50), (2**31 - 1, -2**31), (-2**31, 2**31 - 1)):
        cu, cv = (max(-lim, min(lim, cu0)), max(-lim, min(lim, cv0))) if clamped else (cu0, cv0)
        wrapped = False

        def op(v):
            nonlocal wrapped
            wrapped |= _i32(v) != v
            return _i32(v)
        du = max(max(op(-cu), op(cu - (nu - 1))), 0)
        dv = max(max(op(-cv), op(cv - (nv - 1))), 0)
        R = max(2, du, dv)
        for ring in range(4 * (nu + nv)):
            covers = op(cu - R) <= 0 and op(cu + R) >= nu - 1 and op(cv - R) <= 0 and op(cv + R) >= nv - 1
            if covers:
                break
            R = op(R + 1)
        if clamped:
            assert covers and not wrapped, (cu0, cv0)
        else:
            assert wrapped, (cu0, cv0)
