"""External-query searches and the kernels built on them, against the brute-force numpy references
(tests/golden/query_numpy.py) and the CPU oracle.

- kNN with a query array through every route: k_knnf<16,16> (k <= 16), k_knnf<32,16> (17..32), k_knnf<64,32> (33..64),
  k_search (k > 64) and the one-warp-per-query hand-over kernel; index lists and d² bits must be identical, for
  every query stride.
- Radius search with a query array, counts-only against fill, strict d² < r², the fill call's list limit.
- k_principal_curvatures: against the oracle within a few float32 ulps, against the float64 restatement within a
  conditioning-aware bound, and analytic cases (cylinder, plane, k = 1, k > n, NaN normals).
- k_coverage_mark (ppp_coverage_mark, ppp_coverage_mark_radii): flags identical to the brute-force union.
- Far-away queries (up to +-FLT_MAX) and radii whose float32 square overflows.
- The same searches under the bounds-checked build.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import _lib, api, synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import query_numpy as qn  # noqa: E402
from test_query_reference import EPS32, check_curvatures_f64, lattice_cloud  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
FMAX = float(np.finfo(np.float32).max)
KS = [1, 2, 3, 8, 10, 15, 16, 17, 24, 31, 32, 33, 48, 50, 63, 64, 65, 100, 250]
# largest measured deviations, printed at the end of the module (pytest -s) so the bars below can be checked against them
MEASURED = {}


def _record(key, value):
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(value))


@pytest.fixture(scope="module", autouse=True)
def _print_measured():
    yield
    print("measured:", json.dumps(MEASURED, sort_keys=True))


def cylinder_r(R=20.0, n=20000, seed=31):
    """Cylinder of radius R about the y axis (length 6R) and its exact radial normals."""
    rng = np.random.default_rng(seed)
    th = rng.random(n) * 2 * np.pi
    y = rng.random(n) * 6 * R
    pts = np.stack([R * np.cos(th), y, R * np.sin(th)], axis=1).astype(F32)
    nrm = np.stack([np.cos(th), np.zeros(n), np.sin(th)], axis=1).astype(F32)
    return synth.to_pointxyzrgb(pts), nrm


def nonfinite_cloud():
    """Panel with NaN / inf points and a dense clump 1000 mm away."""
    c = synth.panel(20000, seed=32, noise_sigma=0.05)
    c[::97, 0] = np.nan
    c[5::131, 2] = np.inf
    c[7::173, 1] = -np.inf
    rng = np.random.default_rng(33)
    clump = (c[:300, :3] * F32(0.01) + F32(1000.0)).astype(F32)
    clump += rng.normal(0, 0.01, clump.shape).astype(F32)
    c[-300:, :3] = clump
    return c


def clouds():
    off = synth.panel(20000, seed=34, noise_sigma=0.05)
    off[:, :3] += F32(3000.0)
    tiny = synth.panel(40, seed=35)
    tiny[3, 1] = np.nan
    return {
        "panel": synth.panel(30000, seed=30, noise_sigma=0.05),
        "lattice": lattice_cloud(),
        "cylinder": synth.cylinder(20000, seed=36),
        "box": synth.box_with_walls(20000, seed=37),
        "nonfinite": nonfinite_cloud(),
        "offset": off,
        "tiny": tiny,
    }


def slice_samples(p, n=200):
    """drawpath-like queries: a spline through the points of a slice |x - xc| < 2, sampled at n y positions."""
    fin = np.isfinite(p).all(axis=1)
    xc = float(np.median(p[fin, 0]))
    band = p[fin & (np.abs(p[:, 0] - xc) < 2)]
    band = band[np.argsort(band[:, 1], kind="stable")]
    y = np.linspace(band[0, 1], band[-1, 1], n)
    return np.stack([np.full(n, xc), y, np.interp(y, band[:, 1], band[:, 2])], axis=1).astype(F32)


def query_sets(cloud, seed=0):
    rng = np.random.default_rng(seed)
    p = cloud[:, :3]
    fin = np.isfinite(p).all(axis=1)
    pf = p[fin]
    lo, hi = pf.min(axis=0), pf.max(axis=0)
    n = pf.shape[0]
    on = pf[rng.integers(0, n, 120)]
    sets = {
        "on_points": on,
        "lattice_coords": (np.round(pf[rng.integers(0, n, 60)]) + F32(0.5) * rng.integers(0, 2, (60, 3))).astype(F32),
        "off_surface": (on + rng.uniform(0.01, 5.0, (120, 1)) * rng.normal(0, 1, (120, 3)) / np.sqrt(3)).astype(F32),
        "slice": slice_samples(p, 100) if n > 100 else on[:10],
        "outside": (np.where(rng.random((60, 3)) < 0.5, lo - rng.uniform(1, 100, (60, 3)),
                             hi + rng.uniform(1, 100, (60, 3)))).astype(F32),
        "far": (lo + np.array([[1e4, 0, 0], [0, -1e4, 0], [1e6, 0, 0], [0, 0, -1e6], [1e8, 1e8, 0], [-1e8, 0, 1e8]])).astype(F32),
        "nonfinite": np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [np.nan, np.nan, np.nan]], F32),
    }
    return sets


def all_queries(cloud, seed=0):
    s = query_sets(cloud, seed)
    return np.ascontiguousarray(np.concatenate(list(s.values())).astype(F32))


def with_stride(q, sf):
    out = np.zeros((q.shape[0], sf), F32)
    out[:, :3] = q
    out[:, 3:] = np.nan   # padding must never be read
    return out


CLOUDS = {}


def state(ctx, name):
    """(cloud, GPU cloud, queries, brute-force lists at k = 250) per cloud, built once."""
    if name not in CLOUDS:
        c = clouds()[name]
        q = all_queries(c, seed=len(name))
        ri, rd = qn.knn(c, q, max(KS))
        oc = po.OracleCloud(c)
        oi, od = oc.knn(max(KS), queries=q)
        oc.close()
        assert np.array_equal(ri, oi) and np.array_equal(rd.view(np.uint32), od.view(np.uint32))
        CLOUDS[name] = (c, api.Cloud(ctx, c), q, ri, rd)
    return CLOUDS[name]


# ---------------------------------------------------------------------------------------------------------------------
# kNN route matrix
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["panel", "lattice", "cylinder", "box", "nonfinite", "offset", "tiny"])
@pytest.mark.parametrize("k", KS)
def test_external_knn_route_matrix(ctx, name, k):
    c, gc, q, ri, rd = state(ctx, name)
    nfin = int(np.isfinite(c[:, :3]).all(axis=1).sum())
    kk = min(k, nfin)
    want_i = np.full((q.shape[0], k), -1, np.int32)
    want_d = np.full((q.shape[0], k), np.inf, F32)
    want_i[:, :kk], want_d[:, :kk] = ri[:, :kk], rd[:, :kk]   # (d², idx) lists: the k-list is a prefix of the 250-list
    first = None
    for sf in (3, 4, 8):
        gi, gd = gc.knn(k, queries=with_stride(q, sf))
        assert np.array_equal(gd.view(np.uint32), want_d.view(np.uint32)), (name, k, sf)
        assert np.array_equal(gi, want_i), (name, k, sf)
        if first is None:
            first = (gi, gd)
        else:
            assert gi.tobytes() == first[0].tobytes() and gd.tobytes() == first[1].tobytes()


@pytest.mark.parametrize("k", [10, 16, 32, 50, 64])
def test_hand_over_kernel_runs_for_far_and_wall_queries(ctx, k, monkeypatch, capfd):
    monkeypatch.setenv("PPP_DEBUG", "1")
    for name, sets in (("box", ("on_points", "off_surface")), ("panel", ("far", "outside"))):
        c, gc, _, _, _ = state(ctx, name)
        qs = query_sets(c, seed=len(name))
        q = np.ascontiguousarray(np.concatenate([qs[s] for s in sets]))
        capfd.readouterr()
        gi, gd = gc.knn(k, queries=q)
        err = capfd.readouterr().err
        m = re.findall(r"knn fast path: (\d+) queries, (\d+) handed", err)
        assert m and int(m[-1][0]) == q.shape[0], err
        assert int(m[-1][1]) > 0, (name, err)
        wi, wd = qn.knn(c, q, k)
        assert np.array_equal(gi, wi) and np.array_equal(gd.view(np.uint32), wd.view(np.uint32))


def test_extreme_queries_and_all_infinite_distances(ctx):
    """Queries at +-1e12, +-1e20 and +-FLT_MAX on each axis (cell coordinates far beyond int32 before clamping).
    Where every float32 d² overflows, the row holds the k lowest finite indices at d² = inf."""
    c = synth.box_with_walls(5000, seed=38)
    c[::50, 0] = np.nan
    gc = api.Cloud(ctx, c)
    vals = [1e12, -1e12, 1e20, -1e20, FMAX, -FMAX]
    q = np.array([[v if a == ax else 10.0 for a in range(3)] for v in vals for ax in range(3)] +
                 [[v, v, v] for v in vals], F32)
    fin_ids = np.flatnonzero(np.isfinite(c[:, :3]).all(axis=1))
    for k in (1, 10, 16, 17, 33, 64, 65, 100):
        gi, gd = gc.knn(k, queries=q)
        wi, wd = qn.knn(c, q, k)
        assert np.array_equal(gi, wi) and np.array_equal(gd.view(np.uint32), wd.view(np.uint32)), k
        allinf = ~np.isfinite(wd).any(axis=1)
        assert allinf.sum() >= 12 and (gi[allinf] == fin_ids[None, :k]).all()
    cnt, _, _, _ = gc.radius(7.5, queries=q)
    assert np.array_equal(cnt, qn.radius(c, q, 7.5)[0])
    assert not gc.coverage_mark(q, 7.5).any()
    gc.close()


# ---------------------------------------------------------------------------------------------------------------------
# radius search with a query array
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["panel", "lattice", "cylinder", "box", "nonfinite"])
def test_external_radius(ctx, name):
    c, gc, q, _, _ = state(ctx, name)
    for r in (0.5, 2.5, 7.5, 15.0):
        wc, wo, wi, wd = qn.radius(c, q, r)
        only = np.empty(q.shape[0], np.int32)
        qq = np.ascontiguousarray(q)
        api.check(gc.lib.ppp_radius(gc._h, api._ptr(qq), qq.shape[0], 12, r, api._ptr(only), None, None, None))
        assert np.array_equal(only, wc), (name, r)
        try:
            cnt, off, idx, d2 = gc.radius(r, queries=q)
        except api.PPPError as e:   # the fill call's documented list limit (~900 entries; lattice and box at r = 15)
            assert e.status == _lib.PPP_ERR_UNSUPPORTED and wc.max() > 512, (name, r, wc.max())
            continue
        assert np.array_equal(cnt, wc) and np.array_equal(off, wo), (name, r)
        assert np.array_equal(idx, wi) and np.array_equal(d2.view(np.uint32), wd.view(np.uint32)), (name, r)


def test_radius_ties_on_the_lattice(ctx):
    """d² == float32(r*r) exactly: excluded (strict <)."""
    c = lattice_cloud()
    gc = api.Cloud(ctx, c)
    q = np.array([[10, 10, 0], [20.5, 20, 0], [30, 30, 0], [15, 40, 0.5]], F32)
    for r in (1.0, 2.0, float(np.sqrt(F32(2.0))), 3.0):
        cnt, off, idx, d2 = gc.radius(r, queries=q)
        wc, wo, wi, wd = qn.radius(c, q, r)
        assert np.array_equal(cnt, wc) and np.array_equal(idx, wi) and np.array_equal(d2, wd)
        assert (d2 < F32(r * r)).all()
        # coverage has the same strict membership
        assert np.array_equal(gc.coverage_mark(q, r), qn.coverage(c, q, r)), r
        rr = np.array([r, -r, np.nan, r])
        assert np.array_equal(gc.coverage_mark_radii(q, rr), qn.coverage(c, q, rr)), r
    gc.close()


def test_radius_list_limit_and_overflowing_radius(ctx):
    dense = synth.panel(20000, seed=39, density=4.0, noise_sigma=0.05)
    gc = api.Cloud(ctx, dense)
    q = np.ascontiguousarray(dense[::500, :3])
    cnt = np.empty(q.shape[0], np.int32)
    api.check(gc.lib.ppp_radius(gc._h, api._ptr(q), q.shape[0], 12, 15.0, api._ptr(cnt), None, None, None))
    assert cnt.max() > 900 and np.array_equal(cnt, qn.radius(dense, q, 15.0)[0])
    with pytest.raises(api.PPPError) as e:
        gc.radius(15.0, queries=q)
    assert e.value.status == _lib.PPP_ERR_UNSUPPORTED
    gc.close()
    # radius 2e19: float32(r*r) = inf admits every point at a finite d²
    small = synth.panel(600, seed=40)
    small[::37, 1] = np.nan
    gs = api.Cloud(ctx, small)
    q = np.concatenate([small[:50, :3], [[1e12, 0, 0], [np.nan, 0, 0]]]).astype(F32)
    cnt, off, idx, d2 = gs.radius(2e19, queries=q)
    wc, wo, wi, wd = qn.radius(small, q, 2e19)
    nfin = int(np.isfinite(small[:, :3]).all(axis=1).sum())
    fq = np.isfinite(q).all(axis=1)
    assert (cnt[fq] == nfin).all() and (cnt[~fq] == 0).all() and fq.sum() >= 3
    assert np.array_equal(cnt, wc) and np.array_equal(idx, wi) and np.array_equal(d2.view(np.uint32), wd.view(np.uint32))
    flags = gs.coverage_mark(q[1:4], 2e19)
    assert np.array_equal(flags, np.isfinite(small[:, :3]).all(axis=1).astype(np.uint8))
    with pytest.raises(api.PPPError) as e:
        gs.mls_smooth(2e19)
    assert e.value.status == _lib.PPP_ERR_INVALID
    gs.close()


# ---------------------------------------------------------------------------------------------------------------------
# principal curvatures
# ---------------------------------------------------------------------------------------------------------------------
def ulps(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)).astype(F32)).astype(np.float64)


PC_ULPS = 4            # pc1 / pc2 against the oracle (same float32 arithmetic; measured on a B200: 1 ulp)
PC_DIR_EPS = 4         # direction components against the oracle, in units of eps32 (measured: identical)


def check_pc(gc, c, nrm, q, k, tag, min_well=0.5):
    out, nn0 = gc.principal_curvatures(nrm, q, k)
    wi, _ = qn.knn(c, q, k)
    gi, _ = gc.knn(k, queries=q)
    assert np.array_equal(gi, wi)
    assert np.array_equal(nn0, wi[:, 0])
    oc = po.OracleCloud(c)
    oout, onn0 = oc.principal_curvatures(nrm, q, k)
    oc.close()
    assert np.array_equal(onn0, nn0)
    assert np.array_equal(np.isnan(out), np.isnan(oout)), tag
    ok = np.isfinite(oout).all(axis=1)
    u = ulps(out[ok, 3:5], oout[ok, 3:5]).max() if ok.any() else 0.0
    dd = (np.abs(out[ok, 0:3].astype(np.float64) - oout[ok, 0:3]).max() / EPS32) if ok.any() else 0.0
    _record("pc_vs_oracle_ulps", u)
    _record("pc_dir_vs_oracle_eps", dd)
    assert u <= PC_ULPS, (tag, u)
    assert dd <= PC_DIR_EPS, (tag, dd)
    ref, gap, scale = qn.principal_curvatures_f64(nrm, wi)
    assert np.array_equal(np.isfinite(ref[:, 3]), np.isfinite(out[:, 3]))
    fin = np.isfinite(ref).all(axis=1) & np.isfinite(out).all(axis=1) & (scale > 0)   # k = 1: C = 0, no direction
    ev, ed = check_curvatures_f64(out[fin], ref[fin], gap[fin], scale[fin], (wi[fin] >= 0).sum(axis=1), min_well=min_well)
    _record("pc_vs_f64_value_units", ev.max() if ev.size else 0.0)
    _record("pc_vs_f64_dir_units", ed.max() if ed.size else 0.0)
    return out


@pytest.mark.parametrize("k", [10, 50])
@pytest.mark.parametrize("name", ["panel", "cylinder", "box"])
def test_principal_curvatures_estimated_normals(ctx, name, k):
    c = {"panel": lambda: synth.panel(30000, seed=41, noise_sigma=0.05), "cylinder": lambda: cylinder_r()[0],
         "box": lambda: synth.box_with_walls(20000, seed=42)}[name]()
    gc = api.Cloud(ctx, c)
    nrm = gc.normals_knn(16)
    qs = query_sets(c, seed=43)
    q = np.ascontiguousarray(np.concatenate([qs["on_points"], qs["off_surface"], qs["slice"], qs["outside"]]))
    # box: corners and wall edges make many directions ill-conditioned, fewer rows have a determined direction
    check_pc(gc, c, nrm, q, k, (name, k), min_well=0.2 if name == "box" else 0.5)
    gc.close()


@pytest.mark.parametrize("k", [10, 50])
def test_principal_curvatures_analytic_cylinder(ctx, k):
    """Exact radial normals on a cylinder of radius 20 about y: the direction of largest curvature is perpendicular
    to the axis and pc2 << pc1."""
    c, nrm = cylinder_r()
    gc = api.Cloud(ctx, c)
    q = np.ascontiguousarray(c[::97, :3])
    out = check_pc(gc, c, nrm, q, k, ("cylinder-analytic", k))
    assert np.isfinite(out).all()
    assert np.abs(out[:, 1]).max() < 1e-2
    assert (out[:, 4] < 0.05 * out[:, 3]).all()
    gc.close()


def test_principal_curvatures_degenerate_cases(ctx):
    rng = np.random.default_rng(44)
    plane = synth.to_pointxyzrgb(np.stack([rng.random(3000) * 50, rng.random(3000) * 50, np.zeros(3000)], axis=1).astype(F32))
    up = np.tile(np.array([[0, 0, 1, 0]], F32), (3000, 1))
    gc = api.Cloud(ctx, plane)
    oc = po.OracleCloud(plane)
    q = np.ascontiguousarray(plane[:40, :3] + F32(0.1))
    for k in (1, 10, 50):
        for side in (gc, oc):
            out, _ = side.principal_curvatures(up, q, k)
            assert (out[:, 3:5] == 0).all() and np.isnan(out[:, 0:3]).all(), k
    gc.close()
    oc.close()
    # k = 1 on a curved surface and k > finite points
    c = synth.panel(60, seed=45)
    c[::7, 0] = np.nan
    gc = api.Cloud(ctx, c)
    nrm = gc.normals_knn(8)
    nrm[np.isnan(nrm)] = 0.5
    q = np.ascontiguousarray(np.concatenate([c[1:20, :3], [[np.nan, 0, 0]]]).astype(F32))
    for k in (1, 50, 100):
        check_pc(gc, c, nrm, q, k, ("small", k), min_well=0.0)
    # a neighbour whose normal is NaN poisons the row, the same on both sides
    bad = nrm.copy()
    bad[2, 1] = np.nan
    out, _ = gc.principal_curvatures(bad, q, 10)
    wi, _ = qn.knn(c, q, 10)
    hit = (wi == 2).any(axis=1)
    assert hit.any() and np.isnan(out[hit, 3]).all() and np.isfinite(out[~hit & np.isfinite(q).all(axis=1), 3]).all()
    oout, _ = po.OracleCloud(c).principal_curvatures(bad, q, 10)
    assert np.array_equal(np.isnan(out), np.isnan(oout))
    # normal strides of 12, 16 and 32 bytes
    got = [gc.principal_curvatures(np.ascontiguousarray(with_stride(nrm[:, :3], sf)), q, 10)[0] for sf in (3, 4, 8)]
    assert got[0].tobytes() == got[1].tobytes() == got[2].tobytes()
    gc.close()


# ---------------------------------------------------------------------------------------------------------------------
# coverage
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["panel", "cylinder", "box", "nonfinite"])
def test_coverage_flags(ctx, name):
    c, gc, q, _, _ = state(ctx, name)
    rng = np.random.default_rng(46)
    for r in (0.5, 7.5, 40.0):
        assert np.array_equal(gc.coverage_mark(q, r), qn.coverage(c, q, r)), (name, r)
    # per-query radii on a sparse subset, so that the union is far from the whole cloud and every radius matters
    q = np.ascontiguousarray(q[::13])
    nq = q.shape[0]
    radii = rng.uniform(0.3, 10.0, nq)
    radii[7::19] = 40.0
    radii[::5] *= -1
    radii[1::9] = 0.0
    radii[2::11] = 1e-40
    radii[3::13] = np.nan
    want = qn.coverage(c, q, radii)
    assert 0.01 < want.mean() < 0.7 and not np.array_equal(want, qn.coverage(c, q, np.nanmax(np.abs(radii))))
    assert np.array_equal(gc.coverage_mark_radii(q, radii), want), name
    assert not gc.coverage_mark_radii(q, np.full(nq, np.nan)).any()
    # accumulation: flags no query reaches keep whatever they held (also values other than 0 and 1)
    start = rng.choice(np.array([0, 1, 2, 7, 255], np.uint8), c.shape[0])
    got = gc.coverage_mark_radii(q, radii, flags=start.copy())
    hit = qn.coverage(c, q, radii).astype(bool)
    assert np.array_equal(got, np.where(hit, np.uint8(1), start))
    nan_pts = ~np.isfinite(c[:, :3]).all(axis=1)
    assert np.array_equal(got[nan_pts], start[nan_pts])
    # an infinite radius marks every finite point; so does one whose float32 square overflows
    for big in (np.inf, -np.inf, 3e19):
        rr = np.full(nq, np.nan)
        rr[0] = big
        f = gc.coverage_mark_radii(q[:1].copy(), rr[:1])
        assert np.array_equal(f, (~nan_pts).astype(np.uint8)), big


# ---------------------------------------------------------------------------------------------------------------------
# bounds-checked build
# ---------------------------------------------------------------------------------------------------------------------
def test_bounds_checked_library():
    check_lib = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
    if not os.path.exists(check_lib):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np\n"
            "from polishpathplanning_b200 import api, synth\n"
            "ctx = api.Context(0)\n"
            "for cloud in (synth.panel(20000, 1, noise_sigma=0.05), synth.box_with_walls(20000, 2)):\n"
            "    c = api.Cloud(ctx, cloud)\n"
            "    q = np.concatenate([cloud[::37, :3] + np.float32(0.3), cloud[:20, :3] + np.float32(1e6),\n"
            "                        np.array([[1e20, 0, 0], [0, -3.4e38, 0], [np.nan, 0, 0]], np.float32)]).astype(np.float32)\n"
            "    for k in (1, 10, 16, 17, 32, 33, 64, 65, 100):\n"
            "        c.knn(k, queries=q)\n"
            "    for r in (2.5, 7.5):\n"
            "        c.radius(r, queries=q)\n"
            "    nrm = c.normals_knn(16)\n"
            "    for k in (10, 50):\n"
            "        c.principal_curvatures(nrm, q, k)\n"
            "    c.coverage_mark_radii(q, np.linspace(-40, 40, q.shape[0]))\n"
            "    c.coverage_mark(q, 2e19)\n"
            "    c.sor_mean_distances(50)\n"
            "    c.close()\n"
            "ctx.sync(); print('done')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PPP_GPU_LIB=check_lib), capture_output=True,
                       text=True, timeout=600)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT failed" not in out, out[-2000:]
    assert r.returncode == 0 and "done" in r.stdout, out[-2000:]
