"""ppp_mls_smooth (the reference's smooth(): MovingLeastSquares, order 3, radius 15) against the CPU oracle:
identical rows, points within 2 float32 ulps (>= 99 % bit-identical), normals and curvature within 1e-5; the
mirrors' smooth() flows end in normals and contours bit-exact against the oracle on the smoothed cloud."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from oracle_mls import ppp_oracle_mls as pom
from polishpathplanning_b200 import api, reference_api, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def check_against_oracle(ctx, cloud, radius=15.0, order=3):
    gc = api.Cloud(ctx, np.ascontiguousarray(cloud, np.float32))
    pts, src, nrm = gc.mls_smooth(radius, order, normals=True)
    gc.close()
    oxyz, onrm, osrc, ofit = pom.mls_smooth(cloud, radius, order)
    assert np.array_equal(src, osrc)
    if src.shape[0]:
        a, b = pts[:, 0:3].astype(np.float64), oxyz.astype(np.float64)
        ulps = np.abs(a - b) / np.spacing(np.maximum(np.abs(pts[:, 0:3]), np.abs(oxyz)))
        assert ulps.max() <= 2.0, ulps.max()
        assert np.mean(np.all(pts[:, 0:3] == oxyz, axis=1)) >= 0.99
        assert np.abs(nrm - onrm).max() <= 1e-5
        assert np.array_equal(pts[:, 3:], cloud[src, 3:])   # rgb and padding come from the source records
    return pts, src, ofit


@pytest.mark.parametrize("order", [0, 2, 3])
def test_noisy_panel(ctx, order):
    _, _, fit = check_against_oracle(ctx, synth.panel(200000, seed=11, noise_sigma=0.05), order=order)
    assert fit.all() if order > 1 else not fit.any()


def test_dense_patch_beyond_the_list_limit(ctx):
    """Density 4: ~2,800 neighbours per query, where ppp_radius's fill call refuses (> ~900)."""
    cloud = synth.panel(40000, seed=12, density=4.0, noise_sigma=0.05)
    gc = api.Cloud(ctx, cloud)
    cnt = np.empty(cloud.shape[0], np.int32)
    api.check(gc.lib.ppp_radius(gc._h, None, 0, 0, 15.0, api._ptr(cnt), None, None, None))
    gc.close()
    assert cnt.max() > 900 and np.median(cnt) > 2000
    check_against_oracle(ctx, cloud)


@pytest.mark.parametrize("shape", ["cylinder", "box_with_walls"])
def test_multi_projection_clouds(ctx, shape):
    cloud = synth.cylinder(60000, seed=13) if shape == "cylinder" else synth.box_with_walls(60000, seed=14)
    check_against_oracle(ctx, cloud)


def test_plane_branch_rows(ctx):
    """Clusters of 1..40 points far apart: 0-2 neighbours emit nothing, 3-9 take the plane projection, 10 and more
    the polynomial fit -- the same rows and branches as the oracle."""
    rng = np.random.default_rng(15)
    sizes = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 40]
    pts = np.concatenate([np.array([100.0 * c, 0, 0]) + rng.normal(0, 2.0, (k, 3)) * [1, 1, 0.2]
                          for c, k in enumerate(sizes)]).astype(np.float32)
    _, src, fit = check_against_oracle(ctx, synth.to_pointxyzrgb(pts))
    k = np.repeat(sizes, sizes)[src]
    assert src.shape[0] == sum(s for s in sizes if s >= 3)
    assert np.array_equal(fit == 1, k >= 10)


def test_nan_duplicates_tiny_and_empty(ctx):
    cloud = synth.panel(30000, seed=16, noise_sigma=0.05)
    cloud[::53, 0] = np.nan
    cloud[7::61, 2] = np.inf
    cloud[1000:1200] = cloud[2000:2200]                       # exact duplicates
    check_against_oracle(ctx, cloud)
    check_against_oracle(ctx, synth.panel(5, seed=17))        # tiny: every point sees the others
    check_against_oracle(ctx, synth.panel(2, seed=17))        # fewer than 3 points: no rows
    gc = api.Cloud(ctx, np.zeros((0, 8), np.float32))
    pts, src, nrm = gc.mls_smooth(normals=True)
    assert pts.shape == (0, 8) and src.shape == (0,) and nrm.shape == (0, 4)
    gc.close()


def test_argument_errors(ctx):
    gc = api.Cloud(ctx, synth.panel(1000, seed=18))
    for radius, order in [(0.0, 3), (-1.0, 3), (float("nan"), 3), (float("inf"), 3), (15.0, -1), (15.0, 4)]:
        with pytest.raises(api.PPPError) as e:
            gc.mls_smooth(radius, order)
        assert e.value.status == api._lib.PPP_ERR_INVALID
    out = np.empty((1000, 8), np.float32)
    src = np.empty(1000, np.int32)
    import ctypes as C
    m = C.c_int64(0)
    for stride in (8, 14):
        assert gc.lib.ppp_mls_smooth(gc._h, 15.0, 3, api._ptr(out), stride, None, api._ptr(src), C.byref(m)) == api._lib.PPP_ERR_INVALID
    assert gc.lib.ppp_mls_smooth(gc._h, 15.0, 3, None, 32, None, api._ptr(src), C.byref(m)) == api._lib.PPP_ERR_INVALID
    assert gc.lib.ppp_mls_smooth(gc._h, 15.0, 3, api._ptr(out), 32, None, api._ptr(src), None) == api._lib.PPP_ERR_INVALID
    # a 12-byte record stride (x, y, z only) is accepted
    xyz = np.empty((1000, 3), np.float32)
    api.check(gc.lib.ppp_mls_smooth(gc._h, 15.0, 3, api._ptr(xyz), 12, None, api._ptr(src), C.byref(m)))
    assert m.value == 1000
    gc.close()


def _normals_and_contours_exact(dev_cloud, cloud, normals, variant, mode, tool_radius):
    oc = po.OracleCloud(cloud)
    o = oc.normals(radius=2.5)[0]
    gn = np.concatenate([normals[:, 0:3], normals[:, 4:5]], axis=1)
    assert np.array_equal(np.isnan(gn[:, 0]), np.isnan(o[:, 0]))
    ok = ~np.isnan(o[:, 0])
    assert np.abs(gn[ok] - o[ok]).max() <= 1e-5
    mn, mx = oc.minmax()
    planes = po.planes(variant, mn[0], mx[0], tool_radius)
    goff, gy, gx, gz = dev_cloud.slice_contours(planes, mode)
    ooff, oy, ox, oz = oc.slice_contours(planes, "A" if mode == api.PPP_PAIR_GEN2 else "B")
    assert np.array_equal(goff, ooff)
    assert np.array_equal(gy.view(np.uint64), oy.view(np.uint64)) and np.array_equal(gz.view(np.uint64), oz.view(np.uint64))


def test_reference_api_smooth_flows(ctx, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    pcd = str(tmp_path / "part.pcd")
    synth.write_pcd(pcd, synth.to_pointxyzrgb(synth.panel_metres(40000, 19, noise_sigma=0.05)))
    raw = synth.panel(40000, 19, noise_sigma=0.05)
    oxyz, _, osrc, _ = pom.mls_smooth(raw)
    # SectPath(Smooth = true): smooth in the constructor, then the sweep on the smoothed cloud
    sp = reference_api.SectPath(pcd, 12.0, Smooth=True, ctx=ctx)
    assert np.array_equal(sp.cloud[:, 3:], raw[osrc, 3:])
    assert np.abs(sp.cloud[:, 0:3].astype(np.float64) - oxyz).max() <= 2 * np.spacing(np.abs(oxyz)).max()
    written = synth.read_pcd(str(tmp_path / "smooth_part.pcd"))
    assert np.array_equal(written[:, 0:3], sp.cloud[:, 0:3]) and np.array_equal(written[:, 4], sp.cloud[:, 4])
    nrm = sp.estimate_normal()
    _normals_and_contours_exact(sp._dev(), sp.cloud, nrm, "sectpath", api.PPP_PAIR_SECT, 12.0)
    # path_generater.smooth()
    pg = reference_api.path_generater(pcd, 15.0, ctx=ctx)
    src = pg.smooth()
    assert np.array_equal(src, osrc) and np.array_equal(pg.cloud, sp.cloud)
    nrm = pg.estimate_normal()
    _normals_and_contours_exact(pg._dev(), pg.cloud, nrm, "gen2_contact", api.PPP_PAIR_GEN2, 15.0)


def test_host_adapter_smooth_flow(tmp_path):
    """ppp_main --sect with Smooth = true: smooth_<name>.pcd against the oracle, then normals + sweep on it."""
    host = os.path.join(ROOT, "polishpathplanning_b200", "host")
    subprocess.check_call(["make", "-s", "-C", host])
    pcd = str(tmp_path / "workpiece.pcd")
    synth.write_pcd(pcd, synth.to_pointxyzrgb(synth.panel_metres(40000, 20, noise_sigma=0.05)))
    cfg = str(tmp_path / "config.txt")
    with open(cfg, "w") as f:
        f.write("Tool_Radius = 12\nSmooth = true\nChangeRange = true\nRemoveOutlier = false\n")
    out = str(tmp_path / "sect")
    r = subprocess.run([os.path.join(host, "ppp_main"), "--sect", cfg, pcd, out], capture_output=True, text=True,
                       cwd=str(tmp_path), timeout=300)
    assert r.returncode == 0, r.stderr
    assert "not available" not in r.stderr
    smoothed = synth.read_pcd(str(tmp_path / "smooth_workpiece.pcd"))
    raw = synth.panel(40000, 20, noise_sigma=0.05)
    oxyz, _, osrc, _ = pom.mls_smooth(raw)
    assert smoothed.shape[0] == osrc.shape[0]
    assert np.array_equal(smoothed[:, 4], raw[osrc, 4])
    ulps = np.abs(smoothed[:, 0:3].astype(np.float64) - oxyz) / np.spacing(np.abs(oxyz))
    assert ulps.max() <= 2.0 and np.mean(np.all(smoothed[:, 0:3] == oxyz, axis=1)) >= 0.99
    nrm = np.fromfile(out + ".normals.f32", np.float32).reshape(-1, 8)
    off = np.fromfile(out + ".off.i64", np.int64)
    y = np.fromfile(out + ".y.f64", np.float64)
    z = np.fromfile(out + ".z.f64", np.float64)
    oc = po.OracleCloud(smoothed)
    o = oc.normals(radius=2.5)[0]
    gn = np.concatenate([nrm[:, 0:3], nrm[:, 4:5]], axis=1)
    ok = ~np.isnan(o[:, 0])
    assert np.array_equal(np.isnan(gn[:, 0]), ~ok) and np.abs(gn[ok] - o[ok]).max() <= 1e-5
    mn, mx = oc.minmax()
    ooff, oy, ox, oz = oc.slice_contours(po.planes("sectpath", mn[0], mx[0], 12.0), "B")
    assert np.array_equal(off, ooff) and np.array_equal(y, oy) and np.array_equal(z, oz)


def test_bounds_checked_library():
    check_lib = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
    if not os.path.exists(check_lib):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from polishpathplanning_b200 import api, synth\n"
            "ctx = api.Context(0)\n"
            "for cloud in (synth.panel(20000, 1, noise_sigma=0.05), synth.cylinder(20000, 2), synth.panel(3000, 3, density=4.0)):\n"
            "    for order in (0, 2, 3):\n"
            "        c = api.Cloud(ctx, cloud); c.mls_smooth(15.0, order, normals=True); c.close()\n"
            "ctx.sync(); print('done')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PPP_GPU_LIB=check_lib), capture_output=True,
                       text=True, timeout=600)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT failed" not in out, out[-2000:]
    assert r.returncode == 0 and "done" in r.stdout, out[-2000:]
