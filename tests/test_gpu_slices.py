"""The slicing chain on the GPU -- k_band_count / k_band_fill / k_band_sort, k_contour (variant A), k_pair_nodes
(variant B), k_slice_order / k_slice_order_cl<2,4,8>, k_compact_nodes(_auto) -- against the numpy restatement
tests/golden/slice_numpy.py, bit for bit: band offsets and lists, node offsets and y / x / z.  Bands of tens of
thousands of members, too large for the numpy brute force, are compared with the CPU oracle instead.

Every cloud of tests/test_slice_reference.py runs through slice_bands, slice_contours in modes A and B and insert_point,
on every route the library chooses between:
  - bands: the constant-pitch closed form and the binary search (PPP_BANDS_SEARCH);
  - variant B: the sync-free chain with sorted-position lists, the same with index lists (multi-projection index,
    PPP_PROJECTIONS=3), and the synchronous chain (PPP_SLICE_SYNC);
  - k_contour: bands either side of its 22000-member shared-memory cap;
  - the node ordering: one CTA (PPP_SLICE_CLUSTER=1) or clusters of 2 / 4 / 8 CTAs, node-key counts either side of its
    launch thresholds, equal-y runs across the CTA chunks of a cluster, the persistent 8-CTA clusters for oversized
    bands, and bands beyond a cluster (sorted by CTA 0 alone in global memory).
"""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import api, synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import slice_numpy as sn  # noqa: E402
import test_slice_reference as tr  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
ROUTE_VARS = ("PPP_SLICE_SYNC", "PPP_PROJECTIONS", "PPP_BANDS_SEARCH", "PPP_SLICE_CLUSTER")
# variant B routes: name -> environment
ROUTES_B = {"async_positions": {}, "sync_indices": {"PPP_SLICE_SYNC": "1"},
            "async_projections": {"PPP_PROJECTIONS": "3"}, "sync_projections": {"PPP_PROJECTIONS": "3", "PPP_SLICE_SYNC": "1"}}


def _env(monkeypatch, env):
    for k in ROUTE_VARS:
        if k in env:
            monkeypatch.setenv(k, env[k])
        else:
            monkeypatch.delenv(k, raising=False)


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _assert_same(got, want, what):
    names = ("offsets", "y", "x", "z")
    for n, a, b in zip(names, got, want):
        assert _same(a, b), "%s: %s differ (%s vs %s entries)" % (what, n, np.asarray(a).shape, np.asarray(b).shape)


# ---------------------------------------------------------------------------------------------------------------------
# every cloud, every route
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", tr.CLOUD_NAMES)
def test_bands_and_contours_match_the_reference(ctx, name, monkeypatch):
    cloud, sweeps = tr.clouds()[name]
    ref = sn.Cloud(cloud)
    want = [(sn.slice_bands(cloud, p, hw, tc), {m: ref.slice_contours(p, m, hw, tc) for m in "AB"}) for p, hw, tc in sweeps]
    for route, env in ROUTES_B.items():
        _env(monkeypatch, env)
        gc = api.Cloud(ctx, cloud)
        for (planes, hw, tc), (bands, nodes) in zip(sweeps, want):
            what = "%s/%s hw=%g tc=%d" % (name, route, hw, tc)
            for search in (False, True):
                if search:
                    monkeypatch.setenv("PPP_BANDS_SEARCH", "1")
                else:
                    monkeypatch.delenv("PPP_BANDS_SEARCH", raising=False)
                off, idx = gc.slice_bands(planes, hw, tc)
                assert _same(off, bands[0]) and _same(idx, bands[1]), (what, search)
                for _ in range(2):   # the second sync-free call sizes its launches from the first
                    _assert_same(gc.slice_contours(planes, "B", hw, tc), nodes["B"], what + " B")
                if "PPP_SLICE_SYNC" not in env:   # variant A does not read it
                    _assert_same(gc.slice_contours(planes, "A", hw, tc), nodes["A"], what + " A")
            # insert_point on the two largest bands
            off, idx = bands
            for s in np.argsort(np.diff(off))[-2:]:
                b = idx[off[s]:off[s + 1]]
                for mode in "AB":
                    y, x, z, _, _ = ref.insert_point(b, planes[s], mode)
                    gy, gx, gz = gc.insert_point(b, planes[s], mode)
                    assert _same(gy, y) and _same(gx, x) and _same(gz, z), (what, mode, float(planes[s]))
        gc.close()


def test_launch_names_show_the_routes(ctx, monkeypatch):
    """slice_bands and variant A sort the bands (band_sort); variant A runs contour_gen2; a band beyond what the first
    ordering launch holds goes to slice_order_big."""
    _env(monkeypatch, {})
    c = synth.panel(200000, 51)
    gc = api.Cloud(ctx, c)
    ctx.kernel_profile(True)
    try:
        ctx.kernel_profile_read()
        gc.slice_bands(synth.even_planes(c, 20))
        assert "band_sort" in ctx.kernel_profile_read()
        gc.slice_contours(synth.even_planes(c, 20), "A")
        prof = ctx.kernel_profile_read()
        assert "contour_gen2" in prof and "band_sort" in prof
        mn, mx = gc.bbox()
        planes = np.array([0.5 * (mn[0] + mx[0])], F32)
        gc.slice_contours(planes, "B", half_width=150.0)
        gc.slice_contours(planes, "B", half_width=150.0)
        assert "slice_order_big" in ctx.kernel_profile_read()
    finally:
        ctx.kernel_profile(False)
    gc.close()


# ---------------------------------------------------------------------------------------------------------------------
# bands: plane sets and routes
# ---------------------------------------------------------------------------------------------------------------------
def _plane_sets(c):
    x = c[:, 0]
    x0, x1 = float(np.nanmin(x)), float(np.nanmax(x))
    rng = np.random.default_rng(11)
    even = synth.even_planes(c, 40)
    pitch = float(even[1] - even[0])
    inside = (even.astype(np.float64) + rng.uniform(-0.2, 0.2, even.shape[0]) * pitch).astype(F32)
    outside = even.copy()
    outside[17] += F32(0.3 * pitch)
    sets = {"one": even[:1], "seven": even[:7], "eight": even[:8], "even": even, "irregular_inside": inside,
            "irregular_outside": outside,
            "sectpath_order": po.planes("sectpath", F32(x0), F32(x1), 9.0),
            "duplicated": np.repeat(even[::4], 3),
            "nan_planes": np.concatenate([even[:10], [np.nan, np.inf, -np.inf, 3.0e9], even[10:20], [np.nan]]).astype(F32),
            "integer_pitch": (np.floor(x0) + 3.0 + 2.0 * np.arange(30)).astype(F32)}
    for S in (6144, 6145):   # either side of BAND_SMEM_BINS / 2 (the per-block histograms in shared memory)
        sets["S%d" % S] = (x0 + (x1 - x0) * (np.arange(S) + 0.5) / S).astype(F32)
    return sets


@pytest.mark.parametrize("tc", [True, False])
def test_band_plane_sets(ctx, tc, monkeypatch):
    """Sv < 8 (never the closed form), constant pitch, irregular pitch just inside and just outside the quarter-pitch
    tolerance, the centre-out order of SectPath's Path_set, duplicated planes, non-finite and out-of-range planes, and
    6144 / 6145 planes: both band routes identical to the reference; variant B contours identical to the oracle."""
    c = tr.limits_cloud(synth.even_planes(synth.panel(12000, seed=5), 40), 2.0)
    c = np.concatenate([c, synth.panel(8000, seed=12)])
    oc = po.OracleCloud(c)
    for key, planes in _plane_sets(c).items():
        want = sn.slice_bands(c, planes, 2.0, tc)
        finite = np.isfinite(planes) & (np.abs(planes) < 2e9)
        owant = oc.slice_contours(planes[finite], "B", 2.0, tc) if len(planes) < 6000 else None
        for search in (False, True):
            _env(monkeypatch, {"PPP_BANDS_SEARCH": "1"} if search else {})
            gc = api.Cloud(ctx, c)
            off, idx = gc.slice_bands(planes, 2.0, tc)
            assert _same(off, want[0]) and _same(idx, want[1]), (key, tc, search)
            if owant is not None:
                got = gc.slice_contours(planes, "B", 2.0, tc)
                counts = np.diff(got[0])
                assert (counts[~finite] == 0).all() and np.array_equal(counts[finite], np.diff(owant[0])), key
                for a, b in zip(got[1:], owant[1:]):
                    assert _same(a, b), (key, tc, search)
            gc.close()
    oc.close()


# ---------------------------------------------------------------------------------------------------------------------
# sizes: k_contour's shared-memory cap, the ordering kernels' thresholds, clusters
# ---------------------------------------------------------------------------------------------------------------------
def banded_cloud(sides, seed=13):
    """One slice per entry (nL, nR) at plane 20.5 + 40 s, limits +-2 (truncate_center=False): exactly nL left and nR
    right members, spread over a smooth surface at ~1 point/mm², and nothing else in the band."""
    rng = np.random.default_rng(seed)
    parts = []
    for s, (nl, nr) in enumerate(sides):
        P = 20.5 + 40 * s
        L = max((nl + nr) / 4.0, 4.0)
        for n, a, b in ((nl, P + 0.01, P + 1.99), (nr, P - 1.99, P - 0.01)):
            x = rng.uniform(a, b, n)
            y = rng.uniform(0, L, n)
            parts.append(np.stack([x, y, 3 * np.sin(x / 17.0) * np.cos(y / 23.0)], axis=1))
    p = np.concatenate(parts).astype(F32)
    return synth.to_pointxyzrgb(p[rng.permutation(p.shape[0])]), (20.5 + 40 * np.arange(len(sides))).astype(F32)


def test_contour_gen2_shared_memory_cap(ctx, monkeypatch):
    """k_contour keeps a slice in shared memory up to 22000 members: bands of 21999, 22000, 22001 and 22002 members
    (odd and even), together and alone."""
    _env(monkeypatch, {})
    c, planes = banded_cloud([(11000, 10999), (11000, 11000), (11001, 11000), (11001, 11001)])
    ref = sn.Cloud(c)
    per = [ref.slice_contours(planes[s:s + 1], "A", 2.0, False) for s in range(4)]
    gc = api.Cloud(ctx, c)
    assert np.array_equal(np.diff(gc.slice_bands(planes, 2.0, False)[0]), [21999, 22000, 22001, 22002])
    got = gc.slice_contours(planes, "A", 2.0, False)
    cat = [np.concatenate([[0], np.cumsum([p[0][1] for p in per])])] + [np.concatenate([p[i] for p in per]) for i in (1, 2, 3)]
    _assert_same(got, cat, "gen2 cap, all four")
    for s in (0, 2, 3):
        _assert_same(gc.slice_contours(planes[s:s + 1], "A", 2.0, False), per[s], "gen2 cap, slice %d" % s)
    gc.close()


ORDER_SIDES = [(1, 1), (2, 1), (2, 3), (512, 511), (512, 512), (513, 512), (2304, 2303), (2304, 2304), (2305, 2304),
               (12288, 12287), (12288, 12288), (12289, 12288), (1023, 40), (1025, 40), (4607, 60), (4609, 60)]


@pytest.fixture(scope="module")
def order_case():
    c, planes = banded_cloud(ORDER_SIDES, seed=14)
    ref = sn.Cloud(c)
    return c, planes, [ref.slice_contours(planes[s:s + 1], "B", 2.0, False) for s in range(len(planes))]


@pytest.mark.parametrize("cluster", [None, 1, 2, 4, 8])
def test_slice_order_sizes(ctx, cluster, order_case, monkeypatch):
    """Node-key counts 1 and 2 and bands either side of 1024, 4608 and 24576 members (the thresholds of k_slice_order's
    thread count and shared memory), each alone in a sweep, twice on one handle (the second sync-free call sizes its
    launches from the first), on the sync-free and the synchronous chain, with one CTA or a cluster per slice."""
    c, planes, want = order_case
    for sync in (False, True):
        env = {"PPP_SLICE_SYNC": "1"} if sync else {}
        if cluster:
            env["PPP_SLICE_CLUSTER"] = str(cluster)
        _env(monkeypatch, env)
        gc = api.Cloud(ctx, c)
        for s in range(len(planes)):
            for rep in range(2):
                _assert_same(gc.slice_contours(planes[s:s + 1], "B", 2.0, False), want[s],
                             "sides %s cluster %s sync %d call %d" % (ORDER_SIDES[s], cluster, sync, rep))
        gc.close()


@pytest.fixture(scope="module")
def stacked_case():
    c = tr.stacked_cloud(layers=60, side=48)
    planes = np.array([10.5, 30.5], F32)
    ref = sn.Cloud(c)
    return c, planes, {m: ref.slice_contours(planes, m, 2.0, False) for m in "AB"}


@pytest.mark.parametrize("cluster", [1, 2, 4, 8])
def test_equal_y_runs_across_cluster_chunks(ctx, cluster, stacked_case, monkeypatch):
    """60 stacked lattices in random index order: 5760 node keys per slice in runs of 120 equal y with different z.
    With 2 / 4 / 8 CTAs per slice the chunks hold 4096 / 2048 / 1024 keys, so runs cross chunk boundaries and the last
    insertion of a run can sit in another CTA's shared memory.  The signed-zero slices pin the first-key rule there."""
    c, planes, want = stacked_case
    sz = tr.signed_zero_cloud()
    sz_want = sn.Cloud(sz).slice_contours(tr.SIGNED_ZERO_PLANES, "B", 2.0, True)
    for route, env in ROUTES_B.items():
        _env(monkeypatch, dict(env, PPP_SLICE_CLUSTER=str(cluster)))
        gc = api.Cloud(ctx, c)
        for rep in range(2):
            _assert_same(gc.slice_contours(planes, "B", 2.0, False), want["B"], "stacked %s C=%d" % (route, cluster))
        if "PPP_SLICE_SYNC" not in env:   # variant A does not read it
            _assert_same(gc.slice_contours(planes, "A", 2.0, False), want["A"], "stacked A")
        gc.close()
        gc = api.Cloud(ctx, sz)
        _assert_same(gc.slice_contours(tr.SIGNED_ZERO_PLANES, "B", 2.0, True), sz_want, "signed zero %s C=%d" % (route, cluster))
        gc.close()


@pytest.mark.parametrize("cluster", [None, 2, 4, 8])
def test_bands_beyond_a_cluster(ctx, cluster, monkeypatch):
    """Bands of 66000, 132000 and 262146 members (33000, 66000 and 131073 node keys); the oracle is the reference here.
    - Synchronous chain, and the second sync-free call (sized from the first one's largest band): every band beyond the
      first launch goes to the persistent 8-CTA clusters (slice_order_big, 8 x 16384 keys).  The 131073-key band does not
      fit them either, so CTA 0 sorts it alone in global memory.
    - First sync-free call: the size estimate (uniform spread of the points along x) is far below these bands, so the
      first launch takes all of them, and every band beyond its cluster's capacity is sorted by CTA 0 alone."""
    c, planes = banded_cloud([(33000, 33000), (66000, 66000), (131073, 131073), (300, 200)], seed=15)
    oc = po.OracleCloud(c)
    want = oc.slice_contours(planes, "B", 2.0, False)
    oc.close()
    ctx.kernel_profile(True)
    try:
        for sync in (False, True):
            env = {"PPP_SLICE_SYNC": "1"} if sync else {}
            if cluster:
                env["PPP_SLICE_CLUSTER"] = str(cluster)
            _env(monkeypatch, env)
            gc = api.Cloud(ctx, c)
            for rep in range(2):
                ctx.kernel_profile_read()
                what = "big bands C=%s sync %d call %d" % (cluster, sync, rep)
                _assert_same(gc.slice_contours(planes, "B", 2.0, False), want, what)
                big = "slice_order_big" in ctx.kernel_profile_read()
                assert big == (sync or rep == 1), what
            gc.close()
    finally:
        ctx.kernel_profile(False)


# ---------------------------------------------------------------------------------------------------------------------
# insert_point with explicit lists; the combined call
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("projections", ["1", "3"])
def test_insert_point_lists(ctx, projections, monkeypatch):
    """Lists holding non-finite points (NaN / inf in any coordinate, x = +-inf included: on neither side), lists reaching
    outside the band (membership by the list's bitmap, not the band limits), one-sided, single and empty lists."""
    _env(monkeypatch, {"PPP_PROJECTIONS": projections})
    for cloud in (tr.nonfinite_cloud(with_inf_x=True), tr.duplicates_cloud(), tr.stagger_cloud()):
        ref = sn.Cloud(cloud)
        gc = api.Cloud(ctx, cloud)
        x = cloud[:, 0]
        fin = sn.finite3(cloud)
        bad = np.flatnonzero(~fin)
        rng = np.random.default_rng(21)
        for p in synth.even_planes(cloud[fin], 6):
            band = sn.band(cloud, p, 2.0, True)
            with np.errstate(invalid="ignore"):
                wide = np.flatnonzero(np.abs(x - p) < 7)
                near_bad = bad[~(np.abs(x[bad] - p) >= 6)]
            lists = {"band_nonfinite": np.union1d(band, near_bad), "wide_nonfinite": np.union1d(wide, bad[::3]),
                     "wide": wide, "thinned": band[rng.random(band.shape[0]) < 0.4],
                     "left_only": band[x[band] > p], "right_only": band[x[band] < p],
                     "right_and_nonfinite": np.union1d(band[x[band] < p], near_bad),
                     "single": band[:1], "empty": band[:0]}
            for key, lst in lists.items():
                lst = np.asarray(lst, np.int32)
                for mode in "AB":
                    y, xx, z, _, _ = ref.insert_point(lst, p, mode)
                    gy, gx, gz = gc.insert_point(lst, p, mode)
                    assert _same(gy, y) and _same(gx, xx) and _same(gz, z), (key, mode, float(p), projections)
        gc.close()


@pytest.mark.parametrize("name", ["lattice", "two_faces", "stagger"])
def test_normals_and_contours_combined(ctx, name, monkeypatch):
    _env(monkeypatch, {})
    cloud, sweeps = tr.clouds()[name]
    ref = sn.Cloud(cloud)
    gc = api.Cloud(ctx, cloud)
    for planes, hw, tc in sweeps:
        for mode in "AB":
            nrm, *nodes = gc.normals_and_contours(planes, mode, k=16, half_width=hw, truncate_center=tc)
            _assert_same(nodes, ref.slice_contours(planes, mode, hw, tc), "%s combined %s" % (name, mode))
    gc.close()


# ---------------------------------------------------------------------------------------------------------------------
# bounds-checked build
# ---------------------------------------------------------------------------------------------------------------------
def test_bounds_checked_library():
    check_lib = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
    if not os.path.exists(check_lib):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    code = ("import os, sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import numpy as np\n"
            "from polishpathplanning_b200 import api\n"
            "import test_slice_reference as tr\n"
            "ctx = api.Context(0)\n"
            "cl = tr.clouds()\n"
            "cases = [cl[k] for k in ('stagger', 'duplicates', 'signed_zero', 'far_side', 'nonfinite', 'box')]\n"
            "cases.append((tr.stacked_cloud(layers=60, side=48), [(np.array([10.5, 30.5], np.float32), 2.0, False)]))\n"
            "for env in ({}, {'PPP_SLICE_SYNC': '1'}, {'PPP_PROJECTIONS': '3'}, {'PPP_SLICE_CLUSTER': '2'},\n"
            "            {'PPP_SLICE_CLUSTER': '4'}, {'PPP_SLICE_CLUSTER': '8'}, {'PPP_BANDS_SEARCH': '1'}):\n"
            "    for k in ('PPP_SLICE_SYNC', 'PPP_PROJECTIONS', 'PPP_SLICE_CLUSTER', 'PPP_BANDS_SEARCH'):\n"
            "        os.environ.pop(k, None)\n"
            "    os.environ.update(env)\n"
            "    for cloud, sweeps in cases:\n"
            "        c = api.Cloud(ctx, cloud)\n"
            "        for planes, hw, tc in sweeps:\n"
            "            c.slice_bands(planes, hw, tc)\n"
            "            for mode in 'AB':\n"
            "                c.slice_contours(planes, mode, hw, tc)\n"
            "                c.slice_contours(planes, mode, hw, tc)\n"
            "                c.insert_point(np.arange(0, cloud.shape[0], 3, dtype=np.int32), planes[0], mode)\n"
            "        c.close()\n"
            "ctx.sync(); print('done')\n" % (ROOT, os.path.join(ROOT, "tests")))
    t0 = time.time()
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PPP_GPU_LIB=check_lib), capture_output=True,
                       text=True, timeout=900)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT failed" not in out, out[-2000:]
    assert r.returncode == 0 and "done" in r.stdout, out[-2000:]
    print("bounds-checked slicing pass: %.1f s" % (time.time() - t0))
