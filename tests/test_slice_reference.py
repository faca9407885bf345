"""The numpy restatement of the slicing chain (tests/golden/slice_numpy.py) against the CPU oracle, and small cases with
a known answer (CPU only).

Band lists, left_pair / right_pair of every slice and the node arrays must agree bit for bit on every cloud that
tests/test_gpu_slices.py runs on the GPU: lattices with distance ties in both metrics and equal-y runs, near-duplicates at
float d² == 0 (where NN_full picks the lowest index), stacked faces (equal y, different z), signed zeros, points exactly on
and one ulp outside the band limits, a panel 3000 mm from the origin, bands with a few far-away points on one side,
closed and steep shapes and non-finite points.  Once these pass, the reference is the yardstick of the GPU tests.

Clouds with a point at x = +-inf and finite y, z are left out of the oracle comparison: the oracle follows the
reference's dot product, which puts such a point on a side, while the library drops it (include/ppp_gpu.h)."""
import os
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import slice_numpy as sn  # noqa: E402

F32 = np.float32


# ---------------------------------------------------------------------------------------------------------------------
# clouds (shared with tests/test_gpu_slices.py)
# ---------------------------------------------------------------------------------------------------------------------
def lattice(side=40, stagger=False, z=0.0):
    """side x side points, spacing 1, in index order x-major.  stagger: odd x columns shifted by 0.5 in y, so every
    point has two nearest neighbours at equal distance on the other side of a plane between two columns."""
    g = np.arange(side, dtype=F32)
    xx, yy = np.meshgrid(g, g, indexing="ij")
    if stagger:
        yy = yy + F32(0.5) * (xx % 2)
    return np.stack([xx.ravel(), yy.ravel(), np.full(xx.size, z, F32)], axis=1).astype(F32)


def lattice_cloud():
    return synth.to_pointxyzrgb(lattice())


def stagger_cloud(seed=1):
    """Staggered lattice in random index order: ties between different points in both metrics."""
    p = lattice(48, stagger=True)
    return synth.to_pointxyzrgb(p[np.random.default_rng(seed).permutation(p.shape[0])])


def duplicates_cloud(seed=2):
    """Staggered lattice + exact duplicates + twins of the y = 0 row at float d² == 0 (y = 1e-30, 3e-31, -0.0 and
    z = 1e-30), all in random index order: NN_full maps each of them to the lowest index of its group.
    Appended last: a = (-3e-23, 0, 0), b = (-1e-23, 1e-23, 0), q = (5e-23, 0, 0).  b is at float d² == 0 (every squared
    difference underflows) from a and from the twins at the origin, but not from q, and b is nearer to q than a: at
    plane 0 the left query q finds b, and NN_full(b), a lower index, changes the node's y."""
    p = lattice(40, stagger=True)
    rng = np.random.default_rng(seed)
    dup = p[rng.choice(p.shape[0], 300, replace=False)]
    row = p[p[:, 1] == 0]
    twins = []
    for dy, dz in ((1e-30, 0.0), (3e-31, 0.0), (-0.0, 0.0), (0.0, 1e-30)):
        t = row.copy()
        t[:, 1] = F32(dy)
        t[:, 2] = F32(dz)
        twins.append(t)
    allp = np.concatenate([p, dup] + twins).astype(F32)
    group = np.array([[-3e-23, 0, 0], [-1e-23, 1e-23, 0], [5e-23, 0, 0]], F32)
    return synth.to_pointxyzrgb(np.concatenate([allp[rng.permutation(allp.shape[0])], group]))


def two_faces_cloud():
    """The lattice and a copy 3 mm above it, the copy at higher indices: every node's last insertion has z = 3."""
    p = lattice()
    q = p.copy()
    q[:, 2] += F32(3.0)
    return synth.to_pointxyzrgb(np.concatenate([p, q]))


def stacked_cloud(layers=40, side=48, seed=4):
    """`layers` copies of a side x side lattice, 3 mm apart in z, in random index order: every y of a slice is inserted
    2 x layers times with different z, and the last insertion (the highest left index) decides."""
    p = lattice(side)
    allp = np.concatenate([p + np.array([0, 0, 3.0 * k], F32) for k in range(layers)]).astype(F32)
    return synth.to_pointxyzrgb(allp[np.random.default_rng(seed).permutation(allp.shape[0])])


def signed_zero_cloud():
    """Two slices whose nodes are -0.0 and +0.0 insertions of one key, in both orders, plus a filler panel.
    Plane 1: right (0, -0.0, 0) + left (3, -1.4e-45, 0) gives y = -0.0, z = 0; right (0, 0, 10) + left (3, 1.4e-45, 10)
    gives y = +0.0, z = 10; the -0.0 pair's left point has the lower index.  Plane 101: the same at x + 100 with the
    +0.0 pair first.  Expected: plane 1 -> one node (-0.0, 10); plane 101 -> one node (+0.0, 0)."""
    tiny = float(np.float32(1.4e-45))
    a = [[3, -tiny, 0], [103, tiny, 10], [0, -0.0, 0], [0, 0.0, 10],
         [3, tiny, 10], [103, -tiny, 0], [100, -0.0, 0], [100, 0.0, 10]]
    filler = synth.panel(3000, seed=9)[:, :3] + np.array([200, 0, 0], F32)
    return synth.to_pointxyzrgb(np.concatenate([np.array(a, F32), filler]).astype(F32))


SIGNED_ZERO_PLANES = np.array([1.0, 101.0], F32)


def limits_cloud(planes, half_width, seed=5):
    """A panel whose points are moved exactly onto lo and hi of every plane, and one ulp outside, for both truncate modes."""
    c = synth.panel(12000, seed=seed)
    rng = np.random.default_rng(seed)
    rows = rng.permutation(c.shape[0])
    k = 0
    for p in planes:
        for tc in (True, False):
            lo, hi = sn.band_limits(p, half_width, tc)
            for v in (lo, hi, np.nextafter(lo, F32(-np.inf)), np.nextafter(hi, F32(np.inf))):
                for _ in range(3):
                    c[rows[k], 0] = v
                    k += 1
    return c


def limits_planes():
    return (np.arange(12, dtype=F32) * F32(9.25) + F32(3.3)).astype(F32)


def offset_cloud():
    """A panel 3000 mm from the origin in x and y: the float closed form of the band range is least precise there."""
    c = synth.panel(12000, seed=6)
    c[:, 0] += F32(3000.0)
    c[:, 1] += F32(3000.0)
    return c


def offset_planes(c):
    x = c[:, 0]
    return (np.float64(x.min()) + 0.375 * np.arange(280) + 1.0).astype(F32)


def far_side_cloud(seed=7):
    """Slice at x = 50.5: a dense right side (x in [48.5, 50.5), y in [0, 300)) and three left points 2000 mm away in y,
    so every nearest-left search of a right point runs out of rings and scans the band's member list, and so do the
    searches from the three left points.  Plus a second slice at 80.5 whose left side is dense and right side far."""
    rng = np.random.default_rng(seed)
    right = np.stack([rng.uniform(48.5, 50.49, 3000), rng.uniform(0, 300, 3000), rng.uniform(-1, 1, 3000)], axis=1)
    left = np.array([[51.0, 2300.0, 0.0], [52.0, 2310.0, 0.5], [51.5, 2290.0, 0.0]])
    left2 = np.stack([rng.uniform(80.51, 82.5, 3000), rng.uniform(0, 300, 3000), rng.uniform(-1, 1, 3000)], axis=1)
    right2 = np.array([[79.0, -1700.0, 0.0], [80.0, -1690.0, 1.0]])
    filler = np.stack([rng.uniform(0, 40, 4000), rng.uniform(0, 300, 4000), rng.uniform(-1, 1, 4000)], axis=1)
    allp = np.concatenate([right, left, left2, right2, filler]).astype(F32)
    return synth.to_pointxyzrgb(allp[rng.permutation(allp.shape[0])])


FAR_SIDE_PLANES = np.array([50.5, 80.5], F32)


def nonfinite_cloud(with_inf_x=False, seed=8):
    """A panel with NaN / inf in y or z (and, with_inf_x, x = +-inf with finite y, z) on many rows."""
    c = synth.panel(12000, seed=seed)
    rng = np.random.default_rng(seed)
    rows = rng.choice(c.shape[0], 400, replace=False)
    c[rows[0:80], 1] = np.inf
    c[rows[80:160], 2] = np.nan
    c[rows[160:240], 1] = -np.inf
    c[rows[240:320], 0] = np.nan
    if with_inf_x:
        c[rows[320:360], 0] = np.inf
        c[rows[360:400], 0] = -np.inf
    return c


def clouds():
    """name -> (cloud, [(planes, half_width, truncate_center), ...])."""
    lat = [(np.array([10.5, 10.0, 20.0, 3.25, 38.5, 0.0], F32), 2.0, False),
           (np.array([10.5, 11.0, 25.9, -1.0, 39.0, 0.0], F32), 2.0, True)]
    sz = signed_zero_cloud()
    lp = limits_planes()
    off = offset_cloud()
    cyl = synth.cylinder(20000, seed=22)
    box = synth.box_with_walls(20000, seed=23)
    nf = nonfinite_cloud()
    return {
        "lattice": (lattice_cloud(), lat),
        "stagger": (stagger_cloud(), lat + [(np.array([7.0, 7.5, 8.25, 30.5], F32), 1.5, False)]),
        "duplicates": (duplicates_cloud(), lat),
        "two_faces": (two_faces_cloud(), lat),
        "signed_zero": (sz, [(SIGNED_ZERO_PLANES, 2.0, True), (SIGNED_ZERO_PLANES, 2.0, False)]),
        "limits": (limits_cloud(lp, 2.0), [(lp, 2.0, True), (lp, 2.0, False)]),
        "offset": (off, [(offset_planes(off), 2.0, False), (offset_planes(off)[::7], 2.0, True)]),
        "far_side": (far_side_cloud(), [(FAR_SIDE_PLANES, 2.0, False)]),
        "cylinder": (cyl, [(synth.even_planes(cyl, 30), 2.0, True)]),
        "box": (box, [(synth.even_planes(box, 30), 2.0, True)]),
        "nonfinite": (nf, [(synth.even_planes(nf, 40), 2.0, True), (synth.even_planes(nf, 25), 2.0, False)]),
    }


CLOUD_NAMES = ["lattice", "stagger", "duplicates", "two_faces", "signed_zero", "limits", "offset", "far_side",
               "cylinder", "box", "nonfinite"]


# ---------------------------------------------------------------------------------------------------------------------
# the reference against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.parametrize("name", CLOUD_NAMES)
def test_reference_matches_the_oracle(name):
    cloud, sweeps = clouds()[name]
    ref = sn.Cloud(cloud)
    oc = po.OracleCloud(cloud)
    for planes, hw, tc in sweeps:
        off, idx = sn.slice_bands(cloud, planes, hw, tc)
        ooff, oidx = oc.slice_bands(planes, hw, tc)
        assert _same(off, ooff) and _same(idx, oidx), (name, hw, tc)
        for mode in ("A", "B"):
            for s, p in enumerate(planes):
                b = idx[off[s]:off[s + 1]]
                y, x, z, lp, rp = ref.insert_point(b, p, mode)
                oy, ox, oz, olp, orp = oc.insert_point(b, float(p), mode)
                assert _same(lp, olp) and _same(rp, orp), (name, mode, float(p))
                assert _same(y, oy) and _same(x, ox) and _same(z, oz), (name, mode, float(p))
            got = ref.slice_contours(planes, mode, hw, tc)
            want = oc.slice_contours(planes, mode, hw, tc)
            assert all(_same(a, b) for a, b in zip(got, want)), (name, mode, hw, tc)
    oc.close()


def test_reference_lists_with_nonfinite_points_match_the_oracle():
    """Explicit lists that hold points with an infinite or NaN y or z: the dot product is NaN, neither side."""
    cloud = nonfinite_cloud()
    ref = sn.Cloud(cloud)
    oc = po.OracleCloud(cloud)
    bad = np.flatnonzero(~sn.finite3(cloud) & np.isfinite(cloud[:, 0]))
    for p in synth.even_planes(cloud, 8):
        near = np.flatnonzero(np.abs(cloud[:, 0] - p) < 3)
        lst = np.union1d(near, bad[np.abs(cloud[bad, 0] - p) < 6]).astype(np.int32)
        assert (~sn.finite3(cloud[lst])).any()
        for mode in ("A", "B"):
            got = ref.insert_point(lst, p, mode)
            want = oc.insert_point(lst, float(p), mode)
            assert all(_same(a, b) for a, b in zip(got, want)), (mode, float(p))
    oc.close()


# ---------------------------------------------------------------------------------------------------------------------
# known answers
# ---------------------------------------------------------------------------------------------------------------------
def test_lattice_known_answer():
    """40 x 40 lattice, plane 10.5, limits 8.5 / 12.5: 160 members (x = 9, 10, 11, 12).  Variant A pairs every right
    point of x = 10 with its left neighbour once (40 pairs); variant B pairs every left point (80 pairs).  Both give
    one node per y, y = 0 .. 39, z = 0."""
    cloud = lattice_cloud()
    ref = sn.Cloud(cloud)
    b = sn.band(cloud, 10.5, 2.0, False)
    assert b.shape[0] == 160
    for mode, npairs in (("A", 40), ("B", 80)):
        y, x, z, lp, rp = ref.insert_point(b, 10.5, mode)
        assert lp.shape[0] == npairs and rp.shape[0] == npairs
        assert np.array_equal(y, np.arange(40.0)) and (x == 10.5).all() and (z == 0).all()
        assert (cloud[rp, 0] == 10).all() and (cloud[lp, 0] == 11).all()


def test_two_faces_known_answer():
    """The lattice and a copy 3 mm above it at higher indices: each y is inserted from both faces, the copy last."""
    cloud = two_faces_cloud()
    ref = sn.Cloud(cloud)
    b = sn.band(cloud, 10.5, 2.0, False)
    for mode in ("A", "B"):
        y, x, z, _, _ = ref.insert_point(b, 10.5, mode)
        assert np.array_equal(y, np.arange(40.0)) and (z == 3.0).all(), mode


def test_signed_zero_known_answer():
    ref = sn.Cloud(signed_zero_cloud())
    pts = ref.pts
    # the single pair of the issue: right (0, -0.0, 0), left (3, -1.4e-45, 0), plane 1 -> y = -0.0
    y, _, z, _, _ = ref.insert_point(np.array([0, 2], np.int32), 1.0, "B")
    assert y.shape == (1,) and y[0] == 0 and np.signbit(y[0]) and z[0] == 0
    for mode in ("A", "B"):
        for tc in (True, False):
            off, y, x, z = ref.slice_contours(SIGNED_ZERO_PLANES, mode, 2.0, tc)
            assert np.array_equal(off, [0, 1, 2]), (mode, tc)
            assert y[0] == 0 and np.signbit(y[0]) and z[0] == 10.0, (mode, tc)        # first key -0.0, last z
            assert y[1] == 0 and not np.signbit(y[1]) and z[1] == 0.0, (mode, tc)     # first key +0.0, last z
    assert pts[2, 1] == 0 and np.signbit(pts[2, 1])


def test_band_limit_rules():
    assert sn.band_limits(10.7, 2.0, True) == (F32(8), F32(12))
    assert sn.band_limits(-10.7, 2.0, True) == (F32(-12), F32(-8))             # truncation toward zero
    assert sn.band_limits(10.7, 2.5, False) == (F32(10.7) - F32(2.5), F32(10.7) + F32(2.5))
    for p in (np.nan, np.inf, -np.inf, 2.0e9, -3.0e9):
        assert sn.band_limits(p) is None
    assert sn.band_limits(1.9e9) is not None


def test_nn_full_lowest_index_at_zero_distance():
    cloud = duplicates_cloud()
    ref = sn.Cloud(cloud)
    p = cloud[:, :3]
    n = p.shape[0] - 3                      # the last three points are the a, b, q group
    twins = np.flatnonzero((np.abs(p[:n, 1]) < 1e-20) & (np.abs(p[:n, 2]) < 1e-20))
    got = ref.nn_full(twins)
    for i, g in zip(twins, got):
        same = np.flatnonzero((p[:, 0] == p[i, 0]) & (np.abs(p[:, 1]) < 1e-20) & (np.abs(p[:, 2]) < 1e-20))
        assert g == same.min()
    assert (got != twins).sum() > 40
    # b is at float d² == 0 from a and from the twins at the origin; a and q are not
    g = ref.nn_full([n, n + 1, n + 2])
    assert g[0] == n and g[1] < n and g[2] == n + 2 and p[g[1], 0] == 0
