"""CPU oracle of the MLS pre-filter (smooth(): MovingLeastSquares, order 3, radius 15) against the independent numpy
restatement, plus properties that need no recalled PCL arithmetic."""
import os
import sys

import numpy as np
import pytest

from oracle_mls import ppp_oracle_mls as pom
from polishpathplanning_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import mls_f64_numpy as mls_np  # noqa: E402


def agree(a, b, min_identical=0.99):
    """The parity bar: every coordinate within 2 float32 ulps, at least `min_identical` of the rows bit-identical."""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    ulps = np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.spacing(np.maximum(np.abs(a), np.abs(b)))
    assert ulps.max() <= 2.0, ulps.max()
    assert np.mean(np.all(a == b, axis=1)) >= min_identical


@pytest.mark.parametrize("name", ["noisy_panel", "cylinder"])
def test_oracle_matches_numpy_restatement(name):
    cloud = synth.panel(20000, seed=1, noise_sigma=0.05) if name == "noisy_panel" else synth.cylinder(6000, seed=2)
    xyz, nrm, src, fit = pom.mls_smooth(cloud)
    qs = np.random.default_rng(0).choice(cloud.shape[0], 300, replace=False)
    rows = mls_np.mls_rows(cloud, qs)
    pos = {int(s): i for i, s in enumerate(src)}
    got, ref = [], []
    for q, r in zip(qs, rows):
        assert (r is None) == (int(q) not in pos)
        if r is None:
            continue
        o = pos[int(q)]
        assert r[3] is not None and r[3] == bool(fit[o])
        got.append(xyz[o])
        ref.append(r[0])
        sign = np.sign(np.dot(nrm[o, :3], r[1]))          # eigh's eigenvector sign is arbitrary
        assert np.abs(nrm[o, :3] - sign * r[1]).max() <= 1e-5
        assert abs(nrm[o, 3] - r[2]) <= 1e-5
    assert len(got) == 300
    agree(got, ref)


def test_tilted_plane_stays_on_plane():
    rng = np.random.default_rng(5)
    x, y = rng.random(20000) * 140, rng.random(20000) * 140
    z = 0.3 * x - 0.2 * y + 5.0
    cloud = synth.to_pointxyzrgb(np.stack([x, y, z], axis=1).astype(np.float32))
    xyz, _, src, fit = pom.mls_smooth(cloud)
    assert src.shape[0] == cloud.shape[0] and fit.all()
    p = xyz.astype(np.float64)
    dist = np.abs(0.3 * p[:, 0] - 0.2 * p[:, 1] + 5.0 - p[:, 2]) / np.sqrt(1 + 0.09 + 0.04)
    assert dist.max() <= 1e-4


def test_noisy_panel_rms_drops():
    n, density, sigma = 60000, 1.0, 0.05
    cloud = synth.panel(n, seed=3, noise_sigma=sigma)
    L = np.sqrt(n / density)

    def surface(x, y):   # synth.panel_metres' height field (millimetres)
        return 20.0 * np.sin(2 * np.pi * x / 400.0) * np.cos(2 * np.pi * y / 300.0) + 1e-4 * (x - L / 2) ** 2

    xyz, _, src, _ = pom.mls_smooth(cloud)
    p = xyz.astype(np.float64)
    inner = (p[:, 0] > 20) & (p[:, 0] < L - 20) & (p[:, 1] > 20) & (p[:, 1] < L - 20)
    raw = cloud[src].astype(np.float64)
    rms_raw = np.sqrt(np.mean((raw[inner, 2] - surface(raw[inner, 0], raw[inner, 1])) ** 2))
    rms_mls = np.sqrt(np.mean((p[inner, 2] - surface(p[inner, 0], p[inner, 1])) ** 2))
    assert rms_raw > 0.04 and rms_mls * 4 <= rms_raw, (rms_raw, rms_mls)


def clusters(sizes, spacing=100.0, spread=2.0, seed=0):
    """Clusters of the given sizes, far apart (every point's radius-15 ball holds exactly its own cluster)."""
    rng = np.random.default_rng(seed)
    pts = []
    for c, k in enumerate(sizes):
        centre = np.array([c * spacing, 0.0, 0.0])
        pts.append(centre + rng.normal(0.0, spread, (k, 3)) * np.array([1.0, 1.0, 0.2]))
    return synth.to_pointxyzrgb(np.concatenate(pts).astype(np.float32))


def test_isolated_points_emit_nothing():
    cloud = clusters([1, 2, 1, 2, 30])
    _, _, src, _ = pom.mls_smooth(cloud)
    assert src.tolist() == list(range(6, 36))


def test_few_neighbours_take_the_plane_branch():
    sizes = [3, 4, 5, 6, 7, 8, 9, 10, 40]
    cloud = clusters(sizes)
    xyz, nrm, src, fit = pom.mls_smooth(cloud, order=3)
    assert src.tolist() == list(range(cloud.shape[0]))
    k = np.repeat(sizes, sizes)
    assert np.all(fit[k < 10] == 0) and np.all(fit[k >= 10] == 1)
    # plane branch: the point is the query projected onto its cluster's least-squares plane
    start = 0
    for s in sizes[:7]:
        p = cloud[start:start + s, :3].astype(np.float64)
        c = p.mean(axis=0)
        n = np.linalg.eigh((p - c).T @ (p - c))[1][:, 0]
        assert np.abs((xyz[start:start + s] - c) @ n).max() <= 1e-4
        start += s
    # order 0 and 1: the plane projection for every row
    for order in (0, 1):
        assert not pom.mls_smooth(cloud, order=order)[3].any()


def test_nan_points_emit_nothing():
    cloud = synth.panel(5000, seed=4, noise_sigma=0.05)
    cloud[::97, 1] = np.nan
    cloud[5::101, 2] = np.inf
    _, _, src, _ = pom.mls_smooth(cloud)
    bad = ~np.isfinite(cloud[:, :3]).all(axis=1)
    assert not np.isin(np.flatnonzero(bad), src).any()
    assert np.array_equal(src, np.flatnonzero(~bad))


def test_order_out_of_range():
    with pytest.raises(ValueError):
        pom.mls_smooth(synth.panel(100, seed=0), order=4)
