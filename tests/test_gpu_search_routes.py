"""Search routes that only rare queries take, each against a brute-force reference.

- k_knn_warp on rings whose clamped row span is more than 64 rows: the ring's cell ranges are looked up in several
  batches.  Queries in a small cluster far from the rest of the cloud, on a fine grid, need such rings.
- Radius normals through each stage of normals_radius_launch on one cloud: k_radius_normals32 (up to 32 neighbours),
  the one-warp-per-query k_radius_warp (up to 512) and the generic k_search tail (more than 512).
"""
import os
import re
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from polishpathplanning_b200 import api, synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import query_numpy as qn  # noqa: E402
from test_gpu_parity import NORMAL_TOL, _cmp_normals  # noqa: E402

pytestmark = pytest.mark.gpu
F32 = np.float32


def two_clusters():
    """A 40 x 40 mm panel of 12800 points and, 60 mm away along y, a cluster of 5 points."""
    rng = np.random.default_rng(71)
    n = 12800
    big = np.stack([rng.random(n) * 40, rng.random(n) * 40, rng.normal(0, 0.05, n)], axis=1)
    small = np.array([[20.0, 100.0, 0.0], [20.3, 100.2, 0.01], [19.8, 99.7, -0.02], [20.1, 99.9, 0.0],
                      [20.4, 99.6, 0.03]])
    return synth.to_pointxyzrgb(np.concatenate([big, small]).astype(F32)), small.shape[0]


@pytest.mark.parametrize("k", [16, 32, 64])
def test_hand_over_kernel_past_64_rows_of_ring(ctx, k, monkeypatch, capfd):
    """Cells of 0.5 mm make a grid of 80 x 200 cells.  The small cluster holds fewer than k points, so its queries
    (and those between the clusters) expand their rings until they reach the panel, 120 cells away: past 32 rings a
    ring spans more than 64 cell rows."""
    c, n_small = two_clusters()
    rng = np.random.default_rng(72)
    between = np.stack([np.full(8, 20.0), np.linspace(45.0, 95.0, 8), np.zeros(8)], axis=1)
    q = np.ascontiguousarray(np.concatenate([c[-n_small:, :3], between, c[rng.choice(c.shape[0] - n_small, 400), :3]]),
                             dtype=F32)
    monkeypatch.setenv("PPP_DEBUG", "1")
    gc = api.Cloud(ctx, c)
    gc.set_cell_hint(0.5)
    capfd.readouterr()
    gi, gd = gc.knn(k, queries=q)
    err = capfd.readouterr().err
    m = re.findall(r"knn fast path: (\d+) queries, (\d+) handed", err)
    assert m and int(m[-1][0]) == q.shape[0], err
    assert int(m[-1][1]) >= n_small + between.shape[0], err
    wi, wd = qn.knn(c, q, k)
    assert np.array_equal(gi, wi) and np.array_equal(gd.view(np.uint32), wd.view(np.uint32))
    gc.close()


def three_densities():
    """A curved 200 x 200 mm sheet at 0.8 points / mm^2 (about 16 neighbours at r = 2.5), a 10 x 10 mm patch at
    8 more (about 170) and a 5 x 5 mm patch at 40 more (about 800).  The sheet holds most of the points, so the
    sampled density stays low enough for the fast radius kernel: density * pi * r^2 <= 24."""
    rng = np.random.default_rng(73)

    def patch(n, x0, y0, w):
        return np.stack([x0 + rng.random(n) * w, y0 + rng.random(n) * w], axis=1)

    xy = np.concatenate([patch(32000, 0.0, 0.0, 200.0), patch(800, 50.0, 50.0, 10.0), patch(1000, 150.0, 150.0, 5.0)])
    z = 50.0 + 5.0 * np.sin(xy[:, 0] / 40.0) * np.cos(xy[:, 1] / 50.0) + rng.normal(0, 0.02, xy.shape[0])
    return synth.to_pointxyzrgb(np.concatenate([xy, z[:, None]], axis=1).astype(F32))


@pytest.mark.parametrize("flags", [api.PPP_COV_PCL110, api.PPP_COV_SHIFTED])
def test_radius_normals_through_every_stage(ctx, flags):
    c = three_densities()
    r = 2.5
    o, cnt = po.OracleCloud(c).normals(radius=r, cov_variant=flags)
    assert (cnt <= 32).sum() > 1000 and ((cnt > 32) & (cnt <= 512)).sum() > 100 and (cnt > 512).sum() > 100
    gc = api.Cloud(ctx, c)
    ctx.kernel_profile(True)
    try:
        ctx.kernel_profile_read()
        g = gc.normals_radius(r, flags=flags)
        prof = ctx.kernel_profile_read()
    finally:
        ctx.kernel_profile(False)
    # the fast kernel and its warp hand-over ran; the count launch of the generic tail follows only when the warp
    # kernel handed queries on
    assert "radius_normals" in prof and "radius_redo" in prof, prof
    assert "radius_count" in prof and "knn_redo" in prof, prof
    mx, frac_exact = _cmp_normals(g, o)
    print("three densities flags=%d max|diff|=%.3g bit-exact rows=%.4f" % (flags, mx, frac_exact))
    assert mx <= NORMAL_TOL
    gc.close()
