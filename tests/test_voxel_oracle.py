"""The VoxelGrid oracle (oracle_voxel/, the reference's voxel_down()) against an independent numpy restatement, and
the bound between PCL's summation order and the device's."""
import numpy as np
import pytest

from oracle_voxel import ppp_oracle_voxel as ov
from polishpathplanning_b200 import synth
from voxel_cases import edge_cases, overflow_cloud, pcl_order_bound, voxel_numpy

CASES = edge_cases() + [
    ("panel", synth.panel(30000, 5), 1.0),
    ("panel_dense", synth.panel(30000, 6, density=16.0), 0.5),
    ("cylinder", synth.cylinder(20000, 7), 2.0),
    ("box_with_walls", synth.box_with_walls(20000, 8), (1.0, 2.0, 1.5)),
]


@pytest.mark.parametrize("name,cloud,leaf", CASES, ids=[c[0] for c in CASES])
def test_stable_mode_matches_numpy(name, cloud, leaf):
    rec, off, mem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    nrec, noff, nmem = voxel_numpy(cloud, leaf)
    assert np.array_equal(off, noff)
    assert np.array_equal(mem, nmem)
    assert np.array_equal(rec.view(np.uint32), nrec.view(np.uint32))
    # every finite point in exactly one row, ascending inside each row
    assert np.array_equal(np.sort(mem), np.flatnonzero(np.isfinite(cloud[:, :3]).all(axis=1)))
    assert all(np.all(np.diff(mem[a:b]) > 0) for a, b in zip(off[:-1], off[1:]))


@pytest.mark.parametrize("name,cloud,leaf", CASES, ids=[c[0] for c in CASES])
def test_pcl_order_within_bound(name, cloud, leaf):
    """PCL's std::sort order: the same rows and members per row; centroids within (2n + 1) 2^-24 M of the
    stable order's; colours identical (integer sums)."""
    prec, poff, pmem = ov.voxel_grid(cloud, leaf, ov.PCL_ORDER)
    srec, soff, smem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    assert np.array_equal(poff, soff)
    for a, b in zip(soff[:-1], soff[1:]):
        assert np.array_equal(np.sort(pmem[a:b]), smem[a:b])
    bound = pcl_order_bound(cloud, soff, smem)
    diff = np.abs(prec[:, :3].astype(np.float64) - srec[:, :3].astype(np.float64))
    assert np.all(diff <= bound)
    assert np.array_equal(prec[:, 3:].view(np.uint32), srec[:, 3:].view(np.uint32))


def test_crowded_voxel_sums_in_pcl_order_differ():
    """One voxel of 6,000 members: PCL's introsort visits them out of source order, so the two modes really do sum
    in different orders (the bound above is not checked on identical data only)."""
    name, cloud, leaf = [c for c in edge_cases() if c[0] == "crowded"][0]
    _, _, pmem = ov.voxel_grid(cloud, leaf, ov.PCL_ORDER)
    _, _, smem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    assert not np.array_equal(pmem, smem)


def test_overflow_keeps_the_input():
    cloud, leaf = overflow_cloud()
    with pytest.raises(ov.Overflow, match="Integer indices would overflow"):
        ov.voxel_grid(cloud, leaf)
    with pytest.raises(OverflowError):
        voxel_numpy(cloud, leaf)
    # one voxel more per axis is enough: 1291^3 > INT32_MAX >= 1290^3
    xyz = np.array([[0, 0, 0], [1289.5, 1289.5, 1289.5]], np.float32)
    ov.voxel_grid(synth.to_pointxyzrgb(xyz), 1.0)
    with pytest.raises(ov.Overflow):
        ov.voxel_grid(synth.to_pointxyzrgb(xyz * np.float32(1.001)), 1.0)


@pytest.mark.parametrize("leaf", [0.0, -1.0, np.nan, np.inf, (1.0, 0.0, 1.0), 1e-45])
def test_invalid_leaf(leaf):
    with pytest.raises(ValueError):
        ov.voxel_grid(synth.panel(100, 1), leaf)


def test_no_finite_point_gives_no_rows():
    cloud = synth.to_pointxyzrgb(np.full((5, 3), np.nan, np.float32))
    rec, off, mem = ov.voxel_grid(cloud, 1.0)
    assert rec.shape == (0, 8) and np.array_equal(off, [0]) and mem.shape == (0,)
