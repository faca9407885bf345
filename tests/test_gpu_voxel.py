"""ppp_voxel_grid (the reference's voxel_down(): pcl::VoxelGrid) against the CPU oracle: rows, row offsets, members,
x, y, z and colours bit-identical to the oracle's stable order, and within the documented bound of PCL's own order;
PCL's overflow refusal; the dense-scan flow voxel grid -> normals that the radius-list limit otherwise refuses."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from oracle_voxel import ppp_oracle_voxel as ov
from polishpathplanning_b200 import _lib, api, reference_api, synth
from voxel_cases import edge_cases, overflow_cloud, pcl_order_bound

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECK_LIB = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")


@pytest.fixture(scope="module")
def ctx():
    c = api.Context(0)
    yield c
    c.close()


def check_against_oracle(ctx, cloud, leaf):
    gc = api.Cloud(ctx, np.ascontiguousarray(cloud, np.float32))
    rec, off, mem = gc.voxel_grid(leaf)
    gc.close()
    orec, ooff, omem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    assert np.array_equal(off, ooff)
    assert np.array_equal(mem, omem)
    assert np.array_equal(rec.view(np.uint32), orec.view(np.uint32))   # x, y, z, pad, colours, zero padding
    return rec, off, mem


SHAPES = [
    ("panel", lambda: synth.panel(60000, 1), [0.5, 1.0, 2.5]),
    ("panel_dense", lambda: synth.panel(60000, 2, density=16.0), [0.5, (0.25, 0.5, 1.0)]),
    ("cylinder", lambda: synth.cylinder(60000, 3), [0.5, 2.0]),
    ("box_with_walls", lambda: synth.box_with_walls(60000, 4), [1.0, (2.0, 1.0, 0.5)]),
]


@pytest.mark.parametrize("name,make,leaves", SHAPES, ids=[s[0] for s in SHAPES])
def test_shapes_bit_identical_to_oracle(ctx, name, make, leaves):
    cloud = make()
    for leaf in leaves:
        check_against_oracle(ctx, cloud, leaf)


@pytest.mark.parametrize("name,cloud,leaf", edge_cases(), ids=[c[0] for c in edge_cases()])
def test_edge_cases_bit_identical_to_oracle(ctx, name, cloud, leaf):
    check_against_oracle(ctx, cloud, leaf)


def test_large_cloud_every_pass():
    """2.5M points: a multi-tile digit scan, and keys of more than 24 bits, so that all four radix passes run."""
    c = api.Context(0)
    try:
        cloud = synth.panel(2_500_000, 5, density=16.0)
        gc = api.Cloud(c, cloud)
        mn, mx = gc.bbox()
        leaf = (0.2, 0.2, 0.2)
        ext = np.floor(mx / np.float32(leaf[0])) - np.floor(mn / np.float32(leaf[0])) + 1
        assert 2.0 ** 24 < np.prod(ext.astype(np.float64)) < 2.0 ** 31
        gc.close()
        rec, off, mem = check_against_oracle(c, cloud, leaf)
        assert rec.shape[0] > 1_000_000
        check_against_oracle(c, cloud, 1.0)
    finally:
        c.close()


def test_pcl_order_within_bound(ctx):
    cloud = synth.panel(200000, 6, density=16.0)
    gc = api.Cloud(ctx, cloud)
    rec, off, mem = gc.voxel_grid(0.5)
    prec, poff, pmem = ov.voxel_grid(cloud, 0.5, ov.PCL_ORDER)
    assert np.array_equal(off, poff)
    for a, b in zip(off[:-1], off[1:]):
        assert np.array_equal(mem[a:b], np.sort(pmem[a:b]))
    diff = np.abs(rec[:, :3].astype(np.float64) - prec[:, :3].astype(np.float64))
    assert np.all(diff <= pcl_order_bound(cloud, off, mem))
    assert np.array_equal(rec[:, 3:].view(np.uint32), prec[:, 3:].view(np.uint32))
    same = np.mean(np.all(rec[:, :3] == prec[:, :3], axis=1))
    print("rows bit-identical to PCL's order: %.4f" % same)
    assert same > 0.5


def test_overflow_is_refused_and_the_mirror_keeps_the_cloud(ctx, capsys):
    cloud, leaf = overflow_cloud()
    gc = api.Cloud(ctx, cloud)
    with pytest.raises(api.PPPError, match="Integer indices would overflow") as e:
        gc.voxel_grid(leaf)
    assert e.value.status == _lib.PPP_ERR_UNSUPPORTED
    gc.close()
    pg = reference_api.path_generater(cloud.copy(), 12.0, ctx=ctx)
    before = pg.cloud.copy()
    assert pg.voxel_down(leaf) is None
    assert "Integer indices would overflow" in capsys.readouterr().out
    assert np.array_equal(pg.cloud.view(np.uint32), before.view(np.uint32))
    # voxel coordinates past the int range: refused as well
    far = synth.to_pointxyzrgb(np.array([[3.0e9, 0, 0], [3.0e9, 1, 1]], np.float32))
    gc = api.Cloud(ctx, far)
    with pytest.raises(api.PPPError) as e:
        gc.voxel_grid(1.0)
    assert e.value.status == _lib.PPP_ERR_UNSUPPORTED
    gc.close()


@pytest.mark.parametrize("leaf", [0.0, -0.5, float("nan"), float("inf"), (1.0, 1.0, 0.0), 1e-45])
def test_invalid_leaf(ctx, leaf):
    gc = api.Cloud(ctx, synth.panel(1000, 7))
    with pytest.raises(api.PPPError) as e:
        gc.voxel_grid(leaf)
    assert e.value.status == _lib.PPP_ERR_INVALID
    gc.close()


def test_no_finite_point_and_narrow_records(ctx):
    gc = api.Cloud(ctx, synth.to_pointxyzrgb(np.full((7, 3), np.nan, np.float32)))
    rec, off, mem = gc.voxel_grid(1.0)
    assert rec.shape == (0, 8) and np.array_equal(off, [0]) and mem.shape == (0,)
    gc.close()
    cloud = np.ascontiguousarray(synth.panel(5000, 8)[:, :3])   # 12-byte records: x, y, z only
    gc = api.Cloud(ctx, cloud)
    rec, off, mem = gc.voxel_grid(1.0)
    gc.close()
    orec, ooff, omem = ov.voxel_grid(cloud, 1.0)
    assert rec.shape[1] == 3 and np.array_equal(off, ooff) and np.array_equal(rec, orec)


def test_dense_scan_flow(ctx):
    """A density-64 scan: estimate_normal() (radius 2.5) is refused by the radius-list limit; after voxel_down(0.5) it
    runs and its normals match the oracle's on the downsampled cloud."""
    metres = synth.to_pointxyzrgb(synth.panel_metres(100000, 9, density=64.0))
    pg = reference_api.path_generater(metres, 12.0, ctx=ctx)
    with pytest.raises(api.PPPError) as e:
        pg.estimate_normal()
    assert e.value.status == _lib.PPP_ERR_UNSUPPORTED
    source = pg.cloud.copy()
    off, mem = pg.voxel_down(0.5)
    orec, ooff, omem = ov.voxel_grid(source, 0.5)
    assert np.array_equal(pg.cloud.view(np.uint32), orec.view(np.uint32))
    assert np.array_equal(off, ooff) and np.array_equal(mem, omem)
    assert pg.cloud.shape[0] < source.shape[0] // 4
    g = pg.estimate_normal()
    o, _ = po.OracleCloud(pg.cloud).normals(radius=2.5)
    gn = np.concatenate([g[:, 0:3], g[:, 4:5]], axis=1)
    ok = ~np.isnan(o[:, 0])
    assert ok.mean() > 0.99
    assert np.array_equal(np.isnan(gn[:, 0]), ~ok)
    assert np.abs(gn[ok] - o[ok]).max() <= 1e-5


CPP_PROGRAM = r"""
#include <cstdio>
#include "ppp_adapter.h"
// path_generater::voxel_down on a PCD file, then normals on the result; writes the cloud's records
int main(int argc, char** argv) {
  path_generater pg(argv[1], 12.0);
  const size_t before = pg.cloud->points.size();
  pg.voxel_down((float)atof(argv[3]), (float)atof(argv[4]), (float)atof(argv[5]));
  pg.estimate_normal();   // the device copy is rebuilt from the new cloud
  FILE* f = fopen(argv[2], "wb");
  fwrite(pg.cloud->points.data(), sizeof(PointType), pg.cloud->points.size(), f);
  fclose(f);
  printf("%zu -> %zu\n", before, pg.cloud->points.size());
  return 0;
}
"""


def test_cpp_adapter_voxel_down(tmp_path):
    src = tmp_path / "voxel_main.cpp"
    src.write_text(CPP_PROGRAM)
    exe = str(tmp_path / "voxel_main")
    host = os.path.join(ROOT, "polishpathplanning_b200", "host")
    libdir = os.path.join(ROOT, "polishpathplanning_b200")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", host, "-o", exe, str(src), "-L", libdir,
                           "-lppp_gpu", "-Wl,-rpath," + libdir])
    metres = synth.to_pointxyzrgb(synth.panel_metres(30000, 10, density=4.0))
    metres[:, 4] = np.arange(30000, dtype=np.uint32).view(np.float32)   # distinct colours to average
    pcd = str(tmp_path / "workpiece.pcd")
    synth.write_pcd(pcd, metres)
    scaled = synth.read_pcd(pcd)
    synth.reference_ctor_scale(scaled)   # the constructor's x, y, z *= 1000 and r = g = b = 255
    for leaf, kept in [((0.5, 0.5, 0.5), False), ((1.0, 2.0, 0.25), False), ((1e-4, 1e-4, 1e-4), True)]:
        out = str(tmp_path / "out.bin")
        r = subprocess.run([exe, pcd, out] + [str(v) for v in leaf], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        got = np.fromfile(out, np.float32).reshape(-1, 8)
        if kept:
            assert "Integer indices would overflow" in r.stderr
            assert np.array_equal(got[:, :5].view(np.uint32), scaled[:, :5].view(np.uint32))
        else:
            orec, _, _ = ov.voxel_grid(scaled, leaf)
            assert np.array_equal(got[:, :5].view(np.uint32), orec[:, :5].view(np.uint32))


BOUNDS_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from oracle_voxel import ppp_oracle_voxel as ov
from polishpathplanning_b200 import api, synth
from voxel_cases import edge_cases
ctx = api.Context(0)
cases = edge_cases() + [("panel", synth.panel(300000, 3, density=16.0), 0.1)]
for name, cloud, leaf in cases:
    c = api.Cloud(ctx, cloud)
    rec, off, mem = c.voxel_grid(leaf)
    c.close()
    orec, ooff, omem = ov.voxel_grid(cloud, leaf)
    assert np.array_equal(off, ooff) and np.array_equal(mem, omem) and np.array_equal(rec.view(np.uint32), orec.view(np.uint32)), name
ctx.close()
print("bounds-checked voxel grid ok")
"""


def test_bounds_checked_build():
    if not os.path.exists(CHECK_LIB):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    env = dict(os.environ, PPP_GPU_LIB=CHECK_LIB)
    r = subprocess.run([sys.executable, "-c", BOUNDS_SCRIPT, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "PPP_DEV_ASSERT" not in r.stdout + r.stderr
    assert "bounds-checked voxel grid ok" in r.stdout
