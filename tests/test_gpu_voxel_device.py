"""ppp_dev_voxel_grid (the reference's voxel_down() with the rows left in device memory): whole records -- x, y, z, the
pad float, the averaged rgba word, zeros -- bit-identical to the CPU oracle's stable order and to Cloud.voxel_grid at
every stride; buffers sized as the header asks and nothing written past them; PCL's refusals with rows_dev untouched;
and the device flows smooth -> voxel grid -> normals -> contours equal to the host flows bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ppp_oracle as po
from oracle_voxel import ppp_oracle_voxel as ov
from polishpathplanning_b200 import _lib, api, synth
from voxel_cases import _recs, edge_cases, overflow_cloud

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECK_LIB = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
SENT = -559038737   # 0xDEADBEEF: a word no call may leave behind where it writes, nor overwrite where it must not
GUARD = 64


def _finite(cloud):
    return int(np.isfinite(cloud[:, :3]).all(axis=1).sum())


def dev_voxel(ctx, cloud, leaf):
    """Attaches `cloud` (n, sf) from device records and runs dev_voxel_grid into sentinel-filled buffers of exactly the
    sizes the header asks for (n records, finite points + 1 offsets, one member per finite point), each followed by a
    guard that must stay untouched.  Returns (records, row_offsets, members) as numpy arrays."""
    import torch
    n, sf = cloud.shape
    nf = _finite(cloud)
    src = torch.from_numpy(np.ascontiguousarray(cloud, np.float32)).to("cuda:0")
    rows = torch.full((n + GUARD, sf), SENT, dtype=torch.int32, device="cuda:0")
    off = torch.full((nf + 1 + GUARD,), SENT, dtype=torch.int64, device="cuda:0")
    mem = torch.full((nf + GUARD,), SENT, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    gc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=n, stride_bytes=sf * 4)
    m = gc.dev_voxel_grid(leaf, rows.data_ptr(), sf * 4, offsets_ptr=off.data_ptr(), members_ptr=mem.data_ptr())
    ctx.sync()
    gc.close()
    r, o, k = rows.cpu().numpy(), off.cpu().numpy(), mem.cpu().numpy()
    assert np.all(r[m:] == SENT) and np.all(o[m + 1:] == SENT) and np.all(k[nf:] == SENT)
    return r[:m].view(np.float32), o[:m + 1], k[:nf]


def check_against_oracle(ctx, cloud, leaf):
    rec, off, mem = dev_voxel(ctx, cloud, leaf)
    orec, ooff, omem = ov.voxel_grid(cloud, leaf, ov.STABLE_ORDER)
    assert np.array_equal(off, ooff)
    assert np.array_equal(mem, omem)
    assert np.array_equal(rec.view(np.uint32), orec.view(np.uint32))   # whole records
    return rec


def _coloured(cloud, seed):
    out = np.ascontiguousarray(cloud, np.float32).copy()
    out[:, 4] = np.random.default_rng(seed).integers(0, 2 ** 32, out.shape[0], dtype=np.uint64).astype(np.uint32).view(np.float32)
    return out


SHAPES = [
    ("panel", lambda: synth.panel(60000, 1), [0.5, 1.0, 2.5]),
    ("panel_dense", lambda: synth.panel(60000, 2, density=16.0), [0.5, (0.25, 0.5, 1.0)]),
    ("cylinder", lambda: synth.cylinder(60000, 3), [0.5, 2.0]),
    ("box_with_walls", lambda: synth.box_with_walls(60000, 4), [1.0, (2.0, 1.0, 0.5)]),
]


@pytest.mark.parametrize("name,make,leaves", SHAPES, ids=[s[0] for s in SHAPES])
def test_records_against_oracle_shapes(ctx, name, make, leaves):
    cloud = _coloured(make(), 20)
    for leaf in leaves:
        check_against_oracle(ctx, cloud, leaf)


@pytest.mark.parametrize("name,cloud,leaf", edge_cases(), ids=[c[0] for c in edge_cases()])
def test_records_against_oracle_edge_cases(ctx, name, cloud, leaf):
    check_against_oracle(ctx, cloud, leaf)


def test_crowded_voxel_colour_sums_past_2_24(ctx):
    """One voxel of 100,000 members with bytes of 128..255: its channel sums pass 2^24, where float32 partial sums round
    and only the member order the oracle and the device share gives the same colour."""
    rng = np.random.default_rng(21)
    xyz = np.concatenate([rng.uniform(100.0, 100.9, (100_000, 3)), rng.uniform(103.0, 105.0, (3000, 3))])
    cloud = _recs(xyz, 22)
    cloud[:, 4] = (rng.integers(128, 256, (cloud.shape[0], 4)).astype(np.uint8)).view(np.uint32).reshape(-1).view(np.float32)
    rec = check_against_oracle(ctx, cloud, 1.0)
    bytes_ = np.ascontiguousarray(cloud[:100_000, 4]).view(np.uint32).view(np.uint8).reshape(-1, 4).astype(np.int64)
    assert bytes_.sum(axis=0).min() > 2 ** 24
    assert rec.shape[0] > 1


STRIDES = [12, 16, 20, 32, 48]


@pytest.mark.parametrize("stride", STRIDES)
def test_strides_equal_host_voxel_grid(ctx, stride):
    """Whole records at every stride equal Cloud.voxel_grid on the same records (host centroids and host colour
    averaging); fields other than x, y, z and rgba in the source records are not copied."""
    sf = stride // 4
    base = _coloured(synth.panel(40000, 23, density=16.0), 24)
    cloud = np.random.default_rng(25).uniform(-1e3, 1e3, (base.shape[0], sf)).astype(np.float32)
    cloud[:, :min(sf, 5)] = base[:, :min(sf, 5)]
    cloud[7, 2] = np.nan
    hc = api.Cloud(ctx, cloud)
    href, hoff, hmem = hc.voxel_grid(0.5)
    hc.close()
    rec, off, mem = dev_voxel(ctx, cloud, 0.5)
    assert np.array_equal(off, hoff) and np.array_equal(mem, hmem)
    assert np.array_equal(rec.view(np.uint32), href.view(np.uint32))


def test_unaligned_rows_and_default_scratch(ctx):
    """rows_dev 4 bytes past a 16-byte boundary (no 16-byte stores) and the library's own offsets and members."""
    import torch
    cloud = _coloured(synth.panel(30000, 26, density=16.0), 27)
    href, _, _ = api.Cloud(ctx, cloud).voxel_grid(0.5)
    src = torch.from_numpy(cloud).to("cuda:0")
    rows = torch.full((cloud.shape[0] * 8 + 1,), SENT, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    gc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=cloud.shape[0], stride_bytes=32)
    m = gc.dev_voxel_grid(0.5, rows.data_ptr() + 4, 32)
    ctx.sync()
    r = rows.cpu().numpy()
    assert r[0] == SENT and np.all(r[1 + m * 8:] == SENT)
    assert np.array_equal(r[1:1 + m * 8].reshape(m, 8).view(np.uint32), href.view(np.uint32))
    gc.close()


def test_null_source_is_invalid_from_20_bytes(ctx):
    import torch
    cloud = _coloured(synth.panel(5000, 28), 29)
    for sf in (5, 8):
        recs = np.ascontiguousarray(cloud[:, :sf])
        hc = api.Cloud(ctx, recs)   # a host-uploaded cloud: no device records to default to
        rows = torch.full((recs.shape[0], sf), SENT, dtype=torch.int32, device="cuda:0")
        with pytest.raises(api.PPPError) as e:
            hc.dev_voxel_grid(1.0, rows.data_ptr(), sf * 4)
        assert e.value.status == _lib.PPP_ERR_INVALID
        assert (rows == SENT).all().item()
        hc.close()
    hc = api.Cloud(ctx, np.ascontiguousarray(cloud[:, :4]))   # below 20 bytes the source is not needed
    rows = torch.empty((cloud.shape[0], 4), dtype=torch.float32, device="cuda:0")
    assert hc.dev_voxel_grid(1.0, rows.data_ptr(), 16) > 0
    hc.close()


def test_large_cloud_every_pass(ctx):
    """2.5M points at leaf 0.2: keys of more than 24 bits, so all four radix passes run."""
    cloud = _coloured(synth.panel(2_500_000, 5, density=16.0), 30)
    cloud[::1000, 0] = np.nan   # members hold fewer entries than the cloud has points
    fin = np.isfinite(cloud[:, :3]).all(axis=1)
    inv = np.float32(1.0) / np.float32(0.2)
    ext = np.floor(cloud[fin, :3].max(axis=0) * inv) - np.floor(cloud[fin, :3].min(axis=0) * inv) + 1
    assert 2.0 ** 24 < np.prod(ext.astype(np.float64)) < 2.0 ** 31
    rec = check_against_oracle(ctx, cloud, 0.2)
    assert rec.shape[0] > 1_000_000


def _raw_call(ctx, gc, leaf, rows, stride, off=None, mem=None, src=None):
    lf = np.broadcast_to(np.asarray(leaf, np.float32), (3,)).copy()
    m = C.c_int64(12345)
    st = ctx.lib.ppp_dev_voxel_grid(gc._h, lf.ctypes.data_as(_lib._f32p), src, stride, rows, off, mem, C.byref(m))
    return st, m.value


def test_refusals_overflow_invalid_leaf_no_finite_point(ctx):
    import torch
    cloud, leaf = overflow_cloud()
    src = torch.from_numpy(cloud).to("cuda:0")
    rows = torch.full((cloud.shape[0], 8), SENT, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    gc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=cloud.shape[0], stride_bytes=32)
    st, m = _raw_call(ctx, gc, leaf, rows.data_ptr(), 32, src=src.data_ptr())
    assert st == _lib.PPP_ERR_UNSUPPORTED and m == 0
    assert "Leaf size is too small for the input dataset. Integer indices would overflow." in ctx.lib.ppp_last_error().decode()
    for bad in [0.0, -0.5, float("nan"), float("inf"), (1.0, 1.0, 0.0), 1e-45]:
        st, m = _raw_call(ctx, gc, bad, rows.data_ptr(), 32, src=src.data_ptr())
        assert st == _lib.PPP_ERR_INVALID and m == 0
    ctx.sync()
    assert (rows == SENT).all().item()
    gc.close()
    # voxel coordinates past the int range
    far = synth.to_pointxyzrgb(np.array([[3.0e9, 0, 0], [3.0e9, 1, 1]], np.float32))
    src = torch.from_numpy(far).to("cuda:0")
    torch.cuda.synchronize()
    gc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=2, stride_bytes=32)
    st, m = _raw_call(ctx, gc, 1.0, rows.data_ptr(), 32, src=src.data_ptr())
    assert st == _lib.PPP_ERR_UNSUPPORTED and m == 0
    assert (rows == SENT).all().item()
    gc.close()
    # no finite point: no rows, row_offsets_dev[0] = 0
    nan = synth.to_pointxyzrgb(np.full((7, 3), np.nan, np.float32))
    src = torch.from_numpy(nan).to("cuda:0")
    off = torch.full((8,), SENT, dtype=torch.int64, device="cuda:0")
    torch.cuda.synchronize()
    gc = api.Cloud(ctx, device_ptr=src.data_ptr(), n=7, stride_bytes=32)
    assert gc.dev_voxel_grid(1.0, rows.data_ptr(), 32, offsets_ptr=off.data_ptr()) == 0
    ctx.sync()
    o = off.cpu().numpy()
    assert o[0] == 0 and np.all(o[1:] == SENT) and (rows == SENT).all().item()
    gc.close()


def _downsample_both(ctx, cloud, leaf):
    """(device cloud attached from dev_voxel_grid's rows, its rows tensor, host cloud uploaded from Cloud.voxel_grid's
    records, those records)."""
    import torch
    src = torch.from_numpy(cloud).to("cuda:0")
    torch.cuda.synchronize()
    gd = api.Cloud(ctx, device_ptr=src.data_ptr(), n=cloud.shape[0], stride_bytes=32)
    rows = torch.empty((cloud.shape[0], 8), dtype=torch.float32, device="cuda:0")
    m = gd.dev_voxel_grid(leaf, rows.data_ptr(), 32)
    dc = api.Cloud(ctx, device_ptr=rows.data_ptr(), n=m, stride_bytes=32)
    hrec, _, _ = gd.voxel_grid(leaf)
    hc = api.Cloud(ctx, hrec)
    ctx.sync()
    assert np.array_equal(rows[:m].cpu().numpy().view(np.uint32), hrec.view(np.uint32))
    return dc, (src, rows, gd), hc, hrec


def test_dense_scan_device_flow(ctx):
    """A density-64 scan: radius normals are refused; dev_voxel_grid(0.5) + attach, then normals and both contour
    modes equal the host flow (Cloud.voxel_grid -> upload) bit for bit, and the normals are within 1e-5 of the oracle."""
    cloud = _coloured(synth.panel(100000, 9, density=64.0), 31)
    full = api.Cloud(ctx, cloud)
    with pytest.raises(api.PPPError) as e:
        full.normals_radius(2.5)
    assert e.value.status == _lib.PPP_ERR_UNSUPPORTED
    full.close()
    dc, keep, hc, hrec = _downsample_both(ctx, cloud, 0.5)
    assert hrec.shape[0] < cloud.shape[0] // 4
    gn = dc.normals_radius(2.5)
    assert np.array_equal(gn.view(np.uint32), hc.normals_radius(2.5).view(np.uint32))
    o, _ = po.OracleCloud(hrec).normals(radius=2.5)
    g = np.concatenate([gn[:, 0:3], gn[:, 4:5]], axis=1)
    ok = ~np.isnan(o[:, 0])
    assert ok.mean() > 0.99
    assert np.array_equal(np.isnan(g[:, 0]), ~ok)
    assert np.abs(g[ok] - o[ok]).max() <= 1e-5
    mn, mx = dc.bbox()
    planes = po.planes("gen2_contact", mn[0], mx[0], 15.0)
    for mode in ("A", "B"):
        a = dc.slice_contours(planes, mode)
        b = hc.slice_contours(planes, mode)
        assert a[0][-1] > 0
        for x, y in zip(a, b):   # node offsets, y, x, z
            assert np.array_equal(x.view(np.uint64), y.view(np.uint64))
    dc.close()
    hc.close()


def test_prefilter_chain_smooth_voxel_normals(ctx):
    """dev_mls_smooth + dev_mls_compact -> attach -> dev_voxel_grid -> attach -> normals equals the host chain
    (mls_smooth -> upload -> voxel_grid -> upload -> normals) bit for bit."""
    import torch
    R, ORDER = 15.0, 3
    cloud = _coloured(synth.panel(30000, 48, noise_sigma=0.05), 32)
    cloud[5, 1] = np.nan
    n = cloud.shape[0]
    src = torch.from_numpy(cloud).to("cuda:0")
    recs = torch.empty((n, 8), dtype=torch.float32, device="cuda:0")
    pts = torch.empty_like(src)
    idx = torch.empty(n, dtype=torch.int32, device="cuda:0")
    rows = torch.empty_like(src)
    torch.cuda.synchronize()
    g0 = api.Cloud(ctx, device_ptr=src.data_ptr(), n=n, stride_bytes=32)
    g0.dev_mls_smooth(R, ORDER, recs.data_ptr())
    ms = ctx.dev_mls_compact(recs.data_ptr(), n, src.data_ptr(), 32, 0, 0, pts.data_ptr(), 32, None, idx.data_ptr(), n)
    g1 = api.Cloud(ctx, device_ptr=pts.data_ptr(), n=ms, stride_bytes=32)
    mv = g1.dev_voxel_grid(2.0, rows.data_ptr(), 32)
    g2 = api.Cloud(ctx, device_ptr=rows.data_ptr(), n=mv, stride_bytes=32)
    dn = g2.normals_knn(16)

    hs, _, _ = api.Cloud(ctx, cloud).mls_smooth(R, ORDER)
    hv, _, _ = api.Cloud(ctx, hs).voxel_grid(2.0)
    hn = api.Cloud(ctx, hv).normals_knn(16)
    ctx.sync()
    assert np.array_equal(pts[:ms].cpu().numpy().view(np.uint32), hs.view(np.uint32))
    assert np.array_equal(rows[:mv].cpu().numpy().view(np.uint32), hv.view(np.uint32))
    assert mv < ms
    assert np.array_equal(dn.view(np.uint32), hn.view(np.uint32))
    for c in (g0, g1, g2):
        c.close()


def test_bounds_checked_build():
    """The oracle comparisons and the refusals above, with the library's device-side index assertions compiled in."""
    if not os.path.exists(CHECK_LIB):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    env = dict(os.environ, PPP_GPU_LIB=CHECK_LIB)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "records_against_oracle or refusals"], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=900)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT" not in out, out[-3000:]
    assert r.returncode == 0 and " passed" in r.stdout and "skipped" not in r.stdout, out[-3000:]
