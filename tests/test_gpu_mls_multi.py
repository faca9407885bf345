"""MLS smooth() sharded over the multi-GPU exchange (ppp_dev_mls_smooth + ppp_dev_mls_compact, parallel.mls_smooth_sharded)
against one GPU's ppp_mls_smooth of the whole cloud and against the CPU oracle.  `world` ranks live in this process on
one GPU (Exchange.connect_local), so the exchange kernels, flags, waits and home deliveries run as between GPUs.

Contract: the rows (src_index and every field but x, y, z) are identical; x, y, z within 2 float32 ulps with >= 99 %
bit-identical; normals and curvature within 1e-5 (a slab builds its own grid, so the double sums run in another order)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from exchange_model import exchange_model
from oracle_mls import ppp_oracle_mls as pom
from polishpathplanning_b200 import api, parallel, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R, ORDER = 15.0, 3


def _x_abs_max(cloud):
    fin = np.isfinite(cloud[:, :3]).all(axis=1)
    return float(np.abs(cloud[fin, 0]).max()) if fin.any() else 0.0


class Ranks:
    """world ranks on GPU 0, one Context + Exchange each (32-byte home records)."""

    def __init__(self, world, n, stride_floats=8, normal_stride_bytes=32):
        import torch
        self.world, self.n, self.sf = world, n, stride_floats
        self.starts = parallel.index_ranges(n, world)
        self.ctxs = [api.Context(0) for _ in range(world)]
        self.exs = [parallel.Exchange(self.ctxs[r], r, world, self.starts, n + 1024, 8, 1024, normal_stride_bytes)
                    for r in range(world)]
        parallel.Exchange.connect_local(self.exs)
        self.chunks = [torch.empty((int(self.starts[r + 1] - self.starts[r]), stride_floats), dtype=torch.float32,
                                   device="cuda:0") for r in range(world)]

    def load(self, cloud):
        import torch
        for r in range(self.world):
            self.chunks[r].copy_(torch.from_numpy(np.ascontiguousarray(cloud[self.starts[r]:self.starts[r + 1]])))
        torch.cuda.synchronize()

    def smooth(self, cloud, halo=None, radius=R, order=ORDER):
        """One sharded step into one pinned host buffer; returns (points, src_index, normals) as Cloud.mls_smooth."""
        self.load(cloud)
        if halo is None:
            halo = parallel.mls_halo(radius, _x_abs_max(cloud))
        pts = self.ctxs[0].pinned_empty((self.n, self.sf), np.float32)
        src = self.ctxs[0].pinned_empty((self.n,), np.int32)
        nrm = self.ctxs[0].pinned_empty((self.n, 4), np.float32)
        pts.fill(np.nan)
        out = (pts.ctypes.data, nrm.ctypes.data, src.ctypes.data, self.n, True)
        counts, bases = parallel.mls_smooth_sharded(self.exs, [c.data_ptr() for c in self.chunks], self.sf * 4, radius, order,
                                                    halo, [out] * self.world)
        for c in self.ctxs:
            c.sync()
        for ex in self.exs:
            ex.check()
        assert list(bases) == list(np.concatenate([[0], np.cumsum(counts)[:-1]]))
        return tuple(v.copy() for v in parallel.mls_rows(pts, src, nrm, counts))

    def home_records(self):
        return np.concatenate([ex.read_home_normals() for ex in self.exs], axis=0)

    def close(self):
        for ex in self.exs:
            ex.close()
        for c in self.ctxs:
            c.close()


def single_gpu(cloud, radius=R, order=ORDER):
    ctx = api.Context(0)
    gc = api.Cloud(ctx, np.ascontiguousarray(cloud, np.float32))
    res = gc.mls_smooth(radius, order, normals=True)
    gc.close()
    ctx.close()
    return res


def check_contract(got, ref):
    """Returns the fraction of rows whose x, y, z are bit-identical."""
    pts, src, nrm = got
    rpts, rsrc, rnrm = ref
    assert np.array_equal(src, rsrc)
    assert np.array_equal(pts[:, 3:].view(np.uint32), rpts[:, 3:].view(np.uint32))   # rgb and padding
    if src.shape[0] == 0:
        return 1.0
    a, b = pts[:, 0:3].astype(np.float64), rpts[:, 0:3].astype(np.float64)
    ulps = np.abs(a - b) / np.spacing(np.maximum(np.abs(pts[:, 0:3]), np.abs(rpts[:, 0:3])))
    assert ulps.max() <= 2.0, ulps.max()
    same = float(np.mean(np.all(pts[:, 0:3] == rpts[:, 0:3], axis=1)))
    assert same >= 0.99, same
    assert np.abs(nrm - rnrm).max() <= 1e-5
    return same


def check_oracle(got, cloud, radius=R, order=ORDER, sample=4000):
    """Sampled rows against the CPU oracle with the bars of tests/test_gpu_mls.py."""
    pts, src, nrm = got
    oxyz, onrm, osrc, _ = pom.mls_smooth(cloud, radius, order)
    assert np.array_equal(src, osrc)
    rows = np.random.default_rng(0).choice(src.shape[0], min(sample, src.shape[0]), replace=False) if src.shape[0] else []
    a, b = pts[rows, 0:3].astype(np.float64), oxyz[rows].astype(np.float64)
    ulps = np.abs(a - b) / np.spacing(np.maximum(np.abs(pts[rows, 0:3]), np.abs(oxyz[rows])))
    assert ulps.max() <= 2.0
    assert np.abs(nrm[rows] - onrm[rows]).max() <= 1e-5


_CLOUDS = {
    "panel_d1": lambda: synth.panel(60000, seed=41, noise_sigma=0.05),             # ~700 neighbours
    "panel_d4": lambda: synth.panel(24000, seed=42, density=4.0, noise_sigma=0.05),  # ~2,800 neighbours
    "cylinder": lambda: synth.cylinder(40000, seed=43),                             # not a height field
}
_REF = {}


def _cloud_and_ref(name):
    if name not in _REF:
        cloud = _CLOUDS[name]()
        _REF[name] = (cloud, single_gpu(cloud))
    return _REF[name]


@pytest.mark.parametrize("name", sorted(_CLOUDS))
@pytest.mark.parametrize("world", [2, 3, 5, 8])
def test_ranks_on_one_gpu(world, name):
    cloud, ref = _cloud_and_ref(name)
    ranks = Ranks(world, cloud.shape[0])
    got = ranks.smooth(cloud)
    ranks.close()
    same = check_contract(got, ref)
    print("MLS_MULTI world=%d cloud=%s rows=%d bit_identical=%.6f" % (world, name, got[1].shape[0], same))
    if world == 3:
        check_oracle(got, cloud)


def _halo_edge_cloud():
    """Two ranks cut exactly at x = 11.25: the finite x span [-500.75, 523.25] (1024 mm, so bins are 1 mm wide and the
    bin arithmetic is exact) and as many finite points below the cut as above it, bin 511 not empty.  The probe
    groups sit 100 mm apart in y, the filler points 300 mm away from them."""
    cut = 11.25
    f = np.float32
    groups = []

    def group(y, xs, zs=None):
        # the first two points lie on the line y = const, z = 0 (their float32 distance is their x difference); the
        # others spread over y and sit 0.3 mm higher, so that every neighbour moves the fitted plane
        xs = np.asarray(xs, np.float64)
        zs = np.zeros_like(xs) if zs is None else np.asarray(zs, np.float64)
        ys = np.full_like(xs, y)
        ys[2:] += np.resize([0.7, -0.9, 1.3, -0.4], max(xs.shape[0] - 2, 0))
        zs[2:] += 0.3
        groups.append(np.stack([xs, ys, zs], 1))

    # 1. q on the cut (owned above), p owned below at a float32 distance prev(15) from it: p is q's neighbour and
    #    reaches the upper slab only through a halo of at least 15 - 0.75 ulp(15).
    group(0.0, [cut, -3.75 + 3 * 2.0 ** -22, cut + 0.5, cut + 1.0, cut + 1.5, cut + 2.0, cut + 2.5],
          [0, 0, 0.1, -0.1, 0.05, 0.0, -0.05])
    # 2. q just below the cut (owned below), p above at float32 distance prev(15)
    group(100.0, [np.nextafter(f(cut), f(-1)), 26.25 - 2.0 ** -19, cut - 0.5, cut - 1.0, cut - 1.5, cut - 2.0],
          [0, 0, 0.1, -0.1, 0.05, 0.0])
    # 3. points at cut +- h and one float ulp either side, with company on both sides of the cut
    xs = []
    for c in (f(cut + R), f(cut - R)):
        xs += [np.nextafter(c, f(-1e9)), c, np.nextafter(c, f(1e9))]
    group(200.0, xs + [cut - 1.0, cut + 1.0, cut - 7.0, cut + 7.0], np.linspace(-0.1, 0.1, len(xs) + 4))
    # 4. a point owned below whose only neighbours lie in the upper slab
    group(300.0, [cut - 0.25, cut + 0.25, cut + 0.5, cut + 0.75, cut + 1.0, cut + 1.25], [0, 0.01, -0.01, 0.02, 0, 0.01])
    # 5. clusters of 1 and 2 points (no rows) on either side of the cut
    group(400.0, [cut - 3.0])
    group(500.0, [cut + 3.0, cut + 3.5])
    probes = np.concatenate(groups, 0)
    below = int((probes[:, 0].astype(np.float32) < cut).sum())
    above = probes.shape[0] - below
    rng = np.random.default_rng(44)

    def filler(n, x0, x1):
        return np.stack([rng.uniform(x0, x1, n), rng.uniform(-400.0, -300.0, n), rng.normal(0, 0.05, n)], 1)

    lo = filler(5000 + above - below, -500.75, 10.25)
    hi = filler(5000, 11.25, 523.25)
    lo[0, 0], hi[0, 0] = -500.75, 523.25           # the global x range
    lo[1, 0] = 10.75                                # bin 511 is not empty: the cut is bin 512, x = 11.25
    pts = np.concatenate([lo[:2500], hi[:2500], probes, lo[2500:], hi[2500:]], 0).astype(np.float32)
    bad = np.array([[np.nan, 0, 0], [cut, np.inf, 0], [np.inf, 0, 0], [cut, 600.0, np.nan]], np.float32)
    pts = np.concatenate([pts[:3000], bad, pts[3000:]], 0)
    return synth.to_pointxyzrgb(pts, rgb=7), cut


def test_halo_edge():
    cloud, cut = _halo_edge_cloud()
    world = 2
    starts = parallel.index_ranges(cloud.shape[0], world)
    halo = parallel.mls_halo(R, _x_abs_max(cloud))
    _, info = exchange_model([cloud[starts[r]:starts[r + 1]] for r in range(world)], starts, halo)
    assert info["cuts"][1] == cut                     # the cut the probes were placed around
    ref = single_gpu(cloud)
    ranks = Ranks(world, cloud.shape[0])
    got = ranks.smooth(cloud, halo=halo)
    rec = ranks.home_records()
    ranks.close()
    check_contract(got, ref)
    # the probe q of group 1 has the lower-slab point as a neighbour: without it its row would move
    q = np.nonzero((cloud[:, 0] == np.float32(cut)) & (cloud[:, 1] == 0.0))[0][0]
    assert q in got[1]
    without_p = cloud[np.arange(cloud.shape[0]) != q + 1]     # group 1 is stored as q, p, ...
    assert cloud[q + 1, 0] == np.float32(-3.75 + 3 * 2.0 ** -22)
    moved = single_gpu(without_p)
    assert not np.array_equal(moved[0][moved[1] == q, 0:3], ref[0][ref[1] == q, 0:3])   # p matters to q's row
    # records of points without a row: flag 0 (fewer than 3 neighbours, non-finite)
    has_row = np.zeros(cloud.shape[0], bool)
    has_row[got[1]] = True
    assert np.array_equal(rec[:, 3] == 1.0, has_row) and np.all(rec[~has_row, 3] == 0.0)
    assert not has_row[~np.isfinite(cloud[:, :3]).all(axis=1)].any()


def test_two_steps_through_one_exchange():
    n = 40000
    a = synth.panel(n, seed=45, noise_sigma=0.05)
    b = synth.panel(n, seed=46, noise_sigma=0.05)
    a[n // 3, 0] = np.nan            # non-finite in step 1 only
    gone = 3 * n // 5                # finite in step 1, NaN in step 2; home rank 3, owner of the NaN point rank 0
    b[gone, 2] = np.nan
    b[n // 2:n // 2 + 10, 0] += 3000.0   # and step 2's x range differs
    ranks = Ranks(5, n)
    for cloud in (a, b):
        got = ranks.smooth(cloud)
        check_contract(got, single_gpu(cloud))
    rec = ranks.home_records()
    ranks.close()
    assert gone not in got[1] and rec[gone, 3] == 0.0 and a[gone, 2] == a[gone, 2]
    assert (n // 3) in got[1] and rec[n // 3, 3] == 1.0


def test_refusals():
    import torch
    cloud = synth.panel(20000, seed=47, noise_sigma=0.05)
    need = parallel.mls_halo(R, _x_abs_max(cloud))
    # a 16-byte exchange
    ranks = Ranks(2, cloud.shape[0], normal_stride_bytes=16)
    ranks.load(cloud)
    for p in range(4):
        for ex, ch in zip(ranks.exs, ranks.chunks):
            ex.phase(p, ch.data_ptr(), ch.shape[0], 32, need)
    for ex in ranks.exs:
        _, c = ex.finish_attach(to_rank0=False)
        with pytest.raises(api.PPPError) as e:
            c.dev_mls_smooth(R, ORDER)
        assert e.value.status == api._lib.PPP_ERR_INVALID
        c.close()
    ranks.close()
    # a halo narrower than the rule; the rule's own halo is accepted
    ranks = Ranks(2, cloud.shape[0])
    ranks.load(cloud)
    for halo, ok in ((np.nextafter(need, 0.0), False), (need, True)):
        for p in range(4):
            for ex, ch in zip(ranks.exs, ranks.chunks):
                ex.phase(p, ch.data_ptr(), ch.shape[0], 32, halo)
        clouds = [ex.finish_attach(to_rank0=False)[1] for ex in ranks.exs]
        for c in clouds:
            if ok:
                c.dev_mls_smooth(R, ORDER)
            else:
                with pytest.raises(api.PPPError) as e:
                    c.dev_mls_smooth(R, ORDER)
                assert e.value.status == api._lib.PPP_ERR_INVALID
        # invalid order or radius
        for radius, order in ((R, -1), (R, 4), (0.0, 3), (float("nan"), 3), (2e19, 3)):
            with pytest.raises(api.PPPError) as e:
                clouds[0].dev_mls_smooth(radius, order)
            assert e.value.status == api._lib.PPP_ERR_INVALID
        for ex in ranks.exs:
            ex.results_signal(ex.NORMALS)
        for ex in ranks.exs:
            ex.results_wait(ex.NORMALS)
        for c in clouds:
            c.close()
    # one rank given a narrower halo than the others: the copies it sent are short, so EVERY rank refuses
    for p in range(4):
        for r, (ex, ch) in enumerate(zip(ranks.exs, ranks.chunks)):
            ex.phase(p, ch.data_ptr(), ch.shape[0], 32, need if r == 0 else np.nextafter(need, 0.0))
    clouds = [ex.finish_attach(to_rank0=False)[1] for ex in ranks.exs]
    for c in clouds:
        with pytest.raises(api.PPPError) as e:
            c.dev_mls_smooth(R, ORDER)
        assert e.value.status == api._lib.PPP_ERR_INVALID
    # a slab whose row map was cleared
    clouds[0].dev_set_normal_row_map(None)
    with pytest.raises(api.PPPError) as e:
        clouds[0].dev_mls_smooth(R, ORDER)
    assert e.value.status == api._lib.PPP_ERR_INVALID
    for c in clouds:
        c.close()
    # a correct step again, for the capacity check below
    for p in range(4):
        for ex, ch in zip(ranks.exs, ranks.chunks):
            ex.phase(p, ch.data_ptr(), ch.shape[0], 32, need)
    clouds = [ex.finish_attach(to_rank0=False)[1] for ex in ranks.exs]
    for c in clouds:
        c.dev_mls_smooth(R, ORDER)
    for ex in ranks.exs:
        ex.results_signal(ex.NORMALS)
    for ex in ranks.exs:
        ex.results_wait(ex.NORMALS)
    for c in clouds:
        c.close()
    # output capacity too small: PPP_ERR_CAPACITY, and the count is reported
    ex, ctx = ranks.exs[1], ranks.ctxs[1]
    rows = ctx.dev_mls_compact(ex.home_normals_ptr, ex.home_rows)
    assert rows > 0
    out = torch.empty((rows + 5, 8), dtype=torch.float32, device="cuda:0")
    src = torch.empty(rows + 5, dtype=torch.int32, device="cuda:0")
    import ctypes as C
    m = C.c_int64(0)
    st = ctx.lib.ppp_dev_mls_compact(ctx._h, ex.home_normals_ptr, ex.home_rows, None, 0, 0, 6, out.data_ptr(), 32, None,
                                     src.data_ptr(), rows + 5, C.byref(m))
    assert st == api._lib.PPP_ERR_CAPACITY and m.value == rows
    assert ctx.dev_mls_compact(ex.home_normals_ptr, ex.home_rows, row_base=5, points_ptr=out.data_ptr(),
                               src_index_ptr=src.data_ptr(), cap_rows=rows + 5) == rows
    torch.cuda.synchronize()
    assert np.array_equal(src[5:].cpu().numpy(), np.nonzero(ranks.home_records()[ranks.starts[1]:, 3] == 1.0)[0])
    ranks.close()
    # the plain-cloud form wants a 32-byte record stride and a buffer
    gctx = api.Context(0)
    gc = api.Cloud(gctx, cloud)
    recs = torch.empty((cloud.shape[0], 8), dtype=torch.float32, device="cuda:0")
    for stride, ptr in ((16, recs.data_ptr()), (32, None)):
        with pytest.raises(api.PPPError) as e:
            gc.dev_mls_smooth(R, ORDER, ptr, stride)
        assert e.value.status == api._lib.PPP_ERR_INVALID
    gc.close()
    gctx.close()


def test_plain_cloud_records_equal_mls_smooth():
    """ppp_dev_mls_smooth on one GPU + ppp_dev_mls_compact = ppp_mls_smooth, bit for bit."""
    import torch
    cloud = synth.panel(30000, seed=48, noise_sigma=0.05)
    cloud[5, 1] = np.nan
    ctx = api.Context(0)
    gc = api.Cloud(ctx, cloud)
    ref = gc.mls_smooth(R, ORDER, normals=True)
    recs = torch.full((cloud.shape[0], 8), 7.0, dtype=torch.float32, device="cuda:0")
    src_dev = torch.from_numpy(cloud).to("cuda:0")
    gc.dev_mls_smooth(R, ORDER, recs.data_ptr())
    pts = torch.empty_like(src_dev)
    nrm = torch.empty((cloud.shape[0], 4), dtype=torch.float32, device="cuda:0")
    idx = torch.empty(cloud.shape[0], dtype=torch.int32, device="cuda:0")
    m = ctx.dev_mls_compact(recs.data_ptr(), cloud.shape[0], src_dev.data_ptr(), 32, 0, 0, pts.data_ptr(), 32,
                            nrm.data_ptr(), idx.data_ptr(), cloud.shape[0])
    torch.cuda.synchronize()
    assert m == ref[1].shape[0]
    assert np.array_equal(pts[:m].cpu().numpy().view(np.uint32), ref[0].view(np.uint32))
    assert np.array_equal(idx[:m].cpu().numpy(), ref[1])
    assert np.array_equal(nrm[:m].cpu().numpy().view(np.uint32), ref[2].view(np.uint32))
    r = recs.cpu().numpy()
    assert r[5, 3] == 0.0 and np.isnan(r[5, [0, 1, 2, 4, 5, 6, 7]]).all()
    gc.close()
    ctx.close()


def test_across_processes():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tools", "mls_multi.py"),
                        "--check", "--sizes", "200000", "--steps", "2", "--warmup", "1", "--out", ""],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("check=True") == 2, r.stdout[-2000:]


def test_bounds_checked_library():
    check_lib = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
    if not os.path.exists(check_lib):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "from test_gpu_mls_multi import Ranks\n"
            "from polishpathplanning_b200 import synth\n"
            "for world, cloud in ((3, synth.panel(12000, 1, noise_sigma=0.05)), (2, synth.cylinder(8000, 2))):\n"
            "    rk = Ranks(world, cloud.shape[0]); rk.smooth(cloud); rk.close()\n"
            "print('done')\n" % (ROOT, os.path.join(ROOT, "tests")))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PPP_GPU_LIB=check_lib), capture_output=True,
                       text=True, timeout=600)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT failed" not in out, out[-2000:]
    assert r.returncode == 0 and "done" in r.stdout, out[-2000:]
