"""The device API (ppp_dev_*) as bench.py's headline step and the multi-GPU sharding call it: records already in device
memory, results left in device buffers, query sub-ranges in sorted order, row maps, record strides, caller-owned
contour buffers, and the refusal of ranges and buffers the kernels cannot serve.

Every output buffer starts filled with a sentinel no kernel writes (a NaN with a payload of its own for floats), and
results are compared bit for bit, so that a word written where it should not be and a word left unwritten both show.
The CPU oracle is the reference for what is computed (ids and d2 bit-exact, contours bit-exact, normals within
NORMAL_TOL); where only the plumbing differs (ranges, maps, strides, buffers) the reference is the same library's
full-range or host-API result, and the answer must be identical.

The library enqueues on its own stream: torch.cuda.synchronize() before a call that reads what torch wrote, ctx.sync()
before torch reads what the library wrote."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from oracle import ppp_oracle as po
from polishpathplanning_b200 import api, synth
from test_gpu_parity import NORMAL_TOL, _cmp_normals
from test_gpu_search_routes import three_densities

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENT_F = 0x7FBADBAD              # float words: a NaN whose payload no kernel writes
SENT_I = 0x5A5A5A5A              # int32 words
SENT_L = 0x5A5A5A5A5A5A5A5A      # int64 / double words
R = 2.5                          # the reference's normal radius


def _with_bad_rows(cloud, seed, count=40):
    """NaN / inf coordinates in `count` rows spread over the cloud (first and last row included)."""
    c = cloud.copy()
    rng = np.random.default_rng(seed)
    rows = np.concatenate([[0, c.shape[0] - 1], rng.choice(np.arange(1, c.shape[0] - 1), count - 2, replace=False)])
    for j, r in enumerate(rows):
        c[r, j % 3] = (np.nan, np.inf, -np.inf)[j % 3]
    return c


class Case:
    """A cloud and its oracle; oracle results are computed once per session."""

    def __init__(self, cloud):
        self.cloud = np.ascontiguousarray(cloud, np.float32)
        self.n = self.cloud.shape[0]
        self.finite = np.isfinite(self.cloud[:, :3]).all(axis=1)
        self.nf = int(self.finite.sum())
        self.oc = po.OracleCloud(self.cloud)
        self._memo = {}

    def memo(self, key, fn):
        if key not in self._memo:
            self._memo[key] = fn()
        return self._memo[key]

    def knn(self, k):
        return self.memo(("knn", k), lambda: self.oc.knn(k))

    def normals(self, k=None, radius=None):
        return self.memo(("normals", k, radius), lambda: self.oc.normals(k=k, radius=radius)[0])

    def planes(self, S):
        x = self.cloud[self.finite, 0]
        return bench.make_planes(x.min(), x.max(), S)


_CASES = {}
_MAKERS = {
    "cfg2": lambda: synth.panel(bench.make_cfg("cfg2", 1)["n_total"], seed=0),    # bench.py's cloud
    "box": lambda: synth.box_with_walls(300000, seed=3),                            # multi-projection index
    "nan_panel": lambda: _with_bad_rows(synth.panel(40000, seed=5), 6),
    "cylinder": lambda: synth.cylinder(100000, seed=4),
    "small_box": lambda: synth.box_with_walls(60000, seed=8),
    "three": three_densities,                                                       # all three radius-normal stages
    "dense": lambda: _with_bad_rows(synth.panel(60000, seed=9, density=8.0), 10),   # expect > 24: generic radius kernel
}


def _case(name):
    if name not in _CASES:
        _CASES[name] = Case(_MAKERS[name]())
    return _CASES[name]


def _on_device(case):
    t = torch.from_numpy(case.cloud).cuda()
    torch.cuda.synchronize()
    return t


class Outs:
    """Sentinel-filled device outputs of one normal call: records of sf floats, optionally k ids and k d2 per row."""

    def __init__(self, n, sf=8, k=0, d2=True):
        self.normals = torch.full((n, sf), SENT_F, dtype=torch.int32, device="cuda")
        self.idx = torch.full((n, k), SENT_I, dtype=torch.int32, device="cuda") if k else None
        self.d2 = torch.full((n, k), SENT_F, dtype=torch.int32, device="cuda") if k and d2 else None
        self.sf = sf
        torch.cuda.synchronize()

    def knn(self, c, k, first=0, count=-1, **kw):
        c.dev_normals_knn(k, self.normals.data_ptr(), self.sf * 4, idx_ptr=self.idx.data_ptr() if self.idx is not None else None,
                          d2_ptr=self.d2.data_ptr() if self.d2 is not None else None, first=first, count=count, **kw)

    def radius(self, c, r, first=0, count=-1, **kw):
        c.dev_normals_radius(r, self.normals.data_ptr(), self.sf * 4, first=first, count=count, **kw)

    def read(self, ctx):
        ctx.sync()
        out = {"normals": self.normals.cpu().numpy()}
        if self.idx is not None:
            out["idx"] = self.idx.cpu().numpy()
        if self.d2 is not None:
            out["d2"] = self.d2.cpu().numpy()
        return out


def _sentinel(key):
    return SENT_I if key == "idx" else SENT_F


def _check_against_oracle(case, got, k=None, radius=None):
    """got: Outs.read() of a full-range call at stride 32."""
    g = got["normals"].view(np.float32)
    mx, _ = _cmp_normals(g, case.normals(k=k, radius=radius))
    assert mx <= NORMAL_TOL
    assert np.all(got["normals"][:, [3, 5, 6, 7]] == 0)   # pcl::Normal padding
    if "idx" in got:
        oi, od = case.knn(k)
        assert np.array_equal(got["idx"], oi)
        if "d2" in got:
            assert np.array_equal(got["d2"], od.view(np.int32))


def _profiled(ctx, fn):
    ctx.kernel_profile(True)
    try:
        ctx.kernel_profile_read()
        fn()
        return ctx.kernel_profile_read()
    finally:
        ctx.kernel_profile(False)


def _read_contours(ctx, res, S):
    off = ctx.download(res["node_offsets"], (S + 1,), np.int64)
    t = int(off[-1])
    return (off,) + tuple(ctx.download(res[a], (t,), np.float64) for a in ("y", "x", "z"))


def _same_contours(got, want):
    assert np.array_equal(got[0], want[0])
    for g, w in zip(got[1:], want[1:]):
        assert np.array_equal(g.view(np.uint64), w.view(np.uint64))


# ---------------------------------------------------------------------------------------------------------------------
# a. bench.py's step, cloud after cloud on one context
# ---------------------------------------------------------------------------------------------------------------------
SEQUENCE = [("cfg2", 16), ("box", 16), ("nan_panel", 32), ("cylinder", 64), ("cfg2", 16)]


def test_benchmark_step_over_a_sequence_of_clouds(ctx):
    """attach device records -> dev_normals_knn(k, normals, 32, idx) -> dev_slice_contours(planes, "B") with no
    synchronisation in between -> close, as bench.measure_single's dev_step does, on one context and one set of output
    tensors.  A cloud's self-resetting ingest and scan scratch must not leak into the next.  On the same records: radius
    normals and k = 100 (the generic search kernel), with ids and d2."""
    cfg = bench.make_cfg("cfg2", 1)
    S, n_max, k_max = cfg["S"], cfg["n_total"], 100
    raw = torch.empty((n_max, 8), dtype=torch.float32, device="cuda")
    normals = torch.empty((n_max + 64, 8), dtype=torch.int32, device="cuda")
    idx = torch.empty((n_max + 64) * k_max, dtype=torch.int32, device="cuda")
    d2 = torch.empty((n_max + 64) * k_max, dtype=torch.int32, device="cuda")
    seen = set()
    for name, k in SEQUENCE:
        case = _case(name)
        n = case.n
        planes = case.planes(S)
        raw[:n].copy_(torch.from_numpy(case.cloud))
        normals.fill_(SENT_F)
        idx.fill_(SENT_I)
        torch.cuda.synchronize()
        c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
        c.dev_normals_knn(k, normals.data_ptr(), 32, idx_ptr=idx.data_ptr())
        res = c.dev_slice_contours(planes, bench.PAIRING, bench.HALF_WIDTH, True)
        got_c = _read_contours(ctx, res, S)
        c.close()
        ctx.sync()
        nb = normals[:n + 64].cpu().numpy()
        ib = idx[:(n + 64) * k].cpu().numpy()
        assert np.all(nb[n:] == SENT_F) and np.all(ib[n * k:] == SENT_I), name   # nothing past the cloud's rows
        _check_against_oracle(case, {"normals": nb[:n], "idx": ib[:n * k].reshape(n, k)}, k=k)
        want_c = case.memo(("contours", S), lambda: case.oc.slice_contours(planes, bench.PAIRING, bench.HALF_WIDTH, True))
        _same_contours(got_c, want_c)
        assert res["total_nodes"] == int(want_c[0][-1])
        assert res["total_members"] == int(case.memo(("bands", S), lambda: case.oc.slice_bands(planes)[0][-1])), name
        if name in seen:
            continue
        seen.add(name)
        # the same records: radius normals, then k = 100 with ids and d2
        normals.fill_(SENT_F)
        idx.fill_(SENT_I)
        d2.fill_(SENT_F)
        torch.cuda.synchronize()
        c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
        c.dev_normals_radius(R, normals.data_ptr(), 32)
        ctx.sync()
        _check_against_oracle(case, {"normals": normals[:n].cpu().numpy()}, radius=R)
        c.dev_normals_knn(k_max, normals.data_ptr(), 32, idx_ptr=idx.data_ptr(), d2_ptr=d2.data_ptr())
        c.close()
        ctx.sync()
        oi, od = case.oc.knn(k_max)
        assert np.array_equal(idx[:n * k_max].cpu().numpy().reshape(n, k_max), oi), name
        assert np.array_equal(d2[:n * k_max].cpu().numpy().reshape(n, k_max), od.view(np.int32)), name
        del oi, od
        mx, _ = _cmp_normals(normals[:n].cpu().numpy().view(np.float32), case.oc.normals(k=k_max)[0])
        assert mx <= NORMAL_TOL, name


# ---------------------------------------------------------------------------------------------------------------------
# b. query sub-ranges
# ---------------------------------------------------------------------------------------------------------------------
def _pieces(nf):
    """Uneven tiles of [0, nf): one query, 31, 129, two large ones (the last through count = -1), and empty ranges at
    the end."""
    mid = 161 + (nf - 161) // 2 + 7
    return [(0, 1), (1, 31), (32, 129), (161, mid - 161), (mid, -1), (nf, 0), (nf, -1)]


def _sorted_order(ctx, c, nf):
    p = c.dev_sorted_order()
    assert p
    return ctx.download(p, (nf,), np.int32)


def _tile(ctx, case, c, order, make, call, full):
    """Calls `call(outs, first, count)` on each piece of _pieces into fresh sentinel outputs.  Each piece writes the
    rows of its points (order[first:first + count]) and, on the piece that starts at 0, the defaults of the non-finite
    rows; nothing else.  Together the pieces give `full` bit for bit.  Returns the union of the pieces' kernel
    profiles."""
    union = {key: np.full_like(a, _sentinel(key)) for key, a in full.items()}
    names = set()
    for first, count in _pieces(case.nf):
        o = make()
        prof = _profiled(ctx, lambda: call(o, first, count))
        got = o.read(ctx)
        m = case.nf - first if count < 0 else count
        rows = np.zeros(case.n, bool)
        rows[order[first:first + m]] = True
        if first == 0:
            rows |= ~case.finite
        for key, a in got.items():
            written = a != _sentinel(key)
            assert np.array_equal(written.any(axis=1), rows), (key, first, count)
            assert written[rows].all(), (key, first, count)
            union[key][rows] = a[rows]
        assert ("default_rows" in prof) == (first == 0 and case.nf < case.n), (first, count, prof)
        if m == 0:
            assert not prof, prof
        names |= set(prof)
    for key in full:
        assert np.array_equal(union[key], full[key]), key
    return names


@pytest.mark.parametrize("name,k", [("nan_panel", 16), ("nan_panel", 32), ("nan_panel", 64), ("nan_panel", 100), ("box", 16)])
def test_knn_sub_ranges_tile_the_full_range(ctx, name, k):
    """On the box the full range runs on one grid per axis pair, the pieces on the primary grid: same bits."""
    case = _case(name)
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=case.n, stride_bytes=32)
    c.dev_index(k)
    order = _sorted_order(ctx, c, case.nf)
    o = Outs(case.n, 8, k)
    o.knn(c, k)
    full = o.read(ctx)
    _check_against_oracle(case, full, k=k)
    assert np.array_equal(_sorted_order(ctx, c, case.nf), order)   # the full-range call did not change it
    names = _tile(ctx, case, c, order, lambda: Outs(case.n, 8, k), lambda o, f, n: o.knn(c, k, f, n), full)
    assert "knn_normals" in names
    assert ("knn_redo" in names) == (k <= 64), names   # k <= 64: fixed-point kernel + hand-over; above: k_search
    c.close()


@pytest.mark.parametrize("name", ["three", "dense"])
def test_radius_sub_ranges_tile_the_full_range(ctx, name):
    """three: the fast 32-entry kernel, the one-warp hand-over and the generic tail; dense (8 points / mm^2): straight
    to the generic kernel at the largest neighbour count."""
    case = _case(name)
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=case.n, stride_bytes=32)
    c.dev_index(0, R)
    order = _sorted_order(ctx, c, case.nf)
    o = Outs(case.n)
    full_prof = _profiled(ctx, lambda: o.radius(c, R))
    full = o.read(ctx)
    _check_against_oracle(case, full, radius=R)
    names = _tile(ctx, case, c, order, lambda: Outs(case.n), lambda o, f, n: o.radius(c, R, f, n), full)
    if name == "three":
        stages = {"radius_normals", "radius_redo", "radius_count", "knn_redo"}
    else:
        stages = {"radius_count", "radius_normals"}
        assert "radius_redo" not in names and "radius_redo" not in full_prof
    assert stages <= set(full_prof) and stages <= names, (full_prof, names)
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# c. refusals
# ---------------------------------------------------------------------------------------------------------------------
def _refused(ctx, fn, bufs):
    """fn() is PPP_ERR_INVALID, launches nothing and writes nothing: bufs = [(tensor, sentinel)]."""
    before = ctx.launch_count()
    with pytest.raises(api.PPPError) as e:
        fn()
    assert e.value.status == api._lib.PPP_ERR_INVALID
    assert ctx.launch_count() == before, e.value
    ctx.sync()
    for t, sent in bufs:
        assert torch.all(t == sent), e.value


def test_refused_ranges_and_misaligned_buffers(ctx):
    case = _case("nan_panel")
    n, nf, k = case.n, case.nf, 16
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
    nrm = torch.full((n + 2, 8), SENT_F, dtype=torch.int32, device="cuda")
    idx = torch.full((n + 2, k), SENT_I, dtype=torch.int32, device="cuda")
    d2 = torch.full((n + 2, k), SENT_F, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    N, I, D = nrm.data_ptr(), idx.data_ptr(), d2.data_ptr()
    bufs = [(nrm, SENT_F), (idx, SENT_I), (d2, SENT_F)]
    for first, count in [(-1, -1), (-1, 5), (0, nf + 1), (5, nf - 4), (nf + 1, -1), (nf + 1, 0)]:
        _refused(ctx, lambda: c.dev_normals_knn(k, N, 32, idx_ptr=I, d2_ptr=D, first=first, count=count), bufs)
        _refused(ctx, lambda: c.dev_normals_radius(R, N, 32, first=first, count=count), bufs)
    for off, stride in [(4, 16), (8, 16), (4, 32), (8, 32), (4, 48)]:   # vector stores need 16-byte records
        _refused(ctx, lambda: c.dev_normals_knn(k, N + off, stride, idx_ptr=I), bufs)
        _refused(ctx, lambda: c.dev_normals_radius(R, N + off, stride), bufs)
    _refused(ctx, lambda: c.dev_normals_knn(k, N, 32, idx_ptr=I + 2), bufs)
    _refused(ctx, lambda: c.dev_normals_knn(k, None, 32, idx_ptr=I + 1), bufs)
    _refused(ctx, lambda: c.dev_normals_knn(k, N, 32, idx_ptr=I, d2_ptr=D + 2), bufs)
    _refused(ctx, lambda: api.Cloud(ctx, device_ptr=raw.data_ptr() + 2, n=n - 1, stride_bytes=32), bufs)
    c.close()


@pytest.mark.parametrize("kind", ["knn", "radius"])
def test_accepted_alignments_give_the_same_bits(ctx, kind):
    """Stride 32 from a buffer that is 16- but not 32-byte aligned (the float4 branch of store_normal instead of one
    32-byte store), stride 20 from a 4-byte aligned one: the records of an aligned buffer, nothing before or after."""
    case = _case("nan_panel")
    n = case.n
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
    for sf, off in [(8, 16), (5, 4)]:
        a = Outs(n, sf)
        getattr(a, kind)(c, 16 if kind == "knn" else R)
        want = a.read(ctx)["normals"]
        buf = torch.full((n * sf + 16,), SENT_F, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        p = buf.data_ptr() + off
        assert p % 32 != 0
        if kind == "knn":
            c.dev_normals_knn(16, p, sf * 4)
        else:
            c.dev_normals_radius(R, p, sf * 4)
        ctx.sync()
        got = buf.cpu().numpy()
        w = off // 4
        assert np.all(got[:w] == SENT_F) and np.all(got[w + n * sf:] == SENT_F)
        assert np.array_equal(got[w:w + n * sf].reshape(n, sf), want), (sf, off)
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# d. row map on a plain cloud
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,kind,k", [("nan_panel", "knn", 16), ("box", "knn", 16), ("nan_panel", "knn", 100),
                                         ("three", "radius", 0), ("dense", "radius", 0)])
def test_normal_row_map_on_a_plain_cloud(ctx, name, kind, k, monkeypatch, capfd):
    """Record map[row] receives row's normal (none for a negative entry, non-finite rows included: the default rows go
    through the map as well); ids stay by row.  NULL restores the identity."""
    case = _case(name)
    n = case.n
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
    rng = np.random.default_rng(61)

    def run(m):
        o = Outs(n, 8, k, d2=False)
        c.dev_set_normal_row_map(m.data_ptr() if m is not None else None)
        if kind == "knn":
            o.knn(c, k)
        else:
            o.radius(c, R)
        return o.read(ctx)

    if name == "box":
        monkeypatch.setenv("PPP_DEBUG", "1")
        capfd.readouterr()
    ref = run(None)
    if name == "box":   # the hand-over kernel stored records too
        handed = [int(h) for _, h in re.findall(r"knn fast path: (\d+) queries, (\d+) handed", capfd.readouterr().err)]
        assert handed and sum(handed) > 0, handed
        monkeypatch.delenv("PPP_DEBUG")
    assert not np.any(np.all(ref["normals"] == SENT_F, axis=1))
    perm = rng.permutation(n).astype(np.int32)
    perm_t = torch.from_numpy(perm).cuda()
    torch.cuda.synchronize()
    got = run(perm_t)
    assert np.array_equal(got["normals"][perm], ref["normals"])
    if kind == "knn":
        assert np.array_equal(got["idx"], ref["idx"])
    part = perm.copy()
    drop = rng.random(n) < 0.3
    bad = np.nonzero(~case.finite)[0]
    drop[bad[::2]] = True
    drop[bad[1::2]] = False
    part[drop] = -1
    part_t = torch.from_numpy(part).cuda()
    torch.cuda.synchronize()
    got = run(part_t)
    assert np.array_equal(got["normals"][perm[~drop]], ref["normals"][~drop])
    assert np.all(got["normals"][perm[drop]] == SENT_F)
    got = run(None)
    assert np.array_equal(got["normals"], ref["normals"])
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# e. record strides
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["knn", "radius"])
def test_normal_record_strides(ctx, kind):
    """The fields the header documents at each stride equal the host API's; the device path leaves the others as they
    were: 20 bytes {nx, ny, nz, curvature} + 1 untouched, 48 bytes {nx, ny, nz, 0, curvature} + 7 untouched."""
    case = _case("nan_panel")
    n = case.n
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=n, stride_bytes=32)
    h = api.Cloud(ctx, case.cloud)
    for sf, written in [(4, 4), (5, 4), (8, 8), (12, 5)]:
        o = Outs(n, sf)
        if kind == "knn":
            o.knn(c, 16)
            want = h.normals_knn(16, stride_floats=sf)
        else:
            o.radius(c, R)
            want = h.normals_radius(R, stride_floats=sf)
        got = o.read(ctx)["normals"]
        assert np.array_equal(got[:, :written], want.view(np.int32)[:, :written]), sf
        assert np.all(got[:, written:] == SENT_F), sf
        if sf == 8:
            _check_against_oracle(case, {"normals": got}, **({"k": 16} if kind == "knn" else {"radius": R}))
    h.close()
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# f. caller-owned contour buffers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,sync", [("A", False), ("B", False), ("B", True)])
def test_caller_owned_contour_buffers(ctx, monkeypatch, mode, sync):
    """Node buffers of cap >= total (cap == total included) take the nodes and are the pointers returned; smaller ones
    are left alone and the cloud's own buffers are returned.  An offsets buffer of S + 1 entries receives the offsets,
    one of S is left alone.  Mode B with PPP_SLICE_SYNC runs the chain with host round trips (the chain mode A takes)."""
    if sync:
        monkeypatch.setenv("PPP_SLICE_SYNC", "1")
    case = _case("nan_panel")
    S = 60
    planes = case.planes(S)
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=case.n, stride_bytes=32)
    want = c.slice_contours(planes, mode)   # the host API, before any caller buffer is set
    _same_contours(want, case.oc.slice_contours(planes, mode))
    T = int(want[0][-1])
    own = c.dev_slice_contours(planes, mode)
    _same_contours(_read_contours(ctx, own, S), want)
    for cap in (T, T + 5, T - 1):
        bufs = [torch.full((T + 8,), SENT_L, dtype=torch.int64, device="cuda") for _ in range(3)]
        torch.cuda.synchronize()
        c.dev_set_contour_buffers(*[b.data_ptr() for b in bufs], cap)
        res = c.dev_slice_contours(planes, mode)
        _same_contours(_read_contours(ctx, res, S), want)
        ctx.sync()
        host = [b.cpu().numpy() for b in bufs]
        ptrs = [res[a] for a in ("y", "x", "z")]
        if cap >= T:
            assert ptrs == [b.data_ptr() for b in bufs], cap
            for hb, w in zip(host, want[1:]):
                assert np.array_equal(hb[:T], w.view(np.int64)) and np.all(hb[T:] == SENT_L), cap
        else:
            assert ptrs == [own[a] for a in ("y", "x", "z")], cap
            assert all(np.all(hb == SENT_L) for hb in host), cap
    offb = torch.full((S + 3,), SENT_L, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    c.dev_set_contour_offsets_buffer(offb.data_ptr(), S + 1)
    c.dev_slice_contours(planes, mode)
    ctx.sync()
    ob = offb.cpu().numpy()
    assert np.array_equal(ob[:S + 1], want[0]) and np.all(ob[S + 1:] == SENT_L)
    offb.fill_(SENT_L)
    torch.cuda.synchronize()
    c.dev_set_contour_offsets_buffer(offb.data_ptr(), S)
    c.dev_slice_contours(planes, mode)
    ctx.sync()
    assert np.all(offb.cpu().numpy() == SENT_L)
    c.dev_set_contour_buffers(None, None, None, 0)
    c.dev_set_contour_offsets_buffer(None, 0)
    res = c.dev_slice_contours(planes, mode)
    assert [res[a] for a in ("y", "x", "z")] == [own[a] for a in ("y", "x", "z")]
    _same_contours(_read_contours(ctx, res, S), want)
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# g. ppp_dev_sorted_order
# ---------------------------------------------------------------------------------------------------------------------
def test_sorted_order_describes_the_ranges_of_its_index(ctx):
    """After dev_index(16), a full-range call (which adds one grid per axis pair on a box) and dev_index(64), each
    order returned is a permutation of the finite points and the positions of the ranges of its own k."""
    case = _case("small_box")
    raw = _on_device(case)
    c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=case.n, stride_bytes=32)
    assert c.dev_sorted_order() is None
    finite_rows = np.nonzero(case.finite)[0]
    c.dev_index(16)
    o16 = _sorted_order(ctx, c, case.nf)
    assert np.array_equal(np.sort(o16), finite_rows)
    full = {}
    for k in (16, 64):
        o = Outs(case.n, 8, k)
        o.knn(c, k)
        full[k] = o.read(ctx)
    _check_against_oracle(case, full[16], k=16)
    assert np.array_equal(_sorted_order(ctx, c, case.nf), o16)
    c.dev_index(64)
    o64 = _sorted_order(ctx, c, case.nf)
    assert np.array_equal(np.sort(o64), finite_rows)
    for k, order in ((64, o64), (16, o16)):
        _tile(ctx, case, c, order, lambda: Outs(case.n, 8, k), lambda o, f, n: o.knn(c, k, f, n), full[k])
    c.close()


# ---------------------------------------------------------------------------------------------------------------------
# the sub-range, row-map and stride paths under the bounds-checked build
# ---------------------------------------------------------------------------------------------------------------------
def _bounds_pass():
    ctx = api.Context(0)
    for cloud in (_with_bad_rows(synth.panel(20000, 1, noise_sigma=0.05), 2), synth.box_with_walls(20000, 2)):
        case = Case(cloud)
        raw = _on_device(case)
        c = api.Cloud(ctx, device_ptr=raw.data_ptr(), n=case.n, stride_bytes=32)
        for k in (16, 64, 100):
            c.dev_index(k)
            for first, count in _pieces(case.nf):
                Outs(case.n, 8, k).knn(c, k, first, count)
        c.dev_index(0, R)
        for first, count in _pieces(case.nf):
            Outs(case.n).radius(c, R, first, count)
        m = np.random.default_rng(3).permutation(case.n).astype(np.int32)
        m[::3] = -1
        m_t = torch.from_numpy(m).cuda()
        torch.cuda.synchronize()
        c.dev_set_normal_row_map(m_t.data_ptr())
        for k in (16, 100):
            Outs(case.n, 8, k).knn(c, k)
        Outs(case.n).radius(c, R)
        c.dev_set_normal_row_map(None)
        for sf in (4, 5, 8, 12):
            Outs(case.n, sf).knn(c, 16)
            Outs(case.n, sf).radius(c, R)
        ctx.sync()
        c.close()
    ctx.sync()
    ctx.close()
    print("done")


def test_device_api_paths_under_bounds_checks():
    check_lib = os.path.join(ROOT, "polishpathplanning_b200", "libppp_gpu_check.so")
    if not os.path.exists(check_lib):
        pytest.skip("libppp_gpu_check.so not built (python -m polishpathplanning_b200.build --check)")
    code = ("import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_device_api as t\nt._bounds_pass()\n"
            % (ROOT, os.path.join(ROOT, "tests")))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PPP_GPU_LIB=check_lib), capture_output=True,
                       text=True, timeout=600)
    out = r.stdout + r.stderr
    assert "PPP_DEV_ASSERT failed" not in out, out[-2000:]
    assert r.returncode == 0 and "done" in r.stdout, out[-2000:]
