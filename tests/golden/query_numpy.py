"""Brute-force references for the external-query searches, in plain numpy and sharing nothing with oracle/.

- kNN and radius search: every float32 d² is formed in FLANN's order, ((dx*dx + dy*dy) + dz*dz), one rounding per
  numpy float32 operation, exactly like the kernels (no FMA).  Lists are ordered by (d², index): the d² bits of a
  non-negative float are monotone, so the 64-bit key (bits << 32 | index) orders them with one integer compare.
  Ties at the k-th place, d² = inf included, go to the lower index.
- Radius membership is d² < float32(r * r) (the radius squared in double, then rounded, as PCL does).
- Coverage flags: the union of the radius memberships of the queries; a NaN radius marks nothing.
- Principal curvatures: PCL's computePointPrincipalCurvatures restated in float64 on a given neighbour list (normals
  projected with I - n0 n0^T, centroid, covariance, numpy.linalg.eigh): pc1 = l2 / m, pc2 = l1 / m, direction =
  eigenvector of l2.

Non-finite points are not indexed (they are never neighbours); a query with a non-finite coordinate gets no
neighbours.  Queries are processed in chunks so that 100k points x a few thousand queries fit in memory.
"""
import numpy as np

F32 = np.float32
_CHUNK_ELEMS = 1 << 23   # d² entries per chunk (64 MB of uint64 keys)


def _xyz(a):
    return np.ascontiguousarray(np.asarray(a, F32)[:, :3])


def _indexed(points):
    p = _xyz(points)
    ids = np.flatnonzero(np.isfinite(p).all(axis=1)).astype(np.int64)
    return p[ids], ids


def d2_flann(q, p):
    """(m, 3) x (n, 3) float32 -> (m, n) float32 squared distances in FLANN's summation order."""
    with np.errstate(over="ignore", invalid="ignore"):
        dx = q[:, None, 0] - p[None, :, 0]
        dy = q[:, None, 1] - p[None, :, 1]
        dz = q[:, None, 2] - p[None, :, 2]
        return (dx * dx + dy * dy) + dz * dz


def _chunks(nq, n):
    step = max(1, _CHUNK_ELEMS // max(n, 1))
    for a in range(0, nq, step):
        yield a, min(nq, a + step)


def knn(points, queries, k):
    """(idx int32 (nq, k), d2 float32 (nq, k)): -1 / inf padded beyond min(k, finite points)."""
    p, ids = _indexed(points)
    q = _xyz(queries)
    nq, n = q.shape[0], p.shape[0]
    idx = np.full((nq, k), -1, np.int32)
    d2 = np.full((nq, k), np.inf, F32)
    kk = min(k, n)
    if kk == 0:
        return idx, d2
    qfin = np.isfinite(q).all(axis=1)
    for a, b in _chunks(nq, n):
        rows = np.flatnonzero(qfin[a:b]) + a
        if rows.size == 0:
            continue
        D = d2_flann(q[rows], p)
        key = (D.view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)[None, :]
        if kk < n:
            key = np.partition(key, kk - 1, axis=1)[:, :kk]
        key = np.sort(key, axis=1)[:, :kk]
        idx[rows, :kk] = ids[(key & np.uint64(0xFFFFFFFF)).astype(np.int64)].astype(np.int32)
        d2[rows, :kk] = (key >> np.uint64(32)).astype(np.uint32).view(F32)
    return idx, d2


def radius(points, queries, r):
    """(counts, offsets, idx, d2) with lists sorted by (d², index), membership d² < float32(r * r)."""
    p, ids = _indexed(points)
    q = _xyz(queries)
    r2 = F32(float(r) * float(r))
    nq, n = q.shape[0], p.shape[0]
    counts = np.zeros(nq, np.int32)
    lists_i, lists_d = [[] for _ in range(nq)], [[] for _ in range(nq)]
    qfin = np.isfinite(q).all(axis=1)
    for a, b in _chunks(nq, n):
        rows = np.flatnonzero(qfin[a:b]) + a
        if rows.size == 0:
            continue
        D = d2_flann(q[rows], p)
        for j, t in enumerate(rows):
            m = np.flatnonzero(D[j] < r2)
            o = np.lexsort((ids[m], D[j, m]))
            lists_i[t], lists_d[t] = ids[m][o].astype(np.int32), D[j, m][o]
            counts[t] = m.size
    offsets = np.zeros(nq + 1, np.int64)
    np.cumsum(counts, out=offsets[1:])
    cat = lambda ls, dt: np.concatenate([np.asarray(x, dt) for x in ls]) if nq else np.zeros(0, dt)
    return counts, offsets, cat(lists_i, np.int32), cat(lists_d, F32)


def coverage(points, queries, radii, flags=None):
    """flags (uint8, N) |= 1 for every point with d² < float32(r_i * r_i) from query i; radii: scalar or per query."""
    p, ids = _indexed(points)
    q = _xyz(queries)
    nq, n = q.shape[0], p.shape[0]
    out = np.zeros(np.asarray(points).shape[0], np.uint8) if flags is None else flags.copy()
    rr = np.broadcast_to(np.asarray(radii, np.float64), (nq,))
    with np.errstate(over="ignore", invalid="ignore"):
        r2 = (rr * rr).astype(F32)   # NaN stays NaN: d² < NaN admits nothing
    hit = np.zeros(n, bool)
    qfin = np.isfinite(q).all(axis=1)
    for a, b in _chunks(nq, n):
        rows = np.flatnonzero(qfin[a:b]) + a
        if rows.size:
            hit |= (d2_flann(q[rows], p) < r2[rows, None]).any(axis=0)
    out[ids[hit]] = 1
    return out


def principal_curvatures_f64(normals, idx):
    """float64 restatement on neighbour lists idx (nq, k), -1 padded.  Returns (out (nq, 5): pcx, pcy, pcz, pc1, pc2,
    gap (nq,) = l2 - l1, scale (nq,)): NaN rows where there is no neighbour or a normal is NaN.  scale is what a float32
    evaluation's error is proportional to, per unit roundoff: the largest |C| entry (the eigen solver) plus the sum of
    the |d_j| (each projected normal carries an absolute error of a few roundoffs, since M and n are O(1) -- it
    dominates when the projected normals are nearly equal and C is tiny)."""
    N = np.asarray(normals, np.float64)[:, :3]
    idx = np.asarray(idx)
    nq = idx.shape[0]
    out = np.full((nq, 5), np.nan)
    gap = np.full(nq, np.nan)
    cnorm = np.full(nq, np.nan)
    m_all = (idx >= 0).sum(axis=1)
    for m in np.unique(m_all):
        if m == 0:
            continue
        rows = np.flatnonzero(m_all == m)
        nb = N[idx[rows, :m]]                                   # (r, m, 3)
        n0 = nb[:, 0, :]
        M = np.eye(3)[None] - n0[:, :, None] * n0[:, None, :]   # I - n0 n0^T
        proj = np.einsum("rij,rmj->rmi", M, nb)
        d = proj - proj.mean(axis=1, keepdims=True)
        C = np.einsum("rmi,rmj->rij", d, d)
        ok = np.isfinite(C).all(axis=(1, 2))
        if not ok.any():
            continue
        w, v = np.linalg.eigh(C[ok])                            # ascending eigenvalues
        rr = rows[ok]
        out[rr, 0:3] = v[:, :, 2]
        out[rr, 3] = w[:, 2] / m
        out[rr, 4] = w[:, 1] / m
        gap[rr] = w[:, 2] - w[:, 1]
        cnorm[rr] = np.abs(C[ok]).max(axis=(1, 2)) + np.linalg.norm(d[ok], axis=2).sum(axis=1)
    return out, gap, cnorm
