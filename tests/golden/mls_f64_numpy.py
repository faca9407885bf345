"""Second restatement of the MLS pre-filter (smooth(), src/Path_Generation.cpp:340-360) in vectorised numpy float64,
written independently of oracle_mls/ppp_oracle_mls.cpp: scipy cKDTree neighbours (filtered with the float32
membership rule d2 < (float)(r*r), FLANN's ((dx*dx + dy*dy) + dz*dz)), numpy.linalg.eigh for the plane,
numpy.linalg.cholesky for the weighted least-squares fit.  Test checker only.

The normal of eigh has an arbitrary sign, so normals are only comparable up to sign; points are not affected."""
import numpy as np
from scipy.spatial import cKDTree


def _unit_orthogonal(n):
    # Eigen MatrixBase::unitOrthogonal for 3-vectors
    if not (abs(n[0]) <= abs(n[2]) * 1e-12) or not (abs(n[1]) <= abs(n[2]) * 1e-12):
        return np.array([-n[1], n[0], 0.0]) / np.hypot(n[0], n[1])
    return np.array([0.0, -n[2], n[1]]) / np.hypot(n[1], n[2])


def mls_rows(cloud, queries, radius=15.0, order=3):
    """For each query index: None (no output row) or (xyz float32[3], normal float32[3], curvature float32, fit bool).
    fit is None where numpy's Cholesky refuses the normal equations (not positive definite: the CPU oracle follows
    Eigen there and is not comparable)."""
    xyz32 = np.ascontiguousarray(cloud[:, :3], np.float32)
    finite = np.isfinite(xyz32).all(axis=1)
    idx_f = np.flatnonzero(finite)
    tree = cKDTree(xyz32[idx_f].astype(np.float64))
    nc = (order + 1) * (order + 2) // 2
    expo = [(a, b) for a in range(order + 1) for b in range(order + 1 - a)]
    out = []
    for i in queries:
        if not finite[i]:
            out.append(None)
            continue
        q32 = xyz32[i]
        cand = idx_f[np.asarray(tree.query_ball_point(q32.astype(np.float64), radius * (1 + 1e-5) + 1e-6), np.int64)]
        d = (q32[None, :] - xyz32[cand]).astype(np.float32)
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        nb = cand[d2 < np.float32(radius * radius)]
        m = nb.shape[0]
        if m < 3:
            out.append(None)
            continue
        P = xyz32[nb].astype(np.float64)
        q = q32.astype(np.float64)
        c = P.mean(axis=0)
        D = P - c
        cov = D.T @ D
        evals, evecs = np.linalg.eigh(cov)
        n = evecs[:, 0]
        tr = np.trace(cov)
        curv = abs(evals[0] / tr) if tr != 0 else 0.0
        mean = q - np.dot(q - c, n) * n
        va = _unit_orthogonal(n)
        ua = np.cross(n, va)
        uq, vq = np.dot(q - mean, ua), np.dot(q - mean, va)
        point = mean + uq * ua + vq * va
        normal = n
        fit = False
        if order > 1 and m >= nc:
            E = P - mean
            w = np.exp(-np.einsum("ij,ij->i", E, E) / (radius * radius))
            u, v, f = E @ ua, E @ va, E @ n
            Pm = np.stack([u ** a * v ** b for a, b in expo], axis=1)          # (m, nc)
            A = Pm.T @ (Pm * w[:, None])
            rhs = Pm.T @ (w * f)
            try:
                L = np.linalg.cholesky(A)
            except np.linalg.LinAlgError:
                out.append((point.astype(np.float32), normal.astype(np.float32), np.float32(curv), None))
                continue
            coef = np.linalg.solve(L.T, np.linalg.solve(L, rhs))
            if np.isfinite(coef[0]):
                z = sum(coef[j] * uq ** a * vq ** b for j, (a, b) in enumerate(expo))
                zu = sum(coef[j] * a * uq ** (a - 1) * vq ** b for j, (a, b) in enumerate(expo) if a >= 1)
                zv = sum(coef[j] * b * uq ** a * vq ** (b - 1) for j, (a, b) in enumerate(expo) if b >= 1)
                point = mean + uq * ua + vq * va + z * n
                normal = n - (zu * ua + zv * va)
                normal = normal / np.linalg.norm(normal)
                fit = True
        out.append((point.astype(np.float32), normal.astype(np.float32), np.float32(curv), fit))
    return out
