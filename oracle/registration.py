"""ICP registration: CPU oracle (test infrastructure).

Restates Open3D's tensor ICP (``open3d.t.pipelines.registration.icp`` / ``evaluate_registration``, single scale,
``DoSingleScaleICPIterations``) with the point-to-point and point-to-plane estimations - PARITY UNPINNED: Open3D
itself is not run here.

Choices fixed here:
  * transformed source point ``s' = float32(T s)`` with ``T`` the float64 4x4 accumulated so far: every coordinate
    is ``((T[r,0]*x + T[r,1]*y) + T[r,2]*z) + T[r,3]`` in float64, unfused, ``x, y, z`` promoted from float32, then
    rounded to float32.  Every iteration transforms the ORIGINAL source.  Defined difference: Open3D re-transforms
    its float32 cloud in place after every update, so its rounding builds up;
  * correspondence of source point ``i``: among the target points with ``d2_f32(s'_i, t_j) <= r2``,
    ``r2 = float32(r) * float32(r)`` (``r`` = ``max_correspondence_distance``, ``d2_f32`` the predicate of radius
    outliers and DBSCAN, ``oracle/outliers.py``), the one with the smallest ``(d2, j)``; -1 when there is none.
    Defined difference: Open3D's hybrid search tests ``d2 < r^2`` in its own precision.  A transformed source
    point whose cell on the target's grid cannot be keyed (``|coordinate| / (r (1 + 2^-8))`` beyond 262 143 cells,
    or not finite) has no correspondence;
  * ``fitness = n_corr / n_src``, ``inlier_rmse = sqrt(sum d2 / n_corr)`` summed in float64, both 0 when
    ``n_corr = 0``;
  * point-to-point (Kabsch, no scaling): ``H = sum (s' - mu_s)(t - mu_t)^T = U S V^T``,
    ``R = V diag(1, 1, sign(det(V U^T))) U^T``, ``t = mu_t - R mu_s``;
  * point-to-plane: ``r_i = (s' - t) . n``, ``J_i = [s' x n, n]`` (``n`` the target's float32 normal promoted to
    float64); ``(sum J^T J) x = -(sum J^T r)`` solved by Cholesky for ``x = (alpha, beta, gamma, tx, ty, tz)``;
    the update is ``Rz(gamma) Ry(beta) Rx(alpha)`` with translation ``(tx, ty, tz)`` (Open3D's
    ``PoseToTransformation``).  The system is DEGENERATE (no update, the loop stops) when a Cholesky pivot is not
    above ``1e-12`` times its diagonal entry of ``sum J^T J`` (or is not finite): every normal parallel, for
    example.  Open3D solves whatever it gets;
  * the loop (``icp``):

        T = init; prev_f = prev_r = 0; iterations = 0; converged = False; status = OK
        for j in range(max_iteration):
            corr, d2 = match(source, T)
            if n_corr == 0: status = NO_CORRESPONDENCE; break     # Open3D raises here
            fitness, rmse = metrics(corr, d2)
            update = estimate(...)                                # may set status = DEGENERATE and break
            T = update @ T; iterations = j + 1
            if j > 0 and |prev_f - fitness| < relative_fitness and |prev_r - rmse| < relative_rmse:
                converged = True; break
            prev_f, prev_r = fitness, rmse

    returning ``T`` and the fitness, rmse and correspondences of the LAST matching (0, 0 and all -1 after
    ``NO_CORRESPONDENCE``).  ``max_iteration = 0`` returns ``init``, 0, 0, all -1 and 0 iterations.

``match`` proposes candidates with ``scipy.spatial.cKDTree`` at a slightly inflated float64 radius and decides them
with the float32 predicate and the ``(d2, j)`` order; ``match_brute`` is the same definition by brute force, and
the tests pin the two together.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from .outliers import d2_f32

POINT_TO_POINT, POINT_TO_PLANE = 0, 1
OK, NO_CORRESPONDENCE, DEGENERATE = 0, 1, 2
PIVOT_REL = 1e-12           # Cholesky pivot floor, relative to the diagonal entry
KEY_CELLS = 262143.0        # grid key range of the target's grid, in cells (apc_grid.cuh)


def transform_points(pos: np.ndarray, T: np.ndarray) -> np.ndarray:
    """``float32(T s)`` with the operation order of the definition (numpy does not contract to FMA)."""
    p = np.asarray(pos, np.float32).astype(np.float64)
    T = np.asarray(T, np.float64)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    out = np.empty((p.shape[0], 3), np.float32)
    for r in range(3):
        out[:, r] = (((T[r, 0] * x + T[r, 1] * y) + T[r, 2] * z) + T[r, 3]).astype(np.float32)
    return out


def keyable(q: np.ndarray, r: float) -> np.ndarray:
    """Rows whose cell on the target's grid (cells of ``float32(r) * (1 + 2^-8)``, indexed by one float32 multiply
    with the rounded reciprocal) lies inside the key range."""
    cell = np.float32(np.float32(r) * np.float32(1.00390625))
    inv = np.float32(1.0) / cell
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.floor(q.astype(np.float32) * inv)
        return np.all((c >= -KEY_CELLS) & (c < KEY_CELLS), axis=1)


def match_brute(src_t: np.ndarray, tgt: np.ndarray, r: float):
    """``(corr int32[n], d2 float32[n])`` by the definition, all pairs (small clouds)."""
    r32 = np.float32(r)
    n = src_t.shape[0]
    corr = np.full(n, -1, np.int32)
    d2 = np.zeros(n, np.float32)
    ok = keyable(src_t, r)
    for i in range(n):
        if not ok[i] or tgt.shape[0] == 0:
            continue
        d = d2_f32(src_t[i][None, :], tgt)
        inside = np.flatnonzero(d <= r32 * r32)
        if inside.size:
            j = inside[np.lexsort((inside, d[inside]))[0]]
            corr[i], d2[i] = j, d[j]
    return corr, d2


def match(src_t: np.ndarray, tgt: np.ndarray, r: float, tree=None, k: int = 16):
    """The same with a kd-tree: the ``k`` nearest in float64 within an inflated radius, re-ranked by the float32
    ``(d2, j)``.  A row whose ``k``-th candidate is still within rounding of its nearest (ties, duplicates) is
    decided over every candidate within the radius."""
    r32 = np.float32(r)
    r2 = r32 * r32
    n = src_t.shape[0]
    corr = np.full(n, -1, np.int32)
    d2 = np.zeros(n, np.float32)
    if n == 0 or tgt.shape[0] == 0:
        return corr, d2
    tree = tree if tree is not None else cKDTree(tgt.astype(np.float64))
    k = min(k, tgt.shape[0])
    ok = keyable(src_t, r)
    q = src_t.astype(np.float64)
    q[~ok] = 0.0
    bound = float(r32) * (1.0 + 1e-5) + 1e-6
    dist, idx = tree.query(q, k=k, distance_upper_bound=bound, workers=-1)
    dist, idx = dist.reshape(n, k), idx.reshape(n, k)
    valid = (idx < tgt.shape[0]) & ok[:, None]
    safe = np.where(valid, idx, 0)
    d = d2_f32(src_t[:, None, :], tgt[safe])
    inside = valid & (d <= r2)
    big = np.float32(np.inf)
    key_d = np.where(inside, d, big)
    key_j = np.where(inside, safe, np.iinfo(np.int64).max)
    order = np.lexsort((key_j, key_d), axis=1)[:, 0]
    rows = np.arange(n)
    has = inside[rows, order]
    corr[has] = safe[rows, order][has].astype(np.int32)
    d2[has] = d[rows, order][has]
    # rows the k nearest may not settle: all k within the radius and the last one within rounding of the first
    full = valid[:, k - 1] & (dist[:, k - 1] <= dist[:, 0] * (1.0 + 1e-5) + 1e-6)
    for i in np.flatnonzero(full):
        c = np.asarray(tree.query_ball_point(q[i], bound), np.int64)
        dc = d2_f32(src_t[i][None, :], tgt[c])
        keep = dc <= r2
        c, dc = c[keep], dc[keep]
        if c.size:
            o = np.lexsort((c, dc))[0]
            corr[i], d2[i] = c[o], dc[o]
    return corr, d2


def metrics(corr: np.ndarray, d2: np.ndarray, n_src: int):
    m = corr >= 0
    nc = int(m.sum())
    if nc == 0:
        return 0.0, 0.0
    return nc / n_src, float(np.sqrt(d2[m].astype(np.float64).sum() / nc))


def kabsch(s: np.ndarray, t: np.ndarray) -> np.ndarray:
    """Rigid 4x4 minimising sum |R s + t_ - t|^2 over float64 pairs (no scaling)."""
    mu_s, mu_t = s.mean(axis=0), t.mean(axis=0)
    H = (s - mu_s).T @ (t - mu_t)
    U, _, Vt = np.linalg.svd(H)
    V = Vt.T
    d = 1.0 if np.linalg.det(V @ U.T) >= 0.0 else -1.0
    R = V @ np.diag([1.0, 1.0, d]) @ U.T
    out = np.eye(4)
    out[:3, :3] = R
    out[:3, 3] = mu_t - R @ mu_s
    return out


def pose_to_transformation(x) -> np.ndarray:
    """Open3D's ``PoseToTransformation``: ``Rz(gamma) Ry(beta) Rx(alpha)`` and translation ``(tx, ty, tz)``."""
    a, b, g = x[0], x[1], x[2]
    Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    Ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    Rz = np.array([[np.cos(g), -np.sin(g), 0], [np.sin(g), np.cos(g), 0], [0, 0, 1]])
    out = np.eye(4)
    out[:3, :3] = Rz @ Ry @ Rx
    out[:3, 3] = x[3:6]
    return out


def cholesky_solve(A: np.ndarray, b: np.ndarray):
    """``A x = b`` for symmetric ``A`` by Cholesky; None when a pivot is not above ``PIVOT_REL`` times its
    diagonal entry (not positive definite, up to rounding)."""
    n = A.shape[0]
    L = np.zeros_like(A)
    for j in range(n):
        d = A[j, j] - L[j, :j] @ L[j, :j]
        if not (np.isfinite(d) and d > PIVOT_REL * A[j, j]):
            return None
        L[j, j] = np.sqrt(d)
        for i in range(j + 1, n):
            L[i, j] = (A[i, j] - L[i, :j] @ L[j, :j]) / L[j, j]
    y = np.zeros(n)
    for i in range(n):
        y[i] = (b[i] - L[i, :i] @ y[:i]) / L[i, i]
    x = np.zeros(n)
    for i in reversed(range(n)):
        x[i] = (y[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
    return x


def point_to_plane(s: np.ndarray, t: np.ndarray, n: np.ndarray):
    """The 4x4 update of one Gauss-Newton step, or None when the system is degenerate."""
    r = ((s - t) * n).sum(axis=1)
    J = np.concatenate([np.cross(s, n), n], axis=1)
    x = cholesky_solve(J.T @ J, -(J.T @ r))
    return None if x is None else pose_to_transformation(x)


def evaluate_registration(source, target, r, T=None):
    """``(fitness, inlier_rmse, corr int32[n_src], d2 float32[n_src])`` at ``T`` (identity by default)."""
    src = np.asarray(source, np.float32)
    tgt = np.asarray(target, np.float32)
    T = np.eye(4) if T is None else np.asarray(T, np.float64)
    corr, d2 = match(transform_points(src, T), tgt, r)
    f, rmse = metrics(corr, d2, src.shape[0])
    return f, rmse, corr, d2


def icp(source, target, r, init=None, method=POINT_TO_POINT, target_normals=None, max_iteration=30,
        relative_fitness=1e-6, relative_rmse=1e-6):
    """The loop of the module docstring.  Returns a dict with ``transformation``, ``fitness``, ``inlier_rmse``,
    ``correspondences``, ``iterations``, ``converged`` and ``status``."""
    src = np.asarray(source, np.float32)
    tgt = np.asarray(target, np.float32)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    nrm = None if target_normals is None else np.asarray(target_normals, np.float32).astype(np.float64)
    tree = cKDTree(tgt.astype(np.float64)) if tgt.shape[0] else None
    out = dict(fitness=0.0, inlier_rmse=0.0, correspondences=np.full(src.shape[0], -1, np.int32), iterations=0,
               converged=False, status=OK)
    prev_f = prev_r = 0.0
    for j in range(max_iteration):
        st = transform_points(src, T)
        corr, d2 = match(st, tgt, r, tree)
        out["correspondences"] = corr
        m = corr >= 0
        if not m.any():
            out.update(fitness=0.0, inlier_rmse=0.0, status=NO_CORRESPONDENCE)
            break
        f, rmse = metrics(corr, d2, src.shape[0])
        out.update(fitness=f, inlier_rmse=rmse)
        s64, t64 = st[m].astype(np.float64), tgt[corr[m]].astype(np.float64)
        if method == POINT_TO_POINT:
            update = kabsch(s64, t64)
        else:
            update = point_to_plane(s64, t64, nrm[corr[m]])
            if update is None:
                out["status"] = DEGENERATE
                break
        T = update @ T
        out["iterations"] = j + 1
        if j > 0 and abs(prev_f - f) < relative_fitness and abs(prev_r - rmse) < relative_rmse:
            out["converged"] = True
            break
        prev_f, prev_r = f, rmse
    out["transformation"] = T
    return out
