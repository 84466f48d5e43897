"""Generalized ICP: CPU oracle (test infrastructure).

Restates Open3D's ``TransformationEstimationForGeneralizedICP`` (Segal et al. 2009, plane-to-plane) in the tensor ICP
loop of ``oracle/registration.py`` - PARITY UNPINNED: Open3D itself is not run here.  The transformed source, the
matching, ``fitness`` / ``inlier_rmse``, the loop, its convergence test, the Cholesky solve with its pivot rule and
``pose_to_transformation`` are those of ``oracle/registration.py`` (point-to-plane); only the per-correspondence
system differs:

  * every point's regularisation axis is ``a = normal_from_covariance(float64(C))`` (``oracle/normals.py``) of its
    float32 covariance ``C``, NaN when an entry of ``C`` is not finite: the axis is the only thing taken from a
    covariance.  Segal's ``U diag(1, 1, eps) U^T`` (``eps`` = ``epsilon``, Open3D's "covariance along the normal")
    is then ``I - (1 - eps) a a^T``;
  * for ``s'`` matched to ``t``, with ``R`` the upper-left 3x3 of the accumulated ``T`` and ``m = R a_s``:
    ``M = 2I - (1 - eps)(m m^T + a_t a_t^T)`` (= ``R C_s,reg R^T + C_t,reg``, positive definite for ``eps > 0``),
    ``W = M^-1`` (float64, by its adjugate), ``e = s' - t``, ``J = [-[s']x | I]`` (the pose order of
    point-to-plane); ``(sum J^T W J) x = -(sum J^T W e)``, ``T = pose_to_transformation(x) @ T``;
  * a system the Cholesky rejects, non-finite ones included (a NaN covariance of a matched point), is DEGENERATE.

Quirk, kept: an isotropic covariance has no defined axis.  The identity (what neighbourhoods of fewer than 3 points
get) takes the solver's tie rule, ``(0, 0, 1)``: the point is treated as a horizontal plane; a zero covariance gives
the axis 0 and so ``C_reg = I``.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from .normals import normal_from_covariance
from .registration import (DEGENERATE, NO_CORRESPONDENCE, OK, cholesky_solve, match, metrics,
                           pose_to_transformation, transform_points)


def regularisation_axes(covariances) -> np.ndarray:
    """float64 ``[n, 3]``: the regularisation axis ``normal_from_covariance(float64(C))`` of every float32
    covariance ``C`` (``[n, 3, 3]``, any float dtype, rounded to float32 first); NaN rows where ``C`` has a
    non-finite entry."""
    c = np.asarray(covariances).astype(np.float32).reshape(-1, 9).astype(np.float64)
    out = np.full((c.shape[0], 3), np.nan)
    for i in np.flatnonzero(np.isfinite(c).all(axis=1)):
        out[i] = normal_from_covariance(c[i])
    return out


def regularised_covariance(a: np.ndarray, epsilon: float) -> np.ndarray:
    """Segal's ``U diag(1, 1, eps) U^T`` written with the axis alone: ``I - (1 - eps) a a^T`` (``[n, 3, 3]``)."""
    a = np.asarray(a, np.float64).reshape(-1, 3)
    return np.eye(3) - (1.0 - epsilon) * a[:, :, None] * a[:, None, :]


def system(s: np.ndarray, t: np.ndarray, R: np.ndarray, a_s: np.ndarray, a_t: np.ndarray, epsilon: float):
    """``(H, b, W, J, e)`` of one Gauss-Newton step: ``H = sum J^T W J``, ``b = sum J^T W e`` over the float64
    pairs ``s`` (transformed source), ``t``, with the source axes ``a_s`` (source frame) and the target axes
    ``a_t``."""
    m = np.asarray(a_s, np.float64) @ np.asarray(R, np.float64).T
    k = 1.0 - epsilon
    M = 2.0 * np.eye(3) - k * (m[:, :, None] * m[:, None, :] + a_t[:, :, None] * a_t[:, None, :])
    A = np.empty_like(M)                                     # adjugate: NaN propagates, nothing raises
    A[:, 0, 0] = M[:, 1, 1] * M[:, 2, 2] - M[:, 1, 2] * M[:, 1, 2]
    A[:, 0, 1] = A[:, 1, 0] = M[:, 0, 2] * M[:, 1, 2] - M[:, 0, 1] * M[:, 2, 2]
    A[:, 0, 2] = A[:, 2, 0] = M[:, 0, 1] * M[:, 1, 2] - M[:, 0, 2] * M[:, 1, 1]
    A[:, 1, 1] = M[:, 0, 0] * M[:, 2, 2] - M[:, 0, 2] * M[:, 0, 2]
    A[:, 1, 2] = A[:, 2, 1] = M[:, 0, 1] * M[:, 0, 2] - M[:, 0, 0] * M[:, 1, 2]
    A[:, 2, 2] = M[:, 0, 0] * M[:, 1, 1] - M[:, 0, 1] * M[:, 0, 1]
    det = (M[:, 0, 0] * A[:, 0, 0] + M[:, 0, 1] * A[:, 0, 1]) + M[:, 0, 2] * A[:, 0, 2]
    W = A / det[:, None, None]
    e = s - t
    J = np.zeros((s.shape[0], 3, 6))
    J[:, 0, 1], J[:, 0, 2] = s[:, 2], -s[:, 1]               # -[s']x
    J[:, 1, 0], J[:, 1, 2] = -s[:, 2], s[:, 0]
    J[:, 2, 0], J[:, 2, 1] = s[:, 1], -s[:, 0]
    J[:, :, 3:] = np.eye(3)
    H = np.einsum("nia,nij,njb->ab", J, W, J)
    b = np.einsum("nia,nij,nj->a", J, W, e)
    return H, b, W, J, e


def step(s, t, R, a_s, a_t, epsilon):
    """The 4x4 update of one Gauss-Newton step, or None when the system is degenerate."""
    H, b, _, _, _ = system(s, t, R, a_s, a_t, epsilon)
    x = cholesky_solve(H, -b)
    return None if x is None else pose_to_transformation(x)


def icp(source, target, r, init=None, max_iteration=30, relative_fitness=1e-6, relative_rmse=1e-6,
        source_covariances=None, target_covariances=None, source_axes=None, target_axes=None, epsilon=1e-3):
    """The loop of ``oracle.registration.icp`` with the generalized estimation.  Each cloud takes its covariances
    (``[n, 3, 3]``) or its regularisation axes (float64 ``[n, 3]``, e.g. those the GPU used).  Returns the same
    dict as ``oracle.registration.icp``."""
    src = np.asarray(source, np.float32)
    tgt = np.asarray(target, np.float32)
    T = np.eye(4) if init is None else np.array(init, np.float64)
    ax_s = regularisation_axes(source_covariances) if source_axes is None else np.asarray(source_axes, np.float64)
    ax_t = regularisation_axes(target_covariances) if target_axes is None else np.asarray(target_axes, np.float64)
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
        update = step(st[m].astype(np.float64), tgt[corr[m]].astype(np.float64), T[:3, :3], ax_s[m], ax_t[corr[m]],
                      epsilon)
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
