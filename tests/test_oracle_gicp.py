"""The generalized-ICP oracle (oracle/gicp.py): the regularisation written with the axis alone against
Segal's eigendecomposition, the axes pinned to the analytic solver, the system against point-to-plane's and finite
differences, one Gauss-Newton step, the loop's edges and the recovery of a known transform."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import gicp
from oracle import normals as onrm
from oracle import registration as reg
from test_oracle_registration import planar_patches, pose_error, recovery_pair


def knn_covariances(pos, k=20):
    """float32 covariances of every point's ``k`` nearest (float64 kd-tree), about their mean."""
    p = np.asarray(pos, np.float64)
    _, nb = cKDTree(p).query(p, k=k, workers=-1)
    d = p[nb] - p[:, None, :]
    m = d.mean(axis=1)
    return (np.einsum("nki,nkj->nij", d, d) / k - m[:, :, None] * m[:, None, :]).astype(np.float32)


def separated_covariances(seed, n=200):
    """Random rotations of diag(l0, l1, l2) with l0 < l1 < l2 at least a factor 3 apart."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        Q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        lo = 10.0 ** rng.uniform(-6, -2)
        lam = np.array([lo, lo * rng.uniform(3, 50), lo * rng.uniform(200, 1e4)])
        out.append(Q @ np.diag(lam) @ Q.T)
    return np.asarray(out, np.float32)


@pytest.mark.parametrize("epsilon", [1e-3, 0.1, 0.9])
def test_regularisation_equals_segal_eigendecomposition(epsilon):
    covs = separated_covariances(1)
    a = gicp.regularisation_axes(covs)
    got = gicp.regularised_covariance(a, epsilon)
    for C, G in zip(covs.astype(np.float64), got):
        _, U = np.linalg.eigh(C)                              # ascending: column 0 is the least variance
        ref = U @ np.diag([epsilon, 1.0, 1.0]) @ U.T
        assert np.abs(G - ref).max() < 1e-9


def test_axes_are_the_solver_of_estimate_normals():
    covs = separated_covariances(2, 100)
    a = gicp.regularisation_axes(covs)
    for C, v in zip(covs, a):
        assert np.array_equal(v, onrm.normal_from_covariance(C.astype(np.float64)))
        w, U = np.linalg.eigh(C.astype(np.float64))
        assert abs(v @ U[:, 0]) >= 1 - 1e-12
    # the documented quirks: the identity (fewer than 3 neighbours) -> (0, 0, 1); zero -> 0; non-finite -> NaN
    nan_diag = np.diag([1.0, 2.0, np.nan]).astype(np.float32)
    odd = np.stack([np.eye(3), np.zeros((3, 3)), nan_diag, np.full((3, 3), np.inf)]).astype(np.float32)
    a = gicp.regularisation_axes(odd)
    assert list(a[0]) == [0.0, 0.0, 1.0] and list(a[1]) == [0.0, 0.0, 0.0]
    assert np.isnan(a[2:]).all()
    assert np.array_equal(gicp.regularised_covariance(a[1], 1e-3)[0], np.eye(3))


def pairs(seed, n=300):
    rng = np.random.default_rng(seed)
    s = rng.normal(size=(n, 3)) * 4.0
    t = s + rng.normal(size=(n, 3)) * 0.05
    a_s = rng.normal(size=(n, 3))
    a_t = rng.normal(size=(n, 3))
    a_s /= np.linalg.norm(a_s, axis=1, keepdims=True)
    a_t /= np.linalg.norm(a_t, axis=1, keepdims=True)
    R = reg.pose_to_transformation([0.3, -0.2, 0.5, 0, 0, 0])[:3, :3]
    return s, t, R, a_s, a_t


def test_combined_covariance_and_weight():
    s, t, R, a_s, a_t = pairs(3)
    eps = 1e-3
    _, _, W, _, _ = gicp.system(s, t, R, a_s, a_t, eps)
    Cs, Ct = gicp.regularised_covariance(a_s, eps), gicp.regularised_covariance(a_t, eps)
    M = R @ Cs @ R.T + Ct
    assert np.abs(np.einsum("nij,njk->nik", W, M) - np.eye(3)).max() < 1e-9
    assert (np.linalg.eigvalsh(M) > 0).all()


def test_system_with_the_normal_projector_is_point_to_plane():
    s, t, R, a_s, a_t = pairs(4)
    _, _, _, J, e = gicp.system(s, t, R, a_s, a_t, 1e-3)
    n = a_t
    Wn = n[:, :, None] * n[:, None, :]
    H = np.einsum("nia,nij,njb->ab", J, Wn, J)
    b = np.einsum("nia,nij,nj->a", J, Wn, e)
    Jp = np.concatenate([np.cross(s, n), n], axis=1)
    r = ((s - t) * n).sum(axis=1)
    assert np.abs(H - Jp.T @ Jp).max() < 1e-9 * np.abs(H).max()
    assert np.abs(b - Jp.T @ r).max() < 1e-9 * np.abs(b).max()


def test_jacobian_is_the_derivative_of_the_residual():
    s, t, R, a_s, a_t = pairs(5, 20)
    _, _, _, J, _ = gicp.system(s, t, R, a_s, a_t, 1e-3)

    def e(x):
        U = reg.pose_to_transformation(x)
        return s @ U[:3, :3].T + U[:3, 3] - t

    h = 1e-6
    for k in range(6):
        dx = np.zeros(6)
        dx[k] = h
        fd = (e(dx) - e(-dx)) / (2 * h)
        assert np.abs(fd - J[:, :, k]).max() < 1e-7


def objective(s, t, R, a_s, a_t, eps):
    _, _, W, _, e = gicp.system(s, t, R, a_s, a_t, eps)
    return np.einsum("ni,nij,nj->", e, W, e)


def test_one_step_lowers_the_objective():
    tgt, nrm = planar_patches()
    T = reg.pose_to_transformation([0.01, -0.02, 0.015, 0.03, -0.02, 0.04])
    Ti = np.linalg.inv(T)
    src = reg.transform_points(tgt, Ti)
    a_t = nrm.astype(np.float64)
    a_s = a_t @ Ti[:3, :3].T                                  # the same planes, seen in the source's frame
    corr, _ = reg.match(src, tgt, 0.5)
    m = corr >= 0
    s, t = src[m].astype(np.float64), tgt[corr[m]].astype(np.float64)
    eps, R = 1e-3, np.eye(3)
    before = objective(s, t, R, a_s[m], a_t[corr[m]], eps)
    up = gicp.step(s, t, R, a_s[m], a_t[corr[m]], eps)
    after = objective(s @ up[:3, :3].T + up[:3, 3], t, up[:3, :3] @ R, a_s[m], a_t[corr[m]], eps)
    assert after < 0.05 * before


def test_loop_edges_and_a_nan_covariance():
    tgt, _ = planar_patches()
    init = reg.pose_to_transformation([0.0, 0.0, 0.01, 0.02, 0.0, 0.0])
    src = reg.transform_points(tgt, np.linalg.inv(reg.pose_to_transformation([0.01, 0, 0, 0, 0.05, 0])))
    cs, ct = knn_covariances(src), knn_covariances(tgt)
    kw = dict(source_covariances=cs, target_covariances=ct, init=init)
    out = gicp.icp(src, tgt, 0.5, max_iteration=0, **kw)
    assert np.array_equal(out["transformation"], init) and out["iterations"] == 0 and out["status"] == reg.OK
    assert out["fitness"] == 0.0 and np.all(out["correspondences"] == -1)
    one = gicp.icp(src, tgt, 0.5, max_iteration=1, **kw)
    assert one["iterations"] == 1 and not one["converged"] and one["status"] == reg.OK
    f, rmse, corr, _ = reg.evaluate_registration(src, tgt, 0.5, init)
    assert (one["fitness"], one["inlier_rmse"]) == (f, rmse) and np.array_equal(one["correspondences"], corr)
    m = corr >= 0
    st = reg.transform_points(src, init).astype(np.float64)
    a_s, a_t = gicp.regularisation_axes(cs), gicp.regularisation_axes(ct)
    step = gicp.step(st[m], tgt[corr[m]].astype(np.float64), init[:3, :3], a_s[m], a_t[corr[m]], 1e-3)
    assert np.array_equal(one["transformation"], step @ init)
    loose = gicp.icp(src, tgt, 0.5, max_iteration=5, relative_fitness=10.0, relative_rmse=10.0, **kw)
    assert loose["iterations"] == 2 and loose["converged"]
    # precomputed axes give the same loop as the covariances they come from
    same = gicp.icp(src, tgt, 0.5, max_iteration=1, source_axes=a_s, target_axes=a_t, init=init)
    assert np.array_equal(same["transformation"], one["transformation"])
    bad = ct.copy()
    bad[int(corr[m][0])] = np.diag([1.0, 2.0, np.nan])
    out = gicp.icp(src, tgt, 0.5, source_covariances=cs, target_covariances=bad, init=init)
    assert out["status"] == reg.DEGENERATE and out["iterations"] == 0 and np.array_equal(out["transformation"], init)


def test_recovery():
    src, tgt, T_true = recovery_pair()
    out = gicp.icp(src, tgt, 1.0, source_covariances=knn_covariances(src),
                  target_covariances=knn_covariances(tgt))
    dt, angle = pose_error(out["transformation"], T_true)
    assert out["status"] == reg.OK and dt < 0.02 and angle < 0.2
    assert out["fitness"] > 0.95
