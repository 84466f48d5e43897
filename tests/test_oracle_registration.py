"""The ICP oracle (oracle/registration.py): the kd-tree matcher pinned to brute force, the two estimations, the
loop's semantics and the recovery of a known transform on a C2-shaped scan."""
import numpy as np
import pytest

from oracle import registration as reg


def matcher_cloud(seed):
    """Target with exact duplicates (the tie goes to the lower index) and a source with points exactly float32(r)
    from a target point along an axis, plus random points, around ``origin``."""
    rng = np.random.default_rng(seed)
    r = float(rng.choice([0.2, 0.5, 1.0]))
    origin = np.float32([100.0, -60.0, 40.0]) if seed % 2 else np.float32([0.0, 0.0, 0.0])
    tgt = (rng.uniform(-3 * r, 3 * r, size=(300, 3)) + origin).astype(np.float32)
    dup = rng.integers(0, 300, size=40)
    tgt[rng.integers(0, 300, size=40)] = tgt[dup]
    src = (rng.uniform(-3.5 * r, 3.5 * r, size=(200, 3)) + origin).astype(np.float32)
    e = np.float32(r)
    edge = tgt[rng.integers(0, 300, size=30)].copy()
    for k in range(30):
        edge[k, k % 3] = edge[k, k % 3] + (e if k % 2 else -e)   # float32 add: d2 lands on r2 or next to it
    src = np.concatenate([src, edge, tgt[dup[:10]]])
    return src, tgt, r


def recovery_pair():
    """Target: a C2-shaped scan with 2 cm noise voxelised at 0.1 m.  Source: the same scene with another noise draw,
    voxelised on a grid shifted by a few cm and moved by the inverse of ``T_true`` (0.5 m, 3 degrees): ICP from the
    identity should find ``T_true``."""
    from autodriver_pointcloud_preprocessor_b200 import synth
    from oracle import voxel
    clean = synth.lidar_scan(seed=4, n_beams=128, n_az=2048, nan_frac=0.0, dup_frac=0.0, noise_sigma=0.0)["positions"]
    rng = np.random.default_rng(11)
    tgt = voxel.voxel_down_sample((clean + rng.normal(0, 0.02, clean.shape)).astype(np.float32), 0.1, None,
                                  fixed=True)["positions"]
    shift = np.float32([0.05, 0.03, 0.07])
    moved = (clean + rng.normal(0, 0.02, clean.shape) + shift).astype(np.float32)
    src0 = voxel.voxel_down_sample(moved, 0.1, None, fixed=True)["positions"] - shift
    a = np.deg2rad(3.0)
    T_true = reg.pose_to_transformation([0.2 * a, -0.3 * a, a, 0.4, -0.25, 0.1])
    src = reg.transform_points(src0, np.linalg.inv(T_true))
    return np.ascontiguousarray(src), np.ascontiguousarray(tgt), T_true


def pose_error(T, T_true):
    E = np.linalg.inv(T_true) @ T
    angle = np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1.0) / 2.0, -1.0, 1.0)))
    return np.linalg.norm(T[:3, 3] - T_true[:3, 3]), angle


@pytest.mark.parametrize("seed", range(12))
def test_kdtree_matcher_equals_brute_force(seed):
    src, tgt, r = matcher_cloud(seed)
    a = np.deg2rad(2.0)
    about = np.eye(4)
    about[:3, 3] = src.mean(axis=0)                                  # rotate about the cloud, not the origin
    moved = about @ reg.pose_to_transformation([a, -a, 2 * a, 0.1 * r, 0.0, -0.2 * r]) @ np.linalg.inv(about)
    for T in (np.eye(4), moved):
        st = reg.transform_points(src, T)
        corr, d2 = reg.match(st, tgt, r)
        corr_b, d2_b = reg.match_brute(st, tgt, r)
        assert np.array_equal(corr, corr_b)
        assert np.array_equal(d2.view(np.uint32), d2_b.view(np.uint32))
        assert (corr >= 0).any() and (corr < 0).any()
    # the duplicated target points: the lower index wins
    st = reg.transform_points(src, np.eye(4))
    corr, d2 = reg.match(st, tgt, r)
    for i in range(src.shape[0] - 10, src.shape[0]):
        same = np.flatnonzero(np.all(tgt == st[i], axis=1))
        assert corr[i] == same.min() and d2[i] == 0.0


def test_points_exactly_r_apart_match():
    r = 0.3
    e = np.float32(r)
    tgt = np.float32([[1.0, 2.0, 3.0], [9.0, 9.0, 9.0]])
    src = np.float32([[1.0 + e, 2.0, 3.0], [1.0, 2.0 - e, 3.0], [1.0, 2.0, 3.0 + 2 * e]])
    d2 = reg.d2_f32(src, tgt[0][None, :])
    corr, got = reg.match(src, tgt, r)
    assert list(corr) == [0 if d <= e * e else -1 for d in d2][:2] + [-1]
    assert np.array_equal(corr, reg.match_brute(src, tgt, r)[0])


def test_kabsch_recovers_a_rigid_transform():
    rng = np.random.default_rng(1)
    s = rng.normal(size=(50, 3)) * 5.0
    T = reg.pose_to_transformation([0.3, -0.2, 1.1, 2.0, -1.0, 0.5])
    t = s @ T[:3, :3].T + T[:3, 3]
    assert np.abs(reg.kabsch(s, t) - T).max() < 1e-12


def test_pose_order_is_rz_ry_rx():
    a = 0.4
    T = reg.pose_to_transformation([a, 0.0, 0.0, 1.0, 2.0, 3.0])
    assert np.allclose(T[:3, :3], [[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]], atol=0, rtol=0)
    assert list(T[:3, 3]) == [1.0, 2.0, 3.0]
    al, be, ga = 0.1, -0.2, 0.3
    Rx = reg.pose_to_transformation([al, 0, 0, 0, 0, 0])
    Ry = reg.pose_to_transformation([0, be, 0, 0, 0, 0])
    Rz = reg.pose_to_transformation([0, 0, ga, 0, 0, 0])
    assert np.abs(reg.pose_to_transformation([al, be, ga, 0, 0, 0]) - Rz @ Ry @ Rx).max() < 1e-15
    # Open3D's PoseToTransformation, written out
    T = reg.pose_to_transformation([al, be, ga, 0, 0, 0])
    assert abs(T[0, 1] - (-np.sin(ga) * np.cos(al) + np.cos(ga) * np.sin(be) * np.sin(al))) < 1e-15
    assert abs(T[2, 0] + np.sin(be)) < 1e-15


def planar_patches():
    """Three orthogonal noiseless planes with exact normals: every direction of the 6x6 system is constrained."""
    rng = np.random.default_rng(5)
    u, v = rng.uniform(-2, 2, size=(2, 400))
    pts = np.concatenate([np.stack([u, v, np.zeros_like(u)], 1), np.stack([u, np.full_like(u, 3.0), v + 2], 1),
                          np.stack([np.full_like(u, -3.0), u, v + 2], 1)]).astype(np.float32)
    nrm = np.concatenate([np.tile([0, 0, 1], (400, 1)), np.tile([0, 1, 0], (400, 1)),
                          np.tile([1, 0, 0], (400, 1))]).astype(np.float32)
    return pts, nrm


def test_point_to_plane_step_reduces_the_residual():
    tgt, nrm = planar_patches()
    T = reg.pose_to_transformation([0.01, -0.02, 0.015, 0.03, -0.02, 0.04])
    src = reg.transform_points(tgt, np.linalg.inv(T))
    corr, _ = reg.match(src, tgt, 0.5)
    m = corr >= 0
    s, t, n = src[m].astype(np.float64), tgt[corr[m]].astype(np.float64), nrm[corr[m]].astype(np.float64)
    before = np.abs(((s - t) * n).sum(1)).sum()
    up = reg.point_to_plane(s, t, n)
    s2 = s @ up[:3, :3].T + up[:3, 3]
    after = np.abs(((s2 - t) * n).sum(1)).sum()
    assert after < 0.2 * before


def test_point_to_plane_with_parallel_normals_is_degenerate():
    tgt, _ = planar_patches()
    nrm = np.tile(np.float32([0, 0, 1]), (tgt.shape[0], 1))
    out = reg.icp(tgt, tgt, 0.5, method=reg.POINT_TO_PLANE, target_normals=nrm)
    assert out["status"] == reg.DEGENERATE and out["iterations"] == 0 and not out["converged"]
    assert np.array_equal(out["transformation"], np.eye(4))
    assert out["fitness"] == 1.0 and out["inlier_rmse"] == 0.0


def test_loop_semantics():
    tgt, nrm = planar_patches()
    init = reg.pose_to_transformation([0.0, 0.0, 0.01, 0.02, 0.0, 0.0])
    src = reg.transform_points(tgt, np.linalg.inv(reg.pose_to_transformation([0.01, 0, 0, 0, 0.05, 0])))
    out = reg.icp(src, tgt, 0.5, init=init, max_iteration=0)
    assert np.array_equal(out["transformation"], init) and out["iterations"] == 0
    assert out["fitness"] == 0.0 and out["inlier_rmse"] == 0.0 and np.all(out["correspondences"] == -1)
    # convergence is never declared at j = 0, even with thresholds that any change passes
    out = reg.icp(src, tgt, 0.5, init=init, max_iteration=5, relative_fitness=10.0, relative_rmse=10.0)
    assert out["iterations"] == 2 and out["converged"]
    one = reg.icp(src, tgt, 0.5, init=init, max_iteration=1)
    assert one["iterations"] == 1 and not one["converged"]
    # the metrics and correspondences come from the last matching, T includes the last update
    f, rmse, corr, _ = reg.evaluate_registration(src, tgt, 0.5, init)
    assert (one["fitness"], one["inlier_rmse"]) == (f, rmse) and np.array_equal(one["correspondences"], corr)
    assert not np.array_equal(one["transformation"], init)
    m = corr >= 0
    st = reg.transform_points(src, init)
    step = reg.kabsch(st[m].astype(np.float64), tgt[corr[m]].astype(np.float64))
    assert np.array_equal(one["transformation"], step @ init)
    # no correspondence: the target is 100 m away
    far = reg.icp(src, tgt + np.float32(100.0), 0.5)
    assert far["status"] == reg.NO_CORRESPONDENCE and far["iterations"] == 0 and far["fitness"] == 0.0
    assert np.all(far["correspondences"] == -1)


def test_source_points_outside_the_key_range_have_no_correspondence():
    r = 0.01
    far = np.float32(262143.0 * r * 1.00390625 * 1.001)
    tgt = np.float32([[far, 0.0, 0.0], [0.0, 0.0, 0.0]])
    src = np.float32([[far, 0.0, 0.0], [0.0, 0.0, 0.0], [np.nan, 0.0, 0.0]])
    corr, _ = reg.match(src, tgt, r)
    assert list(corr) == [-1, 1, -1]
    assert np.array_equal(corr, reg.match_brute(src, tgt, r)[0])


@pytest.fixture(scope="module")
def recovery():
    return recovery_pair()


@pytest.mark.parametrize("method", [reg.POINT_TO_POINT, reg.POINT_TO_PLANE])
def test_recovery(recovery, method):
    from oracle import normals as onrm
    src, tgt, T_true = recovery
    nrm = onrm.estimate_normals(tgt, 0.5, 30)[0] if method == reg.POINT_TO_PLANE else None
    out = reg.icp(src, tgt, 1.0, method=method, target_normals=nrm)
    dt, angle = pose_error(out["transformation"], T_true)
    assert out["status"] == reg.OK and dt < 0.02 and angle < 0.2
    assert out["fitness"] > 0.95
