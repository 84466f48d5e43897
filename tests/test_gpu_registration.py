"""ICP registration on the GPU (apc_icp / apc_evaluate_registration; kernels k_icp_match / k_icp_solve) against the
CPU oracle (oracle/registration.py): bit-exact correspondences and distances, the loop's iterations, convergence and
transform, determinism, CUDA-graph capture, n_dev, recovery after errors, the grid shared with the other neighbour
stages, and the ``registration`` module."""
import numpy as np
import pytest

from oracle import registration as reg
from test_gpu_normals_search import dense_patch
from test_oracle_registration import matcher_cloud, planar_patches, recovery_pair

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine
    ctx = engine.Context(max_points=300_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi)
    ctx.close()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


@pytest.fixture(scope="module")
def recovery(env):
    """The recovery pair of the oracle tests, with the target's radius normals computed on the GPU (the oracle's
    point-to-plane loop takes the same normals)."""
    src, tgt, T_true = recovery_pair()
    normals, _, _ = env["ctx"].estimate_normals_radius(to_xyzi(tgt), 0.5)
    env["ctx"].check()
    return src, tgt, T_true, normals.cpu().numpy()


def evaluate(ctx, src, tgt, r, T=None, **kw):
    stats, corr, d2 = ctx.evaluate_registration(to_xyzi(src), to_xyzi(tgt), r, T, **kw)
    ctx.check()
    return stats.cpu().numpy(), corr.cpu().numpy(), d2.cpu().numpy()


def assert_evaluate(got, src, tgt, r, T=None):
    stats, corr, d2 = got
    f, rmse, corr_ref, d2_ref = reg.evaluate_registration(src, tgt, r, T)
    assert np.array_equal(corr, corr_ref)
    assert np.array_equal(d2.view(np.uint32), d2_ref.view(np.uint32))
    assert stats[0] == pytest.approx(f, rel=1e-12, abs=0) and stats[1] == pytest.approx(rmse, rel=1e-12, abs=0)
    return corr_ref


def run_icp(ctx, src, tgt, r, method, normals=None, **kw):
    nrm = torch.from_numpy(np.ascontiguousarray(normals, np.float32)).cuda() if normals is not None else None
    T, stats, info, corr = ctx.icp(to_xyzi(src), to_xyzi(tgt), r, method=method, tgt_normals=nrm, **kw)
    ctx.check()
    return T.cpu().numpy(), stats.cpu().numpy(), info.cpu().numpy(), corr.cpu().numpy()


def test_evaluate_recovery_pair(env, recovery):
    src, tgt, T_true, _ = recovery
    for T in (None, T_true):
        corr = assert_evaluate(evaluate(env["ctx"], src, tgt, 1.0, T), src, tgt, 1.0, T)
        assert (corr >= 0).any()


@pytest.mark.parametrize("seed", range(8))
def test_evaluate_ties_exact_r_and_far_from_origin(env, seed):
    """Duplicate target points, source points exactly r from a target point; odd seeds lie 100 m from the origin."""
    src, tgt, r = matcher_cloud(seed)
    corr = assert_evaluate(evaluate(env["ctx"], src, tgt, r), src, tgt, r)
    assert (corr >= 0).any() and (corr < 0).any()


def test_evaluate_far_from_origin_scan(env, recovery):
    src, tgt, T_true, _ = recovery
    off = np.float32([150.0, -80.0, 20.0])
    s, t = np.ascontiguousarray(src[:40_000] + off), np.ascontiguousarray(tgt + off)
    assert_evaluate(evaluate(env["ctx"], s, t, 0.5), s, t, 0.5)


def test_evaluate_neighbourhoods_above_1024(env):
    from scipy.spatial import cKDTree
    tgt = dense_patch()
    src = reg.transform_points(tgt, reg.pose_to_transformation([0.01, 0.0, -0.02, 0.03, 0.01, 0.0]))
    counts = np.array([len(c) for c in cKDTree(tgt).query_ball_point(src, 0.45)])
    assert counts.max() > 1024
    assert_evaluate(evaluate(env["ctx"], src, tgt, 0.45), src, tgt, 0.45)


@pytest.mark.parametrize("method", [reg.POINT_TO_POINT, reg.POINT_TO_PLANE])
def test_icp_matches_the_oracle_loop(env, recovery, method):
    src, tgt, T_true, normals = recovery
    nrm = normals if method == reg.POINT_TO_PLANE else None
    T, stats, info, corr = run_icp(env["ctx"], src, tgt, 1.0, method, nrm)
    ref = reg.icp(src, tgt, 1.0, method=method, target_normals=nrm)
    assert info[2] == reg.OK and ref["status"] == reg.OK
    assert info[0] == ref["iterations"] and bool(info[1]) == ref["converged"]
    assert np.array_equal(corr, ref["correspondences"])
    assert np.abs(T - ref["transformation"]).max() < 1e-9
    assert stats[0] == pytest.approx(ref["fitness"], rel=1e-12) and stats[1] == pytest.approx(ref["inlier_rmse"], rel=1e-9)
    E = np.linalg.inv(T_true) @ T
    assert np.linalg.norm(T[:3, 3] - T_true[:3, 3]) < 0.02
    assert np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1))) < 0.2


def test_icp_loop_edges(env):
    ctx = env["ctx"]
    tgt, nrm = planar_patches()
    init = reg.pose_to_transformation([0.0, 0.0, 0.01, 0.02, 0.0, 0.0])
    src = reg.transform_points(tgt, np.linalg.inv(reg.pose_to_transformation([0.01, 0, 0, 0, 0.05, 0])))
    T, stats, info, corr = run_icp(ctx, src, tgt, 0.5, reg.POINT_TO_POINT, init=init, max_iteration=0)
    assert np.array_equal(T, init) and list(info) == [0, 0, reg.OK, 0] and not stats.any() and np.all(corr == -1)
    for kw in (dict(max_iteration=1), dict(max_iteration=5, relative_fitness=10.0, relative_rmse=10.0)):
        for method in (reg.POINT_TO_POINT, reg.POINT_TO_PLANE):
            T, stats, info, corr = run_icp(ctx, src, tgt, 0.5, method, nrm, init=init, **kw)
            ref = reg.icp(src, tgt, 0.5, init=init, method=method, target_normals=nrm, **kw)
            assert info[0] == ref["iterations"] and bool(info[1]) == ref["converged"]
            assert np.array_equal(corr, ref["correspondences"]) and np.abs(T - ref["transformation"]).max() < 1e-12
    parallel = np.tile(np.float32([0, 0, 1]), (tgt.shape[0], 1))
    T, stats, info, corr = run_icp(ctx, tgt, tgt, 0.5, reg.POINT_TO_PLANE, parallel)
    assert list(info) == [0, 0, reg.DEGENERATE, 0] and np.array_equal(T, np.eye(4)) and stats[0] == 1.0


def test_determinism(env, recovery):
    src, tgt, _, normals = recovery
    for method in (reg.POINT_TO_POINT, reg.POINT_TO_PLANE):
        a = run_icp(env["ctx"], src, tgt, 1.0, method, normals, max_iteration=10)
        b = run_icp(env["ctx"], src, tgt, 1.0, method, normals, max_iteration=10)
        assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def test_cuda_graph_capture_replays_the_eager_result(env, recovery):
    src, tgt, _, normals = recovery
    ctx = env["ctx"]
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    nrm = torch.from_numpy(normals).cuda()
    eager = ctx.icp(xs, xt, 1.0, method=reg.POINT_TO_PLANE, tgt_normals=nrm)
    ctx.check()
    eager = [t.clone() for t in eager]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ctx.icp(xs, xt, 1.0, method=reg.POINT_TO_PLANE, tgt_normals=nrm)
    for t in out:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    ctx.check()
    assert all(torch.equal(a, b) for a, b in zip(out, eager))
    assert int(eager[2][0]) > 1


def test_n_dev_below_n_max(env, recovery):
    src, tgt, _, normals = recovery
    ctx = env["ctx"]
    ms, mt = 70_000, 120_000
    n_src_dev = torch.tensor([ms], dtype=torch.int32, device="cuda")
    n_tgt_dev = torch.tensor([mt], dtype=torch.int32, device="cuda")
    s, t, nrm = np.ascontiguousarray(src[:ms]), np.ascontiguousarray(tgt[:mt]), np.ascontiguousarray(normals[:mt])
    for method in (reg.POINT_TO_POINT, reg.POINT_TO_PLANE):
        full = run_icp(ctx, src, tgt, 1.0, method, normals, max_iteration=8, n_src_dev=n_src_dev, n_tgt_dev=n_tgt_dev)
        trimmed = run_icp(ctx, s, t, 1.0, method, nrm, max_iteration=8)
        # the launch configuration follows n_max: the sums may round differently, the matching may not
        assert np.abs(full[0] - trimmed[0]).max() < 1e-12
        assert np.array_equal(full[2], trimmed[2]) and np.array_equal(full[3][:ms], trimmed[3])
        assert np.all(full[3][ms:] == -1)
    stats, corr, d2 = evaluate(ctx, src, tgt, 1.0, n_src_dev=n_src_dev, n_tgt_dev=n_tgt_dev)
    assert_evaluate((stats, corr[:ms], d2[:ms]), s, t, 1.0)
    assert np.all(corr[ms:] == -1)


def test_errors_leave_the_context_usable(env, recovery):
    capi, ctx = env["capi"], env["ctx"]
    src, tgt = np.ascontiguousarray(recovery[0][:20_000]), np.ascontiguousarray(recovery[1][:40_000])
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    before = run_icp(ctx, src, tgt, 1.0, reg.POINT_TO_POINT, max_iteration=5)

    def bad(fn, word):
        with pytest.raises(capi.ApcError) as e:
            fn()
        assert e.value.code == capi.APC_ERR_BAD_ARG and word in str(e.value)

    for r in (0.0, -1.0, float("nan"), float("inf"), 1e30):
        bad(lambda: ctx.icp(xs, xt, r), "max_correspondence_distance")
        bad(lambda: ctx.evaluate_registration(xs, xt, r), "max_correspondence_distance")
    bad(lambda: ctx.icp(xs, xt, 1.0, max_iteration=-1), "max_iteration")
    bad(lambda: ctx.icp(xs, xt, 1.0, method=7), "method")
    bad(lambda: ctx.icp(xs, xt, 1.0, method=reg.POINT_TO_PLANE), "normals")
    lib, T16 = capi.lib, (capi.C.c_double * 16)(*np.eye(4).reshape(16))
    out = torch.zeros(64, dtype=torch.float64, device="cuda")
    info = torch.zeros(4, dtype=torch.int32, device="cuda")
    p = lambda t: capi.C.c_void_p(t.data_ptr())
    s = capi.C.c_void_p(torch.cuda.current_stream().cuda_stream)
    calls = [
        (None, 100, p(xt), T16), (p(xs), 100, None, T16), (p(xs), 100, p(xt), None),
        (p(xs), ctx.max_points + 1, p(xt), T16),
    ]
    for src_p, n, tgt_p, t16 in calls:
        rc = lib.apc_icp(ctx.h, src_p, n, None, tgt_p, None, 100, None, 1.0, t16, 0, 5, 1e-6, 1e-6, p(out), p(out[16:]),
                         p(info), None, s)
        assert rc == capi.APC_ERR_BAD_ARG
        rc = lib.apc_evaluate_registration(ctx.h, src_p, n, None, tgt_p, 100, None, 1.0, t16, None, None, p(out), s)
        assert rc == capi.APC_ERR_BAD_ARG
    # no correspondence: the target 100 m away
    T, stats, info_np, corr = run_icp(ctx, src, np.ascontiguousarray(tgt + np.float32(100.0)), 1.0, reg.POINT_TO_POINT)
    assert list(info_np) == [0, 0, reg.NO_CORRESPONDENCE, 0] and np.all(corr == -1) and not stats.any()
    # a target point the grid cannot key
    far = tgt.copy()
    far[5] = [5.0e5, 0.0, 0.0]
    ctx.icp(xs, to_xyzi(far), 1.0)
    with pytest.raises(capi.ApcError) as e:
        ctx.check()
    assert e.value.code == capi.APC_ERR_KEY_RANGE
    after = run_icp(ctx, src, tgt, 1.0, reg.POINT_TO_POINT, max_iteration=5)
    assert all(np.array_equal(a, b) for a, b in zip(before, after))


def bits(*ts):
    return [t.cpu().numpy().copy().view(np.uint8) for t in ts if t is not None]


def test_shared_scratch_interleaved(env, recovery):
    """ICP, DBSCAN, the normals searches and the outlier stages share the context's grids and scratch: interleaved
    on one context, each gives exactly what it gives on a context of its own."""
    engine, ctx = env["engine"], env["ctx"]
    src, tgt, _, normals = recovery
    xs, xt, nrm = to_xyzi(src), to_xyzi(tgt), torch.from_numpy(normals).cuda()
    calls = {
        "icp_p2l": lambda c: c.icp(xs, xt, 1.0, method=reg.POINT_TO_PLANE, tgt_normals=nrm, max_iteration=6),
        "icp_p2p": lambda c: c.icp(xs, xt, 0.5, max_iteration=4),
        "evaluate": lambda c: c.evaluate_registration(xs, xt, 0.7),
        "dbscan": lambda c: c.cluster_dbscan(xt, 0.5, 5, want_counts=True),
        "radius": lambda c: c.radius_outliers(xt, 5, 0.5, want_counts=True),
        "normals_radius": lambda c: c.estimate_normals_radius(xt, 0.5, want_counts=True),
        "normals_knn": lambda c: c.estimate_normals_knn(xs, 20),
        "statistical": lambda c: c.statistical_outliers(xt, 20, 2.0),
    }
    alone = {}
    for name, fn in calls.items():
        c = engine.Context(max_points=max(src.shape[0], tgt.shape[0]))
        alone[name] = bits(*fn(c))
        c.check()
        c.close()
    for name in ("icp_p2l", "dbscan", "icp_p2p", "radius", "evaluate", "normals_radius", "icp_p2l", "statistical",
                 "normals_knn", "icp_p2p", "evaluate", "dbscan"):
        got = bits(*calls[name](ctx))
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(got, alone[name])), name


def cloud(o3d, p, dev, normals=None):
    pcd = o3d.PointCloud(o3d.Device(dev))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p))).to(o3d.Device(dev))
    if normals is not None:
        pcd.point["normals"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(normals))).to(o3d.Device(dev))
    return pcd


def test_carrier(env, recovery):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    src, tgt, T_true, normals = recovery
    crit = o3dreg.ICPConvergenceCriteria(max_iteration=12)
    results = {}
    for dev in ("CUDA:0", "CPU:0"):
        s, t = cloud(o3d, src, dev), cloud(o3d, tgt, dev, normals)
        for est in (o3dreg.TransformationEstimationPointToPoint(), o3dreg.TransformationEstimationPointToPlane()):
            res = o3dreg.icp(s, t, 1.0, np.eye(4), est, crit)
            T = res.transformation
            assert T.device == o3d.Device("CPU:0") and T.dtype == torch.float64 and T.shape == (4, 4)
            c = res.correspondences_
            assert c.dtype == torch.int64 and c.device == o3d.Device(dev) and c.shape == (src.shape[0],)
            results[(dev, repr(est))] = (T.numpy(), c.t.cpu().numpy(), res.fitness, res.inlier_rmse, res.converged,
                                         res.num_iterations)
        ev = o3dreg.evaluate_registration(s, t, 1.0, T_true)
        f, rmse, corr, _ = reg.evaluate_registration(src, tgt, 1.0, T_true)
        assert np.array_equal(ev.correspondences_.t.cpu().numpy(), corr)
        assert ev.fitness == pytest.approx(f, rel=1e-12) and ev.inlier_rmse == pytest.approx(rmse, rel=1e-12)
    for est in ("TransformationEstimationPointToPoint", "TransformationEstimationPointToPlane"):
        a, b = results[("CUDA:0", est)], results[("CPU:0", est)]
        assert all(np.array_equal(x, y) for x, y in zip(a[:2], b[:2])) and a[2:] == b[2:]
        assert a[5] > 1


def test_carrier_voxel_size_and_errors(env, recovery):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    src, tgt, _, normals = recovery
    s, t = cloud(o3d, src, "CUDA:0"), cloud(o3d, tgt, "CUDA:0", normals)
    crit = o3dreg.ICPConvergenceCriteria(max_iteration=6)
    a = o3dreg.icp(s, t, 1.0, None, None, crit, voxel_size=0.3)
    b = o3dreg.icp(s.voxel_down_sample(0.3), t.voxel_down_sample(0.3), 1.0, None, None, crit)
    assert np.array_equal(a.transformation.numpy(), b.transformation.numpy())
    assert torch.equal(a.correspondences_.t, b.correspondences_.t) and a.correspondences_.shape[0] < src.shape[0]
    empty = cloud(o3d, np.zeros((0, 3), np.float32), "CUDA:0")
    for x, y in ((empty, t), (s, empty)):
        with pytest.raises(RuntimeError):
            o3dreg.icp(x, y, 1.0)
        ev = o3dreg.evaluate_registration(x, y, 1.0)
        assert ev.fitness == 0.0 and ev.inlier_rmse == 0.0 and ev.correspondences_.shape == (x._n(),)
        assert torch.all(ev.correspondences_.t == -1)
    with pytest.raises(RuntimeError, match="max_correspondence_distance"):
        o3dreg.icp(s, cloud(o3d, tgt + np.float32(100.0), "CUDA:0"), 1.0)
    with pytest.raises(RuntimeError, match="normals"):
        o3dreg.icp(s, cloud(o3d, tgt, "CUDA:0"), 1.0, estimation_method=o3dreg.TransformationEstimationPointToPlane())
    plane, _ = planar_patches()
    flat = cloud(o3d, plane, "CUDA:0", np.tile(np.float32([0, 0, 1]), (plane.shape[0], 1)))
    with pytest.raises(RuntimeError, match="positive definite"):
        o3dreg.icp(flat, flat, 0.5, estimation_method=o3dreg.TransformationEstimationPointToPlane())
    with pytest.raises(NotImplementedError):
        o3dreg.icp(s, t, 1.0, callback_after_iteration=lambda d: None)
    with pytest.raises(ValueError):
        o3dreg.icp(s, t, 0.0)


def test_kernels_by_name(env, recovery):
    ctx = env["ctx"]
    src, tgt, _, _ = recovery
    ctx.profile(True)
    try:
        ctx.icp(to_xyzi(src), to_xyzi(tgt), 1.0, max_iteration=3)
        ctx.check()
        names = ctx.profile_report()
    finally:
        ctx.profile(False)
    assert {"k_grid_insert", "k_icp_match", "k_icp_solve", "k_grid_clean"} <= set(names)
    assert names["k_icp_match"][1] == 3 and names["k_icp_solve"][1] == 3
