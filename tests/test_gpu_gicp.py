"""Generalized ICP on the GPU (apc_icp_generalized; kernels k_gicp_prep / k_icp_match_gicp / k_icp_solve) against the
CPU oracle (oracle/gicp.py), fed the regularisation axes the GPU used: the axes against the solver, the
loop's iterations, correspondences and transform, determinism, CUDA-graph capture, n_dev, recovery after errors,
the scratch shared with the other neighbour stages, ``PointCloud.estimate_covariances`` and the ``registration``
module."""
import numpy as np
import pytest

from oracle import gicp
from oracle import registration as reg
from test_oracle_registration import pose_error, planar_patches, recovery_pair

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


def knn_cov(ctx, p, k=20):
    """float32 covariances of the KNN-k search on the GPU (what ``estimate_covariances()`` gives)."""
    _, _, cov = ctx.estimate_normals_knn(to_xyzi(p), k, want_cov=True)
    ctx.check()
    return cov.to(torch.float32).contiguous()


@pytest.fixture(scope="module")
def recovery(env):
    src, tgt, T_true = recovery_pair()
    return src, tgt, T_true, knn_cov(env["ctx"], src), knn_cov(env["ctx"], tgt)


@pytest.fixture(scope="module")
def planar(env):
    tgt, _ = planar_patches()
    src = reg.transform_points(tgt, np.linalg.inv(reg.pose_to_transformation([0.01, -0.02, 0.015, 0.03, -0.02, 0.04])))
    return src, tgt, knn_cov(env["ctx"], src), knn_cov(env["ctx"], tgt)


def run(ctx, src, tgt, cs, ct, r, **kw):
    out = ctx.icp_generalized(to_xyzi(src), cs, to_xyzi(tgt), ct, r, **kw)
    ctx.check()
    return [t.cpu().numpy() for t in out]


def separated(cov):
    """Points whose two smallest eigenvalues are clearly apart (the axis is well defined)."""
    w = np.linalg.eigvalsh(cov.astype(np.float64))
    return w[:, 1] > 2.0 * w[:, 0] + 1e-9


def test_axes_are_the_solver(env, recovery):
    src, tgt, _, cs, ct = recovery
    _, _, info, _, ax_s, ax_t = run(env["ctx"], src, tgt, cs, ct, 1.0, max_iteration=0, want_axes=True)
    assert info[0] == 0
    for ax, cov in ((ax_s, cs.cpu().numpy()), (ax_t, ct.cpu().numpy())):
        ok = separated(cov)
        assert ok.mean() > 0.9
        ref = gicp.regularisation_axes(cov[ok])
        assert (np.abs((ax[ok] * ref).sum(1)) >= 1 - 1e-12).all()
    # the documented quirks: identity -> (0, 0, 1), zero -> 0, a non-finite entry -> NaN
    p = np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]])
    odd = np.stack([np.eye(3), np.zeros((3, 3)), np.diag([1.0, 2.0, np.nan]), np.diag([1.0, 2.0, 3.0])])
    odd = torch.from_numpy(odd.astype(np.float32)).cuda()
    _, _, _, _, ax, _ = run(env["ctx"], p, p, odd, odd, 1.0, max_iteration=0, want_axes=True)
    assert list(ax[0]) == [0, 0, 1] and list(ax[1]) == [0, 0, 0] and np.isnan(ax[2]).all() and list(ax[3]) == [1, 0, 0]


def assert_oracle_loop(got, src, tgt, r, **kw):
    T, stats, info, corr, ax_s, ax_t = got
    ref = gicp.icp(src, tgt, r, source_axes=ax_s, target_axes=ax_t, **kw)
    assert info[2] == ref["status"]
    assert info[0] == ref["iterations"] and bool(info[1]) == ref["converged"]
    assert np.array_equal(corr, ref["correspondences"])
    assert np.abs(T - ref["transformation"]).max() < 1e-9
    assert stats[0] == pytest.approx(ref["fitness"], rel=1e-12) and stats[1] == pytest.approx(ref["inlier_rmse"], rel=1e-9)


def test_matches_the_oracle_loop_recovery_pair(env, recovery):
    src, tgt, T_true, cs, ct = recovery
    got = run(env["ctx"], src, tgt, cs, ct, 1.0, want_axes=True)
    assert got[2][2] == reg.OK and got[2][0] > 1
    assert_oracle_loop(got, src, tgt, 1.0)
    dt, angle = pose_error(got[0], T_true)
    assert dt < 0.02 and angle < 0.2


def test_matches_the_oracle_loop_planar_patches(env, planar):
    src, tgt, cs, ct = planar
    init = reg.pose_to_transformation([0.0, 0.0, 0.01, 0.02, 0.0, 0.0])
    for kw in (dict(), dict(max_iteration=1), dict(max_iteration=5, relative_fitness=10.0, relative_rmse=10.0),
               dict(epsilon=0.3)):
        got = run(env["ctx"], src, tgt, cs, ct, 0.5, init=init, want_axes=True, **kw)
        assert_oracle_loop(got, src, tgt, 0.5, init=init, **kw)
    T, stats, info, corr = run(env["ctx"], src, tgt, cs, ct, 0.5, init=init, max_iteration=0)
    assert np.array_equal(T, init) and list(info) == [0, 0, reg.OK, 0] and not stats.any() and np.all(corr == -1)
    # a NaN covariance of a matched point: the system is not finite
    first = run(env["ctx"], src, tgt, cs, ct, 0.5, init=init, max_iteration=1)[3]
    bad = ct.clone()
    bad[int(first[first >= 0][0])] = torch.diag(torch.tensor([1.0, 2.0, float("nan")])).cuda()
    T, stats, info, _ = run(env["ctx"], src, tgt, cs, bad, 0.5, init=init)
    assert list(info) == [0, 0, reg.DEGENERATE, 0] and np.array_equal(T, init) and stats[0] > 0.9


def test_determinism(env, recovery):
    src, tgt, _, cs, ct = recovery
    a = run(env["ctx"], src, tgt, cs, ct, 1.0, max_iteration=10, want_axes=True)
    b = run(env["ctx"], src, tgt, cs, ct, 1.0, max_iteration=10, want_axes=True)
    assert all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


def test_cuda_graph_capture_replays_the_eager_result(env, recovery):
    src, tgt, _, cs, ct = recovery
    ctx = env["ctx"]
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    eager = ctx.icp_generalized(xs, cs, xt, ct, 1.0, want_axes=True)
    ctx.check()
    eager = [t.clone() for t in eager]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ctx.icp_generalized(xs, cs, xt, ct, 1.0, want_axes=True)
    for t in out:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    ctx.check()
    assert all(torch.equal(a, b) for a, b in zip(out, eager))
    assert int(eager[2][0]) > 1


def test_n_dev_below_n_max(env, recovery):
    src, tgt, _, cs, ct = recovery
    ctx = env["ctx"]
    ms, mt = 70_000, 120_000
    n_src_dev = torch.tensor([ms], dtype=torch.int32, device="cuda")
    n_tgt_dev = torch.tensor([mt], dtype=torch.int32, device="cuda")
    s, t = np.ascontiguousarray(src[:ms]), np.ascontiguousarray(tgt[:mt])
    full = run(ctx, src, tgt, cs, ct, 1.0, max_iteration=8, n_src_dev=n_src_dev, n_tgt_dev=n_tgt_dev, want_axes=True)
    trimmed = run(ctx, s, t, cs[:ms].contiguous(), ct[:mt].contiguous(), 1.0, max_iteration=8, want_axes=True)
    # the launch configuration follows n_max: the sums may round differently, the matching may not
    assert np.abs(full[0] - trimmed[0]).max() < 1e-12
    assert np.array_equal(full[2], trimmed[2]) and np.array_equal(full[3][:ms], trimmed[3])
    assert np.all(full[3][ms:] == -1)
    assert np.array_equal(full[4][:ms], trimmed[4]) and not full[4][ms:].any()
    assert np.array_equal(full[5][:mt], trimmed[5]) and not full[5][mt:].any()


def test_errors_leave_the_context_usable(env, recovery):
    capi, ctx = env["capi"], env["ctx"]
    src, tgt = np.ascontiguousarray(recovery[0][:20_000]), np.ascontiguousarray(recovery[1][:40_000])
    cs, ct = recovery[3][:20_000].contiguous(), recovery[4][:40_000].contiguous()
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    before = run(ctx, src, tgt, cs, ct, 1.0, max_iteration=5, want_axes=True)

    def bad(fn, word):
        with pytest.raises(capi.ApcError) as e:
            fn()
        assert e.value.code == capi.APC_ERR_BAD_ARG and word in str(e.value)

    for eps in (0.0, -1e-3, float("nan"), float("inf"), -float("inf")):
        bad(lambda: ctx.icp_generalized(xs, cs, xt, ct, 1.0, epsilon=eps), "epsilon")
    bad(lambda: ctx.icp_generalized(xs, None, xt, ct, 1.0), "covariances")
    bad(lambda: ctx.icp_generalized(xs, cs, xt, None, 1.0), "covariances")
    for r in (0.0, -1.0, float("nan"), float("inf"), 1e30):
        bad(lambda: ctx.icp_generalized(xs, cs, xt, ct, r), "max_correspondence_distance")
    bad(lambda: ctx.icp_generalized(xs, cs, xt, ct, 1.0, max_iteration=-1), "max_iteration")
    lib, T16 = capi.lib, (capi.C.c_double * 16)(*np.eye(4).reshape(16))
    out = torch.zeros(64, dtype=torch.float64, device="cuda")
    info = torch.zeros(4, dtype=torch.int32, device="cuda")
    p = lambda t: capi.C.c_void_p(t.data_ptr())
    s = capi.C.c_void_p(torch.cuda.current_stream().cuda_stream)
    calls = [(None, 100, p(xt), T16, p(out), p(info)), (p(xs), 100, None, T16, p(out), p(info)),
             (p(xs), 100, p(xt), None, p(out), p(info)), (p(xs), ctx.max_points + 1, p(xt), T16, p(out), p(info)),
             (p(xs), 100, p(xt), T16, None, p(info)), (p(xs), 100, p(xt), T16, p(out), None)]
    for src_p, n, tgt_p, t16, out_t, out_info in calls:
        rc = lib.apc_icp_generalized(ctx.h, src_p, p(cs), n, None, tgt_p, p(ct), 100, None, 1.0, t16, 1e-3, 5, 1e-6,
                                     1e-6, out_t, p(out[16:]), out_info, None, None, None, s)
        assert rc == capi.APC_ERR_BAD_ARG
    # no correspondence: the target 100 m away
    T, stats, info_np, corr = run(ctx, src, np.ascontiguousarray(tgt + np.float32(100.0)), cs, ct, 1.0)
    assert list(info_np) == [0, 0, reg.NO_CORRESPONDENCE, 0] and np.all(corr == -1) and not stats.any()
    # an empty target (valid pointers, n_tgt = 0; an empty tensor's data pointer is NULL): nothing to match, the
    # source's axes stay 0
    axes = torch.full((src.shape[0], 3), 7.0, dtype=torch.float64, device="cuda")
    info.fill_(-1)
    rc = lib.apc_icp_generalized(ctx.h, p(xs), p(cs), src.shape[0], None, p(xt), p(ct), 0, None, 1.0, T16, 1e-3, 5,
                                 1e-6, 1e-6, p(out), p(out[16:]), p(info), None, p(axes), None, s)
    assert rc == capi.APC_OK
    ctx.check()
    assert info.tolist() == [0, 0, reg.NO_CORRESPONDENCE, 0] and not axes.any()
    # a target point the grid cannot key
    far = tgt.copy()
    far[5] = [5.0e5, 0.0, 0.0]
    ctx.icp_generalized(xs, cs, to_xyzi(far), ct, 1.0)
    with pytest.raises(capi.ApcError) as e:
        ctx.check()
    assert e.value.code == capi.APC_ERR_KEY_RANGE
    after = run(ctx, src, tgt, cs, ct, 1.0, max_iteration=5, want_axes=True)
    assert all(np.array_equal(a, b) for a, b in zip(before, after))


def bits(*ts):
    return [t.cpu().numpy().copy().view(np.uint8) for t in ts if t is not None]


def test_shared_scratch_interleaved(env, recovery):
    """Generalized ICP, ICP, DBSCAN, the normals searches and the outlier stages share the context's grids and
    scratch: interleaved on one context, each gives exactly what it gives on a context of its own."""
    engine, ctx = env["engine"], env["ctx"]
    src, tgt, _, cs, ct = recovery
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    calls = {
        "gicp": lambda c: c.icp_generalized(xs, cs, xt, ct, 1.0, max_iteration=6, want_axes=True),
        "gicp_eps": lambda c: c.icp_generalized(xs, cs, xt, ct, 0.5, epsilon=0.05, max_iteration=4),
        "icp_p2p": lambda c: c.icp(xs, xt, 0.5, max_iteration=4),
        "dbscan": lambda c: c.cluster_dbscan(xt, 0.5, 5, want_counts=True),
        "radius": lambda c: c.radius_outliers(xt, 5, 0.5, want_counts=True),
        "normals_radius": lambda c: c.estimate_normals_radius(xt, 0.5, want_counts=True, want_cov=True),
        "normals_knn": lambda c: c.estimate_normals_knn(xs, 20, want_cov=True),
        "normals_hybrid": lambda c: c.estimate_normals(xs, 20, 0.5, want_cov=True),
        "statistical": lambda c: c.statistical_outliers(xt, 20, 2.0),
    }
    alone = {}
    for name, fn in calls.items():
        c = engine.Context(max_points=max(src.shape[0], tgt.shape[0]))
        alone[name] = bits(*fn(c))
        c.check()
        c.close()
    for name in ("gicp", "dbscan", "icp_p2p", "gicp_eps", "radius", "normals_radius", "gicp", "statistical",
                 "normals_knn", "gicp_eps", "normals_hybrid", "icp_p2p", "gicp", "dbscan"):
        got = bits(*calls[name](ctx))
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(got, alone[name])), name


def test_kernels_by_name(env, recovery):
    ctx = env["ctx"]
    src, tgt, _, cs, ct = recovery
    ctx.profile(True)
    try:
        ctx.icp_generalized(to_xyzi(src), cs, to_xyzi(tgt), ct, 1.0, max_iteration=3)
        ctx.check()
        names = ctx.profile_report()
    finally:
        ctx.profile(False)
    assert {"k_grid_insert", "k_gicp_prep", "k_icp_match_gicp", "k_icp_solve", "k_grid_clean"} <= set(names)
    assert names["k_gicp_prep"][1] == 1 and names["k_icp_match_gicp"][1] == 3 and names["k_icp_solve"][1] == 3
    assert "k_icp_match" not in names


def cloud(o3d, p, dev, cov=None):
    pcd = o3d.PointCloud(o3d.Device(dev))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p))).to(o3d.Device(dev))
    if cov is not None:
        pcd.point["covariances"] = o3d.Tensor(cov).to(o3d.Device(dev))
    return pcd


def test_estimate_covariances_is_the_engine_covariance(env, recovery):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    ctx = o3d.get_context(300_000)
    src = recovery[0][:50_000]
    xs = to_xyzi(src)
    modes = {(20, None): lambda: ctx.estimate_normals_knn(xs, 20, want_cov=True),
             (None, 0.5): lambda: ctx.estimate_normals_radius(xs, 0.5, want_cov=True),
             (30, 0.5): lambda: ctx.estimate_normals(xs, 30, 0.5, want_cov=True)}
    for (max_nn, radius), engine_call in modes.items():
        want = engine_call()[2].to(torch.float32).cpu()
        ctx.check()
        for dev in ("CUDA:0", "CPU:0"):
            pcd = cloud(o3d, src, dev)
            pcd.point["normals"] = o3d.Tensor(torch.ones((src.shape[0], 3))).to(o3d.Device(dev))
            assert pcd.estimate_covariances(max_nn, radius) is pcd
            cov = pcd.point["covariances"]
            assert cov.dtype == torch.float32 and cov.shape == (src.shape[0], 3, 3) and cov.device == o3d.Device(dev)
            assert torch.equal(cov.t.cpu(), want)
            assert torch.equal(pcd.point["normals"].t.cpu(), torch.ones((src.shape[0], 3)))   # normals left alone
    default = cloud(o3d, src, "CUDA:0").estimate_covariances()
    assert torch.equal(default.point["covariances"].t.cpu(), modes[(20, None)]()[2].to(torch.float32).cpu())
    for dev in ("CUDA:0", "CPU:0"):
        empty = cloud(o3d, np.zeros((0, 3), np.float32), dev).estimate_covariances()
        assert empty.point["covariances"].shape == (0, 3, 3) and empty.point["covariances"].device == o3d.Device(dev)
    with pytest.raises(ValueError):
        cloud(o3d, src, "CUDA:0").estimate_covariances(None, None)


def test_carrier(env, recovery):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    src, tgt, T_true, cs, ct = recovery
    crit = o3dreg.ICPConvergenceCriteria(max_iteration=12)
    est = o3dreg.TransformationEstimationForGeneralizedICP()
    results = {}
    for dev in ("CUDA:0", "CPU:0"):
        s, t = cloud(o3d, src, dev, cs), cloud(o3d, tgt, dev, ct.double())      # any float dtype
        res = o3dreg.icp(s, t, 1.0, np.eye(4), est, crit)
        T = res.transformation
        assert T.device == o3d.Device("CPU:0") and T.dtype == torch.float64 and T.shape == (4, 4)
        c = res.correspondences_
        assert c.dtype == torch.int64 and c.device == o3d.Device(dev) and c.shape == (src.shape[0],)
        results[dev] = (T.numpy(), c.t.cpu().numpy(), res.fitness, res.inlier_rmse, res.converged, res.num_iterations)
    a, b = results["CUDA:0"], results["CPU:0"]
    assert all(np.array_equal(x, y) for x, y in zip(a[:2], b[:2])) and a[2:] == b[2:] and a[5] > 1
    T, stats, info, corr = run(env["ctx"], src, tgt, cs, ct, 1.0, max_iteration=12)
    assert np.array_equal(a[0], T) and np.array_equal(a[1], corr)
    dt, angle = pose_error(a[0], T_true)
    assert dt < 0.02 and angle < 0.2
    # missing covariances: estimate_covariances() defaults on the clouds, which stay as they were
    bare_s, bare_t = cloud(o3d, src, "CUDA:0"), cloud(o3d, tgt, "CUDA:0")
    res = o3dreg.icp(bare_s, bare_t, 1.0, None, est, crit)
    assert "covariances" not in bare_s.point and "covariances" not in bare_t.point
    ref = o3dreg.icp(bare_s.clone().estimate_covariances(), bare_t.clone().estimate_covariances(), 1.0, None, est, crit)
    assert np.array_equal(res.transformation.numpy(), ref.transformation.numpy())
    assert torch.equal(res.correspondences_.t, ref.correspondences_.t)
    eps = o3dreg.icp(bare_s, bare_t, 1.0, None, o3dreg.TransformationEstimationForGeneralizedICP(0.2), crit)
    assert not np.array_equal(eps.transformation.numpy(), res.transformation.numpy())


def test_carrier_voxel_size_and_errors(env, recovery):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    src, tgt, _, cs, ct = recovery
    est = o3dreg.TransformationEstimationForGeneralizedICP()
    s, t = cloud(o3d, src, "CUDA:0", cs), cloud(o3d, tgt, "CUDA:0", ct)
    crit = o3dreg.ICPConvergenceCriteria(max_iteration=6)
    a = o3dreg.icp(s, t, 1.0, None, est, crit, voxel_size=0.3)
    ds, dt = cloud(o3d, src, "CUDA:0").voxel_down_sample(0.3), cloud(o3d, tgt, "CUDA:0").voxel_down_sample(0.3)
    b = o3dreg.icp(ds.estimate_covariances(), dt.estimate_covariances(), 1.0, None, est, crit)
    assert np.array_equal(a.transformation.numpy(), b.transformation.numpy())
    assert torch.equal(a.correspondences_.t, b.correspondences_.t) and a.correspondences_.shape[0] < src.shape[0]
    assert s.point["covariances"].shape == (src.shape[0], 3, 3)
    empty = cloud(o3d, np.zeros((0, 3), np.float32), "CUDA:0")
    for x, y in ((empty, t), (s, empty)):
        with pytest.raises(RuntimeError):
            o3dreg.icp(x, y, 1.0, estimation_method=est)
    with pytest.raises(RuntimeError, match="max_correspondence_distance"):
        o3dreg.icp(s, cloud(o3d, tgt + np.float32(100.0), "CUDA:0"), 1.0, estimation_method=est)
    bad = ct.clone()
    bad[:] = torch.diag(torch.tensor([1.0, 2.0, float("nan")])).cuda()
    with pytest.raises(RuntimeError, match="positive definite"):
        o3dreg.icp(s, cloud(o3d, tgt, "CUDA:0", bad), 1.0, estimation_method=est)
    with pytest.raises(ValueError, match="covariances"):
        o3dreg.icp(s, cloud(o3d, tgt, "CUDA:0", ct[:10]), 1.0, estimation_method=est)
    with pytest.raises(NotImplementedError):
        o3dreg.icp(s, t, 1.0, estimation_method=est, callback_after_iteration=lambda d: None)
    with pytest.raises(ValueError):
        o3dreg.icp(s, t, 0.0, estimation_method=est)
    for eps in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="epsilon"):
            o3dreg.TransformationEstimationForGeneralizedICP(eps)
    with pytest.raises(NotImplementedError):
        o3dreg.TransformationEstimationForGeneralizedICP(kernel=object())
