"""Statistical outlier removal and normal estimation with 64 < k <= APC_MAX_NEIGHBORS (1024): the wide
kernels (k_knn_query_wide / k_knn_stragglers_wide, k_normals_wide) against the oracle, the dispatch that
keeps k <= 64 on the existing kernels, the cap, the fused pipeline and its graph, and the node."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=300_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


def outlier_cloud(env):
    """~18 k voxel centroids of a scan plus isolated far points (the coarse levels and the brute-force
    straggler kernel run); small enough for the oracle's P x (k + 16) candidate array at k = 1024."""
    from oracle import filters, voxel
    synth = env["synth"]
    scan = synth.lidar_scan(seed=5, n_beams=20, n_az=1024, nan_frac=0.0)
    p = scan["positions"][filters.crop_mask(scan["positions"], [-60, -60, -20], [60, 60, 20], False, filters.CROP_OPEN3D)]
    p = voxel.voxel_down_sample(p, 0.1, None, fixed=True)["positions"]
    far = np.array([[300.0, 300.0, 50.0], [-250.0, 40.0, 90.0], [1000.0, -900.0, 5.0]], np.float32)
    return np.ascontiguousarray(np.concatenate([p, far]), dtype=np.float32)


def assert_statistical(ctx, xyzi, host, k, ratio, brute=False):
    from oracle import outliers
    mask, avg, stats = ctx.statistical_outliers(xyzi, k, ratio)
    ctx.check()
    ref_mask, ref_avg = outliers.statistical_mask(host, k, ratio, brute=brute)
    assert np.array_equal(avg.cpu().numpy().view(np.uint32), ref_avg.view(np.uint32))   # float32 means, bit-exact
    if host.shape[0] >= 2:
        mu, sigma, thr = outliers.statistical_threshold(ref_avg, ratio)
        st = stats.cpu().numpy()
        assert st[0] == mu and st[1] == sigma and st[2] == thr
    assert np.array_equal(mask.cpu().numpy().astype(bool), ref_mask)


@pytest.mark.parametrize("k", [65, 100, 256, 1024])
def test_statistical_wide_parity(env, k):
    ctx = env["ctx"]
    host = outlier_cloud(env)
    xyzi = to_xyzi(host)
    for _ in range(2):                                               # the tables clean themselves
        assert_statistical(ctx, xyzi, host, k, 2.0)


def test_statistical_wide_tiny_clouds(env):
    """Fewer points than k: k_eff = min(k, n), down to a single point."""
    ctx = env["ctx"]
    host = outlier_cloud(env)
    for n in (1, 7, 100):
        assert_statistical(ctx, to_xyzi(host[:n].copy()), host[:n], 200, 2.0, brute=True)


def launched(ctx, fn):
    ctx.profile(True)
    try:
        fn()
        ctx.check()
        return set(ctx.profile_report())
    finally:
        ctx.profile(False)


def test_dispatch_keeps_k_up_to_64_on_the_existing_kernels(env):
    ctx = env["ctx"]
    xyzi = to_xyzi(outlier_cloud(env))
    names = launched(ctx, lambda: ctx.statistical_outliers(xyzi, 64, 2.0))
    assert "k_knn_query" in names and "k_knn_stragglers" in names
    assert "k_knn_query_wide" not in names and "k_knn_stragglers_wide" not in names
    names = launched(ctx, lambda: ctx.statistical_outliers(xyzi, 65, 2.0))
    assert "k_knn_query_wide" in names and "k_knn_stragglers_wide" in names
    assert "k_knn_query" not in names and "k_knn_stragglers" not in names
    kernels = {"k_normals_cov", "k_normals_query", "k_normals_wide"}
    for max_nn, want in ((32, "k_normals_cov"), (64, "k_normals_query"), (65, "k_normals_wide")):
        names = launched(ctx, lambda: ctx.estimate_normals(xyzi, max_nn, 0.5))
        assert names & kernels == {want}, (max_nn, names)


def test_cap_is_refused_and_the_context_stays_usable(env):
    capi, ctx = env["capi"], env["ctx"]
    host = outlier_cloud(env)
    xyzi = to_xyzi(host)
    assert capi.APC_MAX_NEIGHBORS == 1024
    with pytest.raises(capi.ApcError) as e:
        ctx.statistical_outliers(xyzi, capi.APC_MAX_NEIGHBORS + 1, 2.0)
    assert e.value.code == capi.APC_ERR_BAD_ARG and "1024" in str(e.value)
    with pytest.raises(capi.ApcError) as e:
        ctx.estimate_normals(xyzi, capi.APC_MAX_NEIGHBORS + 1, 0.5)
    assert e.value.code == capi.APC_ERR_BAD_ARG and "1024" in str(e.value)
    assert_statistical(ctx, xyzi, host, 20, 2.0)


def dense_surface(seed=5):
    """20 k points on a wavy 4 m x 4 m surface (~1000 points per m^2) and a wall: neighbourhoods of
    hundreds of points within half a metre, so max_nn binds; one exact duplicate for distance ties."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-2.0, 2.0, size=(2, 16000))
    ground = np.stack([u, v, 0.1 * np.sin(2.0 * u) * np.cos(3.0 * v)], 1)
    a, b = rng.uniform(-2.0, 2.0, 4000), rng.uniform(0.0, 1.0, 4000)
    wall = np.stack([np.full(4000, 1.5), a, b], 1)
    p = np.concatenate([ground, wall]).astype(np.float32)
    p[0] = p[1]
    return p


@pytest.mark.parametrize("max_nn,radius", [(65, 0.2), (100, 0.25), (512, 0.5)])
def test_normals_wide_parity(env, max_nn, radius):
    from oracle import normals as onrm
    from test_gpu_normals import check_normals
    ctx = env["ctx"]
    p = dense_surface()
    ref, cnt_ref, cov_ref = onrm.estimate_normals(p, radius, max_nn)
    assert (cnt_ref == max_nn).mean() >= 0.25                        # the cap binds
    for _ in range(2):                                               # the grid cleans itself between calls
        got, cnt, cov = ctx.estimate_normals(to_xyzi(p), max_nn, radius, want_counts=True, want_cov=True)
        ctx.check()
        assert np.array_equal(cnt.cpu().numpy(), cnt_ref)            # neighbourhood sizes, bit-exact
        cov = cov.cpu().numpy()
        big = np.abs(cov_ref).max(axis=(1, 2), keepdims=True)
        assert np.all(np.abs(cov - cov_ref) <= 1e-9 * big + 1e-18)
        check_normals(got.cpu().numpy(), cov_ref, ref)


def test_fused_pipeline_and_graph_with_wide_k(env):
    """voxel + statistical (k = 100) + normals (max_nn = 100) + ground through apc_pipeline_run_maps,
    against the oracle pipeline; the same configuration captured as a graph replays the same bytes."""
    from oracle import pipeline as opipe
    from test_gpu_normals import check_normals
    ctx, engine, capi, synth = env["ctx"], env["engine"], env["capi"], env["synth"]
    msg = synth.pack_cloud(synth.lidar_scan(seed=31, n_beams=32, n_az=1024), "xyzirt22")
    n = msg.width
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, n, torch.frombuffer(bytearray(msg.data), dtype=torch.uint8).cuda())
    crop = dict(min=[-60.0, -60.0, -20.0], max=[60.0, 60.0, 20.0], invert=False, mode=capi.CROP_OPEN3D)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True, crop=crop)
    stages = dict(voxel_size=0.1, statistical=dict(nb_neighbors=100, std_ratio=2.0), normals=dict(radius=0.5, max_nn=100),
                  ground=dict(distance_threshold=0.2, ransac_n=5, num_iterations=100, probability=0.99, seed=7))
    pcfg = engine.make_pipeline_cfg(fcfg, **stages)
    out, cnt, _, maps = ctx.pipeline_run_maps([desc], pcfg)
    ctx.check()
    cfg = opipe.default_config()
    cfg.update(crop=crop, **stages)
    ref = opipe.preprocess(msg, cfg)
    c = cnt.cpu().numpy()
    k = int(c[capi.CNT_OUTPUT])
    assert c[capi.CNT_STATUS] == 0 and k == ref["positions"].shape[0]
    assert int(c[capi.CNT_AFTER_STAT]) == int(ref["statistical_mask"].sum())
    rows = out[:k].cpu().numpy()
    assert np.array_equal(rows[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    assert np.array_equal(rows[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    nrm = maps["normals"][:k].cpu().numpy()
    keep = np.ones(ref["normal_counts"].size, dtype=bool)
    keep[ref["ground_inliers"]] = False
    few = ref["normal_counts"][keep] < 3
    assert np.array_equal(nrm[few], np.tile(np.array([0, 0, 1], np.float32), (int(few.sum()), 1)))
    check_normals(nrm[~few], ref["normal_cov"][~few], ref["normals"][~few])
    g_out = torch.zeros((n, 4), device="cuda")
    g_cnt = torch.zeros(8, dtype=torch.int32, device="cuda")
    g_plane = torch.zeros(8, dtype=torch.float64, device="cuda")
    g_maps = {"normals": torch.zeros((n, 3), device="cuda")}
    g = ctx.capture_pipeline([desc], pcfg, g_out, g_cnt, g_plane, maps=g_maps)
    for _ in range(2):
        ctx.launch_graph(g)
        ctx.check()
        assert np.array_equal(g_cnt.cpu().numpy(), c)
        assert np.array_equal(g_out[:k].cpu().numpy().view(np.uint32), rows.view(np.uint32))
        assert np.array_equal(g_maps["normals"][:k].cpu().numpy().view(np.uint32), nrm.view(np.uint32))


NODE_WIDE = {"use_gpu": True, "voxel_size": 0.1, "remove_statistical_outliers": True,
             "remove_statistical_outliers.nb_neighbors": 100, "estimate_normals.max_neighbors": 100,
             "estimate_normals.search_radius": 0.5}


def test_node_publishes_with_wide_neighbourhoods():
    """nb_neighbors = 100 and max_neighbors = 100: the fused ('auto') and the staged ('false') path each
    publish the frame, byte-identical to each other, rows and normals matching the oracle."""
    from oracle import pc2
    from test_gpu_dropin import make_node, oracle_published, scan_msg
    from test_gpu_normals import check_normals
    _, msg = scan_msg("xyzi16", seed=45, n_beams=32, n_az=1024)
    outs = {}
    for fused in ("auto", "false"):
        node = make_node(dict(NODE_WIDE, fused_pipeline=fused))
        node.callback(msg)
        assert len(node.pointcloud_pub.messages) == 1, f"callback dropped the frame ({fused})"
        outs[fused] = node.pointcloud_pub.messages[0]
    a, b = outs["auto"], outs["false"]
    assert a.width == b.width and a.point_step == b.point_step and bytes(a.data) == bytes(b.data)
    ref, _ = oracle_published(msg, dict(voxel_size=0.1, statistical=dict(nb_neighbors=100, std_ratio=2.0),
                                        normals=dict(radius=0.5, max_nn=100)))
    arr = np.frombuffer(a.data, dtype=pc2.dtype_from_fields(a.fields, a.point_step))
    assert a.width == ref["positions"].shape[0]
    assert np.array_equal(np.stack([arr["x"], arr["y"], arr["z"]], 1).view(np.uint32), ref["positions"].view(np.uint32))
    nrm = np.stack([arr["normal_x"], arr["normal_y"], arr["normal_z"]], 1)
    few = ref["normal_counts"] < 3
    assert np.array_equal(nrm[few], np.tile(np.array([0, 0, 1], np.float32), (int(few.sum()), 1)))
    check_normals(nrm[~few], ref["normal_cov"][~few], ref["normals"][~few])


def test_node_reconfigure_to_wide_neighbourhoods():
    from autodriver_pointcloud_preprocessor_b200._ros_compat import Parameter
    from test_gpu_dropin import make_node, scan_msg
    _, msg = scan_msg("xyzi16", seed=46)
    node = make_node({"use_gpu": True, "voxel_size": 0.1, "remove_statistical_outliers": True,
                      "estimate_normals.search_radius": 0.5})
    node.callback(msg)
    assert node.frame_count == 1
    first = node.pointcloud_pub.messages[-1]
    ok = node.parameter_change_callback([Parameter("remove_statistical_outliers.nb_neighbors", value=100),
                                         Parameter("estimate_normals.max_neighbors", value=100)])
    assert ok.successful and node.remove_statistical_outliers_nb_neighbors == 100
    node.callback(msg)
    assert node.frame_count == 2, "callback dropped the frame after the reconfigure"
    second = node.pointcloud_pub.messages[-1]              # (the publisher keeps the newest message only)
    assert second is not first and second.width > 0
