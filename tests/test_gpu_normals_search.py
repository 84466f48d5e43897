"""estimate_normals with one search bound: KNN (max_nn only; apc_estimate_normals_knn, kernels k_normals_knn /
k_normals_knn_stragglers) and radius (radius only; apc_estimate_normals_radius, k_normals_radius) against
the CPU references (test_oracle_normals_search.knn_estimate_normals; oracle/normals.py with max_nn=None), their
determinism, the grids they share with the other neighbour stages, the argument checks and the carrier's choice
of search."""
import numpy as np
import pytest

from test_gpu_normals import check_normals
from test_gpu_wide_neighbors import outlier_cloud
from test_oracle_normals_search import knn_estimate_normals

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

Z = np.array([0, 0, 1], np.float32)


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=300_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


@pytest.fixture(scope="module")
def knn_cloud(env):
    """~18 k voxel centroids of a scan, an exact duplicate (a distance tie) and isolated far points (the coarse
    levels and the brute-force straggler kernel run)."""
    p = outlier_cloud(env).copy()
    p[0] = p[1]
    return p


def dense_patch(seed=9):
    """6 000 points on a wavy 1.6 m x 1.6 m surface (~2 300 points per m^2) and a wall, an exact duplicate, and
    three far points with 0 and 1 neighbours: radius neighbourhoods of more than a thousand points."""
    rng = np.random.default_rng(seed)
    u, v = rng.uniform(-0.8, 0.8, size=(2, 5000))
    ground = np.stack([u, v, 0.05 * np.sin(4.0 * u) * np.cos(5.0 * v)], 1)
    a, b = rng.uniform(-0.8, 0.8, 1000), rng.uniform(0.0, 0.4, 1000)
    wall = np.stack([np.full(1000, 0.7), a, b], 1)
    far = np.array([[20.0, 20.0, 5.0], [20.0, 20.05, 5.0], [-30.0, 10.0, 2.0]])
    p = np.concatenate([ground, wall, far]).astype(np.float32)
    p[0] = p[1]
    return p


def assert_cov(cov, cov_ref, extra=0.0):
    big = np.abs(cov_ref).max(axis=(1, 2), keepdims=True)
    assert np.all(np.abs(cov - cov_ref) <= 1e-9 * big + extra + 1e-18)


def assert_parity(got, cnt, cov, ref, cnt_ref, cov_ref, extra=0.0):
    got, cnt, cov = got.cpu().numpy(), cnt.cpu().numpy(), cov.cpu().numpy()
    assert np.array_equal(cnt, cnt_ref)                              # neighbourhood sizes, bit-exact
    assert_cov(cov, cov_ref, extra)
    few = cnt_ref < 3
    assert np.array_equal(got[few], np.tile(Z, (int(few.sum()), 1)))
    if (~few).sum() > 50:
        check_normals(got[~few], cov_ref[~few], ref[~few])


@pytest.mark.parametrize("k", [1, 2, 3, 30, 64, 65, 100, 1024])
def test_knn_parity(env, knn_cloud, k):
    ctx, p = env["ctx"], knn_cloud
    ref, cnt_ref, cov_ref = knn_estimate_normals(p, k)
    assert np.all(cnt_ref == min(k, p.shape[0]))
    for _ in range(2):                                               # the grid cleans itself between calls
        got, cnt, cov = ctx.estimate_normals_knn(to_xyzi(p), k, want_counts=True, want_cov=True)
        ctx.check()
        assert_parity(got, cnt, cov, ref, cnt_ref, cov_ref)


@pytest.mark.parametrize("n", [1, 2, 3, 7])
def test_knn_tiny_clouds(env, knn_cloud, n):
    """Fewer points than max_nn, tens of metres from the origin: the grid's cells are sized to key them."""
    from oracle import outliers
    p = knn_cloud[1000:1000 + n] + np.float32([40.0, -25.0, 3.0])
    ref, cnt_ref, cov_ref = knn_estimate_normals(p, 30)
    got, cnt, cov = env["ctx"].estimate_normals_knn(to_xyzi(p), 30, want_counts=True, want_cov=True)
    env["ctx"].check()
    assert np.array_equal(cnt.cpu().numpy(), np.full(n, n))
    assert_cov(cov.cpu().numpy(), cov_ref)
    g = got.cpu().numpy()
    if n < 3:
        assert np.array_equal(g, np.tile(Z, (n, 1)))
    else:                                                            # a few points: possibly degenerate, so the
        n64 = g.astype(np.float64)                                   # eigen-residual, not the direction
        assert np.allclose(np.linalg.norm(n64, axis=1), 1.0, atol=1e-5)
        w = np.linalg.eigvalsh(cov_ref)
        rq = np.einsum("ni,nij,nj->n", n64, cov_ref, n64)
        assert np.all(np.abs(rq - w[:, 0]) <= 1e-4 * w[:, 2] + 1e-12)
    mask, avg, _ = env["ctx"].statistical_outliers(to_xyzi(p), 30, 2.0)   # the same grid serves the statistical stage
    env["ctx"].check()
    assert mask.all() and np.array_equal(avg.cpu().numpy(), outliers.knn_avg_distance_brute(p, 30))


@pytest.mark.parametrize("radius", [0.1, 0.45])
def test_radius_parity(env, radius):
    from oracle import normals as onrm
    ctx, p = env["ctx"], dense_patch()
    ref, cnt_ref, cov_ref = onrm.estimate_normals(p, radius, None)
    assert (cnt_ref < 3).any()
    if radius > 0.4:
        assert (cnt_ref > 1024).mean() > 0.2                         # beyond any max_nn the hybrid search takes
    r2 = float(np.float32(radius)) ** 2
    for _ in range(2):
        got, cnt, cov = ctx.estimate_normals_radius(to_xyzi(p), radius, want_counts=True, want_cov=True)
        ctx.check()
        assert_parity(got, cnt, cov, ref, cnt_ref, cov_ref, extra=1e-11 * r2)   # fixed point: 2^-41 r per term


def bits(*ts):
    return [t.cpu().numpy().copy().view(np.uint8) for t in ts]


def test_determinism_and_permutation(env, knn_cloud):
    ctx = env["ctx"]
    xyzi = to_xyzi(knn_cloud)
    a = bits(*ctx.estimate_normals_knn(xyzi, 100, want_counts=True, want_cov=True))
    b = bits(*ctx.estimate_normals_knn(xyzi, 100, want_counts=True, want_cov=True))
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    p = dense_patch()
    got, cnt, cov = ctx.estimate_normals_radius(to_xyzi(p), 0.45, want_counts=True, want_cov=True)
    again = ctx.estimate_normals_radius(to_xyzi(p), 0.45, want_counts=True, want_cov=True)
    assert all(np.array_equal(x, y) for x, y in zip(bits(got, cnt, cov), bits(*again)))
    # the fixed-point moments do not depend on the order of the points: the permuted cloud gives the permuted bits
    perm = np.random.default_rng(1).permutation(p.shape[0])
    g2, c2, v2 = ctx.estimate_normals_radius(to_xyzi(p[perm]), 0.45, want_counts=True, want_cov=True)
    ctx.check()
    assert np.array_equal(c2.cpu().numpy(), cnt.cpu().numpy()[perm])
    assert np.array_equal(g2.cpu().numpy().view(np.uint32), got.cpu().numpy()[perm].view(np.uint32))
    assert np.array_equal(v2.cpu().numpy().view(np.uint64), cov.cpu().numpy()[perm].view(np.uint64))


def test_kernels_by_name(env, knn_cloud):
    ctx = env["ctx"]
    xyzi = to_xyzi(knn_cloud)
    for fn, want in ((lambda: ctx.estimate_normals_knn(xyzi, 30), {"k_normals_knn", "k_normals_knn_stragglers"}),
                     (lambda: ctx.estimate_normals_radius(xyzi, 0.5), {"k_normals_radius"})):
        ctx.profile(True)
        try:
            fn()
            ctx.check()
            names = set(ctx.profile_report())
        finally:
            ctx.profile(False)
        assert want <= names and "k_normals_eigen" in names and "k_grid_clean" in names


def test_shared_scratch_interleaved(env, knn_cloud):
    """Hybrid, KNN, radius and statistical calls share the context's grids: interleaved on one context, each
    gives exactly what it gives on a context of its own."""
    engine, ctx = env["engine"], env["ctx"]
    xyzi = to_xyzi(knn_cloud)
    calls = {
        "hybrid": lambda c: c.estimate_normals(xyzi, 30, 0.5, want_counts=True, want_cov=True),
        "knn": lambda c: c.estimate_normals_knn(xyzi, 65, want_counts=True, want_cov=True),
        "radius": lambda c: c.estimate_normals_radius(xyzi, 0.5, want_counts=True, want_cov=True),
        "statistical": lambda c: c.statistical_outliers(xyzi, 20, 2.0),
        "knn30": lambda c: c.estimate_normals_knn(xyzi, 30, want_counts=True, want_cov=True),
    }
    alone = {}
    for name, fn in calls.items():
        c = engine.Context(max_points=knn_cloud.shape[0])
        alone[name] = bits(*fn(c))
        c.check()
        c.close()
    for name in ("hybrid", "knn", "radius", "statistical", "knn", "knn30", "hybrid", "statistical", "radius", "knn30"):
        got = bits(*calls[name](ctx))
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(got, alone[name])), name


def test_n_dev_below_n_max(env, knn_cloud):
    ctx = env["ctx"]
    m = 5000
    xyzi = to_xyzi(knn_cloud)
    n_dev = torch.tensor([m], dtype=torch.int32, device="cuda")
    head = to_xyzi(knn_cloud[:m].copy())
    for fn, arg in ((ctx.estimate_normals_knn, 100), (ctx.estimate_normals_radius, 0.5)):
        got, cnt, cov = fn(xyzi, arg, want_counts=True, want_cov=True, n_dev=n_dev)
        ref = fn(head, arg, want_counts=True, want_cov=True)
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(bits(got[:m], cnt[:m], cov[:m]), bits(*ref)))
        assert not got[m:].any() and not cnt[m:].any()
    assert np.all(ctx.estimate_normals_knn(xyzi, 100, want_counts=True, n_dev=n_dev)[1][:m].cpu().numpy() == 100)


def test_bad_arguments_and_recovery(env, knn_cloud):
    capi, ctx = env["capi"], env["ctx"]
    xyzi = to_xyzi(knn_cloud)
    before = bits(*ctx.estimate_normals_knn(xyzi, 30, want_counts=True, want_cov=True))
    for k in (0, capi.APC_MAX_NEIGHBORS + 1):
        with pytest.raises(capi.ApcError) as e:
            ctx.estimate_normals_knn(xyzi, k)
        assert e.value.code == capi.APC_ERR_BAD_ARG and "1024" in str(e.value)
    for r in (0.0, -0.5, float("nan"), float("inf")):
        with pytest.raises(capi.ApcError) as e:
            ctx.estimate_normals_radius(xyzi, r)
        assert e.value.code == capi.APC_ERR_BAD_ARG and "radius" in str(e.value)
    after = bits(*ctx.estimate_normals_knn(xyzi, 30, want_counts=True, want_cov=True))
    ctx.check()
    assert all(np.array_equal(x, y) for x, y in zip(before, after))


def test_carrier_selects_the_search(env):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from oracle import normals as onrm
    from oracle import voxel
    scan = env["synth"].lidar_scan(seed=8, n_beams=16, n_az=512, nan_frac=0.0)
    p = voxel.voxel_down_sample(scan["positions"], 0.2, None, fixed=True)["positions"]
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(p).cuda())
    pcd.estimate_normals()                                           # Open3D's default call: KNN, max_nn = 30
    ref, cnt, cov = knn_estimate_normals(p, 30)
    assert np.all(cnt == 30)
    check_normals(pcd.point.normals.cpu().numpy(), cov, ref)
    pcd.estimate_normals(max_nn=None, radius=0.5)
    ref, cnt, cov = onrm.estimate_normals(p, 0.5, None)
    few = cnt < 3
    got = pcd.point.normals.cpu().numpy()
    assert np.array_equal(got[few], np.tile(Z, (int(few.sum()), 1)))
    check_normals(got[~few], cov[~few], ref[~few])
    with pytest.raises(ValueError):
        pcd.estimate_normals(max_nn=None, radius=None)


def test_carrier_knn_full_size_properties(env):
    """C2 size (262 144 points -> ~200 k voxels), KNN with k = 30: unit normals everywhere, +-z on the
    synthetic ground plane (z = -1.8)."""
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from oracle import voxel
    scan = env["synth"].lidar_scan(seed=2, n_beams=128, n_az=2048, nan_frac=0.0)
    p = voxel.voxel_down_sample(scan["positions"], 0.1, None, fixed=True)["positions"]
    assert p.shape[0] > 150_000
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(p).cuda())
    pcd.estimate_normals()
    g = pcd.point.normals.cpu().numpy()
    assert np.allclose(np.linalg.norm(g.astype(np.float64), axis=1), 1.0, atol=1e-5)
    ground = (np.abs(p[:, 2] + 1.8) < 0.03) & (np.hypot(p[:, 0], p[:, 1]) < 15)
    assert ground.sum() > 1000
    assert np.median(np.abs(g[ground][:, 2])) > 0.99
