"""cluster_dbscan on the GPU (apc_cluster_dbscan; kernels k_dbscan_core / _union / _roots / _label) against the
CPU oracle (oracle/dbscan.py): bit-exact labels, cluster counts and neighbour counts, the radius predicate shared
with radius outlier removal, determinism, n_dev, the grid shared with the other neighbour stages, the argument
checks and the carrier."""
import numpy as np
import pytest

from test_gpu_normals_search import dense_patch
from test_oracle_dbscan import border_case

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


def c2_voxels(synth, seed=4):
    """A C2-shaped scan (128 x 2048) voxelised at 0.1 m."""
    from oracle import voxel
    scan = synth.lidar_scan(seed=seed, n_beams=128, n_az=2048, nan_frac=0.0)
    return voxel.voxel_down_sample(scan["positions"], 0.1, None, fixed=True)["positions"]


@pytest.fixture(scope="module")
def nonground(env):
    """The non-ground points of the C2-shaped scan: segment_plane -> select_by_index(inliers, invert=True)."""
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(c2_voxels(env["synth"])).cuda())
    _, inliers = pcd.segment_plane(distance_threshold=0.2, ransac_n=3, num_iterations=200, seed=3)
    rest = pcd.select_by_index(inliers, invert=True)
    p = np.ascontiguousarray(rest.point.positions.cpu().numpy(), dtype=np.float32)
    assert 30_000 < p.shape[0] < 200_000
    return p


def run(ctx, p, eps, min_points, **kw):
    labels, n_clusters, counts = ctx.cluster_dbscan(to_xyzi(p), eps, min_points, want_counts=True, **kw)
    ctx.check()
    return labels.cpu().numpy(), int(n_clusters.item()), counts.cpu().numpy()


def assert_oracle(got, p, eps, min_points):
    from oracle import dbscan as odb
    labels, n_clusters, counts = got
    ref, n_ref, cnt_ref, _ = odb.dbscan(p, eps, min_points)
    assert np.array_equal(counts, cnt_ref.astype(np.int32))
    assert n_clusters == n_ref
    assert np.array_equal(labels, ref)
    return ref


@pytest.mark.parametrize("eps", [0.3, 0.5, 1.0])
@pytest.mark.parametrize("min_points", [1, 5, 10])
def test_parity_c2_nonground(env, nonground, eps, min_points):
    ref = assert_oracle(run(env["ctx"], nonground, eps, min_points), nonground, eps, min_points)
    if min_points > 1:
        assert (ref == -1).any() and ref.max() > 10


@pytest.mark.parametrize("min_points", [10, 1200])
def test_parity_dense_patch(env, min_points):
    """Neighbourhoods of more than 1024 points; at 1200 some points are core, some border, some noise."""
    p = dense_patch()
    got = run(env["ctx"], p, 0.45, min_points)
    assert got[2].max() > 1024
    ref = assert_oracle(got, p, 0.45, min_points)
    if min_points == 1200:
        core = got[2] >= min_points
        assert core.any() and (~core & (ref >= 0)).any() and (ref == -1).any()


def test_parity_border_case(env):
    p, eps, min_points = border_case()
    got = run(env["ctx"], p, eps, min_points)
    assert list(got[0]) == [0, 0, 0, 0, 1, 1, 1, 1, 0]
    assert_oracle(got, p, eps, min_points)


def test_parity_far_from_origin(env, nonground):
    p = np.ascontiguousarray(nonground[:20_000] + np.float32([40.0, -35.0, 6.0]))
    assert_oracle(run(env["ctx"], p, 0.5, 5), p, 0.5, 5)


def test_one_point_and_too_few_points(env, nonground):
    ctx = env["ctx"]
    one = nonground[:1].copy()
    labels, n, counts = run(ctx, one, 0.5, 1)
    assert list(labels) == [0] and n == 1 and list(counts) == [1]
    labels, n, counts = run(ctx, one, 0.5, 2)
    assert list(labels) == [-1] and n == 0
    p = nonground[:500].copy()
    labels, n, counts = run(ctx, p, 1.0, 501)
    assert np.all(labels == -1) and n == 0
    assert_oracle((labels, n, counts), p, 1.0, 501)


def test_counts_are_the_radius_outlier_counts(env, nonground):
    ctx = env["ctx"]
    xyzi = to_xyzi(nonground)
    for eps, min_points in ((0.3, 5), (1.0, 10)):
        labels, _, counts = ctx.cluster_dbscan(xyzi, eps, min_points, want_counts=True)
        mask, rc = ctx.radius_outliers(xyzi, min_points, eps, want_counts=True)
        ctx.check()
        counts = counts.cpu().numpy()
        assert np.array_equal(counts, rc.cpu().numpy())
        assert np.array_equal(counts >= min_points, mask.cpu().numpy().astype(bool))
        # without counts, the core test stops early: the labels do not change
        again, _, none = ctx.cluster_dbscan(xyzi, eps, min_points)
        assert none is None and torch.equal(again, labels)


def test_determinism_and_permutation(env, nonground):
    from oracle import dbscan as odb
    ctx = env["ctx"]
    runs = [run(ctx, nonground, 0.5, 5) for _ in range(3)]
    for r in runs[1:]:
        assert np.array_equal(r[0], runs[0][0]) and r[1] == runs[0][1] and np.array_equal(r[2], runs[0][2])
    perm = np.random.default_rng(2).permutation(nonground.shape[0])
    q = np.ascontiguousarray(nonground[perm])
    got = run(ctx, q, 0.5, 5)
    ref = assert_oracle(got, q, 0.5, 5)
    # the clusters of the core points and the noise are the permuted ones (a border point may change cluster:
    # it takes the lowest id, and the ids follow the new order)
    base = runs[0][0][perm]
    core = got[2] >= 5
    assert np.array_equal(base == -1, ref == -1)
    pairs = np.unique(np.stack([base[core], ref[core]], 1), axis=0)
    assert np.unique(pairs[:, 0]).size == pairs.shape[0] == np.unique(pairs[:, 1]).size


def test_n_dev_below_n_max(env, nonground):
    ctx = env["ctx"]
    m = 7000
    n_dev = torch.tensor([m], dtype=torch.int32, device="cuda")
    labels, n, counts = run(ctx, nonground, 0.5, 5, n_dev=n_dev)
    head = run(ctx, np.ascontiguousarray(nonground[:m]), 0.5, 5)
    assert np.array_equal(labels[:m], head[0]) and n == head[1] and np.array_equal(counts[:m], head[2])
    assert np.all(labels[m:] == -1) and not counts[m:].any()


def bits(*ts):
    return [t.cpu().numpy().copy().view(np.uint8) for t in ts if t is not None]


def test_shared_scratch_interleaved(env, nonground):
    """DBSCAN, radius outliers, radius normals and statistical outliers share the context's grids: interleaved on
    one context, each gives exactly what it gives on a context of its own."""
    engine, ctx = env["engine"], env["ctx"]
    xyzi = to_xyzi(nonground)
    calls = {
        "dbscan": lambda c: c.cluster_dbscan(xyzi, 0.5, 5, want_counts=True),
        "dbscan_nocount": lambda c: c.cluster_dbscan(xyzi, 0.3, 10),
        "radius": lambda c: c.radius_outliers(xyzi, 5, 0.5, want_counts=True),
        "normals_radius": lambda c: c.estimate_normals_radius(xyzi, 0.5, want_counts=True, want_cov=True),
        "statistical": lambda c: c.statistical_outliers(xyzi, 20, 2.0),
    }
    alone = {}
    for name, fn in calls.items():
        c = engine.Context(max_points=nonground.shape[0])
        alone[name] = bits(*fn(c))
        c.check()
        c.close()
    for name in ("dbscan", "radius", "dbscan", "normals_radius", "dbscan_nocount", "statistical", "dbscan", "radius",
                 "normals_radius", "dbscan_nocount"):
        got = bits(*calls[name](ctx))
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(got, alone[name])), name


def test_bad_arguments_and_recovery(env, nonground):
    capi, ctx = env["capi"], env["ctx"]
    p = np.ascontiguousarray(nonground[:5000])
    before = run(ctx, p, 0.5, 5)
    for eps in (0.0, -1.0, float("nan"), float("inf"), 1e30):
        with pytest.raises(capi.ApcError) as e:
            ctx.cluster_dbscan(to_xyzi(p), eps, 5)
        assert e.value.code == capi.APC_ERR_BAD_ARG and "eps" in str(e.value)
    with pytest.raises(capi.ApcError) as e:
        ctx.cluster_dbscan(to_xyzi(p), 0.5, -1)
    assert e.value.code == capi.APC_ERR_BAD_ARG and "min_points" in str(e.value)
    after = run(ctx, p, 0.5, 5)
    assert all(np.array_equal(a, b) for a, b in zip(before, after))


def test_carrier(env, nonground):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from oracle import dbscan as odb
    p = np.ascontiguousarray(nonground[:30_000])
    ref = odb.dbscan(p, 0.5, 10)[0]
    for dev in ("CUDA:0", "CPU:0"):
        pcd = o3d.PointCloud(o3d.Device(dev))
        pcd.point["positions"] = o3d.Tensor(torch.from_numpy(p)).to(o3d.Device(dev))
        labels = pcd.cluster_dbscan(eps=0.5, min_points=10, print_progress=True)
        assert isinstance(labels, o3d.Tensor) and labels.dtype == torch.int32 and labels.device == o3d.Device(dev)
        assert np.array_equal(labels.t.cpu().numpy(), ref)
        empty = o3d.PointCloud(o3d.Device(dev))
        empty.point["positions"] = o3d.Tensor(torch.zeros((0, 3), dtype=torch.float32)).to(o3d.Device(dev))
        e = empty.cluster_dbscan(0.5, 10)
        assert e.shape == (0,) and e.dtype == torch.int32 and e.device == o3d.Device(dev)
    for eps, min_points in ((0.0, 5), (-0.5, 5), (float("nan"), 5), (float("inf"), 5), (0.5, -1)):
        with pytest.raises(ValueError):
            pcd.cluster_dbscan(eps, min_points)
    # min_points above the cloud's size: every point is noise
    assert np.all(pcd.cluster_dbscan(0.5, 2 ** 40).t.numpy() == -1)


def test_carrier_after_ground_removal(env):
    """segment_plane -> select_by_index(inliers, invert=True) -> cluster_dbscan, the Open3D LiDAR idiom."""
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from oracle import dbscan as odb
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(c2_voxels(env["synth"], seed=6)).cuda())
    _, inliers = pcd.segment_plane(distance_threshold=0.2, ransac_n=3, num_iterations=200, seed=1)
    objects = pcd.select_by_index(inliers, invert=True)
    labels = objects.cluster_dbscan(eps=0.5, min_points=10)
    p = objects.point.positions.cpu().numpy()
    ref, n_ref, _, _ = odb.dbscan(p, 0.5, 10)
    assert n_ref > 10 and np.array_equal(labels.t.cpu().numpy(), ref)


def test_kernels_by_name(env, nonground):
    ctx = env["ctx"]
    xyzi = to_xyzi(nonground)
    ctx.profile(True)
    try:
        ctx.cluster_dbscan(xyzi, 0.5, 10)
        ctx.check()
        names = set(ctx.profile_report())
    finally:
        ctx.profile(False)
    assert {"k_dbscan_core", "k_dbscan_union", "k_dbscan_roots", "k_dbscan_label", "k_grid_clean"} <= names
