"""GPU parity tests of normal estimation (pp.py:521-530; csrc/neighbors.cu k_normals_cov / k_normals_wide) against
oracle/normals.py.  Neighbour counts are integer work (bit-exact); covariances and normals are
floating point: covariance within 1e-9 relative to its largest entry, normals within 1e-5 per
component (sign included) wherever the two smallest eigenvalues are separated, and an eigen-residual
bound everywhere."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

T_A = np.array([[0.9986295, -0.0523360, 0.0, 1.5], [0.0523360, 0.9986295, 0.0, -0.25], [0.0, 0.0, 1.0, 1.8],
                [0.0, 0.0, 0.0, 1.0]])


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=300_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


def check_normals(got, cov, ref, atol=1e-5):
    """got / ref float32[N,3]; cov float64[N,3,3] (oracle).

    The bound on the worst deviation: an eigenvector moves by at most |dC| / gap when the matrix moves
    by dC; the GPU's covariance is within 1e-9 of the oracle's (relative to its largest entry, asserted in
    test_normals_parity), so EVERY normal must satisfy
        max_k |got_k - ref_k|  <=  1e-5 + 1e-7 * lambda_max / (lambda_1 - lambda_0)
    i.e. 1e-5 wherever the two smallest eigenvalues are separated by 1 % of the largest, degrading
    gracefully towards degenerate neighbourhoods (collinear points), where the direction itself is
    ill-defined and only the eigen-residual bound below is meaningful."""
    w = np.linalg.eigvalsh(cov)                                   # ascending
    scale = np.maximum(w[:, 2], 1e-300)
    gap = np.maximum(w[:, 1] - w[:, 0], 1e-300)
    separated = gap / scale > 1e-2
    assert separated.sum() > 50
    dev = np.abs(got.astype(np.float64) - ref.astype(np.float64)).max(axis=1)
    assert np.all(dev[separated] <= atol + 1e-5), float(dev[separated].max())
    assert np.all(dev <= atol + 1e-7 * scale / gap), float((dev - 1e-7 * scale / gap).max())
    # everywhere: a unit vector (or exactly one of the axis fallbacks) whose Rayleigh quotient is the smallest eigenvalue
    n64 = got.astype(np.float64)
    assert np.allclose(np.linalg.norm(n64, axis=1), 1.0, atol=1e-5)
    rq = np.einsum("ni,nij,nj->n", n64, cov, n64)
    assert np.all(np.abs(rq - w[:, 0]) <= 1e-4 * scale + 1e-12)


@pytest.mark.parametrize("radius,max_nn", [(0.5, 30), (0.3, 5), (1.0, 64), (0.12, 30)])
def test_normals_parity(env, radius, max_nn):
    from oracle import normals as onrm
    from oracle import voxel
    ctx, synth = env["ctx"], env["synth"]
    scan = synth.lidar_scan(seed=21, n_beams=32, n_az=512, nan_frac=0.0)
    p = voxel.voxel_down_sample(scan["positions"], 0.1, None, fixed=True)["positions"]
    p[0] = p[1]                                                    # an exact duplicate: distance ties broken by index
    ref, cnt_ref, cov_ref = onrm.estimate_normals(p, radius, max_nn)
    for _ in range(2):                                             # the grid cleans itself between calls
        got, cnt, cov = ctx.estimate_normals(to_xyzi(p), max_nn, radius, want_counts=True, want_cov=True)
        ctx.check()
        assert np.array_equal(cnt.cpu().numpy(), cnt_ref)          # neighbourhood sizes, bit-exact
        cov = cov.cpu().numpy()
        big = np.abs(cov_ref).max(axis=(1, 2), keepdims=True)
        assert np.all(np.abs(cov - cov_ref) <= 1e-9 * big + 1e-18)
        few = cnt_ref < 3
        assert few.any() or radius >= 0.5
        assert np.array_equal(got.cpu().numpy()[few], np.tile(np.array([0, 0, 1], np.float32), (int(few.sum()), 1)))
        check_normals(got.cpu().numpy(), cov_ref, ref)


def test_normals_planes_and_edge_cases(env):
    """Exact planes (rank-2 covariance) in three orientations, a line, 1- and 2-point clouds."""
    from oracle import normals as onrm
    ctx = env["ctx"]
    rng = np.random.default_rng(3)
    u, v = rng.uniform(-1, 1, size=(2, 4000)).astype(np.float32)
    for axis in range(3):
        p = np.zeros((4000, 3), np.float32)
        p[:, (axis + 1) % 3], p[:, (axis + 2) % 3] = u, v
        p[:, axis] = np.float32(7.25)
        got, _, _ = ctx.estimate_normals(to_xyzi(p), 30, 0.2)
        ref, cnt, cov = onrm.estimate_normals(p, 0.2, 30)
        g = got.cpu().numpy()
        ok = cnt >= 3
        assert np.allclose(np.abs(g[ok][:, axis]), 1.0, atol=1e-6)
        assert np.allclose(g[ok], ref[ok], atol=1e-5)
    line = np.stack([np.linspace(0, 1, 300, dtype=np.float32), np.zeros(300, np.float32), np.zeros(300, np.float32)], 1)
    got, cnt, _ = ctx.estimate_normals(to_xyzi(line), 30, 0.05, want_counts=True)
    ref, cnt_ref, _ = onrm.estimate_normals(line, 0.05, 30)
    assert np.array_equal(cnt.cpu().numpy(), cnt_ref) and np.allclose(got.cpu().numpy(), ref, atol=1e-6)
    for n in (1, 2):
        got, cnt, _ = ctx.estimate_normals(to_xyzi(line[:n].copy()), 30, 10.0, want_counts=True)
        assert np.array_equal(got.cpu().numpy(), np.tile(np.array([0, 0, 1], np.float32), (n, 1)))
        assert np.array_equal(cnt.cpu().numpy(), np.full(n, n))


def test_normals_full_size_properties(env):
    """C2 size (262 144 points -> ~200k voxels): unit normals everywhere; the synthetic ground plane
    (z = -1.8) gets +-z normals; the estimate does not depend on the point order."""
    from oracle import voxel
    ctx, synth = env["ctx"], env["synth"]
    scan = synth.lidar_scan(seed=2, n_beams=128, n_az=2048, nan_frac=0.0)
    p = voxel.voxel_down_sample(scan["positions"], 0.1, None, fixed=True)["positions"]
    got, cnt, _ = ctx.estimate_normals(to_xyzi(p), 30, 0.5, want_counts=True)
    ctx.check()
    g, c = got.cpu().numpy(), cnt.cpu().numpy()
    assert np.allclose(np.linalg.norm(g.astype(np.float64), axis=1), 1.0, atol=1e-5)
    ground = (np.abs(p[:, 2] + 1.8) < 0.03) & (c >= 10) & (np.hypot(p[:, 0], p[:, 1]) < 15)
    assert ground.sum() > 1000
    assert np.median(np.abs(g[ground][:, 2])) > 0.99
    perm = np.random.default_rng(0).permutation(p.shape[0])
    got2, cnt2, _ = ctx.estimate_normals(to_xyzi(p[perm]), 30, 0.5, want_counts=True)
    assert np.array_equal(cnt2.cpu().numpy(), c[perm])
    # same neighbourhoods (ties are broken by index only between equidistant points), sums in a different order
    same = np.abs(got2.cpu().numpy() - g[perm]).max(axis=1) < 1e-4
    assert same.mean() > 0.999


def test_carrier_normals_and_transform(env):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from oracle import filters
    from oracle import normals as onrm
    from oracle import voxel
    synth = env["synth"]
    scan = synth.lidar_scan(seed=8, n_beams=16, n_az=512, nan_frac=0.0)
    p = voxel.voxel_down_sample(scan["positions"], 0.2, None, fixed=True)["positions"]
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(p).cuda())
    pcd.estimate_normals(max_nn=20, radius=0.6)
    ref, cnt, cov = onrm.estimate_normals(p, 0.6, 20)
    check_normals(pcd.point.normals.cpu().numpy(), cov, ref)
    before = pcd.point.normals.cpu().numpy().copy()
    pcd.transform(o3d.Tensor(T_A, dtype=o3d.float32))
    R = np.eye(4)
    R[:3, :3] = T_A[:3, :3]
    assert np.array_equal(pcd.point.normals.cpu().numpy().view(np.uint32), filters.transform(before, R).view(np.uint32))
    assert np.array_equal(pcd.point.positions.cpu().numpy().view(np.uint32), filters.transform(p, T_A).view(np.uint32))
    # normals travel through selections like any attribute
    sub = pcd.select_by_index(o3d.Tensor(torch.arange(0, p.shape[0], 3).cuda()))
    assert np.array_equal(sub.point.normals.cpu().numpy(), pcd.point.normals.cpu().numpy()[::3])


@pytest.mark.parametrize("with_ground", [False, True])
def test_reference_default_parameter_set_as_one_graph(env, with_ground):
    """The reference's DEFAULT stage set - duplicate removal + non-finite + crop + 0.01 m voxels +
    estimate_normals(0.1, 30) (pp.py:165-178) - captured as ONE CUDA graph (normals are a stage of
    ``apc_pipeline_cfg``), optionally followed by ground removal, through whose selection the normals
    travel (pp.py:542).  Positions bit-exact, normals bounded as in ``check_normals``."""
    from oracle import pipeline as opipe
    ctx, engine, capi, synth = env["ctx"], env["engine"], env["capi"], env["synth"]
    msg = synth.pack_cloud(synth.lidar_scan(seed=31, n_beams=32, n_az=1024), "xyzirt22")
    n = msg.width
    data = torch.frombuffer(bytearray(msg.data), dtype=torch.uint8).cuda()
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, n, data)
    crop = dict(min=[-60.0, -60.0, -20.0], max=[60.0, 60.0, 20.0], invert=False, mode=capi.CROP_OPEN3D)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True, crop=crop)
    # 0.01 m voxels keep nearly every point of a sparse scan; the default radius 0.1 then finds few
    # neighbours - exactly what the reference computes; a second case uses a denser 0.1 / 0.5 setting
    ground = dict(distance_threshold=0.2, ransac_n=5, num_iterations=50, probability=0.99, seed=11) if with_ground else None
    for voxel_size, nrm_cfg in ((0.01, dict(radius=0.1, max_nn=30)), (0.1, dict(radius=0.5, max_nn=30))):
        pcfg = engine.make_pipeline_cfg(fcfg, voxel_size=voxel_size, ground=ground, normals=nrm_cfg)
        out = torch.zeros((n, 4), device="cuda")
        cnt = torch.zeros(8, dtype=torch.int32, device="cuda")
        plane = torch.zeros(8, dtype=torch.float64, device="cuda")
        maps = {"normals": torch.zeros((n, 3), device="cuda")}
        g = ctx.capture_pipeline([desc], pcfg, out, cnt, plane, maps=maps)
        cfg = opipe.default_config()
        cfg.update(crop=crop, voxel_size=voxel_size, ground=ground, normals=nrm_cfg)
        ref = opipe.preprocess(msg, cfg)
        for _ in range(2):                                            # the graph replays cleanly
            out.zero_()
            maps["normals"].zero_()
            ctx.launch_graph(g)
            ctx.check()
            c = cnt.cpu().numpy()
            k = int(c[capi.CNT_OUTPUT])
            assert c[capi.CNT_STATUS] == 0 and k == ref["positions"].shape[0]
            assert np.array_equal(out[:k].cpu().numpy()[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
            got = maps["normals"][:k].cpu().numpy()
            few = ref["normal_counts"] < 3
            if with_ground:
                keep = np.ones(few.shape[0], dtype=bool)
                keep[ref["ground_inliers"]] = False
                few = few[keep]
            assert np.array_equal(got[few], np.tile(np.array([0, 0, 1], np.float32), (int(few.sum()), 1)))
            check_normals(got[~few], ref["normal_cov"][~few], ref["normals"][~few])
        # eager run through apc_pipeline_run_maps gives the same bits as the graph
        out2, cnt2, _, maps2 = ctx.pipeline_run_maps([desc], pcfg)
        ctx.check()
        assert np.array_equal(cnt2.cpu().numpy(), c)
        assert np.array_equal(maps2["normals"][:k].cpu().numpy().view(np.uint32), got.view(np.uint32))
