"""FPFH features and feature matching on the GPU (apc_compute_fpfh / apc_compute_fpfh_knn /
apc_correspondences_from_features) against the CPU oracle (oracle/features.py): SPFH, FPFH and neighbour counts
bit for bit outside the flagged near-edge points, matching bit for bit, determinism, CUDA-graph capture, n_dev,
rejected arguments, the scratch shared with the other neighbour stages, kernel names and the ``registration``
module on CUDA and CPU clouds."""
import warnings

import numpy as np
import pytest

from oracle import features as of
from oracle import normals as onrm
from test_oracle_features import terrain
from test_oracle_normals_search import knn_neighbourhoods

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine
    ctx = engine.Context(max_points=65_536)
    yield dict(ctx=ctx, engine=engine, capi=_capi)
    ctx.close()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


@pytest.fixture(scope="module")
def scene(env):
    """A curved surface with jitter, 40 exact duplicates, and a few NaN and zero normals; normals from the GPU's
    KNN search (the input of both sides)."""
    rng = np.random.default_rng(11)
    p = terrain(seed=3, n_side=60)
    p = p + rng.normal(scale=0.005, size=p.shape).astype(np.float32)
    p = np.concatenate([p, p[rng.choice(len(p), 40, replace=False)]])
    p = np.ascontiguousarray(p[rng.permutation(len(p))])
    nrm, _, _ = env["ctx"].estimate_normals_knn(to_xyzi(p), 20)
    nrm = nrm.cpu().numpy().copy()
    nrm[rng.choice(len(p), 15, replace=False)] = np.nan
    nrm[rng.choice(len(p), 15, replace=False)] = 0.0
    return p, np.ascontiguousarray(nrm)


def gpu_fpfh(ctx, p, nrm, max_nn, radius=None, n_dev=None):
    f, s, c = ctx.compute_fpfh(to_xyzi(p), torch.from_numpy(nrm).cuda(), max_nn, radius, want_spfh=True,
                               want_counts=True, n_dev=n_dev)
    ctx.check()
    return f.cpu().numpy(), s.cpu().numpy(), c.cpu().numpy()


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def check_against_oracle(got, p, nrm, nbs):
    """Counts exactly; the SPFH bit for bit outside the points with a pair near an interior bin edge (rare), where
    CUDA's and libm's atan2 may differ in the last ulp; the FPFH bit for bit everywhere against the oracle's FPFH
    of the GPU's SPFH, and outside the points that read a flagged SPFH against the oracle's own."""
    feat, sp, counts, near = of.compute_fpfh(p, nrm, nbs)
    _, _, flag = of.spfh(p, nrm, nbs)
    assert np.array_equal(got[2], counts)
    assert flag.mean() < 0.005, flag.mean()
    assert same_bits(got[1][~flag], sp[~flag])
    assert same_bits(got[0], of.fpfh(p, got[1], nbs))
    assert same_bits(got[0][~near], feat[~near])


@pytest.mark.parametrize("max_nn,radius", [(1, 0.3), (2, 0.3), (3, 0.3), (30, 0.3), (64, 0.3), (100, 0.5), (1024, 1.3)])
def test_hybrid_matches_the_oracle(env, scene, max_nn, radius):
    p, nrm = scene
    got = gpu_fpfh(env["ctx"], p, nrm, max_nn, radius)
    nbs = onrm.neighbourhoods(p, radius, max_nn)
    if max_nn == 1024:
        assert max(len(nb) for nb in nbs) == 1024        # the cap binds
    check_against_oracle(got, p, nrm, nbs)


@pytest.mark.parametrize("max_nn", [1, 30, 100, 1024])
def test_knn_matches_the_oracle(env, scene, max_nn):
    p, nrm = scene
    got = gpu_fpfh(env["ctx"], p, nrm, max_nn)
    check_against_oracle(got, p, nrm, knn_neighbourhoods(p, max_nn))


@pytest.mark.parametrize("n", [0, 1, 2, 7])
def test_knn_more_neighbours_than_points(env, scene, n):
    p, nrm = scene
    p, nrm = np.ascontiguousarray(p[:n]), np.ascontiguousarray(nrm[:n])
    f, s, c = env["ctx"].compute_fpfh(to_xyzi(p), torch.from_numpy(nrm).cuda(), 30, want_spfh=True, want_counts=True)
    env["ctx"].check()
    assert tuple(f.shape) == (n, 33) and tuple(s.shape) == (n, 33)
    if n:
        check_against_oracle((f.cpu().numpy(), s.cpu().numpy(), c.cpu().numpy()), p, nrm, knn_neighbourhoods(p, 30))
        assert (c.cpu().numpy() == n).all()


def test_unkeyable_points_get_zeros(env, scene):
    p, nrm = scene
    far = p.copy()
    far[7] = [5.0e5, 0.0, 0.0]
    ctx = env["ctx"]
    ctx.compute_fpfh(to_xyzi(far), torch.from_numpy(nrm).cuda(), 30, 0.3)
    with pytest.raises(env["capi"].ApcError) as e:
        ctx.check()
    assert e.value.code == env["capi"].APC_ERR_KEY_RANGE
    f, s, c = ctx.compute_fpfh(to_xyzi(far), torch.from_numpy(nrm).cuda(), 30, 0.3, want_spfh=True, want_counts=True)
    try:
        ctx.check()
    except env["capi"].ApcError:
        pass
    assert not f[7].any() and not s[7].any() and int(c[7]) == 0


@pytest.mark.parametrize("radius", [0.3, None])
def test_determinism_graph_and_n_dev(env, scene, radius):
    p, nrm = scene
    ctx = env["ctx"]
    xyzi, nt = to_xyzi(p), torch.from_numpy(nrm).cuda()
    a = [t.clone() for t in ctx.compute_fpfh(xyzi, nt, 50, radius, want_spfh=True, want_counts=True)]
    b = ctx.compute_fpfh(xyzi, nt, 50, radius, want_spfh=True, want_counts=True)
    ctx.check()
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ctx.compute_fpfh(xyzi, nt, 50, radius, want_spfh=True, want_counts=True)
    for t in out:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    ctx.check()
    assert all(torch.equal(x, y) for x, y in zip(out, a))
    m = 2000
    n_dev = torch.tensor([m], dtype=torch.int32, device="cuda")
    full = gpu_fpfh(ctx, p, nrm, 50, radius, n_dev=n_dev)
    trimmed = gpu_fpfh(ctx, np.ascontiguousarray(p[:m]), np.ascontiguousarray(nrm[:m]), 50, radius)
    for x, y in zip(full, trimmed):
        assert same_bits(x[:m], y) and not x[m:].any()


def test_errors_leave_the_context_usable(env, scene):
    capi, ctx = env["capi"], env["ctx"]
    p, nrm = scene
    xyzi, nt = to_xyzi(p), torch.from_numpy(nrm).cuda()
    before = gpu_fpfh(ctx, p, nrm, 30, 0.3)

    def bad(fn, word):
        with pytest.raises(capi.ApcError) as e:
            fn()
        assert e.value.code == capi.APC_ERR_BAD_ARG and word in str(e.value)

    for k in (0, -1, 1025):
        bad(lambda: ctx.compute_fpfh(xyzi, nt, k, 0.3), "max_nn")
        bad(lambda: ctx.compute_fpfh(xyzi, nt, k), "max_nn")
    for r in (0.0, -1.0, float("nan"), float("inf"), 1e30):
        bad(lambda: ctx.compute_fpfh(xyzi, nt, 30, r), "radius")
    bad(lambda: ctx.compute_fpfh(xyzi, None, 30, 0.3), "NULL")
    bad(lambda: ctx.compute_fpfh(xyzi, None, 30), "NULL")
    f = torch.zeros((4, 33), device="cuda")
    info = torch.zeros(2, dtype=torch.int32, device="cuda")
    pairs = torch.zeros((4, 2), dtype=torch.int32, device="cuda")
    lib = capi.lib
    ptr = lambda t: capi.C.c_void_p(t.data_ptr())
    s = capi.C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.apc_compute_fpfh(ctx.h, None, ptr(nt), 4, None, 30, 0.3, ptr(f), None, None, s) == capi.APC_ERR_BAD_ARG
    assert lib.apc_compute_fpfh(ctx.h, ptr(xyzi), ptr(nt), 4, None, 30, 0.3, None, None, None, s) == capi.APC_ERR_BAD_ARG
    assert lib.apc_compute_fpfh_knn(ctx.h, ptr(xyzi), ptr(nt), ctx.max_points + 1, None, 30, ptr(f), None, None,
                                    s) == capi.APC_ERR_BAD_ARG
    a = torch.rand((4, 33), device="cuda")
    for dim in (0, 65):
        assert lib.apc_correspondences_from_features(ctx.h, ptr(a), 4, None, ptr(a), 4, None, dim, 0, 0.1, ptr(pairs),
                                                     None, ptr(info), s) == capi.APC_ERR_BAD_ARG
    for ratio in (-0.1, float("nan"), float("inf")):
        bad(lambda: ctx.correspondences_from_features(a, a, True, ratio), "ratio")
    calls = [(None, ptr(a), ptr(pairs), ptr(info), 4), (ptr(a), None, ptr(pairs), ptr(info), 4),
             (ptr(a), ptr(a), None, ptr(info), 4), (ptr(a), ptr(a), ptr(pairs), None, 4),
             (ptr(a), ptr(a), ptr(pairs), ptr(info), ctx.max_points + 1)]
    for sp, tp, pp, ip, n in calls:
        assert lib.apc_correspondences_from_features(ctx.h, sp, n, None, tp, 4, None, 33, 1, 0.1, pp, None, ip,
                                                     s) == capi.APC_ERR_BAD_ARG
    after = gpu_fpfh(ctx, p, nrm, 30, 0.3)
    assert all(same_bits(x, y) for x, y in zip(before, after))


def random_features(rng, n, dim, levels=3):
    """Small integers: exact ties between rows are common; a few NaN rows."""
    f = rng.integers(0, levels, size=(n, dim)).astype(np.float32)
    f[rng.choice(n, max(1, n // 200), replace=False), rng.integers(0, dim)] = np.nan
    return f


def gpu_match(ctx, a, b, mutual=False, ratio=0.1):
    pairs, info, nearest = ctx.correspondences_from_features(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda(),
                                                             mutual, ratio, want_nearest=True)
    ctx.check()
    info = info.cpu().numpy()
    return pairs[:int(info[0])].cpu().numpy(), nearest.cpu().numpy(), bool(info[1])


@pytest.mark.parametrize("dim", [1, 33, 64])
@pytest.mark.parametrize("mutual", [False, True])
def test_matching_matches_the_oracle(env, dim, mutual):
    rng = np.random.default_rng(dim)
    levels = 40 if dim == 1 else 3
    a, b = random_features(rng, 3000, dim, levels), random_features(rng, 5000, dim, levels)
    b[17] = np.arange(dim) % levels                               # a planted tie across target splits
    b[4000] = b[17]
    a[5] = b[17]
    pairs, nearest, fb = gpu_match(env["ctx"], a, b, mutual)
    rp, rn, rfb = of.correspondences(a, b, mutual, 0.1)
    assert np.array_equal(nearest, rn) and (nearest[5] == 17 or dim == 1)
    assert fb == rfb and np.array_equal(pairs, rp)


def test_matching_fallback_and_empty(env):
    ctx = env["ctx"]
    rng = np.random.default_rng(5)
    b = rng.normal(size=(100, 33)).astype(np.float32)
    a = (np.repeat(b[:3], 20, axis=0) + rng.normal(scale=1e-3, size=(60, 33))).astype(np.float32)
    for ratio, want_fb in ((3 / 60, True), (2.99 / 60, False), (0.0, False)):
        pairs, _, fb = gpu_match(ctx, a, b, True, ratio)
        rp, _, rfb = of.correspondences(a, b, True, ratio)
        assert fb == rfb == want_fb and np.array_equal(pairs, rp)
    pairs, nearest, fb = gpu_match(ctx, a, b[:0], True)             # an empty target: no pairs, and so the fallback
    rp, rn, rfb = of.correspondences(a, b[:0], True, 0.1)
    assert len(pairs) == len(rp) == 0 and (nearest == -1).all() and np.array_equal(nearest, rn) and fb == rfb
    nan_tgt = np.full((10, 33), np.nan, np.float32)
    pairs, nearest, _ = gpu_match(ctx, a, nan_tgt)
    assert len(pairs) == 0 and (nearest == -1).all()


def bits(*ts):
    return [t.cpu().numpy().copy().view(np.uint8) for t in ts if t is not None]


def test_shared_scratch_interleaved(env, scene):
    """FPFH and matching share the context's grids and scratch with the normals searches and ICP: interleaved on one
    context, each gives exactly what it gives on a context of its own."""
    engine, ctx = env["engine"], env["ctx"]
    p, nrm = scene
    xyzi, nt = to_xyzi(p), torch.from_numpy(nrm).cuda()
    fa = torch.from_numpy(random_features(np.random.default_rng(1), 2000, 33)).cuda()
    fb = torch.from_numpy(random_features(np.random.default_rng(2), 2500, 33)).cuda()
    calls = {
        "fpfh_hybrid": lambda c: c.compute_fpfh(xyzi, nt, 40, 0.3, want_spfh=True, want_counts=True),
        "fpfh_knn": lambda c: c.compute_fpfh(xyzi, nt, 100, want_spfh=True, want_counts=True),
        "match": lambda c: c.correspondences_from_features(fa, fb, True, 0.1, want_nearest=True),
        "normals_knn": lambda c: c.estimate_normals_knn(xyzi, 20, want_cov=True),
        "normals_hybrid": lambda c: c.estimate_normals(xyzi, 20, 0.3, want_cov=True),
        "icp": lambda c: c.icp(xyzi, xyzi, 0.3, max_iteration=3),
    }
    alone = {}
    for name, fn in calls.items():
        c = engine.Context(max_points=len(p))
        alone[name] = bits(*fn(c))
        c.check()
        c.close()
    for name in ("fpfh_hybrid", "normals_knn", "fpfh_knn", "match", "icp", "fpfh_hybrid", "normals_hybrid",
                 "fpfh_knn", "match", "fpfh_hybrid"):
        got = bits(*calls[name](ctx))
        ctx.check()
        assert all(np.array_equal(x, y) for x, y in zip(got, alone[name])), name


def test_kernels_by_name(env, scene):
    ctx = env["ctx"]
    p, nrm = scene
    xyzi, nt = to_xyzi(p), torch.from_numpy(nrm).cuda()
    fa = torch.rand((500, 33), device="cuda")
    ctx.profile(True)
    try:
        ctx.compute_fpfh(xyzi, nt, 30, 0.3)
        ctx.check()
        hybrid = ctx.profile_report()
        ctx.compute_fpfh(xyzi, nt, 30)
        ctx.check()
        knn = ctx.profile_report()
        ctx.correspondences_from_features(fa, fa, False)
        ctx.check()
        single = ctx.profile_report()
        ctx.correspondences_from_features(fa, fa, True)
        ctx.check()
        mutual = ctx.profile_report()
    finally:
        ctx.profile(False)
    assert hybrid["k_fpfh_hybrid_spfh"][1] == 1 and hybrid["k_fpfh_hybrid"][1] == 1
    assert not any(k.startswith("k_fpfh_knn") or k.startswith("k_normals") for k in hybrid)
    for k in ("k_fpfh_knn_spfh", "k_fpfh_knn_stragglers_spfh", "k_fpfh_knn", "k_fpfh_knn_stragglers"):
        assert knn[k][1] == 1, k
    assert single["k_feat_nn"][1] == 1 and mutual["k_feat_nn"][1] == 2
    for r in (single, mutual):
        assert r["k_feat_pairs"][1] == 1 and r["k_feat_select"][1] == 1


def cloud(o3d, p, dev, nrm=None):
    pcd = o3d.PointCloud(o3d.Device(dev))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p))).to(o3d.Device(dev))
    if nrm is not None:
        pcd.point["normals"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(nrm))).to(o3d.Device(dev))
    return pcd


@pytest.mark.parametrize("dev", ["CUDA:0", "CPU:0"])
def test_carrier(env, scene, dev):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    p, nrm = scene
    pcd = cloud(o3d, p, dev, nrm)
    f = o3dreg.compute_fpfh_feature(pcd, max_nn=40, radius=0.3)
    assert f.device == o3d.Device(dev) and tuple(f.shape) == (len(p), 33) and f.t.dtype == torch.float32
    ref, _, _ = gpu_fpfh(env["ctx"], p, nrm, 40, 0.3)
    assert same_bits(f.t.cpu().numpy(), ref)
    fk = o3dreg.compute_fpfh_feature(pcd, max_nn=40)
    assert same_bits(fk.t.cpu().numpy(), gpu_fpfh(env["ctx"], p, nrm, 40)[0])
    half = len(p) // 2
    corr = o3dreg.correspondences_from_features(f, o3d.Tensor(f.t[:half]), mutual_filter=True)
    assert corr.device == o3d.Device(dev) and corr.t.dtype == torch.int64
    rp, _, _ = of.correspondences(ref, ref[:half], True, 0.1)
    assert np.array_equal(corr.t.cpu().numpy(), rp)
    a = np.repeat(ref[:3], 20, axis=0)
    with pytest.warns(RuntimeWarning, match="fall back"):
        fb = o3dreg.correspondences_from_features(o3d.Tensor(torch.from_numpy(a)).to(o3d.Device(dev)), f, True, 0.5)
    assert len(fb) == 60
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        o3dreg.correspondences_from_features(f, f, True, 0.1)
    # empty, no normals, not modelled
    empty = o3dreg.compute_fpfh_feature(cloud(o3d, p[:0], dev, nrm[:0]))
    assert tuple(empty.shape) == (0, 33) and empty.device == o3d.Device(dev)
    with pytest.raises(RuntimeError):
        o3dreg.compute_fpfh_feature(cloud(o3d, p, dev))
    with pytest.raises(NotImplementedError):
        o3dreg.compute_fpfh_feature(pcd, max_nn=None, radius=0.3)
    with pytest.raises(NotImplementedError):
        o3dreg.compute_fpfh_feature(pcd, indices=[0, 1])


def test_registration_scene_correspondences(env):
    """The oracle's rigid-motion scene run through the GPU: the mutual FPFH pairs are mostly the true ones."""
    from scipy.spatial.transform import Rotation

    from test_oracle_features import oriented
    ctx = env["ctx"]
    p = terrain()
    R = Rotation.from_euler("zyx", [40, 15, -20], degrees=True).as_matrix()
    perm = np.random.default_rng(1).permutation(len(p))
    q = np.ascontiguousarray((p.astype(np.float64) @ R.T + np.array([3.0, -1.0, 0.5])).astype(np.float32)[perm])
    up = np.array([0.0, 0.0, 1.0])
    ns = np.ascontiguousarray(oriented(ctx.estimate_normals(to_xyzi(p), 30, 0.25)[0].cpu().numpy(), up))
    nt = np.ascontiguousarray(oriented(ctx.estimate_normals(to_xyzi(q), 30, 0.25)[0].cpu().numpy(), R @ up))
    fs = gpu_fpfh(ctx, p, ns, 100, 0.5)[0]
    ft = gpu_fpfh(ctx, q, nt, 100, 0.5)[0]
    pairs, _, fb = gpu_match(ctx, fs, ft, True)
    assert not fb and len(pairs) > 0.5 * len(p)
    assert (np.argsort(perm)[pairs[:, 0]] == pairs[:, 1]).mean() > 0.9
