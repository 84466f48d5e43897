"""Fast Global Registration on the GPU (apc_fgr_from_features / apc_fgr; kernels k_fgr_*) against the CPU oracle
(oracle/fgr.py): the mutual set, the tuple test's pairs and trials, iterations and status exactly, the transform within
1e-9; options, seeds and sizes; determinism, CUDA-graph capture, device counts, errors, scratch shared with the other
registration stages, kernel names, the ``registration`` functions, and FGR + ICP recovering a motion ICP alone misses."""
import numpy as np
import pytest

from oracle import fgr
from oracle import registration as reg
from test_oracle_fgr import hard_terrain, motion, moved, pose_error

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

BAD_ARG = -2


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine
    ctx = engine.Context(max_points=200_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi)
    ctx.close()


@pytest.fixture(scope="module")
def terrain_case():
    return hard_terrain()


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


def dev(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a if dtype is None else a.astype(dtype))).cuda()


def run_features(ctx, p, q, fs, ft, **kw):
    T, info, used = ctx.fgr_from_features(to_xyzi(p), to_xyzi(q), dev(fs, np.float32), dev(ft, np.float32), **kw)
    ctx.check()
    info = info.cpu().numpy()
    return T.cpu().numpy(), info, used[:info[2]].cpu().numpy().astype(np.int64)


def run_pairs(ctx, p, q, pairs, **kw):
    T, info, used = ctx.fgr(to_xyzi(p), to_xyzi(q), dev(np.asarray(pairs).reshape(-1, 2), np.int32), **kw)
    ctx.check()
    info = info.cpu().numpy()
    return T.cpu().numpy(), info, used[:info[2]].cpu().numpy().astype(np.int64)


def assert_result(got, ref, trials, n_in, tol=1e-9):
    T, info, used = got
    assert np.array_equal(used, ref["pairs_used"].reshape(-1, 2))
    assert info.tolist() == [ref["iterations"], n_in, len(ref["pairs_used"]), ref["status"], trials, info[5]]
    assert np.abs(T - ref["transformation"]).max() <= tol, np.abs(T - ref["transformation"]).max()


OPTIONS = [dict(), dict(use_absolute_scale=True), dict(decrease_mu=False), dict(tuple_test=False), dict(seed=1),
           dict(seed=123456789012345), dict(maximum_tuple_count=7, iteration_number=5),
           dict(division_factor=2.0, maximum_correspondence_distance=0.1, tuple_scale=0.9, iteration_number=0)]


@pytest.mark.parametrize("opt", OPTIONS, ids=[str(o) for o in OPTIONS])
def test_features_match_the_oracle(env, terrain_case, opt):
    p, q, fs, ft, T_true, _ = terrain_case
    tuple_on = opt.get("tuple_test", True)
    gpu_kw = dict(opt)
    ref = fgr.fgr_from_features(p, q, fs, ft, tuple_test_on=tuple_on,
                                **{k: v for k, v in opt.items() if k != "tuple_test"})
    got = run_features(env["ctx"], p, q, fs, ft, **gpu_kw)
    assert_result(got, ref, ref["trials"], len(ref["pairs_in"]))
    assert got[1][5] == 0
    if opt in (dict(), dict(seed=1)):
        dt, ang = pose_error(got[0], T_true)
        assert dt < 0.1 and ang < 2.0


@pytest.mark.parametrize("K", [0, 5, 9, 10, 1000, 30000])
def test_correspondence_entry_matches_the_oracle(env, K):
    rng = np.random.default_rng(K)
    n = max(K, 1)
    p = (rng.normal(size=(n, 3)) * [20.0, 20.0, 2.0]).astype(np.float32)
    T_true = motion(75.0, 4.0, -3.0, (10.0, -4.0, 1.0))
    q = moved(p + rng.normal(0, 0.02, p.shape).astype(np.float32), T_true)
    pairs = np.stack([np.arange(K), rng.permutation(n)[:K]], 1)
    pairs[: K // 2, 1] = pairs[: K // 2, 0]                      # half true pairs, half random
    for absolute in (False, True):
        ref = fgr.fgr(p, q, pairs, use_absolute_scale=absolute)
        ref.update(pairs_used=pairs)
        got = run_pairs(env["ctx"], p, q, pairs, use_absolute_scale=absolute)
        assert_result(got, ref, 0, K)
        assert got[1][5] == 0
        if K >= 1000:
            dt, ang = pose_error(got[0], T_true)
            assert dt < 0.05 and ang < 0.2


def test_out_of_range_pairs_are_dropped_and_counted(env):
    rng = np.random.default_rng(2)
    p = rng.normal(size=(500, 3)).astype(np.float32) * 5
    q = moved(p[:400], motion(30.0))
    pairs = np.stack([np.arange(400), np.arange(400)], 1)
    bad = np.array([[-1, 3], [500, 3], [3, 400], [7, -5], [1 << 30, 1]])
    mixed = np.concatenate([pairs[:100], bad, pairs[100:], bad[::-1]])
    ref = fgr.fgr(p, q, pairs)
    ref.update(pairs_used=pairs)
    got = run_pairs(env["ctx"], p, q, mixed)
    assert_result(got, ref, 0, len(mixed))
    assert got[1][5] == 2 * len(bad)


def test_large_mutual_set_and_tuple_cut(env):
    """K ~ 30 000 mutual pairs (3-dim features, a permuted noisy copy): the mutual set equals the existing matching's,
    the tuple test equals the oracle's on it with the cut reached (1000) and not reached (all 100 K trials)."""
    ctx = env["ctx"]
    rng = np.random.default_rng(9)
    n = 30000
    p = rng.uniform(-30, 30, size=(n, 3)).astype(np.float32)
    perm = rng.permutation(n)
    q = moved(p[perm] + rng.normal(0, 0.01, (n, 3)).astype(np.float32), motion(140.0))
    fs, ft = p / np.float32(30), (p[perm] + rng.normal(0, 0.05, (n, 3)).astype(np.float32)) / np.float32(30)
    T0, info0, mutual = run_features(ctx, p, q, fs, ft, tuple_test=False)
    pairs, cinfo, _ = ctx.correspondences_from_features(dev(fs), dev(ft), True, 0.0)
    ctx.check()
    want = pairs[:int(cinfo[0])].cpu().numpy().astype(np.int64)
    assert int(cinfo[1]) == 0 and np.array_equal(mutual, want) and len(want) > 20000
    ref = fgr.fgr(p, q, want)
    ref.update(pairs_used=want)
    assert_result((T0, info0, mutual), ref, 0, len(want))
    q_far = rng.uniform(-30, 30, size=(n, 3)).astype(np.float32)    # unrelated target: few tuples pass
    for tgt, count in ((q, 1000), (q_far, 60000)):
        used, trials = fgr.tuple_test(p, tgt, want, 0, 0.95, count)
        got = run_features(ctx, p, tgt, fs, ft, maximum_tuple_count=count)
        assert np.array_equal(got[2], used) and got[1][4] == trials and got[1][2] == len(used)
        if count == 60000:
            assert trials == 100 * len(want) and len(used) < 3 * count
        ref = fgr.fgr(p, tgt, used)
        assert got[1][0] == ref["iterations"] and got[1][3] == ref["status"]
        # the unrelated target's optimum is flat: 64 steps amplify the summation order's last bits
        assert np.abs(got[0] - ref["transformation"]).max() <= (1e-9 if count == 1000 else 1e-6)


def test_mutual_set_where_matching_falls_back(env):
    """A feature at the centre of the source's features (the other target rows spread three times wider) is nearly
    every source row's nearest: 20 planted rows (and perhaps the centre row's own) are the only mutual pairs, so
    correspondences_from_features falls back while FGR keeps them."""
    ctx = env["ctx"]
    rng = np.random.default_rng(4)
    fs = rng.normal(size=(400, 33)).astype(np.float32)
    ft = np.concatenate([rng.normal(size=(300, 33)) * 3, np.zeros((1, 33)), fs[:20] + 1e-3]).astype(np.float32)
    p = rng.normal(size=(400, 3)).astype(np.float32) * 4
    q = np.concatenate([rng.normal(size=(301, 3)) * 4, moved(p[:20], motion(50.0))]).astype(np.float32)
    _, cinfo, _ = ctx.correspondences_from_features(dev(fs), dev(ft), True, 0.1)
    ctx.check()
    assert int(cinfo[1]) == 1
    for tuple_on in (False, True):
        ref = fgr.fgr_from_features(p, q, fs, ft, tuple_test_on=tuple_on)
        assert 20 <= len(ref["pairs_in"]) <= 21                # the centre row may pair with the smallest source row
        got = run_features(ctx, p, q, fs, ft, tuple_test=tuple_on)
        assert_result(got, ref, ref["trials"], len(ref["pairs_in"]))


def test_too_few_and_degenerate(env):
    ctx = env["ctx"]
    p = (np.random.default_rng(1).normal(size=(50, 3)) * 3).astype(np.float32)
    q = moved(p, motion(20.0))
    pairs = np.stack([np.arange(50), np.arange(50)], 1)
    T, info, _ = run_pairs(ctx, p, q, pairs[:9])
    assert info[3] == fgr.TOO_FEW and info[0] == 0 and np.array_equal(T, np.eye(4))
    T, info, _ = run_pairs(ctx, p, q, pairs[:10], iteration_number=0)
    want = np.eye(4)
    want[:3, 3] = q.astype(np.float64).mean(0) - p.astype(np.float64).mean(0)
    assert info[3] == fgr.OK and np.abs(T - want).max() < 1e-12
    line = np.zeros((30, 3), np.float32)
    line[:, 0] = np.arange(30)
    T, info, _ = run_pairs(ctx, line, line + np.float32(1), np.stack([np.arange(30), np.arange(30)], 1))
    assert info[3] == fgr.DEGENERATE and info[0] == 0
    bad = p.copy()
    bad[49, 1] = np.nan
    T, info, _ = run_pairs(ctx, bad, q, pairs[:20])
    assert info[3] == fgr.DEGENERATE and info[0] == 0
    T, info, _ = run_pairs(ctx, p, np.zeros((0, 3), np.float32), pairs)
    assert info[3] == fgr.TOO_FEW and info[5] == 50


def test_determinism_and_graph_capture(env, terrain_case):
    ctx = env["ctx"]
    p, q, fs, ft, _, _ = terrain_case
    xs, xt, ds, dt = to_xyzi(p), to_xyzi(q), dev(fs), dev(ft)
    pairs = dev(np.stack([np.arange(len(q)), np.arange(len(q))], 1), np.int32)
    calls = (lambda: ctx.fgr_from_features(xs, xt, ds, dt), lambda: ctx.fgr(xs, xt, pairs))
    for call in calls:
        a = [t.clone() for t in call()]
        b = [t.clone() for t in call()]
        ctx.check()
        assert all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(a, b))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = call()
        for t in out:
            t.zero_()
        g.replay()
        torch.cuda.synchronize()
        ctx.check()
        n = int(a[1][2])
        assert torch.equal(out[0], a[0]) and torch.equal(out[1], a[1]) and torch.equal(out[2][:n], a[2][:n])
        assert int(a[1][0]) == 64


def test_n_dev_below_n_max(env, terrain_case):
    ctx = env["ctx"]
    p, q, fs, ft, _, _ = terrain_case
    ms, mt = 3000, 1800
    nsd = torch.tensor([ms], dtype=torch.int32, device="cuda")
    ntd = torch.tensor([mt], dtype=torch.int32, device="cuda")
    ref = fgr.fgr_from_features(p[:ms], q[:mt], fs[:ms], ft[:mt])
    T, info, used = ctx.fgr_from_features(to_xyzi(p), to_xyzi(q), dev(fs), dev(ft), n_src_dev=nsd, n_tgt_dev=ntd)
    ctx.check()
    info = info.cpu().numpy()
    assert_result((T.cpu().numpy(), info, used[:info[2]].cpu().numpy()), ref, ref["trials"], len(ref["pairs_in"]))
    pairs = ref["pairs_in"]
    npd = torch.tensor([len(pairs) // 2], dtype=torch.int32, device="cuda")
    half = pairs[:len(pairs) // 2]
    ref = fgr.fgr(p[:ms], q[:mt], half)
    ref.update(pairs_used=half)
    T, info, used = ctx.fgr(to_xyzi(p), to_xyzi(q), dev(pairs, np.int32), n_src_dev=nsd, n_tgt_dev=ntd, n_pairs_dev=npd)
    ctx.check()
    info = info.cpu().numpy()
    assert_result((T.cpu().numpy(), info, used[:info[2]].cpu().numpy()), ref, 0, len(half))


def test_errors_leave_the_context_usable(env, terrain_case):
    ctx, lib = env["ctx"], env["capi"].lib
    p, q, fs, ft, _, _ = terrain_case
    xs, xt, ds, dt = to_xyzi(p), to_xyzi(q), dev(fs), dev(ft)
    good = run_features(ctx, p, q, fs, ft)
    T = torch.empty((4, 4), dtype=torch.float64, device="cuda")
    info = torch.empty(6, dtype=torch.int32, device="cuda")
    P = lambda t: t.data_ptr() if t is not None else None
    base = dict(src=xs, n_src=len(p), tgt=xt, n_tgt=len(q), fs=ds, ft=dt, dim=33, div=1.4, mcd=0.025, it=64,
                ts=0.95, mtc=1000, T=T, info=info)

    def feat(**kw):
        a = dict(base, **kw)
        return lib.apc_fgr_from_features(ctx.h, P(a["src"]), a["n_src"], None, P(a["tgt"]), a["n_tgt"], None,
                                         P(a["fs"]), P(a["ft"]), a["dim"], a["div"], 0, 1, a["mcd"], a["it"], a["ts"],
                                         a["mtc"], 1, 0, P(a["T"]), P(a["info"]), None, None)
    cases = [dict(src=None), dict(tgt=None), dict(fs=None), dict(ft=None), dict(T=None), dict(info=None),
             dict(n_src=200_001), dict(n_tgt=200_001), dict(dim=0), dict(dim=65), dict(div=1.0),
             dict(div=float("inf")), dict(div=float("nan")), dict(mcd=0.0), dict(mcd=float("nan")), dict(it=-1),
             dict(ts=0.0), dict(ts=1.0000001), dict(ts=float("nan")), dict(mtc=0), dict(mtc=200_001)]
    for kw in cases:
        assert feat(**kw) == BAD_ARG, kw
    pairs = dev(np.stack([np.arange(100), np.arange(100)], 1), np.int32)
    ok = lib.apc_fgr(ctx.h, P(xs), len(p), None, P(xt), len(q), None, P(pairs), 100, None, 1.4, 0, 1, 0.025, 64,
                     P(T), P(info), None, None)
    assert ok == 0
    assert lib.apc_fgr(ctx.h, P(xs), len(p), None, P(xt), len(q), None, None, 100, None, 1.4, 0, 1, 0.025, 64,
                       P(T), P(info), None, None) == BAD_ARG
    assert lib.apc_fgr(ctx.h, P(xs), len(p), None, P(xt), len(q), None, P(pairs), 200_001, None, 1.4, 0, 1, 0.025,
                       64, P(T), P(info), None, None) == BAD_ARG
    assert lib.apc_fgr(ctx.h, P(xs), len(p), None, P(xt), len(q), None, P(pairs), 100, None, 0.5, 0, 1, 0.025, 64,
                       P(T), P(info), None, None) == BAD_ARG
    after = run_features(ctx, p, q, fs, ft)
    assert all(np.array_equal(a, b) for a, b in zip(good, after))


def test_shared_scratch_interleaved(env, terrain_case):
    ctx = env["ctx"]
    p, q, fs, ft, _, _ = terrain_case
    alone = run_features(ctx, p, q, fs, ft)
    pairs = alone[2]
    alone_pairs = run_pairs(ctx, p, q, pairs)
    nrm, _, _ = ctx.estimate_normals(to_xyzi(q), 30, 0.25)
    f1, _, _ = ctx.compute_fpfh(to_xyzi(q), nrm.contiguous(), 100, 0.5)
    c1 = ctx.correspondences_from_features(dev(fs), dev(ft), True, 0.1)
    ctx.check()
    mid = run_features(ctx, p, q, fs, ft)
    i1 = ctx.icp(to_xyzi(p), to_xyzi(p), 0.5, max_iteration=3)
    c2 = ctx.correspondences_from_features(dev(fs), dev(ft), True, 0.1)
    f2, _, _ = ctx.compute_fpfh(to_xyzi(q), nrm.contiguous(), 100, 0.5)
    ctx.check()
    end = run_pairs(ctx, p, q, pairs)
    i2 = ctx.icp(to_xyzi(p), to_xyzi(p), 0.5, max_iteration=3)
    ctx.check()
    assert all(np.array_equal(a, b) for a, b in zip(alone, mid))
    assert all(np.array_equal(a, b) for a, b in zip(alone_pairs, end))
    assert torch.equal(f1, f2) and torch.equal(c1[0], c2[0]) and torch.equal(c1[1], c2[1])
    assert all(torch.equal(a, b) for a, b in zip(i1, i2))


def test_kernels_by_name(env, terrain_case):
    ctx = env["ctx"]
    p, q, fs, ft, _, _ = terrain_case
    ctx.profile(True)
    try:
        ctx.fgr_from_features(to_xyzi(p), to_xyzi(q), dev(fs), dev(ft), iteration_number=5)
        ctx.check()
        a = ctx.profile_report()
        ctx.fgr(to_xyzi(p), to_xyzi(q), dev(np.zeros((50, 2)), np.int32), iteration_number=3)
        ctx.check()
        b = ctx.profile_report()
    finally:
        ctx.profile(False)
    assert a["k_feat_nn"][1] == 2 and a["k_feat_pairs"][1] == 1 and a["k_fgr_tuples"][1] == 1
    assert a["k_fgr_norm"][1] == 1 and a["k_fgr_accum"][1] == 5 and a["k_icp_solve"][1] == 5
    assert a["k_fgr_final"][1] == 1 and "k_fgr_pairs" not in a and "k_feat_select" not in a
    assert b["k_fgr_pairs"][1] == 1 and b["k_fgr_accum"][1] == 3 and "k_fgr_tuples" not in b
    assert "k_feat_nn" not in b


def cloud(o3d, p, device):
    pcd = o3d.PointCloud(o3d.Device(device))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p))).to(o3d.Device(device))
    return pcd


def test_registration_functions(env, terrain_case):
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    p, q, fs, ft, T_true, _ = terrain_case
    ref = fgr.fgr_from_features(p, q, fs, ft, seed=3)
    opt = o3dreg.FastGlobalRegistrationOption(seed=3)
    assert "seed=3" in repr(opt) and "tuple_test=True" in repr(opt)
    out = {}
    for device in ("CUDA:0", "CPU:0"):
        s, t = cloud(o3d, p, device), cloud(o3d, q, device)
        feats = [o3d.Tensor(torch.from_numpy(f)).to(o3d.Device(device)) for f in (fs, ft)]
        res = o3dreg.registration_fgr_based_on_feature_matching(s, t, feats[0], feats[1], opt)
        T = res.transformation
        assert T.device == o3d.Device("CPU:0") and T.dtype == torch.float64 and T.shape == (4, 4)
        assert res.fitness == 0.0 and res.inlier_rmse == 0.0 and res.num_iterations == 64
        assert res.correspondences_.device == o3d.Device(device) and torch.all(res.correspondences_.t == -1)
        assert np.abs(T.numpy() - ref["transformation"]).max() <= 1e-9
        corres = o3d.Tensor(torch.from_numpy(ref["pairs_in"])).to(o3d.Device(device))
        r2 = o3dreg.registration_fgr_based_on_correspondence(s, t, corres)
        ref2 = fgr.fgr(p, q, ref["pairs_in"])
        assert np.abs(r2.transformation.numpy() - ref2["transformation"]).max() <= 1e-9
        out[device] = (T.numpy(), r2.transformation.numpy())
    assert all(np.array_equal(a, b) for a, b in zip(out["CUDA:0"], out["CPU:0"]))
    s, t = cloud(o3d, p, "CUDA:0"), cloud(o3d, q, "CUDA:0")
    with pytest.raises(ValueError):
        o3dreg.registration_fgr_based_on_feature_matching(s, t, fs[:10], ft)
    with pytest.raises(ValueError):
        o3dreg.registration_fgr_based_on_correspondence(s, t, np.array([[0, len(q)]]))
    with pytest.raises(ValueError):
        o3dreg.registration_fgr_based_on_correspondence(s, t, np.array([[-1, 0]]))
    for bad in (dict(division_factor=1.0), dict(maximum_correspondence_distance=0), dict(iteration_number=-1),
                dict(tuple_scale=0), dict(tuple_scale=1.5), dict(maximum_tuple_count=0)):
        with pytest.raises(ValueError):
            o3dreg.FastGlobalRegistrationOption(**bad)
    with pytest.warns(RuntimeWarning):
        res = o3dreg.registration_fgr_based_on_correspondence(s, t, np.stack([np.arange(9), np.arange(9)], 1))
    assert np.array_equal(res.transformation.numpy(), np.eye(4)) and res.num_iterations == 0
    line = np.zeros((30, 3), np.float32)
    line[:, 0] = np.arange(30)
    with pytest.raises(RuntimeError, match="positive definite"):
        o3dreg.registration_fgr_based_on_correspondence(cloud(o3d, line, "CUDA:0"), cloud(o3d, line + 1, "CUDA:0"),
                                                        np.stack([np.arange(30), np.arange(30)], 1))


def test_end_to_end_fgr_then_icp_recovers_what_icp_alone_misses(terrain_case):
    """The hard terrain pair (170 degrees of yaw; the target a noisy, 60 % subsample of the source, so only ~11 % of
    the mutual FPFH pairs are true), all on CUDA clouds: estimate_normals (oriented to the vertical, as a user does
    before FPFH) -> compute_fpfh_feature -> FGR -> point-to-point ICP lands within 2 cm / 0.2 degrees, where ICP
    from the identity does not (given a 2 m window, wide enough on this 4 m patch to find pairs at all, it settles
    about 180 degrees off)."""
    from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
    from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
    p, q, _, _, T_true, _ = terrain_case
    s, t = cloud(o3d, p, "CUDA:0"), cloud(o3d, q, "CUDA:0")
    for c, up in ((s, np.array([0.0, 0.0, 1.0])), (t, T_true[:3, :3] @ np.array([0.0, 0.0, 1.0]))):
        c.estimate_normals(30, 0.25)
        n = c.point["normals"].t
        sign = torch.where(n.double() @ torch.from_numpy(up).cuda() < 0, -1.0, 1.0).to(n.dtype)[:, None]
        c.point["normals"] = o3d.Tensor((n * sign).contiguous())
    fs, ft = o3dreg.compute_fpfh_feature(s, 100, 0.5), o3dreg.compute_fpfh_feature(t, 100, 0.5)
    g = o3dreg.registration_fgr_based_on_feature_matching(s, t, fs, ft)
    crit = o3dreg.ICPConvergenceCriteria(max_iteration=50)
    fine = o3dreg.icp(s, t, 0.1, g.transformation, None, crit)
    alone = o3dreg.icp(s, t, 2.0, np.eye(4), None, crit)
    dt_g, ang_g = pose_error(g.transformation.numpy(), T_true)
    dt, ang = pose_error(fine.transformation.numpy(), T_true)
    dt_a, ang_a = pose_error(alone.transformation.numpy(), T_true)
    print(f"fgr {dt_g:.4f} m {ang_g:.4f} deg; +icp {dt:.4f} m {ang:.4f} deg; icp alone {dt_a:.3f} m {ang_a:.2f} deg")
    assert dt_g < 0.1 and ang_g < 2.0, (dt_g, ang_g)
    assert dt < 0.02 and ang < 0.2, (dt, ang)
    assert dt_a > 1.0 or ang_a > 10.0
