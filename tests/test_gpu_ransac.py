"""RANSAC plane segmentation on the GPU against ``oracle/ransac.py`` where the kernels are delicate: the
float32 pre-test's rounding band and its float64 re-decision (queued, or inline once the queue is
full), the packed per-thread count + error accumulator, the prefix-record selection with its early
stop, the final pass, and the argument checks.  Every case asserts, through the band model of
``ransac_cases``, that it reaches the path it targets, and prints the counts."""
import contextlib

import numpy as np
import pytest

import ransac_cases as rc

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
NONE = 0xFFFFFFFF


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=310_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


@contextlib.contextmanager
def scored_once():
    """``oracle.ransac.score`` is a pure function of (points, plane, thr): while the oracle runs, a
    plane that recurs in a sample table (permuted anchors, copied rows) is scored once."""
    from oracle import ransac
    orig, cache = ransac.score, {}

    def score(P64, plane, thr):
        k = (id(P64), plane.tobytes(), float(thr))
        if k not in cache:
            cache[k] = orig(P64, plane, thr)
        return cache[k]

    ransac.score = score
    try:
        yield
    finally:
        ransac.score = orig


def to_dev(pts):
    x = np.zeros((pts.shape[0], 4), dtype=np.float32)
    x[:, :3] = pts[:, :3]
    return torch.from_numpy(x).cuda()


def run_gpu(ctx, xyzi, thr, ransac_n, iters, prob, seed, table, nd):
    plane8, mask, info = ctx.segment_plane(xyzi, thr, ransac_n, iters, prob, seed=seed, sample_table=table, n_dev=nd)
    ctx.check()
    scores = ctx.segment_plane_scores(iters)
    return (plane8.cpu().numpy().copy(), mask.cpu().numpy().copy(), info.cpu().numpy().astype(np.int64) & NONE,
            scores.cpu().numpy().copy())


def compare(ctx, pts, thr, ransac_n, iters, prob=0.99, seed=0, table=None, n_dev=None):
    """``ctx.segment_plane`` twice (bit-identical runs) against ``oracle.ransac.segment_plane`` on the first
    ``n_dev`` points.  Returns the oracle's info dict (``None`` when there is no hypothesis)."""
    from oracle import ransac
    n_max = pts.shape[0]
    P = n_max if n_dev is None else n_dev
    xyzi = to_dev(pts)
    nd = None if n_dev is None else torch.tensor([n_dev], dtype=torch.int32, device="cuda")
    a = run_gpu(ctx, xyzi, thr, ransac_n, iters, prob, seed, table, nd)
    b = run_gpu(ctx, xyzi, thr, ransac_n, iters, prob, seed, table, nd)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))           # deterministic
    plane8, mask, info, scores = a
    assert not mask[P:].any()
    if P < ransac_n:
        assert info[0] == NONE and info[1] == 0 and not mask.any() and not plane8.any()
        return None
    with scored_once():
        ref_plane, ref_inl, ri = ransac.segment_plane(np.ascontiguousarray(pts[:P, :3]), thr, ransac_n, iters, prob,
                                                      seed=seed, samples=table)
    valid = np.any(ri["planes"] != 0.0, axis=1)
    ref_scores = np.array(ri["scores"], dtype=np.int64).reshape(iters, 2)
    assert np.array_equal(scores[valid], ref_scores[valid])               # (count, err) of every valid hypothesis
    best = ri["best_it"]
    assert info[0] == (NONE if best < 0 else best)
    assert info[1] == ref_inl.size
    assert np.array_equal(np.flatnonzero(mask[:P]), ref_inl)
    if best < 0:
        assert not plane8.any()
        return ri
    assert np.array_equal(plane8[4:].view(np.uint64), ri["best_plane"].view(np.uint64))
    if ref_inl.size >= 3:                     # fewer inliers fit no plane: the refit is undefined there
        assert np.allclose(plane8[:4], ref_plane, rtol=0, atol=1e-5)
    return ri


def report(name, b, n_max):
    q = rc.queue_entries(n_max, b["in_band"], b["ch"])
    print(f"{name}: CH={b['ch']} in-band={int(b['in_band'].sum())} disagreements={int(b['disagree'].sum())} "
          f"sure-inliers={int(b['sure_in'].sum())} CTAs overflowing the queue={int((q > rc.QCAP).sum())}/{q.size}")
    return q


# ---- 1. rounding band near the origin ----------------------------------------------------------------
@pytest.mark.parametrize("thr", [0.25, 0.2, 0.0137])
def test_rounding_band_near_origin(env, thr):
    pts, table, meta = rc.band_cloud(thr)
    b = rc.band(pts, rc.planes_of(pts, table), thr)
    report(f"band thr={thr}", b, pts.shape[0])
    assert b["disagree"].sum() >= 50
    assert (meta["exact_ties"] > 0) == (thr == 0.25)
    compare(env["ctx"], pts, thr, 3, 40, table=table)


# ---- 2. queue overflow ----------------------------------------------------------------------------------
def test_queue_overflow(env):
    pts, table, thr = rc.all_ambiguous_cloud()
    b = rc.band(pts, rc.planes_of(pts, table), thr)
    q = report("all ambiguous", b, pts.shape[0])
    assert b["in_band"][0].all() and q.min() > rc.QCAP
    compare(env["ctx"], pts, thr, 3, 20, table=table)


# ---- 3. far from the origin -----------------------------------------------------------------------------
FAR = [(30000.0, -20000.0, 5.0), (-65000.0, 65000.0, -100.0)]


@pytest.mark.parametrize("centre", FAR)
@pytest.mark.parametrize("thr", [0.2, 0.01])
def test_far_from_origin(env, centre, thr):
    scan = env["synth"].lidar_scan(seed=9, n_beams=32, n_az=1024, nan_frac=0.0)
    pts = (scan["positions"].astype(np.float64) + np.asarray(centre)).astype(np.float32)
    ri = compare(env["ctx"], pts, thr, 3, 100, seed=11)
    b = rc.band(pts, ri["planes"], thr)
    report(f"far {centre} thr={thr}", b, pts.shape[0])
    assert b["in_band"].sum() > 5000
    if thr == 0.01:
        assert not b["sure_in"].any()                                      # m > thr: every inlier via float64


@pytest.mark.parametrize("graph", [False, True])
def test_far_from_origin_pipeline(env, graph):
    """C1 stages (voxel 0.1 + ground) with the scan moved to (30000, -20000, 0), eager and replayed."""
    from oracle import pipeline as opipe
    ctx, engine, synth, capi = env["ctx"], env["engine"], env["synth"], env["capi"]
    msg = synth.pack_cloud(synth.lidar_scan(seed=31, n_beams=32, n_az=1024), "xyzirt22")
    data = torch.frombuffer(bytearray(msg.data), dtype=torch.uint8).cuda()
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, data)
    T = np.eye(4)
    T[:3, 3] = (30000.0, -20000.0, 0.0)
    crop = dict(min=[29940.0, -20060.0, -20.0], max=[30060.0, -19940.0, 20.0], invert=False, mode=capi.CROP_OPEN3D)
    stages = dict(voxel_size=0.1, ground=dict(distance_threshold=0.2, ransac_n=5, num_iterations=100, probability=0.99,
                                              seed=7))
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                                  transforms=[T], crop=crop)
    pcfg = engine.make_pipeline_cfg(fcfg, **stages)
    out = torch.zeros((msg.width, 4), device="cuda")
    counts = torch.zeros(8, dtype=torch.int32, device="cuda")
    plane = torch.zeros(8, dtype=torch.float64, device="cuda")
    if graph:
        g = ctx.capture_pipeline([desc], pcfg, out, counts, plane)
        out.zero_(); counts.zero_()
        for _ in range(2):
            ctx.launch_graph(g)
    else:
        ctx.pipeline_run([desc], pcfg, out, counts, plane)
    ctx.check()
    cfg = opipe.default_config()
    cfg.update(transforms=[T], crop=crop, voxel_size=0.1, ground=stages["ground"])
    ref = opipe.preprocess(msg, cfg)
    c = counts.cpu().numpy()
    assert c[capi.CNT_STATUS] == 0 and c[capi.CNT_FILTERED] == ref["n_filtered"]
    n_out = int(c[capi.CNT_OUTPUT])
    assert n_out == ref["positions"].shape[0]
    got = out[:n_out].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    assert int(c[capi.CNT_GROUND_INLIERS]) == ref["ground_inliers"].size > 1000
    assert np.allclose(plane.cpu().numpy()[:4], ref["plane"], rtol=0, atol=1e-5)


# ---- 4. early stop ------------------------------------------------------------------------------------
@pytest.mark.parametrize("target,winner,later,iters,n", [(60, 20, 90, 128, 3), (300, 150, 420, 1000, 4)])
def test_early_stop(env, target, winner, later, iters, n):
    pts, table, meta = rc.planted_ground_cloud(target, winner, later, iters, ransac_n=n)
    ri = compare(env["ctx"], pts, 0.2, n, iters, table=table)
    sc = ri["scores"]
    print(f"early stop: winner {winner} ({sc[winner][0]} inliers), bound {meta['bound']:.6f}, "
          f"row {later} has {sc[later][0]}")
    assert ri["best_it"] == winner < meta["bound"] < later and sc[later][0] > sc[winner][0]


# ---- 5. selection over many chunks ----------------------------------------------------------------------
@pytest.mark.parametrize("winner", [127, 128, 255, 256, 4095])
def test_selection_over_many_chunks(env, winner):
    pts, table, meta = rc.selection_cloud(winner)
    assert pts.shape[0] >= 40 * 1024
    ri = compare(env["ctx"], pts, 0.2, 3, 4096, prob=1.0, table=table)
    sc = ri["scores"]
    print(f"selection: winner {winner}, ties {meta['tie_rows']}, copies {meta['dup_rows']}")
    assert ri["best_it"] == winner
    assert all(sc[r] == sc[winner] for r in meta["dup_rows"])
    assert all(sc[r][0] == sc[winner][0] and sc[r][1] > sc[winner][1] for r in meta["tie_rows"])


# ---- 6. accumulator saturation --------------------------------------------------------------------------
def test_accumulator_saturation(env):
    pts, table = rc.saturation_cloud()
    b = rc.band(pts, rc.planes_of(pts, table[:16]), 0.2, ch=16)
    report("saturation (first chunk)", b, pts.shape[0])
    assert b["sure_in"].all()
    ri = compare(env["ctx"], pts, 0.2, 3, 4096, table=table)
    assert ri["best_it"] == 0 and ri["scores"][0][0] == pts.shape[0]


# ---- 7. degenerate hypotheses and extreme outcomes ----------------------------------------------------
def test_degenerate_rows_are_never_selected(env):
    pts = rc.ground_clutter_cloud(3000, seed=6)
    pts[:3] = [[1, 1, 1], [2, 2, 2], [3, 3, 3]]                           # collinear
    rng = np.random.default_rng(6)
    table = rng.integers(3, 3000, size=(60, 3)).astype(np.int32)
    table[::3] = [0, 1, 2]
    table[1::3, 1] = table[1::3, 0]                                       # a repeated index
    ri = compare(env["ctx"], pts, 0.2, 3, 60, table=table)
    planes = ri["planes"]
    assert not planes[::3].any() and not planes[1::3].any()
    assert ri["best_it"] % 3 == 2


def test_all_hypotheses_degenerate(env):
    pts = rc.ground_clutter_cloud(2000, seed=7)
    table = np.tile(np.array([[5, 5, 9], [1, 2, 2], [7, 7, 7]], dtype=np.int32), (10, 1))
    ri = compare(env["ctx"], pts, 0.2, 3, 30, table=table)
    assert ri["best_it"] == -1


def test_every_point_an_inlier(env):
    """inl == P sets the bound to 0: the first valid record wins, even over later rows with a smaller error."""
    rng = np.random.default_rng(8)
    xy = rng.integers(-4096, 4096, size=(5000, 2)) / 256.0
    on = np.concatenate([xy, 0.5 * xy[:, :1] + 0.25 * xy[:, 1:]], 1).astype(np.float32)   # exactly on z = x/2 + y/4
    table = rng.integers(0, 5000, size=(64, 3)).astype(np.int32)
    table[0] = [3, 3, 4]
    ri = compare(env["ctx"], on, 0.2, 3, 64, table=table)
    assert ri["best_it"] == 1 and ri["scores"][1][0] == 5000
    near = on + np.float32([0, 0, 1]) * rng.uniform(-0.01, 0.01, size=(5000, 1)).astype(np.float32)
    ri = compare(env["ctx"], near, 0.2, 3, 64, table=table)
    sc = ri["scores"]
    assert ri["best_it"] == 1 and sc[1][0] == 5000
    assert any(s[0] == 5000 and s[1] < sc[1][1] for s in sc[2:])             # a later row would win without the stop


def test_tiny_probability(env):
    """p = 1e-6: the bound is below 1, so the first row with inliers wins."""
    pts = rc.ground_clutter_cloud(4000, seed=9)
    table = np.random.default_rng(9).integers(0, 4000, size=(50, 3)).astype(np.int32)
    table[:3] = [[2, 2, 2], [0, 0, 1], [4, 5, 5]]
    ri = compare(env["ctx"], pts, 0.2, 3, 50, prob=1e-6, table=table)
    valid = np.any(ri["planes"] != 0.0, axis=1)
    first = min(it for it in range(50) if valid[it] and ri["scores"][it][0] > 0)
    assert ri["best_it"] == first >= 3
    assert any(s[0] > ri["scores"][first][0] for s in ri["scores"][first + 1:])


def test_non_finite_points(env):
    pts = rc.ground_clutter_cloud(5000, seed=10)
    pts[[10, 500, 1023, 1024, 4999]] = [[np.nan, 1, 1], [1, np.inf, 1], [-np.inf, 0, 0], [0, 0, np.nan],
                                        [np.inf, -np.inf, np.nan]]
    rng = np.random.default_rng(10)
    table = rng.integers(0, 5000, size=(40, 3)).astype(np.int32)
    table[5] = [10, 20, 30]
    table[17] = [500, 1024, 40]
    ri = compare(env["ctx"], pts, 0.2, 3, 40, table=table)
    assert not ri["planes"][5].any() and not ri["planes"][17].any()     # a non-finite sample: a zero plane
    compare(env["ctx"], pts, 0.2, 5, 100, seed=3)


# ---- 8. shapes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ransac_n", [3, 4, 15, 16])
@pytest.mark.parametrize("P", ["n", "n+1", 1023, 1024, 1025])
def test_shapes(env, ransac_n, P):
    P = {"n": ransac_n, "n+1": ransac_n + 1}.get(P, P)
    pts = rc.ground_clutter_cloud(P, seed=100 + P + ransac_n)
    for iters in (1, 15, 16, 17, 20, 21, 127, 128, 129):
        compare(env["ctx"], pts, 0.2, ransac_n, iters, seed=iters)


# ---- 9. device count and arguments ----------------------------------------------------------------------
def test_device_count(env):
    ctx = env["ctx"]
    pts = rc.ground_clutter_cloud(6000, seed=11)
    compare(ctx, pts, 0.2, 5, 100, seed=4, n_dev=4321)
    table = np.random.default_rng(11).integers(0, 900, size=(40, 3)).astype(np.int32)
    compare(ctx, pts, 0.2, 3, 40, table=table, n_dev=900)
    compare(ctx, pts, 0.2, 5, 100, seed=4, n_dev=4)                       # fewer points than ransac_n
    compare(ctx, pts, 0.2, 5, 100, seed=4, n_dev=0)
    empty = torch.zeros((0, 4), device="cuda")
    plane8, mask, info = ctx.segment_plane(empty, 0.2, 3, 10, 0.99, n_dev=torch.zeros(1, dtype=torch.int32, device="cuda"))
    ctx.check()
    assert (int(info[0]) & NONE) == NONE and int(info[1]) == 0 and not plane8.cpu().numpy().any()


def test_bad_arguments_and_recovery(env):
    capi, ctx = env["capi"], env["ctx"]
    pts = rc.ground_clutter_cloud(3000, seed=12)
    xyzi = to_dev(pts)
    good = dict(distance_threshold=0.2, ransac_n=5, num_iterations=50, probability=0.99)
    bad = [(dict(ransac_n=2), capi.APC_ERR_BAD_ARG), (dict(ransac_n=17), capi.APC_ERR_BAD_ARG),
           (dict(num_iterations=0), capi.APC_ERR_BAD_ARG), (dict(num_iterations=4097), capi.APC_ERR_BAD_ARG),
           (dict(probability=0.0), capi.APC_ERR_BAD_ARG), (dict(probability=1.5), capi.APC_ERR_BAD_ARG),
           (dict(probability=float("nan")), capi.APC_ERR_BAD_ARG), (dict(distance_threshold=0.0), capi.APC_ERR_BAD_ARG),
           (dict(distance_threshold=-1.0), capi.APC_ERR_BAD_ARG),
           (dict(distance_threshold=float("nan")), capi.APC_ERR_BAD_ARG)]
    for k, (kw, code) in enumerate(bad):
        args = dict(good, **kw)
        with pytest.raises(capi.ApcError) as e:
            ctx.segment_plane(xyzi, args["distance_threshold"], args["ransac_n"], args["num_iterations"],
                              args["probability"], seed=k)
        assert e.value.code == code, kw
        compare(ctx, pts, 0.2, 5, 50, seed=k)
    with pytest.raises(capi.ApcError) as e:
        ctx.segment_plane(xyzi[:4].contiguous(), 0.2, 5, 50, 0.99)
    assert e.value.code == capi.APC_ERR_TOO_FEW
    compare(ctx, pts, 0.2, 5, 50, seed=99)

