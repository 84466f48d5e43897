"""GPU tests at the BASELINE.json sizes (C2 262k, C3 4x262k, C4 1.5M, C5 batched replay):
direct comparison with the oracle where it finishes in seconds, and size-independent
properties (conservation, ordering, sampled brute-force checks, replay == single-shot)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def big():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=1_600_000)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


def dev_bytes(msg):
    return torch.frombuffer(bytearray(msg.data), dtype=torch.uint8).cuda()


def test_c2_full_pipeline_262k(big):
    """configs[1]: the bench workload itself, bit-exact against the oracle."""
    import bench
    from oracle import pipeline as opipe
    ctx, engine, capi = big["ctx"], big["engine"], big["capi"]
    msg = bench.make_frames(1, seed0=77)[0]
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, dev_bytes(msg))
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                                  transforms=[bench.TF], crop=bench.CROP)
    out, counts, plane = ctx.pipeline_run([desc], engine.make_pipeline_cfg(fcfg, **bench.STAGES))
    ctx.check()
    ref = opipe.preprocess(msg, bench.oracle_config())
    c = counts.cpu().numpy()
    assert c[capi.CNT_FILTERED] == ref["n_filtered"] and c[capi.CNT_VOXELS] == ref["voxel_positions"].shape[0]
    assert c[capi.CNT_AFTER_RADIUS] == int(ref["radius_mask"].sum())
    assert c[capi.CNT_GROUND_INLIERS] == ref["ground_inliers"].size
    n = int(c[capi.CNT_OUTPUT])
    assert n == ref["positions"].shape[0]
    got = out[:n].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    assert np.allclose(plane.cpu().numpy()[:4], ref["plane"], atol=1e-5, rtol=0)


def test_c3_concat_4x262k_then_voxel(big):
    """configs[2]: 4 LiDARs (different byte layouts) merged in one launch, then 0.1 m voxels."""
    from oracle import pipeline as opipe
    from oracle import voxel
    ctx, engine, synth = big["ctx"], big["engine"], big["synth"]
    T = synth.sensor_extrinsics(4)
    scans = [synth.lidar_scan(seed=90 + s, nan_frac=0.0) for s in range(4)]
    msgs = [synth.pack_cloud(sc, lay) for sc, lay in zip(scans, ["xyzi16", "xyzirt22", "ouster48", "xyzi16"])]
    bufs = [dev_bytes(m) for m in msgs]
    descs = [engine.make_cloud_desc(m.fields, m.point_step, m.width, b, transform=T[s])
             for s, (m, b) in enumerate(zip(msgs, bufs))]
    out, counts, _ = ctx.pipeline_run(descs, engine.make_pipeline_cfg(engine.make_filter_cfg(), voxel_size=0.1))
    ctx.check()
    c = counts.cpu().numpy()
    assert c[big["capi"].CNT_INPUT] == 4 * 262144 == c[big["capi"].CNT_FILTERED]
    merged = opipe.concat(scans, list(T))
    ref = voxel.voxel_down_sample(merged["positions"], 0.1, merged["intensity"], fixed=True)
    v = int(c[big["capi"].CNT_OUTPUT])
    assert v == ref["positions"].shape[0]
    got = out[:v].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))


def test_c4_dense_1p5m_voxel_and_statistical(big):
    """configs[3]: 1.5 M points, 0.05 m voxels, statistical outlier removal k=20."""
    from oracle import outliers
    from oracle import voxel
    ctx, synth = big["ctx"], big["synth"]
    scan = synth.lidar_scan(seed=5, n_points=1_500_000, nan_frac=0.0, dup_frac=0.0)
    pos = scan["positions"]
    xyzi = torch.from_numpy(np.concatenate([pos, scan["intensity"][:, None]], 1)).cuda()
    out, p2v, vc, cnt = ctx.voxel_downsample(xyzi, 0.05, want_p2v=True, want_counts=True)
    ctx.check()
    v = int(cnt.item())
    p2v_h, vc_h = p2v.cpu().numpy(), vc[:v].cpu().numpy()
    # size-independent properties: conservation, membership consistency, first-occurrence order
    assert vc_h.sum() == pos.shape[0] and p2v_h.min() == 0 and p2v_h.max() == v - 1
    assert np.array_equal(np.bincount(p2v_h, minlength=v), vc_h)
    first = np.full(v, pos.shape[0], dtype=np.int64)
    np.minimum.at(first, p2v_h, np.arange(pos.shape[0]))
    assert np.all(np.diff(first) > 0)                                   # voxels numbered by first occurrence
    keys = voxel.pack_key(voxel.voxel_index(pos, 0.05))
    assert np.array_equal(keys, keys[first][p2v_h])                     # every point sits in its voxel's cell
    ref = voxel.voxel_down_sample(pos, 0.05, scan["intensity"], fixed=True)
    assert np.array_equal(out[:v].cpu().numpy()[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    # statistical outliers on the voxelised cloud (about 1.2 M points)
    cloud = out[:v].contiguous()
    host = cloud.cpu().numpy()[:, :3]
    mask, avg, stats = ctx.statistical_outliers(cloud, 20, 2.0)
    ctx.check()
    ref_mask, ref_avg = outliers.statistical_mask(host, 20, 2.0)
    assert np.array_equal(avg.cpu().numpy().view(np.uint32), ref_avg.view(np.uint32))
    assert np.array_equal(mask.cpu().numpy().astype(bool), ref_mask)
    # sampled exhaustive check, independent of the kd-tree: 64 queries against all points
    rng = np.random.default_rng(0)
    q = rng.choice(v, size=64, replace=False)
    d2 = outliers.d2_f32(host[q][:, None, :], host[None, :, :])
    d2.partition(19, axis=1)
    d = np.sqrt(np.sort(d2[:, :20], axis=1)).astype(np.float32)
    s = d[:, 0].copy()
    for j in range(1, 20):
        s = s + d[:, j]
    assert np.array_equal((s / np.float32(20)).view(np.uint32), avg.cpu().numpy()[q].view(np.uint32))


def test_c5_batched_replay_matches_single_shot(big):
    """configs[4] in small: multi-lane graph replay == one-scan-at-a-time pipeline, resident and
    host-to-host, repeated (tables must self-clean between scans)."""
    import bench
    from autodriver_pointcloud_preprocessor_b200 import replay
    ctx, engine, capi = big["ctx"], big["engine"], big["capi"]
    msgs = bench.make_frames(6, seed0=300)
    filter_kw = dict(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                     transforms=[bench.TF], crop=bench.CROP)
    pipe = replay.ScanPipeline(msgs[0].fields, bench.POINT_STEP, bench.N_POINTS, filter_kw, bench.STAGES, lanes=3)
    assert pipe.kernels_per_scan >= 10
    h_frames = [torch.frombuffer(bytearray(m.data), dtype=torch.uint8).pin_memory() for m in msgs]
    want = []
    for m in msgs:
        desc = engine.make_cloud_desc(m.fields, m.point_step, m.width, dev_bytes(m))
        out, counts, _ = ctx.pipeline_run([desc], pipe.pcfg)
        n = int(counts.cpu().numpy()[capi.CNT_OUTPUT])
        want.append(out[:n].cpu().numpy())
    for rep in range(2):
        outs, counts, d2h = pipe.process_host(h_frames)
        for f in range(len(msgs)):
            assert counts[f, capi.CNT_STATUS] == 0
            assert np.array_equal(outs[f].view(np.uint32), want[f].view(np.uint32)), (rep, f)
        assert d2h == sum(w.shape[0] * 16 + 32 for w in want)
    # views of the lanes' pinned output buffers: one frame per lane per call
    outs, _, _ = pipe.process_host(h_frames[:3], keep_outputs="view")
    for f in range(3):
        assert not outs[f].flags.owndata and np.array_equal(outs[f].view(np.uint32), want[f].view(np.uint32)), f
    with pytest.raises(ValueError):
        pipe.process_host(h_frames, keep_outputs="view")
    pool = torch.stack([h.cuda() for h in h_frames])
    arena = torch.zeros((len(msgs), bench.N_POINTS, 4), device="cuda")
    carena = torch.zeros((len(msgs), 8), dtype=torch.int32, device="cuda")
    pipe.prepare_resident(pool, arena, carena)
    for rep in range(2):
        arena.zero_()
        pipe.run_resident(list(range(len(msgs))))
        torch.cuda.synchronize()
        pipe.check()
        for f in range(len(msgs)):
            n = int(carena[f, capi.CNT_OUTPUT])
            assert np.array_equal(arena[f, :n].cpu().numpy().view(np.uint32), want[f].view(np.uint32)), (rep, f)
    # the multi-GPU path: graphs write the lanes' own buffers, every lane stages the frame's rows
    # into the send slab right behind the graph
    pipe.prepare_resident(pool, None, carena)
    rows = max(w.shape[0] for w in want) + 7
    slab = torch.zeros((len(msgs), rows, 4), device="cuda")
    pipe.run_resident(list(range(len(msgs))), stage_to=slab)
    torch.cuda.synchronize()
    for f in range(len(msgs)):
        n = int(carena[f, capi.CNT_OUTPUT])
        assert n == want[f].shape[0]
        assert np.array_equal(slab[f, :n].cpu().numpy().view(np.uint32), want[f].view(np.uint32)), f
    pipe.close()


def test_bench_dump_outputs_are_the_last_steps_results(big, tmp_path):
    """bench.py --dump-outputs: the counters of every frame and the rows / plane of each lane's last frame,
    as the timed steps left them, equal one-scan-at-a-time runs of the same frames; --steps sets the
    number of timed steps."""
    import json
    import os
    import subprocess
    import sys
    import bench
    ctx, engine, capi = big["ctx"], big["engine"], big["capi"]
    FT, lanes, steps = 10, 3, 2
    r = subprocess.run([sys.executable, os.path.abspath(bench.__file__), "--steps", str(steps), "--frames-total", str(FT),
                        "--lanes", str(lanes), "--no-configs", "--no-cpu-baseline", "--no-e2e",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == steps
    counts = np.load(tmp_path / "counts.npy")
    assert counts.dtype == np.float64 and counts.shape == (FT, 8)
    assert sorted(os.listdir(tmp_path)) == ["counts.npy"] + [f"{k}_{f:05d}.npy" for k in ("plane", "xyzi")
                                                             for f in range(FT - lanes, FT)]
    block = bench.make_c5_block(0, FT, workers=1)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                                  transforms=[bench.TF], crop=bench.CROP)
    pcfg = engine.make_pipeline_cfg(fcfg, **bench.STAGES)
    fields = bench.frame_msg(b"").fields
    for f in range(FT):
        data = torch.from_numpy(block[f].copy()).cuda()
        out, c, plane = ctx.pipeline_run([engine.make_cloud_desc(fields, bench.POINT_STEP, bench.N_POINTS, data)], pcfg)
        ctx.check()
        c = c.cpu().numpy()
        assert np.array_equal(counts[f], c.astype(np.float64)), f
        if f >= FT - lanes:
            rows = np.load(tmp_path / f"xyzi_{f:05d}.npy")
            assert rows.dtype == np.float32
            assert np.array_equal(rows.view(np.uint32), out[:int(c[capi.CNT_OUTPUT])].cpu().numpy().view(np.uint32)), f
            assert np.array_equal(np.load(tmp_path / f"plane_{f:05d}.npy"), plane.cpu().numpy()), f


def test_c1_full_size_131072_crop_voxel_ground(big):
    """configs[0] at its own size: 64 x 2048 = 131 072 points, crop_box + 0.1 m voxels + RANSAC ground
    removal, every intermediate count and the published rows bit-exact against the oracle."""
    import bench
    from oracle import pipeline as opipe
    ctx, engine, capi, synth = big["ctx"], big["engine"], big["capi"], big["synth"]
    msg = synth.pack_cloud(synth.lidar_scan(seed=64, n_beams=64, n_az=2048), "xyzi16")
    assert msg.width == 131072
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, dev_bytes(msg))
    ground = dict(distance_threshold=0.2, ransac_n=5, num_iterations=100, probability=0.99, seed=7)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                                  crop=bench.CROP)
    out, counts, plane = ctx.pipeline_run([desc], engine.make_pipeline_cfg(fcfg, voxel_size=0.1, ground=ground))
    ctx.check()
    cfg = opipe.default_config()
    cfg.update(crop=bench.CROP, voxel_size=0.1, ground=ground)
    ref = opipe.preprocess(msg, cfg)
    c = counts.cpu().numpy()
    assert c[capi.CNT_INPUT] == 131072 and c[capi.CNT_FILTERED] == ref["n_filtered"]
    assert c[capi.CNT_VOXELS] == ref["voxel_positions"].shape[0]
    assert c[capi.CNT_GROUND_INLIERS] == ref["ground_inliers"].size
    n = int(c[capi.CNT_OUTPUT])
    assert n == ref["positions"].shape[0]
    got = out[:n].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    assert np.allclose(plane.cpu().numpy()[:4], ref["plane"], atol=1e-5, rtol=0)


def test_concat_eight_sensors_at_the_cloud_limit(big):
    """APC_MAX_CLOUDS = 8 sensors of three byte layouts, ragged sizes (one empty), each with its own
    extrinsic, merged in one launch and voxelised: sensor order and point order preserved."""
    from oracle import pipeline as opipe
    from oracle import voxel
    ctx, engine, capi, synth = big["ctx"], big["engine"], big["capi"], big["synth"]
    layouts = ["xyzi16", "xyzirt22", "ouster48", "xyzi16", "xyzirt22", "ouster48", "xyzi16", "xyzirt22"]
    sizes = [(32, 1024), (16, 777), (8, 1), (64, 512), (32, 333), (16, 1024), (128, 256), (32, 1025)]
    T = np.concatenate([synth.sensor_extrinsics(4), synth.sensor_extrinsics(4)])
    T[4:, :3, 3] += np.array([3.0, -2.0, 0.5], dtype=np.float32)
    scans, msgs = [], []
    for s, ((nb, na), lay) in enumerate(zip(sizes, layouts)):
        sc = synth.lidar_scan(seed=200 + s, n_beams=nb, n_az=na, nan_frac=0.0, dup_frac=0.0)
        if s == 2:                                              # an empty sensor in the middle
            sc = {k: v[:0] for k, v in sc.items()}
        scans.append(sc)
        msgs.append(synth.pack_cloud(sc, lay))
    bufs = [dev_bytes(m) if m.width else torch.zeros(16, dtype=torch.uint8, device="cuda") for m in msgs]
    descs = [engine.make_cloud_desc(m.fields, m.point_step, m.width, b, transform=T[s])
             for s, (m, b) in enumerate(zip(msgs, bufs))]
    assert len(descs) == capi.APC_MAX_CLOUDS
    fcfg = engine.make_filter_cfg()
    xyzi, src, _, cnt = ctx.frontend(descs, fcfg, want_src=True)
    ctx.check()
    merged = opipe.concat(scans, list(T))
    n = int(cnt.item())
    assert n == merged["positions"].shape[0] == sum(m.width for m in msgs)
    got = xyzi[:n].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), merged["positions"].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), merged["intensity"].view(np.uint32))
    assert np.array_equal(src[:n].cpu().numpy(), np.arange(n))
    out, counts, _ = ctx.pipeline_run(descs, engine.make_pipeline_cfg(fcfg, voxel_size=0.1))
    ctx.check()
    ref = voxel.voxel_down_sample(merged["positions"], 0.1, merged["intensity"], fixed=True)
    v = int(counts.cpu().numpy()[capi.CNT_OUTPUT])
    assert v == ref["positions"].shape[0]
    assert np.array_equal(out[:v].cpu().numpy()[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    # a ninth sensor is refused
    with pytest.raises(capi.ApcError):
        ctx.frontend(descs + [descs[0]], fcfg, want_src=False)


def test_low_latency_mode_is_bit_identical(big):
    """apc_ctx_set_low_latency (programmatic dependent launches): same counters, rows and plane as the
    ordinary launches, eager and as a replayed graph, C2 size, five replays."""
    import bench
    from autodriver_pointcloud_preprocessor_b200 import engine as eng
    capi = big["capi"]
    msg = bench.make_frames(1, seed0=91)[0]
    data = dev_bytes(msg)
    fcfg = eng.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True,
                               transforms=[bench.TF], crop=bench.CROP)
    pcfg = eng.make_pipeline_cfg(fcfg, **bench.STAGES)
    res = {}
    for mode in (False, True):
        ctx = eng.Context(max_points=msg.width)
        ctx.set_low_latency(mode)
        desc = eng.make_cloud_desc(msg.fields, msg.point_step, msg.width, data)
        out, counts, plane = ctx.pipeline_run([desc], pcfg)
        ctx.check()
        c = counts.cpu().numpy().copy()
        n = int(c[capi.CNT_OUTPUT])
        res[mode] = (c, out[:n].cpu().numpy().copy(), plane.cpu().numpy().copy())
        o2 = torch.zeros_like(out)
        c2 = torch.zeros_like(counts)
        p2 = torch.zeros_like(plane)
        g = ctx.capture_pipeline([desc], pcfg, o2, c2, p2)
        for _ in range(5):
            o2.zero_()
            ctx.launch_graph(g)
            ctx.check()
            assert np.array_equal(c2.cpu().numpy(), c)
            assert np.array_equal(o2[:n].cpu().numpy().view(np.uint32), res[mode][1].view(np.uint32))
        ctx.close()
    assert np.array_equal(res[False][0], res[True][0])
    assert np.array_equal(res[False][1].view(np.uint32), res[True][1].view(np.uint32))
    assert np.array_equal(res[False][2], res[True][2])
