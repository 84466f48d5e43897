"""The open-addressing tables under every stage, fed inputs built to collide: the duplicate table of the open3d back
end (k_dedup_insert / k_frontend, k_dup_insert_soa), the voxel table (k_voxel_insert / k_voxel_finalize) and the
single-level and KNN neighbour grids (grid_insert_*, grid_resolve).

Realistic scans keep these tables at a load of at most 0.25, so probe chains stay one or two slots long, seldom wrap
from the last slot to slot 0, and the fingerprint-collision branch of the duplicate table never runs.  The inputs here
come from the numpy models in ``test_hash_models.py`` (the hashes are bijections, so exact collisions can be computed):
  * distinct points with one identical 64-bit duplicate hash (same fingerprint, same home slot: the table's last),
    so every insert confirms the fingerprint by reading the representative's x/y/z back and probes on;
  * voxels of 64 distinct 2x2 blocks whose block hash lands in the table's last block, so the voxel chains wrap;
  * isolated decoy points whose cells home onto the slots of a dense cloud's cells and of their empty neighbours, so
    lookups walk past foreign keys before they find their key or an empty slot;
  * coordinates, voxel sizes and intensities at the edges of the voxel stage's fixed-point domain, and fixed-point
    sums above 2^53 where the int64 -> float64 conversion rounds.
Every assertion compares with the CPU oracle; the models only choose the inputs.  Each adversarial call is followed by
an ordinary one through the same context: a slot left occupied by the self-cleaning shows up there."""
import numpy as np
import pytest

import test_hash_models as hm
from test_gpu_normals_search import assert_parity, dense_patch
from test_gpu_stages import dev_bytes, oracle_frontend

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

MAXP = 32768                    # small tables: a wrapping chain costs a few thousand atomics


@pytest.fixture(scope="module")
def env():
    from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth
    ctx = engine.Context(max_points=MAXP)
    yield dict(ctx=ctx, engine=engine, capi=_capi, synth=synth)
    ctx.close()


def to_xyzi(p, w=None):
    w = np.zeros(p.shape[0], np.float32) if w is None else w
    return torch.from_numpy(np.ascontiguousarray(np.concatenate([p, w[:, None]], 1), np.float32)).cuda()


# ==== 1. duplicate table ============================================================================================
def chain_points(rng, k, low32):
    """k distinct finite points with one 64-bit duplicate hash whose low 32 bits are ``low32``."""
    h = (int(rng.integers(1, 2**32)) << 32) | low32
    kz = np.unique(np.float32(rng.uniform(-4.0, 4.0, 2 * k + 64)).view(np.uint32))
    p = hm.same_hash_points(h, rng.permutation(kz))[:k]
    assert p.shape[0] == k and np.all(hm.dedup_hash(p) == np.uint64(h))
    return p


def collision_cloud(synth, seed):
    """Chains of 1000, 33 and 2 same-hash points (homes: the last slot, 16 slots before it, anywhere), 1-3 exact
    duplicates of each, one in ten rows with a NaN intensity (dropped by read_points' NaN skip), and a small scan,
    shuffled over 11 tiles of 1024 so that duplicates often come before the point they copy."""
    rng = np.random.default_rng(seed)
    distinct = np.concatenate([chain_points(rng, 1000, 0xffffffff), chain_points(rng, 33, 0xfffffff0),
                               chain_points(rng, 2, int(rng.integers(0, 2**32)))])
    rows = np.concatenate([distinct, np.repeat(distinct, rng.integers(1, 4, distinct.shape[0]), axis=0)])
    inten = rng.uniform(0.0, 255.0, rows.shape[0]).astype(np.float32)
    inten[rng.random(rows.shape[0]) < 0.1] = np.nan
    scan = synth.lidar_scan(seed=seed, n_beams=16, n_az=512)
    pos = np.concatenate([rows, scan["positions"]])
    inten = np.concatenate([inten, scan["intensity"]])
    perm = rng.permutation(pos.shape[0])
    return dict(positions=np.ascontiguousarray(pos[perm]), intensity=inten[perm],
                ring=np.zeros(pos.shape[0], np.uint16), time=np.zeros(pos.shape[0], np.float32))


def pack(synth, cloud, layout):
    with np.errstate(invalid="ignore", over="ignore"):            # ouster48's range field of x, y up to 3e38
        return synth.pack_cloud(cloud, layout)


def run_frontend(env, descs):
    cfg = env["engine"].make_filter_cfg(skip_nans=True, dedup_mode=env["capi"].DEDUP_OPEN3D)
    xyzi, src, stage, cnt = env["ctx"].frontend(descs, cfg, want_src=True, want_stage=True)
    env["ctx"].check()
    m = int(cnt.item())
    return xyzi[:m].cpu().numpy(), src[:m].cpu().numpy().astype(np.uint32), stage.cpu().numpy()


def assert_frontend(got, ref):
    (xyzi, src, stage), (p_ref, i_ref, src_ref, stage_ref) = got, ref
    assert np.array_equal(stage, stage_ref)                        # per-point stage mask, bit-exact
    assert np.array_equal(src, src_ref)                            # surviving indices, in order
    assert np.array_equal(xyzi[:, :3].view(np.uint32), p_ref.view(np.uint32))
    assert np.array_equal(xyzi[:, 3].view(np.uint32), i_ref.view(np.uint32))


def ordinary_frontend(env, seed=90):
    """An ordinary scan through the same context: a duplicate slot left occupied merges or drops its points."""
    msg = env["synth"].pack_cloud(env["synth"].lidar_scan(seed=seed, n_beams=32, n_az=512), "xyzi16")
    desc = env["engine"].make_cloud_desc(msg.fields, msg.point_step, msg.width, dev_bytes(msg))
    assert_frontend(run_frontend(env, [desc]), oracle_frontend(msg, dict(skip_nans=True), dedup=True))


@pytest.fixture(scope="module")
def collisions(env):
    return collision_cloud(env["synth"], 7)


@pytest.mark.parametrize("layout", ["xyzi16", "xyzirt22", "ouster48", "xyzi16+1"])
def test_dedup_same_hash_chains(env, collisions, layout):
    """k_dedup_insert / k_frontend on wrapping chains of same-fingerprint distinct points, through the FAST16 path
    (xyzi16), the generic staged path (unaligned 22-byte records, 48-byte records) and a 16-byte layout whose device
    pointer is one byte off (neither FAST16 nor bulk-copied)."""
    synth, engine = env["synth"], env["engine"]
    msg = pack(synth, collisions, layout.split("+")[0])
    data = dev_bytes(msg)
    if layout.endswith("+1"):
        buf = torch.zeros(data.numel() + 1, dtype=torch.uint8, device="cuda")
        buf[1:] = data
        data = buf[1:]
        assert data.data_ptr() % 16 == 1
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, data)
    ref = oracle_frontend(msg, dict(skip_nans=True), dedup=True)
    assert ref[2].size > 2000
    for _ in range(2):
        assert_frontend(run_frontend(env, [desc]), ref)
    ordinary_frontend(env)


def test_dedup_across_segments(env):
    """Representatives in sensor 0 (xyzi16), same-hash distinct points in sensors 2 (ouster48) and 3 (xyzirt22),
    true duplicates of sensor 0's points in sensor 3, and an empty sensor 1 in between: the fingerprint confirm must
    read each representative with its own sensor's record layout."""
    synth, engine = env["synth"], env["engine"]
    rng = np.random.default_rng(11)
    same = chain_points(rng, 240, 0xffffffff)
    reps, far2, far3 = same[:80], same[80:160], same[160:]
    scans = [synth.lidar_scan(seed=40 + s, n_beams=16, n_az=256) for s in range(3)]

    def seg(pts, scan):
        pos = np.concatenate([pts, scan["positions"]])
        inten = np.concatenate([rng.uniform(0.0, 255.0, pts.shape[0]).astype(np.float32), scan["intensity"]])
        inten[rng.random(pos.shape[0]) < 0.05] = np.nan
        perm = rng.permutation(pos.shape[0])
        return dict(positions=np.ascontiguousarray(pos[perm]), intensity=inten[perm],
                    ring=np.zeros(pos.shape[0], np.uint16), time=np.zeros(pos.shape[0], np.float32))

    empty = dict(positions=np.zeros((0, 3), np.float32), intensity=np.zeros(0, np.float32))
    clouds = [seg(reps, scans[0]), seg(empty["positions"], empty), seg(far2, scans[1]),
              seg(np.concatenate([far3, reps, reps[::3]]), scans[2])]
    msgs = [pack(synth, c, lay) for c, lay in zip(clouds, ["xyzi16", "xyzirt22", "ouster48", "xyzirt22"])]
    datas = [dev_bytes(m) if m.width else torch.zeros(16, dtype=torch.uint8, device="cuda") for m in msgs]
    descs = [engine.make_cloud_desc(m.fields, m.point_step, m.width, d) for m, d in zip(msgs, datas)]
    from oracle import dedup as odedup
    from oracle import filters, pc2
    pos, inten, skip = [], [], []
    for m in msgs:
        arr = pc2.read_points(m, skip_nans=False)
        pos.append(np.vstack((arr["x"], arr["y"], arr["z"])).T.astype(np.float32))
        inten.append(arr["intensity"].astype(np.float32))
        skip.append(pc2.read_points_mask(m, skip_nans=True))
    pos, inten = np.concatenate(pos), np.concatenate(inten)
    p_ref, src_ref, stage_ref = filters.frontend(pos, nanskip_mask=np.concatenate(skip), dedup_mask_fn=odedup.open3d_mask,
                                                 remove_nan=False, remove_infinite=False)
    n0 = msgs[0].width
    rep_bits = {r.tobytes() for r in reps}
    assert sum(r.tobytes() in rep_bits for r in pos[n0:]) >= 80   # sensor 3 holds copies of sensor 0's points
    for _ in range(2):
        assert_frontend(run_frontend(env, descs), (p_ref, inten[src_ref], src_ref, stage_ref))
    ordinary_frontend(env)


def test_duplicate_mask_same_hash_chains(env, collisions):
    """The stand-alone SoA table (k_dup_insert_soa / k_dup_mask_soa) on the same chains."""
    from oracle import dedup as odedup
    ctx = env["ctx"]
    pos = collisions["positions"]
    xyzi = to_xyzi(pos, collisions["intensity"])
    ref = odedup.open3d_mask(pos)
    for _ in range(2):
        m = ctx.duplicate_mask(xyzi)
        ctx.check()
        assert np.array_equal(m.cpu().numpy().astype(bool), ref)
    plain = env["synth"].lidar_scan(seed=91, n_beams=32, n_az=512)["positions"]
    m = ctx.duplicate_mask(to_xyzi(plain))
    ctx.check()
    assert np.array_equal(m.cpu().numpy().astype(bool), odedup.open3d_mask(plain))


def test_dedup_pipeline_eager_and_graph(env, collisions):
    from oracle import pipeline as opipe
    ctx, engine, capi = env["ctx"], env["engine"], env["capi"]
    msg = pack(env["synth"], collisions, "xyzirt22")
    data = dev_bytes(msg)
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, data)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True)
    pcfg = engine.make_pipeline_cfg(fcfg, voxel_size=0.0)
    cfg = opipe.default_config()
    cfg.update(crop=None, voxel_size=0.0)
    ref = opipe.preprocess(msg, cfg)
    out = torch.zeros((msg.width, 4), device="cuda")
    counts = torch.zeros(8, dtype=torch.int32, device="cuda")
    plane = torch.zeros(8, dtype=torch.float64, device="cuda")
    for mode in ("eager", "graph"):
        out.zero_(); counts.zero_()
        if mode == "graph":
            g = ctx.capture_pipeline([desc], pcfg, out, counts, plane)
            out.zero_(); counts.zero_()
            ctx.launch_graph(g)
            ctx.launch_graph(g)
        else:
            ctx.pipeline_run([desc], pcfg, out, counts, plane)
        ctx.check()
        c = counts.cpu().numpy()
        assert c[capi.CNT_STATUS] == 0 and c[capi.CNT_FILTERED] == ref["n_filtered"], mode
        n = int(c[capi.CNT_OUTPUT])
        assert n == ref["positions"].shape[0], mode
        got = out[:n].cpu().numpy()
        assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32)), mode
        assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32)), mode
    ordinary_frontend(env)


# ==== 2. voxel table ================================================================================================
VS_CHAIN = 0.05


def voxel_chain_cloud(synth, seed, vs=VS_CHAIN):
    """64 distinct 2x2 blocks whose block hash lands in the LAST block of the voxel table (the chains wrap to block
    0), 1-4 filled voxels per block, 1-50 interior points per voxel, mixed with a small scan and shuffled."""
    rng = np.random.default_rng(seed)
    cap = hm.hash_cap(MAXP)
    last = cap // 4 - 1
    q = rng.integers(-200_000, 200_000, size=(1 << 22, 3))
    q[:, :2] &= ~np.int64(1)
    hit = q[hm.voxel_home_block(hm.voxel_key(q), cap) == last]
    hit = np.unique(hit, axis=0)[:64]
    assert hit.shape[0] == 64
    pts, subs = [], []
    for b in hit:
        for sub in rng.permutation(4)[:rng.integers(1, 5)]:
            qv = b + np.array([sub & 1, sub >> 1, 0])
            u = rng.uniform(0.05, 0.95, size=(int(rng.integers(1, 51)), 3))
            p = ((qv + u) * vs).astype(np.float32)
            p = p[np.all(hm.voxel_index(p, vs) == qv, axis=1)]
            pts.append(p)
            subs.append(sub)
    pts = np.concatenate(pts)
    assert np.all(hm.voxel_home_block(hm.voxel_key(hm.voxel_index(pts, vs)), cap) == last)
    assert len(set(subs)) == 4
    scan = synth.lidar_scan(seed=seed, n_beams=16, n_az=512, nan_frac=0.0)["positions"]
    pos = np.concatenate([pts, scan])
    inten = rng.uniform(0.0, 255.0, pos.shape[0]).astype(np.float32)
    perm = rng.permutation(pos.shape[0])
    return np.ascontiguousarray(pos[perm]), inten[perm]


def assert_voxel(ctx, xyzi, pos, inten, vs):
    from oracle import voxel as ovox
    out, p2v, vc, cnt = ctx.voxel_downsample(xyzi, vs, want_p2v=True, want_counts=True)
    ctx.check()
    ref = ovox.voxel_down_sample(pos, vs, inten, fixed=True)
    v = int(cnt.item())
    assert v == ref["positions"].shape[0]
    assert np.array_equal(p2v.cpu().numpy(), ref["p2v"])           # membership and first-occurrence order
    assert np.array_equal(vc[:v].cpu().numpy().astype(np.uint32), ref["counts"])
    got = out[:v].cpu().numpy()
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    return ref


def assert_voxel_sorted(ctx, xyzi, pos, inten, vs, ref):
    """The sort-based path: the same rows in ascending voxel-key order."""
    from oracle import voxel as ovox
    out, vc, cnt = ctx.voxel_downsample_sorted(xyzi, vs, want_counts=True)
    ctx.check()
    v = int(cnt.item())
    order = np.argsort(ovox.pack_key(ovox.voxel_index(pos[ref["first_idx"]], vs)), kind="stable")
    assert v == order.size
    got = out[:v].cpu().numpy()
    assert np.array_equal(vc[:v].cpu().numpy().astype(np.uint32), ref["counts"][order])
    assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"][order].view(np.uint32))
    assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"][order].view(np.uint32))


def ordinary_voxel(env, seed=92):
    """An ordinary scan through the same voxel table: a slot left occupied by finalize corrupts it."""
    scan = env["synth"].lidar_scan(seed=seed, n_beams=32, n_az=512, nan_frac=0.0)
    for vs in (VS_CHAIN, 0.3):
        assert_voxel(env["ctx"], to_xyzi(scan["positions"], scan["intensity"]), scan["positions"], scan["intensity"], vs)


def test_voxel_wrapping_block_chains(env):
    """k_voxel_insert probes block by block from the table's last block; k_voxel_finalize resets every slot, also
    those of voxels with several points, or the second call (same keys) and the ordinary scan go wrong."""
    ctx = env["ctx"]
    pos, inten = voxel_chain_cloud(env["synth"], 21)
    xyzi = to_xyzi(pos, inten)
    for _ in range(2):
        ref = assert_voxel(ctx, xyzi, pos, inten, VS_CHAIN)
    assert (ref["counts"] > 1).sum() > 100
    ordinary_voxel(env)
    assert_voxel_sorted(ctx, xyzi, pos, inten, VS_CHAIN, ref)


def test_voxel_chains_feed_the_radius_grid(env):
    """The pipeline's voxel finalize inserts the centroids into the radius grid (k_voxel_finalize<true>)."""
    from oracle import pipeline as opipe
    ctx, engine, capi = env["ctx"], env["engine"], env["capi"]
    pos, inten = voxel_chain_cloud(env["synth"], 22)
    cloud = dict(positions=pos, intensity=inten, ring=np.zeros(pos.shape[0], np.uint16),
                 time=np.zeros(pos.shape[0], np.float32))
    msg = env["synth"].pack_cloud(cloud, "xyzi16")
    data = dev_bytes(msg)
    desc = engine.make_cloud_desc(msg.fields, msg.point_step, msg.width, data)
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True)
    radius = dict(nb_points=2, radius=0.12)
    pcfg = engine.make_pipeline_cfg(fcfg, voxel_size=VS_CHAIN, radius=radius)
    cfg = opipe.default_config()
    cfg.update(crop=None, voxel_size=VS_CHAIN, radius=radius)
    ref = opipe.preprocess(msg, cfg)
    assert ref["radius_mask"].any() and not ref["radius_mask"].all()
    for _ in range(2):
        out, counts, _ = ctx.pipeline_run([desc], pcfg)
        ctx.check()
        c = counts.cpu().numpy()
        assert c[capi.CNT_STATUS] == 0 and c[capi.CNT_VOXELS] == ref["voxel_counts"].size
        n = int(c[capi.CNT_OUTPUT])
        assert n == ref["positions"].shape[0]
        got = out[:n].cpu().numpy()
        assert np.array_equal(got[:, :3].view(np.uint32), ref["positions"].view(np.uint32))
        assert np.array_equal(got[:, 3].view(np.uint32), ref["intensity"].view(np.uint32))
    ordinary_voxel(env)


def _on_axis(v, axis, w=1.0):
    row = [0.5, 0.5, 0.5, w]
    row[axis] = v
    return [row]


def _edge_cases():
    """(id, rows, voxel size, expected acceptance or None: whatever the oracle says)."""
    f = np.float32
    below = np.nextafter(f(65536.0), f(0.0))
    vs1 = np.nextafter(f(0.0625), f(0.0))
    vs2 = np.nextafter(vs1, f(0.0))
    cases = []
    for x, acc in ((below, True), (-below, True), (f(65536.0), False), (f(-65536.0), False)):
        for axis in range(3):
            cases.append((f"{'xyz'[axis]}={x}@1", _on_axis(x, axis), 1.0, acc))        # |x| < 2^16
            cases.append((f"{'xyz'[axis]}={x}@0.05", _on_axis(x, axis), 0.05, False))  # index beyond 2^20
    # index 2^20 - 1 / -2^20 (accepted), 2^20 (rejected), -2^20 - 1 (rejected)
    for vs, acc_pos, acc_neg in ((f(0.0625), True, True), (vs1, False, True), (vs2, False, False)):
        for axis in range(3):
            cases.append((f"{'xyz'[axis]}={below}@{vs}", _on_axis(below, axis), vs, acc_pos))
            cases.append((f"{'xyz'[axis]}={-below}@{vs}", _on_axis(-below, axis), vs, acc_neg))
    cases.append(("signed zeros", [[-0.0, 0.5, 0.5, 1.0], [0.0, 0.5, -0.0, 2.0], [0.0, -0.0, 0.5, 4.0]], 0.1, True))
    for vs in (0.0625, 0.25):
        k = np.arange(1, 9, dtype=np.float32)
        cases.append((f"negative multiples@{vs}", np.stack([-k * f(vs), -k * f(vs) * 2, -k * f(vs), k], 1), vs, True))
    # x just below (above) a boundary k * vs whose float32 quotient rounds onto k: the index is k (-k), not k - 1
    for vs in (0.1, 0.05, 0.3):
        vs32, rows = f(vs), []
        for k in range(1, 200_000, 997):
            b = k * np.float64(vs32)
            lo = np.nextafter(f(b), f(-np.inf)) if np.float64(f(b)) >= b else f(b)
            hi = np.nextafter(f(b), f(np.inf)) if np.float64(f(b)) <= b else f(b)
            if lo / vs32 == f(k) and np.float64(lo) < b:
                rows.append([lo, 0.5, 0.5, 1.0])
            if hi / vs32 == f(k) and np.float64(hi) > b:
                rows.append([-hi, 0.5, 0.5, 1.0])
        assert len(rows) >= 20
        cases.append((f"rounds onto k@{vs}", rows, vs, True))
    top = np.nextafter(f(2.0**20), f(0.0))
    for w, acc in ((top, True), (-top, True), (f(2.0**20), False), (f(-2.0**20), False), (f(np.nan), False),
                   (f(np.inf), False)):
        cases.append((f"w={w}", [[1.5, 0.5, 0.5, w]], 0.1, acc))
    for x in (np.nan, np.inf, -np.inf):
        cases.append((f"x={x}", [[x, 0.5, 0.5, 1.0]], 0.1, False))
    return cases


EDGE = _edge_cases()


@pytest.mark.parametrize("name,rows,vs,accept", EDGE, ids=[c[0] for c in EDGE])
def test_voxel_domain_edges(env, name, rows, vs, accept):
    """Accept / reject agrees with oracle.voxel.in_domain (and |intensity| < 2^20); accepted inputs are bit-exact,
    rejected ones raise APC_ERR_KEY_RANGE and leave a usable context.  One edge per case and axis, so that a bound
    that is wrong on one axis only is caught."""
    from oracle import voxel as ovox
    ctx, capi = env["ctx"], env["capi"]
    context = np.array([[1.0, 2.0, 3.0, 10.0], [1.01, 2.0, 3.0, 20.0], [-7.0, 0.3, -1.0, 5.0]], np.float32)
    a = np.concatenate([np.asarray(rows, np.float32), context])
    pos, inten = np.ascontiguousarray(a[:, :3]), np.ascontiguousarray(a[:, 3])
    with np.errstate(invalid="ignore"):
        ok = bool(ovox.in_domain(pos, vs).all() and (np.abs(inten) < ovox.ATTR_LIMIT).all())
    assert ok == accept                                            # the edge the case is named for
    xyzi = to_xyzi(pos, inten)
    if ok:
        for _ in range(2):
            assert_voxel(ctx, xyzi, pos, inten, vs)
    else:
        ctx.voxel_downsample(xyzi, vs)
        with pytest.raises(capi.ApcError) as e:
            ctx.check()
        assert e.value.code == capi.APC_ERR_KEY_RANGE
        assert_voxel(ctx, to_xyzi(context[:, :3], context[:, 3]), context[:, :3], context[:, 3], vs)


def big_sum_cloud(seed):
    """Two voxels of 2^14 points each (voxel size 65536: [0, 65536)^3 and [-65536, 0)^3), whose fixed-point x and
    intensity sums lie above 2^53 (magnitude) and are built so that the int64 -> float64 conversion decides the float32
    mean (see test_hash_models.rounding_sum_values); the negative voxel's sums are large negative numbers carried
    through unsigned 64-bit atomics.  (Within a voxel of 4096 m next to 2^16 m every rint(x 2^24) is a multiple of
    2^16 and the sum never rounds: the voxel must hold coordinates near 2^16 m and small ones.)"""
    rng = np.random.default_rng(seed)
    n = 1 << 14
    out = []
    for sign in (1.0, -1.0):
        x = hm.rounding_sum_values(rng, n, 65024.0, 65500.0, 2.0**-8, 1.0 - 2.0**-24, 24)
        w = hm.rounding_sum_values(rng, n, 2.0**20 - 1024.0, 2.0**20 - 64.0, 2.0**-4, 1.0 - 2.0**-20, 20)
        yz = rng.uniform(0.001, 300.0, size=(n, 2)).astype(np.float32)
        p = np.concatenate([x[:, None], yz], 1) * np.float32(sign)
        perm = rng.permutation(n)
        out.append(np.concatenate([p[perm], (w[perm] * np.float32(sign))[:, None]], 1))
    a = np.concatenate(out).astype(np.float32)
    return np.ascontiguousarray(a[:, :3]), np.ascontiguousarray(a[:, 3])


def test_voxel_sums_beyond_2_53(env):
    ctx = env["ctx"]
    pos, inten = big_sum_cloud(23)
    assert pos.shape[0] == MAXP
    for col, fb in ((pos[:MAXP // 2, 0], 24), (pos[MAXP // 2:, 0], 24), (inten[:MAXP // 2], 20), (inten[MAXP // 2:], 20)):
        rn, s = hm.fixed_mean_model(col, fb, "rn")
        assert abs(s) > 2**53 and rn != hm.fixed_mean_model(col, fb, "rz")[0]
    xyzi = to_xyzi(pos, inten)
    ref = assert_voxel(ctx, xyzi, pos, inten, 65536.0)
    assert np.array_equal(ref["counts"], [MAXP // 2] * 2)
    assert_voxel_sorted(ctx, xyzi, pos, inten, 65536.0, ref)
    ordinary_voxel(env)


@pytest.mark.parametrize("frac_bits", [0, 20, 30])
def test_voxel_mean_attr_range(env, frac_bits):
    """apc_voxel_mean_attr accumulates rint(v 2^frac_bits) below 2^40: values just below are bit-exact against
    centroids_fixed, a value at 2^40 raises APC_ERR_KEY_RANGE."""
    from oracle import voxel as ovox
    ctx, capi = env["ctx"], env["capi"]
    rng = np.random.default_rng(frac_bits)
    lim = np.float32(2.0 ** (40 - frac_bits))
    top = np.nextafter(lim, np.float32(0.0))
    pos = (rng.integers(0, 4, size=(4000, 3)) + 0.5).astype(np.float32)
    attr = (top * rng.choice([1.0, -1.0, 0.999, -0.75], size=4000)).astype(np.float32)
    small = rng.random(4000) < 0.3
    attr[small] = rng.uniform(-3.0, 3.0, int(small.sum()))
    xyzi = to_xyzi(pos)
    out, p2v, _, cnt = ctx.voxel_downsample(xyzi, 1.0, want_p2v=True)
    ctx.check()
    v = int(cnt.item())
    ref_p2v = ovox.membership(pos, 1.0)[0]
    assert np.array_equal(p2v.cpu().numpy(), ref_p2v)
    got = ctx.voxel_mean_attr(torch.from_numpy(attr).cuda(), p2v, cnt, pos.shape[0], frac_bits)
    ctx.check()
    ref = ovox.centroids_fixed(attr, ref_p2v, v, scale=float(1 << frac_bits))
    assert np.array_equal(got[:v].cpu().numpy().view(np.uint32), ref.view(np.uint32))
    for bad in (lim, -lim):
        a2 = attr.copy()
        a2[1234] = bad
        ctx.voxel_mean_attr(torch.from_numpy(a2).cuda(), p2v, cnt, pos.shape[0], frac_bits)
        with pytest.raises(capi.ApcError) as e:
            ctx.check()
        assert e.value.code == capi.APC_ERR_KEY_RANGE


# ==== 3. neighbour grids ============================================================================================
R = 0.3


def decoys(blob, cell, cap, rng, recip_inv=None, per_target=30, level=0, box=190.0, keep_out=40.0, spacing=10 * R):
    """Isolated points, one per cell, at cell centres, whose cells' grid_key home onto the slots of the blob's
    occupied cells, of their empty 27-neighbour cells and of the table's last slot.  They claim those slots first
    (lower indices), so the blob's cells sit behind runs of foreign keys and empty-neighbour lookups walk those runs
    to their end.  ``recip_inv``: the grid indexes by multiplying with this host-rounded reciprocal (else divides)."""
    def index(p):
        return hm.cell_recip(p, recip_inv) if recip_inv is not None else hm.cell_div(p, cell)

    occ = np.unique(index(blob), axis=0)
    off = np.stack(np.meshgrid([-1, 0, 1], [-1, 0, 1], [-1, 0, 1], indexing="ij"), -1).reshape(-1, 3)
    nbr = np.unique((occ[:, None, :] + off[None]).reshape(-1, 3), axis=0)
    occ_keys = set(hm.grid_key(level, occ).tolist())
    empty = nbr[[k not in occ_keys for k in hm.grid_key(level, nbr).tolist()]]
    targets = np.concatenate([hm.grid_home(hm.grid_key(level, occ[rng.permutation(len(occ))[:12]]), cap),
                              hm.grid_home(hm.grid_key(level, empty[rng.permutation(len(empty))[:12]]), cap),
                              [np.uint32(cap - 1)]])
    lim = int(box / float(cell))
    picked = [[] for _ in targets]
    for _ in range(16):                                            # batches of 4 M candidate cells
        cand = rng.integers(-lim, lim, size=(1 << 22, 3))
        cand = cand[np.abs(cand).max(axis=1) * float(cell) > keep_out]
        home = hm.grid_home(hm.grid_key(level, cand), cap)
        for j, t in enumerate(targets):
            picked[j].extend(cand[home == t][:per_target - len(picked[j])])
        if min(len(x) for x in picked) >= per_target:
            break
    cells = np.unique(np.asarray([c for x in picked for c in x]), axis=0)
    p = ((cells + 0.5) * np.float64(cell)).astype(np.float32)
    ok = np.all(hm.cell_div(p, cell) == cells, axis=1)
    if recip_inv is not None:
        ok &= np.all(hm.cell_recip(p, recip_inv) == cells, axis=1)
    p = p[ok]
    kept = []
    for q in p[rng.permutation(p.shape[0])]:
        if not kept or np.min(np.linalg.norm(np.asarray(kept) - q, axis=1)) >= spacing:
            kept.append(q)
    kept = np.asarray(kept, np.float32)
    homes = hm.grid_home(hm.grid_key(level, index(kept)), cap)
    assert (homes == cap - 1).sum() >= per_target // 2
    assert min(np.isin(homes, targets[:12]).sum(), np.isin(homes, targets[12:24]).sum()) >= 6 * per_target
    return kept


@pytest.fixture(scope="module")
def blob():
    """dense_patch: 6 000 points on a 1.6 m wavy patch and a wall, plus three far points."""
    return dense_patch()


@pytest.fixture(scope="module")
def radius_decoys(blob):
    """Decoys for radius_outliers' grid: cells of 2 r (1 + 2^-10), indexed with the host-rounded reciprocal."""
    c, inv = hm.radius_cell(R)
    return np.concatenate([decoys(blob, c, hm.grid_cap(MAXP, 1), np.random.default_rng(31), recip_inv=inv), blob])


@pytest.fixture(scope="module")
def nb_decoys(blob):
    """Decoys for the grid of estimate_normals_radius, cluster_dbscan and icp at r: cells of r (1 + 2^-8), indexed
    with the host-rounded reciprocal."""
    c, inv = hm.nb_cell(R)
    return np.concatenate([decoys(blob, c, hm.grid_cap(MAXP, 1), np.random.default_rng(32), recip_inv=inv), blob])


def twice_then_plain(cloud, blob, oracle):
    """(cloud, its oracle result) twice, then the plain blob: a grid slot left dirty shows up in the next call."""
    ref, ref_blob = oracle(cloud), oracle(blob)
    return ((cloud, ref), (cloud, ref), (blob, ref_blob))


def test_radius_outliers_past_decoys(env, radius_decoys, blob):
    from oracle import outliers
    ctx = env["ctx"]
    for p, ref in twice_then_plain(radius_decoys, blob, lambda q: outliers.radius_counts_brute(q, R)):
        for nb in (2, 40):
            mask, counts = ctx.radius_outliers(to_xyzi(p), nb, R, want_counts=True)
            ctx.check()
            assert np.array_equal(counts.cpu().numpy().astype(np.uint32), ref)
            assert np.array_equal(mask.cpu().numpy().astype(bool), ref >= nb)
            mask2, _ = ctx.radius_outliers(to_xyzi(p), nb, R, want_counts=False)
            ctx.check()
            assert np.array_equal(mask2.cpu().numpy().astype(bool), ref >= nb)


def test_normals_radius_past_decoys(env, nb_decoys, blob):
    from oracle import normals as onrm
    ctx = env["ctx"]
    r2 = float(np.float32(R)) ** 2
    for p, (ref, cnt_ref, cov_ref) in twice_then_plain(nb_decoys, blob, lambda q: onrm.estimate_normals(q, R, None)):
        got, cnt, cov = ctx.estimate_normals_radius(to_xyzi(p), R, want_counts=True, want_cov=True)
        ctx.check()
        assert_parity(got, cnt, cov, ref, cnt_ref, cov_ref, extra=1e-11 * r2)


def test_dbscan_past_decoys(env, nb_decoys, blob):
    from oracle import dbscan as odb
    ctx = env["ctx"]
    for p, (ref, n_ref, cnt_ref, _) in twice_then_plain(nb_decoys, blob, lambda q: odb.dbscan(q, R, 10)):
        labels, n_clusters, counts = ctx.cluster_dbscan(to_xyzi(p), R, 10, want_counts=True)
        ctx.check()
        assert np.array_equal(counts.cpu().numpy(), cnt_ref.astype(np.int32))
        assert int(n_clusters.item()) == n_ref
        assert np.array_equal(labels.cpu().numpy(), ref)


def test_icp_past_decoys(env, nb_decoys, blob):
    """The decoys are in the target, whose grid every source point's lookups walk, and in the source: the decoys
    that share a home slot are displaced along its chain, and each must still find its twin."""
    from oracle import registration as reg
    ctx = env["ctx"]
    moved = reg.transform_points(blob, reg.pose_to_transformation([0.01, 0.0, -0.02, 0.03, 0.01, 0.0]))
    src = np.concatenate([moved, nb_decoys[:nb_decoys.shape[0] - blob.shape[0]]])
    for tgt, ref in twice_then_plain(nb_decoys, blob, lambda q: reg.icp(src, q, R, max_iteration=8)):
        T, stats, info, corr = ctx.icp(to_xyzi(src), to_xyzi(tgt), R, max_iteration=8)
        ctx.check()
        T, stats, info, corr = T.cpu().numpy(), stats.cpu().numpy(), info.cpu().numpy(), corr.cpu().numpy()
        assert info[2] == ref["status"] and info[0] == ref["iterations"] and bool(info[1]) == ref["converged"]
        assert np.array_equal(corr, ref["correspondences"])
        assert np.abs(T - ref["transformation"]).max() < 1e-9
        assert stats[0] == pytest.approx(ref["fitness"], rel=1e-12)


def test_statistical_outliers_past_level0_decoys(env, blob):
    """Level 0 of the 12-level KNN grid only: its cell sizes are computed on the device from the bounding box, so
    two anchor points at +-200 m pin level 0 to 400 / 4096 m and the decoys target that level.  The coarser levels
    get whatever slots their keys hash to."""
    from oracle import outliers
    ctx = env["ctx"]
    anchors = np.array([[-200.0, -200.0, -200.0], [200.0, 200.0, 200.0]], np.float32)
    f = np.float32
    c0 = max(max(f(400.0) * f(1.0 / 4096.0), f(1.0e-4)), f(200.0) * f(1.0 / 262000.0))
    d = decoys(blob, f(c0), hm.grid_cap(MAXP, hm.KNN_LEVELS), np.random.default_rng(33), per_target=8)
    p = np.concatenate([anchors, d, blob])
    for q, (ref_mask, ref_avg) in twice_then_plain(p, blob, lambda c: outliers.statistical_mask(c, 8, 1.5)):
        mask, avg, _ = ctx.statistical_outliers(to_xyzi(q), 8, 1.5)
        ctx.check()
        assert np.array_equal(avg.cpu().numpy().view(np.uint32), ref_avg.view(np.uint32))
        assert np.array_equal(mask.cpu().numpy().astype(bool), ref_mask)
