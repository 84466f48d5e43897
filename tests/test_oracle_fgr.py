"""Fast Global Registration oracle (oracle/fgr.py): the vectorised tuple sampler against ``oracle.ransac.splitmix64``,
the tuple test at constructed edges, the ``par`` schedule, one iteration's system against finite differences, exact
recovery in both scale modes, the TOO_FEW / DEGENERATE / zero-iteration edges, and a hard terrain case."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

from oracle import fgr
from oracle import features as of
from oracle import normals as onrm
from oracle import registration as reg
from oracle.ransac import M64, splitmix64
from test_oracle_features import oriented, terrain


def pose_error(T, T_true):
    E = np.linalg.inv(T_true) @ T
    ang = np.degrees(np.arccos(np.clip((np.trace(E[:3, :3]) - 1.0) / 2.0, -1.0, 1.0)))
    return float(np.linalg.norm(T[:3, 3] - T_true[:3, 3])), float(ang)


def motion(yaw, pitch=10.0, roll=-5.0, t=(5.0, -2.0, 0.3)):
    T = np.eye(4)
    T[:3, :3] = Rotation.from_euler("zyx", [yaw, pitch, roll], degrees=True).as_matrix()
    T[:3, 3] = t
    return T


def moved(p, T):
    return (p.astype(np.float64) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)


@pytest.mark.parametrize("seed", [0, 7, (1 << 64) - 5])
def test_vectorised_sampler_is_the_ransac_stream(seed):
    rng = np.random.default_rng(3)
    t = np.concatenate([np.arange(50), rng.integers(0, 400_000_000, 50), [(1 << 32) - 1, 1 << 32, (1 << 40) + 3]])
    for K in (1, 3, 1000, 4_000_000):
        for k in range(3):
            got = fgr.draws(seed, t.astype(np.uint64), k, K)
            want = [((splitmix64((seed + (int(x) << 32) + k) & M64) >> 32) * K) >> 32 for x in t]
            assert got.tolist() == want
            assert np.all((got >= 0) & (got < K))


def lattice(n=12, seed=0):
    """Distinct integer points (exact float32 products with powers of two)."""
    rng = np.random.default_rng(seed)
    return rng.choice(64, size=(n, 3), replace=True).astype(np.float32) + np.arange(n, dtype=np.float32)[:, None] * 64


def distinct_draws(seed, K, trials, pairs):
    t = np.arange(trials, dtype=np.uint64)
    c = np.stack([fgr.draws(seed, t, k, K) for k in range(3)], 1)
    s = pairs[c, 0]
    return (s[:, 0] != s[:, 1]) & (s[:, 1] != s[:, 2]) & (s[:, 0] != s[:, 2]), c


@pytest.mark.parametrize("factor,accepts", [(0.5, False), (2.0, False), (0.75, True), (1.0, True)])
def test_tuple_edges_are_strict(factor, accepts):
    """The target is the source scaled by ``factor``: with scale 0.5, ``lj == li * 0.5`` and ``lj == li / 0.5`` are
    both exact and rejected; inside the band every tuple of three distinct points is accepted."""
    p = lattice()
    q = (p * np.float32(factor)).astype(np.float32)
    pairs = np.stack([np.arange(len(p)), np.arange(len(p))], 1)
    used, trials = fgr.tuple_test(p, q, pairs, seed=5, tuple_scale=0.5, maximum_tuple_count=10 ** 9)
    assert trials == 100 * len(p)
    ok, c = distinct_draws(5, len(p), trials, pairs)
    if not accepts:
        assert used.shape == (0, 2)
    else:
        assert np.array_equal(used, pairs[c[ok].reshape(-1)])


def test_repeated_draws_and_shared_points_are_rejected():
    p = lattice(6)
    # pairs 0 and 1 share source point 0, pairs 2 and 3 target point 2; every pair maps its source point onto equal
    # coordinates, so only zero edges reject
    pairs = np.array([[0, 0], [0, 1], [2, 2], [3, 2], [4, 4], [5, 5]])
    p[3] = p[2]
    q = p.copy()
    q[1] = p[0]
    used, trials = fgr.tuple_test(p, q, pairs, seed=11, tuple_scale=0.9, maximum_tuple_count=10 ** 9)
    t = np.arange(trials, dtype=np.uint64)
    c = np.stack([fgr.draws(11, t, k, len(pairs)) for k in range(3)], 1)
    s, d = pairs[c, 0], pairs[c, 1]
    ok = np.ones(len(c), bool)
    for a, b in ((0, 1), (1, 2), (2, 0)):
        ok &= (s[:, a] != s[:, b]) & (d[:, a] != d[:, b])
    assert (~ok).sum() > 50 and ok.sum() > 10
    assert np.array_equal(used, pairs[c[ok].reshape(-1)])


def test_maximum_tuple_count_cut_in_trial_order():
    p = lattice(40)
    pairs = np.stack([np.arange(40), np.arange(40)], 1)
    full, trials_full = fgr.tuple_test(p, p, pairs, seed=2, tuple_scale=0.95, maximum_tuple_count=10 ** 9)
    ok, _ = distinct_draws(2, 40, trials_full, pairs)
    acc = np.flatnonzero(ok)
    assert trials_full == 4000 and len(full) == 3 * len(acc)
    for m in (1, 2, 17, len(acc) - 1, len(acc)):
        used, trials = fgr.tuple_test(p, p, pairs, seed=2, tuple_scale=0.95, maximum_tuple_count=m, chunk=64)
        assert np.array_equal(used, full[:3 * m])
        assert trials == acc[m - 1] + 1
    used, trials = fgr.tuple_test(p, p, pairs, seed=2, maximum_tuple_count=len(acc) + 1, chunk=64)
    assert np.array_equal(used, full) and trials == 4000


@pytest.mark.parametrize("absolute", [False, True])
@pytest.mark.parametrize("decrease_mu", [False, True])
def test_par_schedule(monkeypatch, absolute, decrease_mu):
    p = terrain(n_side=12)
    q = moved(p, motion(20.0))
    pairs = np.stack([np.arange(len(p)), np.arange(len(p))], 1)
    seen = []
    real = fgr.system
    monkeypatch.setattr(fgr, "system", lambda a, b, T, par: seen.append(par) or real(a, b, T, par))
    fgr.fgr(p, q, pairs, division_factor=1.4, use_absolute_scale=absolute, decrease_mu=decrease_mu,
            maximum_correspondence_distance=0.025, iteration_number=64)
    D = fgr.normalise(p, q, absolute)[4]
    par, want = (D if absolute else 1.0), []
    for itr in range(64):
        if decrease_mu and itr % 4 == 0 and par > 0.025:
            par = par / 1.4
        want.append(par)
    assert seen == want
    if decrease_mu and not absolute:
        assert len(set(want)) == 11 and want[40] < 0.025 < want[39] and want[40] == want[63]   # 1.4^-11 < 0.025
    if not decrease_mu:
        assert set(want) == {D if absolute else 1.0}


def test_system_matches_finite_differences():
    rng = np.random.default_rng(4)
    p = rng.normal(size=(50, 3))
    q = p @ motion(25.0)[:3, :3].T * 0.3 + rng.normal(0, 0.05, (50, 3))
    T = motion(-10.0, 3.0, 2.0, (0.1, 0.2, -0.1))
    par = 0.7
    A, b = fgr.system(p, q, T, par)
    qt = q @ T[:3, :3].T + T[:3, 3]
    s = (par / (((p - qt) ** 2).sum(1) + par)) ** 2

    def res(x):
        U = reg.pose_to_transformation(x) @ T
        return p - (q @ U[:3, :3].T + U[:3, 3])

    h = 1e-6
    J = np.empty((50, 3, 6))
    g = np.empty(6)
    for k in range(6):
        e = np.zeros(6)
        e[k] = h
        J[:, :, k] = (res(e) - res(-e)) / (2 * h)
        g[k] = (0.5 * (s * (res(e) ** 2).sum(1)).sum() - 0.5 * (s * (res(-e) ** 2).sum(1)).sum()) / (2 * h)
    A_fd = np.einsum("n,nak,nal->kl", s, J, J)
    assert np.allclose(A, A_fd, rtol=1e-6, atol=1e-8)
    assert np.allclose(b, g, rtol=1e-6, atol=1e-8)


@pytest.mark.parametrize("absolute", [False, True])
@pytest.mark.parametrize("offset", [0.0, 150.0])
def test_noiseless_recovery(absolute, offset):
    p = terrain(n_side=20) + np.float32(offset)
    T_true = motion(60.0, 12.0, -8.0, (3.0, -1.0, 0.5))
    q = moved(p, T_true)
    perm = np.random.default_rng(0).permutation(len(p))
    pairs = np.stack([perm, perm], 1)
    out = fgr.fgr(p, q, pairs, use_absolute_scale=absolute)
    assert out["status"] == fgr.OK and out["iterations"] == 64
    # q is float32-rounded: the exact motion of the rounded points is not T_true, so compare with Kabsch on them
    T_ref = reg.kabsch(p.astype(np.float64), q.astype(np.float64))
    assert np.abs(out["transformation"] - T_ref).max() < 1e-9 * max(1.0, offset)
    assert np.abs(out["transformation"] - T_true).max() < 1e-4


def test_edges_zero_iterations_too_few_degenerate():
    p = terrain(n_side=10)
    q = moved(p, motion(30.0))
    pairs = np.stack([np.arange(len(p)), np.arange(len(p))], 1)
    out = fgr.fgr(p, q, pairs, iteration_number=0)
    want = np.eye(4)
    want[:3, 3] = q.astype(np.float64).mean(0) - p.astype(np.float64).mean(0)
    assert out["status"] == fgr.OK and out["iterations"] == 0 and np.array_equal(out["transformation"], want)
    few = fgr.fgr(p, q, pairs[:9])
    assert few["status"] == fgr.TOO_FEW and few["iterations"] == 0 and np.array_equal(few["transformation"], np.eye(4))
    ten = fgr.fgr(p, q, pairs[:10])
    assert ten["status"] == fgr.OK and ten["iterations"] == 64
    line = np.zeros((30, 3), np.float32)
    line[:, 0] = np.arange(30, dtype=np.float32)
    lp = np.stack([np.arange(30), np.arange(30)], 1)
    deg = fgr.fgr(line, line + np.float32(1.0), lp)
    assert deg["status"] == fgr.DEGENERATE and deg["iterations"] == 0
    bad = p.copy()
    bad[len(p) - 1, 2] = np.nan                      # not in any pair: the normalisation still becomes NaN
    nan = fgr.fgr(bad, q, pairs[:20])
    assert nan["status"] == fgr.DEGENERATE and nan["iterations"] == 0


def test_mutual_pairs_have_no_fallback():
    rng = np.random.default_rng(5)
    a = rng.normal(size=(40, 8)).astype(np.float32)
    b = rng.normal(size=(60, 8)).astype(np.float32)
    pairs = fgr.mutual_pairs(a, b)
    fwd, back = of.nearest(a, b), of.nearest(b, a)
    want = [(i, fwd[i]) for i in range(40) if fwd[i] >= 0 and back[fwd[i]] == i]
    assert pairs.tolist() == [list(x) for x in want]
    _, _, fell_back = of.correspondences(a, b, True, 0.5)
    assert fell_back                                  # correspondences_from_features would return all 40


def hard_terrain(yaw=170.0, keep=0.6, seed=3):
    p = terrain(n_side=60)
    rng = np.random.default_rng(seed)
    T_true = motion(yaw)
    sel = rng.random(len(p)) < keep
    q = ((p[sel].astype(np.float64) + rng.normal(0, 0.01, (sel.sum(), 3))) @ T_true[:3, :3].T
         + T_true[:3, 3]).astype(np.float32)
    up = np.array([0.0, 0.0, 1.0])
    ns = oriented(onrm.estimate_normals(p, 0.25, 30)[0], up)
    nt = oriented(onrm.estimate_normals(q, 0.25, 30)[0], T_true[:3, :3] @ up)
    fs = of.compute_fpfh(p, ns, onrm.neighbourhoods(p, 0.5, 100))[0]
    ft = of.compute_fpfh(q, nt, onrm.neighbourhoods(q, 0.5, 100))[0]
    return p, q, fs, ft, T_true, np.flatnonzero(sel)


def test_hard_terrain_needs_the_tuple_test():
    p, q, fs, ft, T_true, truth = hard_terrain()
    out = fgr.fgr_from_features(p, q, fs, ft)
    pairs = out["pairs_in"]
    good = np.mean(np.linalg.norm(p[pairs[:, 0]] - p[truth[pairs[:, 1]]], axis=1) < 0.1)
    assert good < 0.2
    dt, ang = pose_error(out["transformation"], T_true)
    assert out["status"] == fgr.OK and dt < 0.1 and ang < 2.0, (dt, ang)
    plain = fgr.fgr_from_features(p, q, fs, ft, tuple_test_on=False)
    assert pose_error(plain["transformation"], T_true)[1] > 90.0
    icp = reg.icp(p, q, 0.1, out["transformation"], max_iteration=30)
    dt2, ang2 = pose_error(icp["transformation"], T_true)
    assert dt2 < dt and dt2 < 0.02 and ang2 < 0.5, (dt2, ang2)
