"""CPU checks of the FPFH / feature-matching oracle (``oracle/features.py``): the pair feature against a Darboux
frame built independently, bins, SPFH, FPFH, matching against brute force and a kd-tree, and a registration
scene on which the mutual FPFH correspondences are mostly the true ones."""
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree
from scipy.spatial.transform import Rotation

from oracle import features as of
from oracle import normals as onrm
from test_oracle_normals_search import knn_neighbourhoods
from test_oracle_wide_k import cloud_with_duplicates


def unit(rng, n):
    v = rng.normal(size=(n, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def darboux(p1, n1, p2, n2):
    """Open3D's pair feature from an explicit frame: the source is the point whose normal makes the smaller angle
    with the line (``acos`` test, as Open3D), frame rows ``u = n_s``, ``v = (p_t - p_s) x u / |.|``, ``w = u x v``;
    the target normal in that frame gives ``f0 = atan2(n_w, n_u)`` and ``f1 = n_v``."""
    p1, n1, p2, n2 = (np.asarray(x, np.float64) for x in (p1, n1, p2, n2))
    dp = p2 - p1
    d = np.linalg.norm(dp)
    if d == 0:
        return np.zeros(3)
    a1, a2 = n1 @ dp / d, n2 @ dp / d
    if math.acos(min(abs(a1), 1.0)) > math.acos(min(abs(a2), 1.0)):
        u, t, line, f2 = n2, n1, -dp, -a2
    else:
        u, t, line, f2 = n1, n2, dp, a1
    v = np.cross(line, u)
    if np.linalg.norm(v) == 0:
        return np.zeros(3)
    v /= np.linalg.norm(v)
    frame = np.stack([u, v, np.cross(u, v)])
    tl = frame @ t
    return np.array([math.atan2(tl[2], tl[0]), tl[1], f2])


def test_pair_feature_matches_darboux_frame():
    rng = np.random.default_rng(0)
    n = 400
    p1, p2 = rng.normal(size=(n, 3)).astype(np.float32), rng.normal(size=(n, 3)).astype(np.float32)
    n1, n2 = unit(rng, n), unit(rng, n)
    got = of.pair_features(p1, n1, p2, n2)
    ref = np.stack([darboux(p1[i], n1[i], p2[i], n2[i]) for i in range(n)])
    assert np.allclose(got, ref, atol=1e-12, rtol=0)
    assert np.all(np.abs(got[:, 1:]) <= 1 + 1e-12) and np.all(np.abs(got[:, 0]) <= math.pi)


def test_pair_feature_swap_symmetry_is_exact():
    rng = np.random.default_rng(1)
    n = 500
    p1, p2 = rng.normal(size=(n, 3)).astype(np.float32), rng.normal(size=(n, 3)).astype(np.float32)
    n1, n2 = unit(rng, n), unit(rng, n)
    a = of.pair_features(p1, n1, p2, n2)
    b = of.pair_features(p2, n2, p1, n1)
    assert np.array_equal(a, b)


def test_pair_feature_zero_cases():
    z = np.zeros((1, 3), np.float32)
    n = np.array([[0, 0, 1]], np.float32)
    assert np.array_equal(of.pair_features(z, n, z, n), np.zeros((1, 3)))          # d == 0
    p2 = np.array([[0, 0, 2]], np.float32)
    assert np.array_equal(of.pair_features(z, n, p2, n), np.zeros((1, 3)))         # dp parallel to the normal
    # a zero normal is ordinary input: finite features
    f = of.pair_features(z, np.zeros((1, 3), np.float32), np.array([[1, 0, 0]], np.float32), np.array([[0.6, 0.8, 0]], np.float32))
    assert np.isfinite(f).all()
    f = of.pair_features(z, np.full((1, 3), np.nan, np.float32), np.array([[1, 0, 0]], np.float32), n)
    assert not np.isfinite(f).all()


def test_bins_edges_and_clamping():
    f = np.array([[-math.pi, -1.0, -1.0],          # lowest edges: bin 0 (an ulp below clamps to it too: not flagged)
                  [math.pi, 1.0, 1.0],             # argument 11: clamped to 10
                  [0.0, 0.0, 0.0],                 # the zero feature: bins 5, 16, 27
                  [4.0, 1.5, -1.5],                # outside the ranges: clamped
                  [0.1, 0.3, -0.2],
                  [0.1, -5.0 / 11.0, 0.3]])        # f1's argument within rounding of the interior edge 3: flagged
    b, finite, near = of.bins(f)
    assert finite.all()
    assert b[0].tolist() == [0, 11, 22] and not near[0]
    assert b[1].tolist() == [10, 21, 32] and not near[1]
    assert near[5] and not near[:5].any()
    assert b[2].tolist() == [5, 16, 27] and not near[2]
    assert b[3].tolist() == [10, 21, 22]
    x = of.bin_arguments(f[4:])[0]
    assert b[4].tolist() == [int(math.floor(x[0])), 11 + int(math.floor(x[1])), 22 + int(math.floor(x[2]))]
    # just below and above an interior edge
    e = (2.0 * 3 / 11.0) - 1.0
    b2, _, _ = of.bins(np.array([[0, np.nextafter(e, -2), 0], [0, np.nextafter(e, 2), 0]]))
    x2 = of.bin_arguments(np.array([[0, np.nextafter(e, -2), 0], [0, np.nextafter(e, 2), 0]]))[:, 1]
    assert (b2[:, 1] - 11).tolist() == np.floor(x2).astype(int).tolist()
    _, fin, _ = of.bins(np.array([[np.nan, 0, 0], [0, np.inf, 0]]))
    assert not fin.any()


def _cloud(seed=2, n=600):
    rng = np.random.default_rng(seed)
    p = rng.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    p[:, 2] = (0.3 * np.sin(2 * p[:, 0]) * np.cos(3 * p[:, 1])).astype(np.float32)
    return p


def test_spfh_counts_and_normalisation():
    p = _cloud()
    nrm, _, _ = onrm.estimate_normals(p, 0.3, 30)
    nbs = onrm.neighbourhoods(p, 0.3, 40)
    sp, counts, _ = of.spfh(p, nrm, nbs)
    assert np.array_equal(counts, [len(nb) for nb in nbs])
    for i in range(0, len(p), 37):
        m = counts[i]
        if m <= 1:
            assert not sp[i].any()
            continue
        incr = 100.0 / (m - 1)
        c = np.round(sp[i].astype(np.float64) / incr)
        assert np.array_equal(sp[i], (c * incr).astype(np.float32))
        for g in range(3):
            assert c[11 * g:11 * g + 11].sum() == m - 1      # every pair lands once per group
        assert np.allclose(sp[i].reshape(3, 11).astype(np.float64).sum(axis=1), 100.0, rtol=1e-6)


def test_spfh_skip_first_equals_skip_query_with_duplicates():
    p = cloud_with_duplicates(n=300)
    rng = np.random.default_rng(3)
    nrm = unit(rng, len(p))
    for k in (2, 5, 30):
        nbs = knn_neighbourhoods(p, k)
        sp, counts, _ = of.spfh(p, nrm, nbs)
        dups = 0
        for i, nb in enumerate(nbs):
            if i not in nb:                                # only when lower-index duplicates fill the list
                assert (of._d2(p, i, np.asarray(nb)) == 0).all()
                continue
            if nb[0] != i:
                dups += 1
            others = np.asarray([j for j in nb if j != i], np.int64)
            f = of.pair_features(np.repeat(p[i:i + 1], len(others), 0), np.repeat(nrm[i:i + 1], len(others), 0),
                                 p[others], nrm[others])
            b, fin, _ = of.bins(f)
            h = np.zeros(33)
            for g in range(3):
                np.add.at(h, b[fin, g], 1)
            incr = 100.0 / (len(nb) - 1) if len(nb) > 1 else 0.0
            assert np.array_equal(sp[i], (h * incr).astype(np.float32)), (k, i)
        assert dups > 0                                    # the lists do start with a duplicate before the query


def test_spfh_small_neighbourhoods_and_bad_normals():
    p = _cloud(n=200)
    nrm, _, _ = onrm.estimate_normals(p, 0.3, 30)
    # m <= 1: zeros
    sp, counts, _ = of.spfh(p, nrm, [np.array([i]) for i in range(len(p))])
    assert not sp.any() and (counts == 1).all()
    nbs = onrm.neighbourhoods(p, 0.4, 30)
    bad = nrm.copy()
    bad[::5] = np.nan
    bad[1::5] = 0.0
    sp, counts, _ = of.spfh(p, bad, nbs)
    assert np.isfinite(sp).all()
    i = next(i for i in range(0, len(p), 5) if len(nbs[i]) > 2)
    assert not sp[i].any() and counts[i] == len(nbs[i])        # a NaN query normal: no pair is binned, m counts
    # a zero query normal bins every pair (v = dp x 0 = 0: the zero feature, even against a NaN normal)
    j = next(j for j in range(1, len(p), 5) if len(nbs[j]) > 2)
    assert np.allclose(sp[j].reshape(3, 11).astype(np.float64).sum(axis=1), 100.0, rtol=1e-6)
    # a NaN neighbour normal drops that pair only
    j = next(j for j in range(2, len(p), 5) if len(nbs[j]) > 2 and any(np.isnan(bad[k]).any() for k in nbs[j][1:]))
    sums = sp[j].reshape(3, 11).astype(np.float64).sum(axis=1)
    n_nan = sum(1 for k in nbs[j][1:] if np.isnan(bad[k]).any())
    assert np.allclose(sums, 100.0 * (len(nbs[j]) - 1 - n_nan) / (len(nbs[j]) - 1), rtol=1e-6)


def test_fpfh_restates_open3d_loop():
    p = _cloud(seed=4, n=300)
    nrm, _, _ = onrm.estimate_normals(p, 0.3, 30)
    nbs = onrm.neighbourhoods(p, 0.35, 25)
    feat, sp, _, _ = of.compute_fpfh(p, nrm, nbs)
    for i in range(0, len(p), 23):                 # Open3D's interleaved loop: equal up to summation order
        f = np.zeros(33)
        s = np.zeros(3)
        for k in nbs[i][1:]:
            d2 = float(of._d2(p, i, np.array([k]))[0])
            if d2 == 0:
                continue
            v = sp[k].astype(np.float64) / d2
            f += v
            s += v.reshape(3, 11).sum(axis=1)
        s = np.where(s != 0, 100.0 / np.where(s != 0, s, 1), 0.0)
        ref = f * np.repeat(s, 11) + sp[i]
        assert np.allclose(feat[i], ref, rtol=1e-5, atol=1e-4)


def test_fpfh_invariant_under_rigid_motion():
    p = _cloud(seed=5, n=800)
    nrm, _, _ = onrm.estimate_normals(p, 0.3, 30)
    R = Rotation.from_euler("zyx", [30, -20, 50], degrees=True).as_matrix()
    t = np.array([5.0, -2.0, 1.0])
    q = (p.astype(np.float64) @ R.T + t).astype(np.float32)
    m = (nrm.astype(np.float64) @ R.T).astype(np.float32)
    fa = of.compute_fpfh(p, nrm, knn_neighbourhoods(p, 30))[0]
    fb = of.compute_fpfh(q, m, knn_neighbourhoods(q, 30))[0]
    close = np.all(np.abs(fa - fb) <= 1e-3 * 200, axis=1)
    assert close.mean() > 0.97, close.mean()


def test_matching_against_brute_force_and_kdtree():
    rng = np.random.default_rng(6)
    a = rng.uniform(0, 100, size=(300, 33)).astype(np.float32)
    b = rng.uniform(0, 100, size=(400, 33)).astype(np.float32)
    nn = of.nearest(a, b)
    d2 = np.array([[float(((a[i].astype(np.float64) - b[j]) ** 2).sum()) for j in range(len(b))] for i in range(len(a))])
    assert np.array_equal(nn, np.argmin(d2, axis=1))
    _, kd = cKDTree(b.astype(np.float64)).query(a.astype(np.float64), k=1)
    assert np.array_equal(nn, kd)


def test_matching_ties_go_to_lower_index_and_nan_rows():
    rng = np.random.default_rng(7)
    b = rng.integers(0, 4, size=(50, 8)).astype(np.float32)
    b[30] = b[10]                                      # exact duplicate rows: the lower index wins
    a = np.concatenate([b[[10, 30]], rng.integers(0, 4, size=(20, 8)).astype(np.float32)])
    a[5, 3] = np.nan                                   # no finite distance: no match
    nn = of.nearest(a, b)
    assert nn[0] == 10 and nn[1] == 10 and nn[5] == -1
    d2 = of.feature_d2(a, b)
    for i in range(len(a)):
        if i == 5:
            continue
        best = d2[i].min()
        assert nn[i] == np.flatnonzero(d2[i] == best)[0]
    bn = b.copy()
    bn[10, 0] = np.nan                                 # a NaN target row never wins
    assert of.nearest(a[:1], bn)[0] == 30
    pairs, near, fb = of.correspondences(a, b)
    assert not fb and 5 not in pairs[:, 0] and np.array_equal(pairs[:, 0], np.sort(pairs[:, 0]))
    assert len(pairs) == len(a) - 1


def test_mutual_filter_and_fallback():
    rng = np.random.default_rng(8)
    b = rng.normal(size=(100, 33)).astype(np.float32)
    a = (b[rng.permutation(100)[:60]] + rng.normal(scale=0.01, size=(60, 33))).astype(np.float32)
    pairs, nn, fb = of.correspondences(a, b, True, 0.1)
    assert not fb and len(pairs) == 60                 # every row is its match's match
    back = of.nearest(b, a)
    # many sources onto one target: only one survives the filter
    a2 = np.repeat(b[:3], 20, axis=0) + rng.normal(scale=1e-3, size=(60, 33)).astype(np.float32)
    pairs2, nn2, fb2 = of.correspondences(a2, b, True, 0.0)
    back2 = of.nearest(b, a2)
    assert not fb2 and len(pairs2) == 3 and all(back2[j] == i for i, j in pairs2)
    # ratio: kept only when count > ratio * n_src
    pairs3, _, fb3 = of.correspondences(a2, b, True, 3 / 60)
    assert fb3 and len(pairs3) == 60
    pairs4, _, fb4 = of.correspondences(a2, b, True, 2.99 / 60)
    assert not fb4 and len(pairs4) == 3
    assert back is not None


def terrain(seed=0, n_side=40):
    """A smooth height field of seven Gaussian bumps on a jittered grid: every point has its own curvature."""
    rng = np.random.default_rng(seed)
    g = np.linspace(-2.0, 2.0, n_side)
    x, y = np.meshgrid(g, g)
    x = x + rng.uniform(-0.02, 0.02, x.shape)
    y = y + rng.uniform(-0.02, 0.02, y.shape)
    z = np.zeros_like(x)
    for _ in range(7):
        c = rng.uniform(-1.8, 1.8, 2)
        s = rng.uniform(0.3, 0.8)
        z += rng.uniform(-0.8, 0.8) * np.exp(-((x - c[0]) ** 2 + (y - c[1]) ** 2) / s ** 2)
    return np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32)


def oriented(normals, up):
    n = normals.copy()
    n[(n.astype(np.float64) @ up) < 0] *= -1
    return n


def test_mutual_fpfh_correspondences_are_mostly_true():
    p = terrain()
    R = Rotation.from_euler("zyx", [40, 15, -20], degrees=True).as_matrix()
    t = np.array([3.0, -1.0, 0.5])
    perm = np.random.default_rng(1).permutation(len(p))
    q = (p.astype(np.float64) @ R.T + t).astype(np.float32)[perm]
    up = np.array([0.0, 0.0, 1.0])
    ns = oriented(onrm.estimate_normals(p, 0.25, 30)[0], up)
    nt = oriented(onrm.estimate_normals(q, 0.25, 30)[0], R @ up)
    fs = of.compute_fpfh(p, ns, onrm.neighbourhoods(p, 0.5, 100))[0]
    ft = of.compute_fpfh(q, nt, onrm.neighbourhoods(q, 0.5, 100))[0]
    pairs, _, fb = of.correspondences(fs, ft, True, 0.1)
    true = np.argsort(perm)[pairs[:, 0]] == pairs[:, 1]
    assert not fb and len(pairs) > 0.5 * len(p)
    assert true.mean() > 0.9, true.mean()
