"""The closed-form DBSCAN oracle (oracle.dbscan.dbscan) against Open3D's sequential loop restated literally
(oracle.dbscan.dbscan_open3d), label for label, and the border rule on a hand-built case."""
import numpy as np
import pytest

from oracle import dbscan as odb
from oracle.outliers import radius_counts_brute

MIN_POINTS = (0, 1, 2, 3, 5, 10)


def blobs_with_bridges(rng, eps):
    """A few Gaussian blobs, sparse bridges between some of them, scattered noise, exact duplicates and pairs
    exactly float32(eps) apart along an axis."""
    parts = []
    centres = rng.uniform(-6 * eps, 6 * eps, size=(rng.integers(2, 5), 3))
    for c in centres:
        parts.append(c + rng.normal(scale=rng.uniform(0.3, 1.2) * eps, size=(rng.integers(5, 40), 3)))
    for a, b in zip(centres[:-1], centres[1:]):
        if rng.random() < 0.6:
            t = np.linspace(0.0, 1.0, rng.integers(3, 12))[:, None]
            parts.append(a + t * (b - a))
    parts.append(rng.uniform(-8 * eps, 8 * eps, size=(rng.integers(0, 15), 3)))
    p = np.concatenate(parts).astype(np.float32)
    dup = rng.integers(0, p.shape[0], size=3)
    p[rng.integers(0, p.shape[0], size=3)] = p[dup]
    e = np.float32(eps)
    base = p[rng.integers(0, p.shape[0], size=4)]
    edge = base.copy()
    for k in range(4):
        edge[k, k % 3] = base[k, k % 3] + e                      # float32 add: d2 lands on r2 or next to it
    p = np.concatenate([p, edge])
    return p[rng.permutation(p.shape[0])]


@pytest.mark.parametrize("seed", range(40))
def test_closed_form_equals_the_open3d_loop(seed):
    rng = np.random.default_rng(seed)
    eps = float(rng.choice([0.1, 0.25, 0.5, 1.0]))
    p = blobs_with_bridges(rng, eps)
    for min_points in MIN_POINTS:
        ref = odb.dbscan_open3d(p, eps, min_points)
        labels, n_clusters, counts, tests = odb.dbscan(p, eps, min_points)
        assert np.array_equal(labels, ref), (seed, min_points)
        assert n_clusters == (ref.max() + 1 if ref.size else 0)
        assert np.array_equal(counts, radius_counts_brute(p, eps))
        assert tests == int(counts.sum())


def test_pairs_exactly_eps_apart_are_neighbours():
    e = np.float32(0.3)
    p = np.array([[1.0, 2.0, 3.0], [1.0 + e, 2.0, 3.0], [1.0, 2.0 - e, 3.0], [50.0, 0.0, 0.0]], np.float32)
    lists = odb.neighbour_lists_brute(p, 0.3)
    labels, n, counts, _ = odb.dbscan(p, 0.3, 2)
    assert np.array_equal(counts, [len(x) for x in lists])
    assert np.array_equal(labels, odb.dbscan_open3d(p, 0.3, 2))


def border_case():
    """Cluster 0 (points 0-3) and cluster 1 (points 4-7) at eps = 1, min_points = 4; point 8 is not core and lies
    within eps of one point of each, 0.95 from cluster 0 and 0.5 from cluster 1."""
    x = [0.0, 0.1, 0.2, 0.3, 1.75, 2.3, 2.35, 2.4, 1.25]
    p = np.zeros((len(x), 3), np.float32)
    p[:, 0] = x
    return p, 1.0, 4


def test_border_point_takes_the_lower_id():
    p, eps, min_points = border_case()
    counts = radius_counts_brute(p, eps)
    assert np.all(counts[:8] >= min_points) and counts[8] == 3
    d2 = odb.d2_f32(p[8], p[:8])
    assert d2[4] < d2[3] <= np.float32(eps) ** 2                            # nearer to cluster 1
    labels, n, _, _ = odb.dbscan(p, eps, min_points)
    assert n == 2 and list(labels) == [0, 0, 0, 0, 1, 1, 1, 1, 0]
    assert np.array_equal(labels, odb.dbscan_open3d(p, eps, min_points))
