"""The statistical-outlier oracle at the wide neighbourhood sizes (64 < k <= 1024): the kd-tree version
(candidates with a margin, re-ranked in float32) equals the exhaustive one bit for bit, duplicates
included, so the GPU parity tests at these k compare against a pinned reference."""
import numpy as np
import pytest

from oracle import outliers


def cloud_with_duplicates(n=2000, seed=3):
    rng = np.random.default_rng(seed)
    p = rng.normal(0.0, 1.0, size=(n, 3)).astype(np.float32)
    p[: n // 20] = p[n // 20: n // 10]                 # 5 % exact duplicates: tied distances
    p[-5:] = np.float32(40.0) + p[-5:]                 # a few far points
    return p


@pytest.mark.parametrize("k", [100, 1024])
def test_kdtree_avg_distance_equals_brute_force(k):
    p = cloud_with_duplicates()
    a = outliers.knn_avg_distance(p, k)
    b = outliers.knn_avg_distance_brute(p, k)
    assert a.dtype == np.float32 and a.shape == (p.shape[0],)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
