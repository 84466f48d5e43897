"""CPU reference of estimate_normals with one search bound, and its checks.

Open3D picks the search from the arguments of ``estimate_normals`` (the hybrid search, both arguments, is
``oracle/normals.py``).  With the float32 ``d2 = (dx*dx + dy*dy) + dz*dz`` of the outlier stages, query
included, the covariance and eigensolver of ``oracle/normals.py`` unchanged:

* KNN (``max_nn`` only): the ``min(max_nn, N)`` points first in the total order ``(d2, index)``, no distance
  bound - :func:`knn_estimate_normals` below;
* radius (``radius`` only): every point with ``d2 <= float32(radius)**2``, no cap on the count - the hybrid
  oracle with ``max_nn=None`` (``oracle.normals.estimate_normals(pos, radius, None)``).

The checks: the kd-tree KNN neighbourhoods equal the exhaustive ones index for index, duplicates and far
points included, and the radius search equals the hybrid search whenever max_nn does not bind."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import normals as onrm
from test_oracle_wide_k import cloud_with_duplicates


def _d2(pos, i, c):
    d = pos[c] - pos[i]                                       # float32
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def knn_neighbourhoods(pos, max_nn, margin=16):
    """For every point the ``min(max_nn, N)`` first points in the order ``(d2, index)``, in that order.  The
    kd-tree proposes ``max_nn + margin`` candidates in float64; they are re-ranked by the float32 ``d2``.
    Where the k-th float32 distance comes within rounding of the farthest candidate (a point outside the
    candidates might tie or beat it), every point within that distance is fetched and re-ranked instead."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    n = pos.shape[0]
    k = min(int(max_nn), n)
    kq = min(n, k + margin)
    p64 = pos.astype(np.float64)
    tree = cKDTree(p64)
    dist, nn = tree.query(p64, k=kq, workers=-1)
    dist, nn = dist.reshape(n, kq), nn.reshape(n, kq)
    out = []
    for i in range(n):
        c = nn[i]
        d2 = _d2(pos, i, c)
        order = np.lexsort((c, d2))[:k]
        kth = float(d2[order[-1]])
        if kq < n and not kth < dist[i, -1] ** 2 * (1.0 - 1e-5):
            c = np.asarray(tree.query_ball_point(p64[i], np.sqrt(kth) * (1.0 + 1e-5) + 1e-7), dtype=np.int64)
            d2 = _d2(pos, i, c)
            order = np.lexsort((c, d2))[:k]
        out.append(c[order])
    return out


def knn_neighbourhoods_brute(pos, max_nn):
    """The KNN search by exhaustive float32 distances (small N only): pins :func:`knn_neighbourhoods`."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    k = min(int(max_nn), pos.shape[0])
    d = pos[:, None, :] - pos[None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    order = np.argsort(d2, axis=1, kind="stable")             # stable: equal d2 stay in index order
    return list(order[:, :k].astype(np.int64))


def knn_estimate_normals(pos, max_nn):
    """KNN search; returns ``(normals float32[N,3], counts int32[N], covariances float64[N,3,3])`` like
    ``oracle.normals.estimate_normals``."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    n = pos.shape[0]
    normals = np.zeros((n, 3), dtype=np.float32)
    counts = np.zeros(n, dtype=np.int32)
    covs = np.zeros((n, 3, 3), dtype=np.float64)
    for i, nb in enumerate(knn_neighbourhoods(pos, max_nn)):
        C = onrm.covariance(pos, i, nb)
        covs[i] = C
        counts[i] = nb.size
        normals[i] = np.asarray(onrm.normal_from_covariance(C), dtype=np.float64).astype(np.float32)
    return normals, counts, covs


@pytest.mark.parametrize("k", [30, 100, 1024])
def test_kdtree_knn_equals_brute_force(k):
    p = cloud_with_duplicates()
    b = knn_neighbourhoods_brute(p, k)
    for margin in (16, 0):                             # margin 0: every query takes the re-ranked ball
        a = knn_neighbourhoods(p, k, margin=margin)
        assert len(a) == len(b) == p.shape[0]
        for i, (x, y) in enumerate(zip(a, b)):
            assert x.size == k and np.array_equal(x, y), (margin, i)
    normals, counts, cov = knn_estimate_normals(p, k)
    assert np.all(counts == k) and normals.dtype == np.float32 and cov.shape == (p.shape[0], 3, 3)


def test_knn_fewer_points_than_max_nn():
    p = cloud_with_duplicates(n=40)
    for n in (1, 2, 3, 7):
        normals, counts, _ = knn_estimate_normals(p[:n], 30)
        assert np.all(counts == n)
        if n < 3:
            assert np.array_equal(normals, np.tile(np.array([0, 0, 1], np.float32), (n, 1)))


@pytest.mark.parametrize("radius", [0.4, 1.0])
def test_radius_equals_hybrid_without_cap(radius):
    p = cloud_with_duplicates()
    got = onrm.estimate_normals(p, radius, None)
    big = int(got[1].max())
    assert big >= 20 and (got[1] < 3).any()
    ref = onrm.estimate_normals(p, radius, big)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)
