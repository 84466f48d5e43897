"""DBSCAN clustering: CPU oracle (test infrastructure).

Restates Open3D ``PointCloud::ClusterDBSCAN`` (legacy; the tensor ``cluster_dbscan`` calls it) - PARITY
UNPINNED: Open3D itself is not run here.

Choices fixed here:
  * neighbourhood ``N(i) = {j : d2_f32(p_i, p_j) <= r2}`` with ``r2 = float32(eps) * float32(eps)`` and
    ``d2 = (dx*dx + dy*dy) + dz*dz`` in float32, unfused, ``i`` included - the radius predicate of
    ``oracle/outliers.py``.  Open3D's kd-tree keeps ``j`` when the float64 ``d2 < eps^2`` (strict); the two
    differ only for pairs within rounding of ``eps`` apart;
  * ``core(i)`` iff ``|N(i)| >= min_points`` (``min_points`` 0 and 1 both make every point core);
  * clusters are the connected components of the core points, core ``i`` and core ``j`` linked when
    ``j in N(i)``; ids ``0, 1, ...`` in the order of each component's lowest core index;
  * a core point gets its component's id, a non-core point the smallest id among the components of the core
    points in ``N(i)``, otherwise ``-1`` (noise).

``dbscan_open3d`` is Open3D's sequential loop itself (small clouds, brute-force neighbour lists); ``dbscan`` is
the closed form above at scan size.  The tests pin the two together label for label.
"""
from __future__ import annotations

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

from .outliers import d2_f32


def neighbour_lists_brute(pos: np.ndarray, eps: float) -> list:
    r32 = np.float32(eps)
    d2 = d2_f32(pos[:, None, :], pos[None, :, :])
    return [np.flatnonzero(row) for row in d2 <= r32 * r32]


def dbscan_open3d(pos: np.ndarray, eps: float, min_points: int) -> np.ndarray:
    """Open3D's ``ClusterDBSCAN`` loop with the neighbour lists above: points in index order; a non-core point
    still unlabelled becomes noise; an unlabelled core point starts a new cluster that expands through core
    points; the expansion relabels noise points it reaches and leaves points of earlier clusters alone."""
    nbs = neighbour_lists_brute(pos, eps)
    labels = np.full(pos.shape[0], -2, dtype=np.int64)              # -2: undefined
    cluster_label = 0
    for idx in range(pos.shape[0]):
        if labels[idx] != -2:
            continue
        if len(nbs[idx]) < min_points:
            labels[idx] = -1
            continue
        nbs_next = set(nbs[idx].tolist())
        nbs_visited = {idx}
        labels[idx] = cluster_label
        while nbs_next:
            nb = nbs_next.pop()
            nbs_visited.add(nb)
            if labels[nb] == -1:
                labels[nb] = cluster_label
            if labels[nb] != -2:
                continue
            labels[nb] = cluster_label
            if len(nbs[nb]) >= min_points:
                nbs_next.update(q for q in nbs[nb].tolist() if q not in nbs_visited)
        cluster_label += 1
    return labels.astype(np.int32)


def neighbour_pairs(pos: np.ndarray, eps: float):
    """Pairs ``i < j`` with ``d2_f32 <= r2``: proposed by the kd-tree at a slightly larger float64 radius,
    decided in float32."""
    r32 = np.float32(eps)
    tree = cKDTree(pos.astype(np.float64))
    pairs = tree.query_pairs(float(r32) * (1.0 + 1e-5) + 1e-7, output_type="ndarray")
    if pairs.size == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    i, j = pairs[:, 0].astype(np.int64), pairs[:, 1].astype(np.int64)
    keep = d2_f32(pos[i], pos[j]) <= r32 * r32
    return i[keep], j[keep]


def dbscan(pos: np.ndarray, eps: float, min_points: int):
    """Returns ``(labels int32[P], n_clusters, counts uint32[P], tests)``: ``counts = |N(i)|`` and ``tests`` =
    ``sum |N(i)|``, the distance tests a walk over exactly the neighbourhoods makes."""
    P = pos.shape[0]
    if P == 0:
        return np.zeros(0, np.int32), 0, np.zeros(0, np.uint32), 0
    i, j = neighbour_pairs(pos, eps)
    counts = (1 + np.bincount(i, minlength=P) + np.bincount(j, minlength=P)).astype(np.uint32)
    core = counts >= min_points
    cc = core[i] & core[j]
    graph = coo_matrix((np.ones(int(cc.sum()), np.int8), (i[cc], j[cc])), shape=(P, P))
    _, comp = connected_components(graph, directed=False)
    # rank the components that hold core points by their lowest core index
    core_idx = np.flatnonzero(core)
    first = np.full(comp.max() + 1, P, np.int64)
    np.minimum.at(first, comp[core_idx], core_idx)
    roots = np.flatnonzero(first < P)
    order = roots[np.argsort(first[roots])]
    cid = np.full(comp.max() + 1, -1, np.int64)
    cid[order] = np.arange(order.size)
    labels = np.full(P, -1, np.int64)
    labels[core_idx] = cid[comp[core_idx]]
    # border points: the smallest id among their core neighbours
    big = np.iinfo(np.int64).max
    best = np.full(P, big, np.int64)
    for a, b in ((i, j), (j, i)):                                    # a non-core, b core
        m = ~core[a] & core[b]
        np.minimum.at(best, a[m], labels[b[m]])
    border = ~core & (best != big)
    labels[border] = best[border]
    return labels.astype(np.int32), int(order.size), counts, int(counts.astype(np.int64).sum())
