"""FPFH features and feature matching: CPU oracle (test infrastructure; never imported by the product path).

Restates Open3D's ``t.pipelines.registration.compute_fpfh_feature`` and ``correspondences_from_features``
(``t/pipelines/kernel/Feature*``, legacy ``Feature.cpp``) as recalled from Open3D 0.18/0.19: Open3D is not
installable here, PARITY UNPINNED.  Neighbourhoods are inputs, so nothing of the search is restated: the hybrid
lists of ``oracle.normals.neighbourhoods`` or the KNN lists of ``knn_neighbourhoods`` (``tests/
test_oracle_normals_search.py``), each ordered by ``(d2, index)`` with the float32 ``d2 = (dx*dx + dy*dy) + dz*dz``.

* **Pair feature** ``(p1, n1, p2, n2)``, Open3D ``ComputePairFeatures``, float64 from the float32 inputs:
  ``dp = p2 - p1``, ``d = |dp|`` (zero feature when ``d == 0``); ``a1 = n1.dp / d``, ``a2 = n2.dp / d``; when
  ``|a1| < |a2|`` the roles swap (``n1 <-> n2``, ``dp = -dp``, ``f2 = -a2``), else ``f2 = a1``.  Open3D tests
  ``acos|a1| > acos|a2|``: the same except where ``acos`` rounds two values to one (deviation, so that no libm
  call decides a swap).  ``v = dp x n1`` (zero feature when ``|v| == 0``), normalised; ``w = n1 x v``;
  ``f1 = v.n2``, ``f0 = atan2(w.n2, n1.n2)``.  Dot products are ``(x0*y0 + x1*y1) + x2*y2``.
* **Bins** 3 x 11: ``floor((11 (f0 + pi)) / (2 pi))`` and ``floor((11 (f + 1)) * 0.5)`` for ``f1``, ``f2``, each
  clamped to 0..10, at offsets 0, 11, 22.  A pair with a non-finite feature (a NaN normal) adds to no bin.  A zero
  normal is an ordinary input (it gives finite features).  Near a bin edge CUDA's and libm's ``atan2`` may differ in
  the last ulp: :func:`spfh` flags every point with a bin argument within 1e-9 of an interior edge (1..10; the
  outer edges 0 and 11 clamp to the same bin either way).
* **SPFH** of a point whose neighbourhood has ``m`` entries: zeros for ``m <= 1``, else the bin counts of its pairs
  with entries ``1..m-1`` times ``float64(100 / (m - 1))``, rounded to float32.  Open3D adds ``100 / (m - 1)``
  once per pair (a few ulp apart: deviation).  Entry 0 is skipped, as Open3D skips the first neighbour: it is at
  ``d2 == 0`` (the query, or a duplicate of it with a lower index), so its pair feature is zero.  Skipping the
  query itself instead gives the same histogram whenever the query is in its list; it is absent only when ``m``
  duplicates with lower indices fill the list, and skipping entry 0 keeps ``m - 1`` pairs there too.
* **FPFH** (float64, rounded to float32 at the end): ``raw[j] = sum spfh[k][j] / d2_k`` over the entries ``1..m-1``
  with ``d2_k > 0``, sequentially in list order; ``sum_g`` = the sequential sum of ``raw`` over group ``g``'s 11
  bins (Open3D interleaves the group sums with the bins: a fixed-order deviation); ``scale_g = 100 / sum_g`` when
  ``sum_g != 0``, else 0; ``feature[j] = raw[j] * scale_g + spfh[i][j]``.
* **Matching**: ``d2 = sum_j (a_j - b_j)^2`` in float32, increasing ``j``; a row's match is the other set's row
  with the smallest ``(d2, index)`` among the finite ``d2``, none when there is none.  Pairs ``(i, nn_st[i])``
  in ascending ``i`` for the rows with a match; with the mutual filter only those with ``nn_ts[nn_st[i]] == i``,
  unless there are not more than ``ratio * n_src`` (float64) of them (recalled: ``>``), when Open3D warns and
  returns the unfiltered set.
"""
from __future__ import annotations

import math

import numpy as np

BINS = 33


def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def _cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1],
                     a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)


def pair_features(p1, n1, p2, n2) -> np.ndarray:
    """float64 ``[k, 3]`` = ``(f0, f1, f2)`` of every row of the float32 ``[k, 3]`` inputs."""
    p1, n1, p2, n2 = (np.asarray(x, np.float32).reshape(-1, 3).astype(np.float64) for x in (p1, n1, p2, n2))
    with np.errstate(invalid="ignore", divide="ignore"):
        dp = p2 - p1
        d = np.sqrt(_dot(dp, dp))
        a1 = _dot(n1, dp) / d
        a2 = _dot(n2, dp) / d
        swap = (np.abs(a1) < np.abs(a2))[:, None]
        u = np.where(swap, n2, n1)
        t = np.where(swap, n1, n2)
        e = np.where(swap, -dp, dp)
        f2 = np.where(swap[:, 0], -a2, a1)
        v = _cross(e, u)
        vn = np.sqrt(_dot(v, v))
        v = v / vn[:, None]
        w = _cross(u, v)
        f1 = _dot(v, t)
        f0 = np.arctan2(_dot(w, t), _dot(u, t))
    out = np.stack([f0, f1, f2], axis=1)
    out[(d == 0.0) | (vn == 0.0)] = 0.0
    return out


def bin_arguments(f: np.ndarray) -> np.ndarray:
    """The values whose floor is the bin, ``[k, 3]``."""
    f = np.asarray(f, np.float64).reshape(-1, 3)
    return np.stack([(11.0 * (f[:, 0] + math.pi)) / (2.0 * math.pi),
                     (11.0 * (f[:, 1] + 1.0)) * 0.5,
                     (11.0 * (f[:, 2] + 1.0)) * 0.5], axis=1)


def bins(f: np.ndarray):
    """``(bins int64[k, 3] with the group offsets, finite bool[k], near_edge bool[k])``."""
    x = bin_arguments(f)
    finite = np.isfinite(f).all(axis=1)
    with np.errstate(invalid="ignore"):
        b = np.clip(np.floor(np.where(finite[:, None], x, 0.0)), 0, 10).astype(np.int64) + np.array([0, 11, 22])
        r = np.round(x)
        near = finite & ((np.abs(x - r) < 1e-9) & (r >= 1) & (r <= 10)).any(axis=1)   # interior edges: 0, 11 clamp
    return b, finite, near


def _d2(pos, i, c):
    d = pos[c] - pos[i]                                       # float32
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def spfh(pos, normals, nbs):
    """``(spfh float32[n, 33], counts int32[n], near_edge bool[n])`` from the ``(d2, index)``-ordered lists."""
    pos = np.ascontiguousarray(pos, np.float32)
    normals = np.ascontiguousarray(normals, np.float32)
    n = pos.shape[0]
    counts = np.array([len(nb) for nb in nbs], np.int32)
    qi = np.concatenate([np.full(max(len(nb) - 1, 0), i, np.int64) for i, nb in enumerate(nbs)] + [np.zeros(0, np.int64)])
    ki = np.concatenate([np.asarray(nb[1:], np.int64) for nb in nbs] + [np.zeros(0, np.int64)])
    f = pair_features(pos[qi], normals[qi], pos[ki], normals[ki])
    b, finite, near = bins(f)
    hist = np.zeros((n, BINS), np.int64)
    for g in range(3):
        np.add.at(hist, (qi[finite], b[finite, g]), 1)
    flag = np.zeros(n, bool)
    flag[qi[near]] = True
    with np.errstate(divide="ignore"):
        incr = np.where(counts > 1, 100.0 / np.maximum(counts - 1, 1).astype(np.float64), 0.0)
    return (hist.astype(np.float64) * incr[:, None]).astype(np.float32), counts, flag


def fpfh(pos, spfh_f32, nbs) -> np.ndarray:
    """float32 ``[n, 33]`` FPFH from the SPFH and the same lists."""
    pos = np.ascontiguousarray(pos, np.float32)
    sp = np.asarray(spfh_f32, np.float32)
    out = np.zeros((pos.shape[0], BINS), np.float32)
    for i, nb in enumerate(nbs):
        ks = np.asarray(nb[1:], np.int64)
        raw = np.zeros(BINS)
        if ks.size:
            d2 = _d2(pos, i, ks)
            ks, d2 = ks[d2 > 0], d2[d2 > 0]
            if ks.size:
                raw = np.cumsum(sp[ks].astype(np.float64) / d2.astype(np.float64)[:, None], axis=0)[-1]
        scale = np.zeros(BINS)
        for g in range(3):
            s = np.cumsum(raw[11 * g:11 * g + 11])[-1]
            scale[11 * g:11 * g + 11] = 100.0 / s if s != 0.0 else 0.0
        out[i] = (raw * scale + sp[i].astype(np.float64)).astype(np.float32)
    return out


def compute_fpfh(pos, normals, nbs):
    """``(features float32[n, 33], spfh float32[n, 33], counts int32[n], near_edge bool[n])``.  ``near_edge``
    flags the points whose FPFH reads an SPFH with a pair near a bin edge (their own or a neighbour's)."""
    sp, counts, flag = spfh(pos, normals, nbs)
    feat = fpfh(pos, sp, nbs)
    near = np.array([bool(flag[np.asarray(nb, np.int64)].any()) or bool(flag[i]) for i, nb in enumerate(nbs)], bool)
    return feat, sp, counts, near


def feature_d2(a, b) -> np.ndarray:
    """float32 ``[na, nb]``: ``sum_j (a_j - b_j)^2`` accumulated in increasing ``j``."""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    d2 = np.zeros((a.shape[0], b.shape[0]), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for j in range(a.shape[1]):
            x = a[:, j][:, None] - b[:, j][None, :]
            d2 = d2 + x * x
    return d2


def nearest(a, b) -> np.ndarray:
    """int64 ``[na]``: the row of ``b`` with the smallest ``(d2, index)`` among the finite ``d2``, -1 for none."""
    if b.shape[0] == 0:
        return np.full(a.shape[0], -1, np.int64)
    d2 = feature_d2(a, b)
    d2 = np.where(np.isfinite(d2), d2, np.inf)
    nn = np.argmin(d2, axis=1)                      # first occurrence: the lower index
    return np.where(np.isfinite(d2[np.arange(a.shape[0]), nn]), nn, -1).astype(np.int64)


def correspondences(src, tgt, mutual_filter=False, ratio=0.1):
    """``(pairs int64[K, 2], nearest int64[n_src], fell_back bool)``."""
    src = np.asarray(src, np.float32)
    tgt = np.asarray(tgt, np.float32)
    nn = nearest(src, tgt)
    rows = np.flatnonzero(nn >= 0)
    pairs = np.stack([rows, nn[rows]], axis=1).astype(np.int64).reshape(-1, 2)
    if not mutual_filter:
        return pairs, nn, False
    back = nearest(tgt, src)
    keep = back[pairs[:, 1]] == pairs[:, 0]
    if keep.sum() > ratio * float(src.shape[0]):
        return pairs[keep], nn, False
    return pairs, nn, True
