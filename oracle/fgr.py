"""Fast Global Registration: CPU oracle (test infrastructure).

Restates Fast Global Registration (Zhou, Park, Koltun, ECCV 2016) as Open3D runs it
(``registration_fgr_based_on_feature_matching`` / ``registration_fgr_based_on_correspondence``,
``FastGlobalRegistration.cpp`` of 0.18/0.19, and the authors' code) - PARITY UNPINNED: recalled, Open3D itself is
not run here.  Inputs are float32 positions promoted to float64; all arithmetic is float64 and unfused.

  1. initial matching (feature entry): the mutual set of ``oracle.features.correspondences(..., mutual_filter=True)``
     before its ratio fallback - the source rows ``i`` whose nearest target row ``j`` (``features.nearest``) has
     ``i`` as its nearest source row, in ascending ``i`` (Open3D's ``InitialMatching`` cross check; no fallback);
  2. tuple test (feature entry, ``tuple_test``): ``K`` pairs, trials ``t = 0 .. 100 K - 1``; draw ``k`` of trial
     ``t`` is ``((z >> 32) * K) >> 32`` with ``z = splitmix64(seed + (t << 32) + k)`` (mod 2^64; the RANSAC stream's
     index formula without its rejection of repeats).  With the source points ``p_k`` and target points ``q_k`` of
     the three pairs, ``l = sqrt((dx*dx + dy*dy) + dz*dz)`` over the edges (0,1), (1,2), (2,0); the tuple is
     accepted iff ``li * scale < lj`` and ``lj < li / scale`` on all three edges (each product or quotient rounded
     once).  A repeated draw or a shared point gives a zero edge and is rejected.  Accepted tuples append their
     three pairs in draw order; the test stops after ``maximum_tuple_count`` accepted tuples, and ``trials`` is the
     index of the last trial examined + 1.  Duplicated pairs stay;
  3. normalisation: ``mu_s``, ``mu_t`` the means of ALL points of each cloud, ``D`` the largest norm of a centred
     point of either cloud; relative scale divides the centred points by ``D`` and starts with ``par = 1``,
     absolute scale keeps metres and starts with ``par = D``;
  4. ``iteration_number`` iterations from ``T = I``: if ``decrease_mu and itr % 4 == 0 and
     par > maximum_correspondence_distance``, ``par /= division_factor`` (before the step); ``q' = T q`` from the
     ORIGINAL normalised target, ``r = p - q'``, ``s = (par / (|r|^2 + par))^2``; with the Jacobian rows
     x ``(0, -q'z, q'y, -1, 0, 0)``, y ``(q'z, 0, -q'x, 0, -1, 0)``, z ``(-q'y, q'x, 0, 0, 0, -1)``,
     ``A = sum s J J^T``, ``b = sum s J r``; ``A x = -b`` by ``registration.cholesky_solve`` (DEGENERATE when it
     fails: the loop stops), ``T = pose_to_transformation(x) T``;
  5. result: with ``R, t`` of the final ``T``, the source-to-target transform in metres is ``[R^T | mu_t - R^T mu_s
     - g R^T t]`` (``g = D`` relative, 1 absolute): the inverse, since the optimiser moves the target onto the
     source.  ``iteration_number = 0`` gives ``[I | mu_t - mu_s]``.  Fewer than ``MIN_PAIRS`` pairs reaching step
     4 is TOO_FEW: the identity, 0 iterations.  A non-finite coordinate makes the normalisation non-finite and the
     first iteration DEGENERATE.

Defined deviations from Open3D: the tuple draws come from the counter-based stream above (Open3D uses its own RNG;
``seed=None`` means 0 here, so results are reproducible); ``T`` accumulates and the original target is transformed
every iteration (Open3D re-transforms its copy of the target in place); the TOO_FEW result is a defined choice.
"""
from __future__ import annotations

import numpy as np

from . import features
from . import registration as reg

OK, TOO_FEW, DEGENERATE = 0, 1, 2
MIN_PAIRS = 10
TRIALS_PER_PAIR = 100
_C1, _C2, _C3 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)


def splitmix64_vec(x) -> np.ndarray:
    """``oracle.ransac.splitmix64`` on a uint64 array (wrapping arithmetic)."""
    z = np.asarray(x, np.uint64) + _C1
    z = (z ^ (z >> np.uint64(30))) * _C2
    z = (z ^ (z >> np.uint64(27))) * _C3
    return z ^ (z >> np.uint64(31))


def draws(seed: int, t, k: int, K: int) -> np.ndarray:
    """int64 draw ``k`` of the trials ``t`` (uint64 array) among ``K`` pairs."""
    x = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + (np.asarray(t, np.uint64) << np.uint64(32)) + np.uint64(k)
    return (((splitmix64_vec(x) >> np.uint64(32)) * np.uint64(K)) >> np.uint64(32)).astype(np.int64)


def edge_lengths(P: np.ndarray) -> np.ndarray:
    """``[m, 3]`` lengths of the edges (0,1), (1,2), (2,0) of ``m`` triangles ``P [m, 3, 3]`` (float64)."""
    out = np.empty(P.shape[:2])
    for e in range(3):
        d = P[:, e] - P[:, (e + 1) % 3]
        out[:, e] = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
    return out


def tuple_test(src, tgt, pairs, seed=0, tuple_scale=0.95, maximum_tuple_count=1000, chunk=1 << 18):
    """``(pairs_used int64[3 * accepted, 2], trials)`` of step 2."""
    P = np.asarray(src, np.float32).astype(np.float64)
    Q = np.asarray(tgt, np.float32).astype(np.float64)
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    K = pairs.shape[0]
    n_trials = TRIALS_PER_PAIR * K
    out, got, trials = [], 0, n_trials
    for t0 in range(0, n_trials, chunk):
        t = np.arange(t0, min(t0 + chunk, n_trials), dtype=np.uint64)
        c = np.stack([draws(seed, t, k, K) for k in range(3)], axis=1)          # [m, 3] pair indices
        li = edge_lengths(P[pairs[c, 0]])
        lj = edge_lengths(Q[pairs[c, 1]])
        ok = np.all((li * tuple_scale < lj) & (lj < li / tuple_scale), axis=1)
        acc = np.flatnonzero(ok)
        if got + acc.size >= maximum_tuple_count:
            acc = acc[:maximum_tuple_count - got]
            out.append(c[acc])
            got = maximum_tuple_count
            trials = int(t[acc[-1]]) + 1
            break
        out.append(c[acc])
        got += acc.size
    idx = np.concatenate(out, axis=0).reshape(-1) if out else np.zeros(0, np.int64)
    return pairs[idx].reshape(-1, 2), trials


def par_schedule(par0, iteration_number, division_factor=1.4, decrease_mu=True, maximum_correspondence_distance=0.025):
    """``par`` used by each iteration (after that iteration's schedule step)."""
    out, par = [], float(par0)
    for itr in range(iteration_number):
        if decrease_mu and itr % 4 == 0 and par > maximum_correspondence_distance:
            par /= division_factor
        out.append(par)
    return out


def normalise(src, tgt, use_absolute_scale=False):
    """``(P, Q, mu_s, mu_t, D, g, par0)`` of step 3 (``P``, ``Q`` the normalised float64 clouds)."""
    P = np.asarray(src, np.float32).astype(np.float64)
    Q = np.asarray(tgt, np.float32).astype(np.float64)
    mu_s, mu_t = P.mean(axis=0), Q.mean(axis=0)
    P, Q = P - mu_s, Q - mu_t
    norms = np.concatenate([np.sqrt((P * P).sum(axis=1)), np.sqrt((Q * Q).sum(axis=1))])
    D = float(np.max(norms))
    g, par0 = (1.0, D) if use_absolute_scale else (D, 1.0)
    return P / g, Q / g, mu_s, mu_t, D, g, par0


def system(p, q, T, par):
    """``(A [6, 6], b [6])`` of one iteration: pairs ``p`` (source) and ``q`` (original target), normalised."""
    qt = np.empty_like(q)
    for r in range(3):
        qt[:, r] = ((T[r, 0] * q[:, 0] + T[r, 1] * q[:, 1]) + T[r, 2] * q[:, 2]) + T[r, 3]
    res = p - qt
    s = (par / (((res[:, 0] * res[:, 0] + res[:, 1] * res[:, 1]) + res[:, 2] * res[:, 2]) + par)) ** 2
    A, b = np.zeros((6, 6)), np.zeros(6)
    zero, one = np.zeros(len(q)), np.ones(len(q))
    rows = (np.stack([zero, -qt[:, 2], qt[:, 1], -one, zero, zero], 1),
            np.stack([qt[:, 2], zero, -qt[:, 0], zero, -one, zero], 1),
            np.stack([-qt[:, 1], qt[:, 0], zero, zero, zero, -one], 1))
    for ax, J in enumerate(rows):
        A += (J * s[:, None]).T @ J
        b += (J * (s * res[:, ax])[:, None]).sum(axis=0)
    return A, b


def fgr(src, tgt, pairs, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
        maximum_correspondence_distance=0.025, iteration_number=64):
    """Steps 3-5 on the pairs that reach the optimiser.  Returns a dict with ``transformation``, ``iterations`` and
    ``status``."""
    pairs = np.asarray(pairs, np.int64).reshape(-1, 2)
    if pairs.shape[0] < MIN_PAIRS:
        return dict(transformation=np.eye(4), iterations=0, status=TOO_FEW)
    P, Q, mu_s, mu_t, D, g, par = normalise(src, tgt, use_absolute_scale)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        p, q = P[pairs[:, 0]], Q[pairs[:, 1]]
        T, status, iterations = np.eye(4), OK, 0
        for itr in range(iteration_number):
            if decrease_mu and itr % 4 == 0 and par > maximum_correspondence_distance:
                par /= division_factor
            A, b = system(p, q, T, par)
            x = reg.cholesky_solve(A, -b)
            if x is None:
                status = DEGENERATE
                break
            T = reg.pose_to_transformation(x) @ T
            iterations = itr + 1
        R, t = T[:3, :3], T[:3, 3]
        out = np.eye(4)
        out[:3, :3] = R.T
        out[:3, 3] = mu_t - R.T @ mu_s - g * (R.T @ t)
    return dict(transformation=out, iterations=iterations, status=status)


def mutual_pairs(src_feat, tgt_feat) -> np.ndarray:
    """int64 ``[K, 2]``: step 1, the mutual set without its fallback."""
    pairs, _, _ = features.correspondences(src_feat, tgt_feat, mutual_filter=True, ratio=-1.0)   # never falls back
    return pairs


def fgr_from_features(src, tgt, src_feat, tgt_feat, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
                      maximum_correspondence_distance=0.025, iteration_number=64, tuple_scale=0.95,
                      maximum_tuple_count=1000, tuple_test_on=True, seed=None):
    """Steps 1-5.  The dict of :func:`fgr` plus ``pairs_in`` (the mutual set), ``pairs_used`` and ``trials``."""
    pairs = mutual_pairs(src_feat, tgt_feat)
    used, trials = pairs, 0
    if tuple_test_on:
        used, trials = tuple_test(src, tgt, pairs, 0 if seed is None else int(seed), tuple_scale, maximum_tuple_count)
    out = fgr(src, tgt, used, division_factor, use_absolute_scale, decrease_mu, maximum_correspondence_distance,
              iteration_number)
    out.update(pairs_in=pairs, pairs_used=used, trials=trials)
    return out
