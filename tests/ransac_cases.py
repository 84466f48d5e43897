"""Seeded clouds and sample tables for the RANSAC plane segmentation tests, and a float32 model of
which evaluations ``k_rs_score`` finds ambiguous.

The band model restates the scoring kernel's pre-test (``csrc/ransac.cu``): a hypothesis chunk of
``CH`` planes, ``hm = RS_EPS * (max |float32(d_h)| over the chunk + float32(thr) + 1)`` and, per
point, ``m = RS_EPS * (|x| + |y| + |z|) + hm``, all in float32 in that order.  An evaluation is in
band when ``thr32 - m <= |d32| < thr32 + m``; the kernel re-decides those in float64.  The model
only shows that a case reaches the path it targets: what the tests pass on is equality with
``oracle/ransac.py``.

Every hypothesis is planted through an explicit sample table whose indices are in range (the
kernel clamps an out-of-range index to ``P - 1``; the oracle does not).
"""
from __future__ import annotations

import math
import os

import numpy as np

from oracle import ransac

RS_EPS = np.float32(5e-7)
TILE_POINTS, TILE_THREADS, TILE_ITEMS = 1024, 256, 4
SM_COUNT = 148
QCAP = 128


def chunk_size(iters: int, knob: int | None = None) -> int:
    """Hypotheses per scoring CTA: 20 or 16, whichever pads ``iters`` less (the default), or 10 / 8
    under ``APC_RS_CH=10``."""
    knob = int(os.environ.get("APC_RS_CH", "20")) if knob is None else knob
    up = lambda a, b: -(-a // b) * b
    if knob in (20, 16):
        return 20 if up(iters, 20) < up(iters, 16) else 16
    return 10 if up(iters, 10) <= up(iters, 8) else 8


def score_grid(n_max: int, iters: int, ch: int) -> tuple[int, int]:
    """``(CTAs striding over the point tiles, chunks)`` of the scoring launch."""
    n_tiles = -(-n_max // TILE_POINTS)
    n_chunks = -(-iters // ch)
    gx0 = min(n_tiles, max(1, SM_COUNT * (2 if ch <= 10 else 1) // n_chunks))
    return -(-n_tiles // -(-n_tiles // gx0)), n_chunks


def band(pts: np.ndarray, planes: np.ndarray, thr: float, ch: int | None = None) -> dict:
    """Band model of every (point, valid hypothesis) evaluation.

    Returns boolean ``[iters, P]`` arrays ``in_band``, ``disagree`` (float32 and float64 decisions
    differ) and ``sure_in`` (below the band: counted by the float32 pre-test alone), plus ``valid``."""
    iters = planes.shape[0]
    ch = chunk_size(iters) if ch is None else ch
    P32 = np.ascontiguousarray(pts[:, :3], dtype=np.float32)
    P64 = P32.astype(np.float64)
    thr32 = np.float32(thr)
    with np.errstate(invalid="ignore", over="ignore"):
        s = (np.abs(P32[:, 0]) + np.abs(P32[:, 1])) + np.abs(P32[:, 2])
        pm = (RS_EPS * s).astype(np.float32)
        valid = np.any(planes != 0.0, axis=1)
        in_band = np.zeros((iters, P32.shape[0]), dtype=bool)
        disagree = np.zeros_like(in_band)
        sure_in = np.zeros_like(in_band)
        for c0 in range(0, iters, ch):
            dmax = np.float32(0.0)
            for h in range(c0, min(c0 + ch, iters)):                # padding rows are zero planes
                dmax = np.fmax(dmax, np.abs(np.float32(planes[h, 3])))   # fmaxf: NaN ignored
            hm = RS_EPS * ((dmax + thr32) + np.float32(1.0))
            m = (pm + hm).astype(np.float32)
            lo, hi = (thr32 - m).astype(np.float32), (thr32 + m).astype(np.float32)
            for h in range(c0, min(c0 + ch, iters)):
                if not valid[h]:
                    continue
                ad = np.abs(ransac.plane_distance_f32(P32, planes[h]))
                d64 = ransac.plane_distance(P64, planes[h])
                in_band[h] = (lo <= ad) & (ad < hi)
                sure_in[h] = ad < lo
                disagree[h] = (ad < thr32) != (d64 < np.float64(thr))
    return dict(in_band=in_band, disagree=disagree, sure_in=sure_in, valid=valid, ch=ch)


def queue_entries(n_max: int, in_band: np.ndarray, ch: int) -> np.ndarray:
    """Entries each scoring CTA puts in its float64 queue: a thread with an in-band evaluation in a
    tile queues all its ``TILE_ITEMS`` points of that tile.  Shape ``[chunks, CTAs]``."""
    iters, P = in_band.shape
    gx, n_chunks = score_grid(n_max, iters, ch)
    n_tiles = -(-n_max // TILE_POINTS)
    out = np.zeros((n_chunks, gx), dtype=np.int64)
    idx = np.arange(P)
    tile, thread = idx // TILE_POINTS, idx % TILE_THREADS
    for c in range(n_chunks):
        amb = in_band[c * ch:(c + 1) * ch].any(axis=0)
        per_thread = np.zeros((n_tiles, TILE_THREADS), dtype=bool)
        np.logical_or.at(per_thread, (tile[amb], thread[amb]), True)
        queued = per_thread.sum(axis=1) * TILE_ITEMS
        np.add.at(out[c], np.arange(n_tiles) % gx, queued)
    return out


def planes_of(pts: np.ndarray, table: np.ndarray) -> np.ndarray:
    P64 = np.asarray(pts[:, :3], dtype=np.float32).astype(np.float64)
    return np.stack([ransac.hypothesis(P64, row) for row in table])


def early_stop_bound(inl: int, P: int, ransac_n: int, iters: int, probability: float) -> float:
    """The bound the oracle's ``select`` sets when a hypothesis with ``inl`` inliers becomes the best."""
    if inl >= P:
        return 0.0
    fitness = np.float64(inl) / np.float64(P)
    fn = fitness
    for _ in range(ransac_n - 1):
        fn = fn * fitness
    denom = math.log(1.0 - float(fn))
    log1mp = math.log(1.0 - probability) if probability < 1.0 else -math.inf
    cand = math.inf if denom == 0.0 else log1mp / denom
    return min(cand, float(iters))


def _unit(v):
    return v / np.linalg.norm(v)


def _basis(n):
    u = _unit(np.cross(n, [1.0, 0.0, 0.0] if abs(n[0]) < 0.9 else [0.0, 1.0, 0.0]))
    return u, np.cross(n, u)


def _perms3(a, b, c):
    return [(a, b, c), (a, c, b), (b, a, c), (b, c, a), (c, a, b), (c, b, a)]


# ---- band cloud --------------------------------------------------------------------------------
def band_cloud(thr: float, seed: int = 0, n_planes: int = 4, per_plane: int = 1200, n_clutter: int = 1500,
               iters: int = 40, ulps: int = 4):
    """Tilted planes with float64 coefficients that float32 cannot hold, each with points at float64
    distance within ``ulps`` float32 ulps of ``thr`` on both sides, plus the exact plane z = 0 with
    points at |z| = thr32 + k ulps, k in -3..3 (with thr = 0.25 those lie at d64 == thr exactly:
    outliers, the test being strict).  The table holds the 6 anchor orders of every plane (distinct
    float64 fits of nearly one plane: a point in band for one is in band for all six) and random
    clutter triangles, shuffled over ``iters`` rows.  Returns ``(pts float32[P, 3], table, meta)``."""
    rng = np.random.default_rng(seed)
    thr32 = np.float32(thr)
    tol = ulps * float(np.spacing(thr32))
    parts, rows = [], []
    base = 0
    for _ in range(n_planes):
        n = _unit(np.array([rng.uniform(-0.4, 0.4), rng.uniform(-0.4, 0.4), 1.0]))
        u, v = _basis(n)
        centre = np.array([rng.uniform(-4, 4), rng.uniform(-4, 4), rng.uniform(-1, 1)])
        ang = rng.uniform(0, 2 * np.pi) + np.array([0.0, 2.1, 4.2])
        anchors = (centre + 3.0 * (np.cos(ang)[:, None] * u + np.sin(ang)[:, None] * v)).astype(np.float32)
        plane = ransac.triangle_plane(*anchors.astype(np.float64))
        assert np.all(plane[:3].astype(np.float32).astype(np.float64) != plane[:3])   # not float32 values
        got = []
        while sum(len(g) for g in got) < per_plane:
            st = rng.uniform(-5, 5, size=(400_000, 2))
            side = rng.choice([-1.0, 1.0], size=400_000)
            cand = (centre + st[:, :1] * u + st[:, 1:] * v + (side * thr)[:, None] * n).astype(np.float32)
            d64 = ransac.plane_distance(cand.astype(np.float64), plane)
            got.append(cand[np.abs(d64 - thr) <= tol])
        pts = np.concatenate(got)[:per_plane]
        parts.append(np.concatenate([anchors, pts]))
        rows += _perms3(base, base + 1, base + 2)
        base += 3 + per_plane
    # the exact plane z = 0: every distance is exact in float64 and in float32
    anchors = np.array([[-3, -3, 0], [3, -3, 0], [-3, 3, 0]], dtype=np.float32)
    k = np.arange(-3, 4)
    zs = np.concatenate([thr32 + k * np.spacing(thr32), -(thr32 + k * np.spacing(thr32))]).astype(np.float32)
    ex = np.zeros((zs.size * 20, 3), dtype=np.float32)
    ex[:, :2] = rng.uniform(-5, 5, size=(ex.shape[0], 2))
    ex[:, 2] = np.repeat(zs, 20)
    parts.append(np.concatenate([anchors, ex]))
    rows += _perms3(base, base + 1, base + 2)
    base += 3 + ex.shape[0]
    clutter = rng.uniform([-8, -8, -3], [8, 8, 3], size=(n_clutter, 3)).astype(np.float32)
    parts.append(clutter)
    while len(rows) < iters:
        rows.append(tuple(base + rng.choice(n_clutter, 3, replace=False)))
    pts = np.concatenate(parts)
    table = np.array(rows, dtype=np.int32)[rng.permutation(len(rows))][:iters]
    exact_ties = int(np.sum(np.abs(ex[:, 2].astype(np.float64)) == thr))
    return pts, table, dict(exact_ties=exact_ties)


# ---- all-ambiguous cloud ---------------------------------------------------------------------------
AMBIGUOUS_THR = 2e-5


def all_ambiguous_cloud(P: int = 300_332, seed: int = 1, iters: int = 20):
    """Every point lies in the rounding band of hypothesis 0, anchors included: the points sit at
    |d64| within 0.4 m of ``thr`` (their own band half-width) of a tilted plane through three anchors
    at the far corners of a 100 m patch, where m > thr.  So every thread of every tile queues its
    points and every CTA overflows its queue.  ``P`` is ragged (300 332 = 293 tiles + 300 points), so
    the last tile queues past-the-end entries.  The other ``iters - 1`` rows are random triangles of
    the cloud: planes within microradians of the first.  Returns ``(pts, table, thr)``."""
    rng = np.random.default_rng(seed)
    thr = AMBIGUOUS_THR
    n = _unit(np.array([0.03, -0.02, 1.0]))
    u, v = _basis(n)
    centre = np.array([0.0, 0.0, 0.5])
    anchors = (centre + np.array([[-45, -45], [45, -40], [-40, 45]]) @ np.stack([u, v])).astype(np.float32)
    plane = ransac.triangle_plane(*anchors.astype(np.float64))
    out = [anchors]
    have = 3
    while have < P:
        k = 2 * (P - have) + 1000
        st = rng.uniform(-50, 50, size=(k, 2))
        foot = centre + st[:, :1] * u + st[:, 1:] * v
        s = (np.abs(foot).sum(axis=1) * float(RS_EPS))
        off = rng.choice([-1.0, 1.0], size=k) * (thr + rng.uniform(-0.4, 0.4, size=k) * s)
        cand = (foot + off[:, None] * plane[:3]).astype(np.float32)
        b = band(cand, plane[None, :], thr, ch=chunk_size(iters))
        keep = cand[b["in_band"][0]]
        out.append(keep[:P - have])
        have += out[-1].shape[0]
    pts = np.concatenate(out)
    rows = [(0, 1, 2)] + [tuple(rng.choice(P, 3, replace=False)) for _ in range(iters - 1)]
    return pts, np.array(rows, dtype=np.int32), thr


# ---- planted ground: the early-stop bound falls at a chosen iteration ----------------------------
def planted_ground_cloud(target_bound: float, winner_it: int, later_it: int, iters: int, ransac_n: int = 3,
                         probability: float = 0.99, P: int = 4000, seed: int = 2, thr: float = 0.2):
    """Ground G1 (|z| <= 0.04) on the plane z = 0, a second layer G2 at z in [0.25, 0.33], clutter at
    z >= 1.  Row ``winner_it`` fits z = 0 through anchors on it (inliers: G1 and the anchors of the
    other plane); row ``later_it`` fits z = 0.15 through its own anchors (inliers: G1 + G2 + both sets
    of anchors - more).  |G1| is chosen so that the oracle's bound after ``winner_it`` is the one
    closest to ``target_bound`` that is not within 1e-9 (relative) of an integer.  Every other row is a
    random clutter triangle.  Returns ``(pts, table, meta)``."""
    rng = np.random.default_rng(seed)
    na = ransac_n
    best = None
    for g1 in range(na, P // 2):
        b = early_stop_bound(g1 + na, P, ransac_n, iters, probability)
        frac = abs(b - round(b))
        if frac <= 1e-9 * max(1.0, b) or not b < iters:
            continue
        if best is None or abs(b - target_bound) < abs(best[1] - target_bound):
            best = (g1, b)
    g1, bound = best
    n_g2 = 60
    n_clutter = P - g1 - n_g2 - na
    ang = np.linspace(0, 2 * np.pi, na, endpoint=False) + 0.3
    ring = np.stack([6 * np.cos(ang), 6 * np.sin(ang)], 1)
    anchors0 = np.concatenate([ring, np.zeros((na, 1))], 1).astype(np.float32)           # part of G1
    anchors1 = np.concatenate([ring * 0.7, np.full((na, 1), 0.15)], 1).astype(np.float32)
    G1 = np.concatenate([rng.uniform(-15, 15, (g1 - na, 2)), rng.uniform(-0.04, 0.04, (g1 - na, 1))], 1)
    G2 = np.concatenate([rng.uniform(-15, 15, (n_g2, 2)), rng.uniform(0.25, 0.33, (n_g2, 1))], 1)
    clutter = rng.uniform([-20, -20, 1.0], [20, 20, 8.0], size=(n_clutter, 3))
    pts = np.concatenate([anchors0, G1.astype(np.float32), anchors1, G2.astype(np.float32),
                          clutter.astype(np.float32)])
    c0 = P - n_clutter
    table = np.array([c0 + rng.choice(n_clutter, ransac_n, replace=False) for _ in range(iters)], dtype=np.int32)
    table[winner_it] = np.arange(na)
    table[later_it] = g1 + np.arange(na)
    return pts, table, dict(bound=bound, winner_it=winner_it, later_it=later_it, inliers=g1 + na)


# ---- selection over many chunks --------------------------------------------------------------------
def selection_cloud(winner_it: int, iters: int = 4096, P: int = 41_000, seed: int = 3):
    """A symmetric ground (z and -z both present, |z| <= 0.04) and clutter at z >= 1.  Row ``winner_it``
    fits z = 0; rows fitting z = +-0.02 / +-0.03 (the same inliers - the ground and every anchor - and a
    larger error) sit before and after it; copies of the winner's row follow it (an equal key: the
    earlier row wins); every other row is a random clutter triangle.  Returns ``(pts, table, meta)``."""
    rng = np.random.default_rng(seed)
    levels = [0.0, 0.02, -0.02, 0.03, -0.03]
    ang = np.array([0.3, 2.4, 4.4])
    anchors = np.concatenate([np.concatenate([np.stack([(5 + i) * np.cos(ang), (5 + i) * np.sin(ang)], 1),
                                              np.full((3, 1), z)], 1) for i, z in enumerate(levels)]).astype(np.float32)
    half = np.concatenate([rng.uniform(-15, 15, (9000, 2)), rng.uniform(0.0, 0.04, (9000, 1))], 1).astype(np.float32)
    mirror = half * np.float32([1, 1, -1])
    ground = np.concatenate([half, mirror])
    n_clutter = P - anchors.shape[0] - ground.shape[0]
    clutter = rng.uniform([-20, -20, 1.0], [20, 20, 12.0], size=(n_clutter, 3)).astype(np.float32)
    pts = np.concatenate([anchors, ground, clutter])
    c0 = P - n_clutter
    table = np.array([c0 + rng.choice(n_clutter, 3, replace=False) for _ in range(iters)], dtype=np.int32)
    win = np.array([0, 1, 2], dtype=np.int32)
    tie_rows = [r for r in (0, 1, winner_it - 1, winner_it - 129, winner_it + 2, winner_it + 128, iters - 2)
                if 0 <= r < iters and r != winner_it]
    for k, r in enumerate(tie_rows):
        lvl = 1 + k % 4
        table[r] = 3 * lvl + np.array(_perms3(0, 1, 2)[k % 6], dtype=np.int32)
    dup_rows = [r for r in (winner_it + 1, winner_it + 127, winner_it + 300, iters - 1) if winner_it < r < iters]
    for k, r in enumerate(dup_rows):
        table[r] = win if k % 2 == 0 else win[::-1]
    table[winner_it] = win
    return pts, table, dict(tie_rows=tie_rows, dup_rows=dup_rows)


# ---- accumulator saturation ------------------------------------------------------------------------
def saturation_cloud(thr: float = 0.2, P: int = 67_001, iters: int = 4096, seed: int = 4):
    """Every point a sure inlier of every hypothesis at the largest float32 distance the pre-test still
    accepts: the plane is z = 0 exactly (three anchors at z = 0, the 6 anchor orders cycling through
    the table) and every other point sits at z = +-(the largest float32 below thr32 - m), so each point
    adds rint(u) ~ 65 500 to its thread's packed error sum, and a 128-point window carries nearly
    2^23.  With 4096 rows there is one scoring CTA per chunk and 66 tiles of points: every thread
    flushes its accumulator twice with full windows.  Returns ``(pts, table)``."""
    rng = np.random.default_rng(seed)
    thr32 = np.float32(thr)
    anchors = np.array([[-9, -9, 0], [9, -9, 0], [-9, 9, 0]], dtype=np.float32)
    xy = rng.uniform(-10, 10, size=(P - 3, 2)).astype(np.float32)
    hm = RS_EPS * ((np.float32(0.0) + thr32) + np.float32(1.0))
    z = np.full(P - 3, thr32, dtype=np.float32)
    for _ in range(3):                                           # m depends on |z|: settle it
        m = (RS_EPS * ((np.abs(xy[:, 0]) + np.abs(xy[:, 1])) + z) + hm).astype(np.float32)
        z = np.nextafter((thr32 - m).astype(np.float32), np.float32(0))
    sign = rng.choice(np.float32([-1, 1]), size=P - 3)
    pts = np.concatenate([anchors, np.concatenate([xy, (sign * z)[:, None]], 1)]).astype(np.float32)
    perms = _perms3(0, 1, 2)
    table = np.array([perms[i % 6] for i in range(iters)], dtype=np.int32)
    return pts, table


# ---- generic ground + clutter ----------------------------------------------------------------------
def ground_clutter_cloud(P: int, seed: int = 5, ground_frac: float = 0.6, centre=(0.0, 0.0, 0.0)):
    """A tilted, noisy ground plane and clutter above it, around ``centre``."""
    rng = np.random.default_rng(seed)
    ng = int(P * ground_frac)
    xy = rng.uniform(-25, 25, size=(ng, 2))
    g = np.concatenate([xy, (0.02 * xy[:, :1] - 0.01 * xy[:, 1:] + rng.normal(0, 0.05, (ng, 1)))], 1)
    c = rng.uniform([-25, -25, 0.5], [25, 25, 6.0], size=(P - ng, 3))
    pts = np.concatenate([g, c])[rng.permutation(P)] + np.asarray(centre)
    return pts.astype(np.float32)
