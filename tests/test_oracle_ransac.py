"""CPU checks of the RANSAC oracle's building blocks and of the RANSAC case builders: the float32 FMA
emulation against exact rational arithmetic, the scoring kernel's selection algorithm (prefix records
of a packed key, then a walk that stops at the early-stop bound) against the oracle's sequential
loop, and the preconditions each case builder claims."""
import math
from fractions import Fraction

import numpy as np
import pytest

import ransac_cases as rc
from oracle import ransac


def round_f32(q: Fraction) -> np.float32:
    """``q`` rounded to the nearest float32, ties to even (normal and subnormal range)."""
    if q == 0:
        return np.float32(0.0)
    sign, a = (-1 if q < 0 else 1), abs(q)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    if Fraction(2) ** e > a:
        e -= 1
    quantum = Fraction(2) ** (max(e, -126) - 23)
    n, rem = divmod(a, quantum)
    if rem * 2 > quantum or (rem * 2 == quantum and n % 2 == 1):
        n += 1
    v = n * quantum
    if v >= Fraction(2) ** 128:
        return np.float32(sign * np.inf)
    return np.float32(sign * float(v))


def exact_fma(a, b, c) -> np.float32:
    return round_f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def test_fma32_random_triples():
    rng = np.random.default_rng(0)
    n = 4000
    mant = rng.uniform(1.0, 2.0, size=(3, n)) * rng.choice([-1.0, 1.0], size=(3, n))
    a = (mant[0] * 2.0 ** rng.integers(-20, 20, n)).astype(np.float32)
    b = (mant[1] * 2.0 ** rng.integers(-20, 20, n)).astype(np.float32)
    c = (mant[2] * 2.0 ** rng.integers(-40, 40, n)).astype(np.float32)
    c[: n // 4] = (-(a[: n // 4].astype(np.float64) * b[: n // 4])).astype(np.float32)   # cancellation
    got = ransac.fma32(a, b, c)
    want = np.array([exact_fma(x, y, z) for x, y, z in zip(a, b, c)], dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_fma32_float64_sum_on_a_float32_midpoint():
    """a*b + c built so that the float64 sum lands exactly on a float32 midpoint while the exact sum
    does not: a = 1 + s*2^-j, b = -s*t*2^-24*(1 - s*2^-j)*2^E, so a*b = -s*t*2^(E-24)*(1 - 2^-2j), and
    c in [2^E, 2^(E+1)).  Rounding the float64 sum to float32 naively is then wrong whenever the
    exact sum sits on the other side of the midpoint than ties-to-even goes."""
    rng = np.random.default_rng(1)
    A, B, Cs = [], [], []
    for _ in range(3000):
        j = int(rng.integers(15, 24))
        s = float(rng.choice([-1.0, 1.0]))
        t = float(rng.choice([-1.0, 1.0]))
        E = int(rng.integers(-10, 10))
        A.append(1.0 + s * 2.0 ** -j)
        B.append(-s * t * 2.0 ** (E - 24) * (1.0 - s * 2.0 ** -j))
        Cs.append((1.0 + int(rng.integers(0, 1 << 23)) * 2.0 ** -23) * 2.0 ** E)
    a, b, c = (np.array(v, dtype=np.float32) for v in (A, B, Cs))
    assert np.array_equal(a.astype(np.float64), A) and np.array_equal(b.astype(np.float64), B)
    s64 = a.astype(np.float64) * b + c.astype(np.float64)
    on_mid = (s64.view(np.uint64) & np.uint64((1 << 29) - 1)) == np.uint64(1 << 28)
    exact = [Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z)) for x, y, z in zip(a, b, c)]
    residual = np.array([e != Fraction(float(s)) for e, s in zip(exact, s64)])
    assert np.sum(on_mid & residual) > 2500
    want = np.array([round_f32(e) for e in exact], dtype=np.float32)
    naive = s64.astype(np.float32)
    assert np.sum(naive.view(np.uint32) != want.view(np.uint32)) > 500      # double rounding goes wrong here
    assert np.array_equal(ransac.fma32(a, b, c).view(np.uint32), want.view(np.uint32))


KEY_ERR_MAX = (1 << 40) - 1


def kernel_select(scores, valid, P, ransac_n, iters, probability):
    """The selection of ``rs_select_cta``: the key ``(inl << 40) | (2^40 - 1 - min(err, 2^40 - 1))``
    (0 for an invalid hypothesis or no inliers), the strict prefix maxima of the key sequence as
    records, then a walk over the records that stops at the first beyond the current bound."""
    records, best = [], 0
    for it in range(iters):
        inl, err = scores[it]
        key = (inl << 40) | (KEY_ERR_MAX - min(err, KEY_ERR_MAX)) if valid[it] and inl > 0 else 0
        if key > best:
            records.append(it)
            best = key
    log1mp = math.log(1.0 - probability) if probability < 1.0 else -math.inf
    best_it, break_it = -1, float(iters)
    for it in records:
        if it > break_it:
            break
        best_it = it
        inl = scores[it][0]
        if inl < P:
            fitness = inl / P
            fn = fitness
            for _ in range(ransac_n - 1):
                fn = fn * fitness
            denom = math.log(1.0 - fn)
            cand = math.inf if denom == 0.0 else log1mp / denom
            break_it = cand if cand < iters else float(iters)
        else:
            break_it = 0.0
    return best_it


def test_kernel_selection_equals_sequential_select():
    rng = np.random.default_rng(2)
    lengths = [1, 2, 127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 512, 513, 640, 1000]
    stops = 0
    for case in range(3000):
        iters = int(lengths[case % len(lengths)] if case % 3 else rng.integers(1, 700))
        P = int(rng.choice([10, 50, 200, 5000, 10 ** 6]))
        n = int(rng.integers(3, 17))
        prob = float(rng.choice([1.0, 0.99, 1e-6]))
        hi = int(rng.choice([3, 10, P]))
        inl = rng.integers(0, min(hi, P) + 1, size=iters)
        inl[rng.random(iters) < 0.02] = P
        err = rng.integers(0, int(rng.choice([3, 1000, 1 << 38])), size=iters)
        valid = rng.random(iters) > 0.1
        scores = [(int(i), int(e)) for i, e in zip(inl, err)]
        want = ransac.select(scores, valid, P, n, iters, prob)
        assert kernel_select(scores, valid, P, n, iters, prob) == want, (case, iters, P, n, prob)
        later_better = [it for it in range(want + 1, iters) if valid[it] and
                        (scores[it][0] > scores[want][0] or
                         (scores[it][0] == scores[want][0] > 0 and scores[it][1] < scores[want][1]))]
        stops += bool(want >= 0 and later_better)
    assert stops > 300           # the early stop decided many of them


# ---- the case builders deliver what they claim -------------------------------------------------
@pytest.mark.parametrize("thr", [0.25, 0.2, 0.0137])
def test_band_cloud_reaches_the_band(thr):
    pts, table, meta = rc.band_cloud(thr)
    assert table.min() >= 0 and table.max() < pts.shape[0]
    planes = rc.planes_of(pts, table)
    b = rc.band(pts, planes, thr)
    assert b["ch"] == 20 and table.shape[0] == 40
    assert b["disagree"].sum() >= 50
    per_hyp = b["in_band"].sum(axis=1)
    assert (per_hyp >= 280).sum() >= 30                          # every planted hypothesis
    for c in range(2):                                           # both chunks hold several at once
        assert (b["in_band"][20 * c:20 * (c + 1)].sum(axis=0) >= 3).sum() > 1000
    assert (meta["exact_ties"] > 0) == (thr == 0.25)


def test_all_ambiguous_cloud_overflows_every_queue():
    pts, table, thr = rc.all_ambiguous_cloud()
    P = pts.shape[0]
    assert P % 1024 % 256 != 0                                   # a thread with live and past-the-end items
    planes = rc.planes_of(pts, table)
    b = rc.band(pts, planes, thr)
    assert b["in_band"][0].all()
    q = rc.queue_entries(P, b["in_band"], b["ch"])
    assert q.min() > 8 * rc.QCAP


@pytest.mark.parametrize("target,winner,later,iters,n", [(60, 20, 90, 128, 3), (300, 150, 420, 1000, 4)])
def test_planted_ground_stops_before_a_better_hypothesis(target, winner, later, iters, n):
    pts, table, meta = rc.planted_ground_cloud(target, winner, later, iters, ransac_n=n)
    b = meta["bound"]
    assert abs(b - target) < 1.0 and winner < b < later
    assert abs(b - round(b)) > 1e-9 * b
    _, _, info = ransac.segment_plane(pts, 0.2, n, iters, 0.99, samples=table)
    sc = info["scores"]
    assert info["best_it"] == winner and sc[winner][0] == meta["inliers"]
    assert sc[later][0] > sc[winner][0]
    assert rc.early_stop_bound(sc[winner][0], pts.shape[0], n, iters, 0.99) == b


def test_selection_cloud_winner_and_ties():
    pts, table, meta = rc.selection_cloud(255)
    P64 = pts.astype(np.float64)
    planes = rc.planes_of(pts, table)
    win = ransac.score(P64, planes[255], 0.2)
    for r in meta["tie_rows"]:
        s = ransac.score(P64, planes[r], 0.2)
        assert s[0] == win[0] and s[1] > win[1]
    for r in meta["dup_rows"]:
        assert ransac.score(P64, planes[r], 0.2) == win
    rest = [r for r in range(0, 4096, 97) if r not in meta["tie_rows"] + meta["dup_rows"] + [255]]
    assert max(ransac.score(P64, planes[r], 0.2)[0] for r in rest) < win[0] // 4


def test_saturation_cloud_is_all_sure_inliers():
    pts, table = rc.saturation_cloud()
    planes = rc.planes_of(pts, table[:12])
    b = rc.band(pts, planes, 0.2, ch=16)
    assert b["sure_in"].all()
    P64 = pts.astype(np.float64)
    q = np.rint(np.float64(ransac.err_scale(0.2)) * (pts[3:, 2].astype(np.float64) ** 2))
    assert q.min() > 65_000 and 128 * q.max() <= 2 ** 23          # a full window stays below 2^24
    assert ransac.score(P64, planes[0], 0.2)[0] == pts.shape[0]
    assert pts.shape[0] > 64 * 1024
