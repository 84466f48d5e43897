"""Numpy models of the hash functions and table geometry behind the duplicate, voxel and neighbour-grid tables, the
constructions of colliding inputs that ``test_gpu_hash_tables.py`` feeds the kernels, and CPU-only guards.

The models restate:
  * ``mix64`` (csrc/apc_common.cuh), the splitmix64 finaliser every table hashes with, and its inverse;
  * ``dedup_hash`` (csrc/frontend.cu): the 64-bit hash of the x/y/z bit patterns; the duplicate table's home slot is
    its low bits, the slot's fingerprint its high 32 bits;
  * the voxel key and slot (csrc/voxel.cu): 21-bit indices with a 2^20 bias, 2x2 (x, y) blocks of four slots whose
    block hash picks a block, probing block by block;
  * ``grid_key`` (csrc/apc_grid.cuh) and the grid's home slot;
  * the capacities: ``hash_cap`` (csrc/ctx.cu) and the single-level and 12-level grids (csrc/neighbors.cu);
  * the float32 cell sizes and reciprocals of the single-level grids.

The GPU tests never assert against these models: every assertion there compares with the CPU oracle.  The models only
choose which inputs are adversarial (same 64-bit hash, same voxel block, same grid home slot).  Were a model to drift
from the kernels, those tests would still pass but lose their aim; the source-pinning test below fails instead.
"""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "autodriver_pointcloud_preprocessor_b200", "csrc")

U64 = np.uint64
MIX_SHIFTS = (30, 27, 31)
MIX_MULS = (0xBF58476D1CE4E5B9, 0x94D049BB133111EB)
DEDUP_KZ_ADD = 0x9E3779B97F4A7C15
SLOTS_PER_POINT = 4
VOX_BIAS = 1 << 20              # voxel index bias; indices must lie in [-2^20, 2^20)
VOX_SHIFTS = (42, 21)
VOX_POS_LIMIT = 65536.0
GRID_BIAS = 262144
GRID_SHIFTS = (57, 38, 19)
GRID_INDEX_LIMIT = 262143.0     # grid cell indices must lie in [-262143, 262143)
KNN_LEVELS = 12
RADIUS_CELL_MULT = 2.0          # radius outlier grid: cells of 2 r (1 + 2^-10)
RADIUS_CELL_SLACK = 1.0009765625
NB_CELL_SLACK = 1.00390625      # normals-radius / DBSCAN / ICP grid: cells of r (1 + 2^-8)


def _unxorshift(y, s):
    x = y.copy()
    for _ in range(64 // s + 1):
        x = y ^ (x >> U64(s))
    return x


def mix64(z):
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> U64(MIX_SHIFTS[0]))) * U64(MIX_MULS[0])
        z = (z ^ (z >> U64(MIX_SHIFTS[1]))) * U64(MIX_MULS[1])
    return z ^ (z >> U64(MIX_SHIFTS[2]))


def mix64_inv(h):
    z = np.atleast_1d(np.asarray(h, dtype=np.uint64))
    with np.errstate(over="ignore"):
        z = _unxorshift(z, MIX_SHIFTS[2]) * U64(pow(MIX_MULS[1], -1, 1 << 64))
        z = _unxorshift(z, MIX_SHIFTS[1]) * U64(pow(MIX_MULS[0], -1, 1 << 64))
    return _unxorshift(z, MIX_SHIFTS[0])


def dedup_hash(pos):
    """64-bit hash of every row's x/y/z float32 bit patterns (frontend.cu dedup_hash)."""
    k = np.ascontiguousarray(pos, dtype=np.float32).reshape(-1, 3).view(np.uint32).astype(np.uint64)
    with np.errstate(over="ignore"):
        return mix64((k[:, 0] | (k[:, 1] << U64(32))) ^ mix64(k[:, 2] + U64(DEDUP_KZ_ADD)))


def _finite_normal(bits):
    e = (bits >> np.uint32(23)) & np.uint32(0xff)
    return (e != 0) & (e != 0xff)


def same_hash_points(h, kz):
    """Distinct points whose 64-bit dedup hash is exactly ``h``: z takes the bit patterns ``kz``, x and y follow from
    inverting the hash.  Rows whose x or y would be zero, subnormal, infinite or NaN are dropped."""
    kz = np.asarray(kz, dtype=np.uint32)
    with np.errstate(over="ignore"):
        a = mix64_inv(np.uint64(h)) ^ mix64(kz.astype(np.uint64) + U64(DEDUP_KZ_ADD))
    kx = (a & U64(0xffffffff)).astype(np.uint32)
    ky = (a >> U64(32)).astype(np.uint32)
    ok = _finite_normal(kx) & _finite_normal(ky) & _finite_normal(kz)
    return np.stack([kx[ok], ky[ok], kz[ok]], 1).view(np.float32)


def next_pow2(v):
    p = 1024
    while p < v:
        p <<= 1
    return p


def hash_cap(max_points):
    """Capacity of the duplicate and voxel tables (ctx.cu)."""
    lf = os.environ.get("APC_HASH_SLOTS_PER_POINT")
    spp = int(lf) if lf and lf.lstrip("-").isdigit() and int(lf) >= 2 else SLOTS_PER_POINT
    return next_pow2(spp * max_points)


def grid_cap(max_points, levels):
    """Capacity of the single-level (levels = 1) and KNN (levels = 12) neighbour grids (neighbors.cu)."""
    cap = next_pow2(levels * max_points * 4 // 3 + 1024)
    return max(cap, hash_cap(max_points)) if levels == 1 else cap


# ---- voxel table ------------------------------------------------------------------------------------------------
def voxel_index(pos, vs):
    return np.floor(np.asarray(pos, np.float32) / np.float32(vs)).astype(np.int64)


def voxel_key(q):
    u = (np.asarray(q, np.int64) + VOX_BIAS).astype(np.uint64).reshape(-1, 3)
    return (u[:, 0] << U64(VOX_SHIFTS[0])) | (u[:, 1] << U64(VOX_SHIFTS[1])) | u[:, 2]


def voxel_block(key):
    return key & ~U64((1 << VOX_SHIFTS[0]) | (1 << VOX_SHIFTS[1]))


def voxel_sub(key):
    return ((key >> U64(VOX_SHIFTS[0])) & U64(1)) | (((key >> U64(VOX_SHIFTS[1])) & U64(1)) << U64(1))


def voxel_home_block(key, cap):
    """Block (slot // 4) the key's first probe lands in: the 32-bit block hash shifted by 2, masked."""
    h32 = mix64(voxel_block(key)).astype(np.uint32)
    return ((h32 << np.uint32(2)) & np.uint32(cap - 1)) >> np.uint32(2)


def voxel_slot(key, cap):
    return (voxel_home_block(key, cap) << np.uint32(2)) | voxel_sub(key).astype(np.uint32)


# ---- neighbour grids --------------------------------------------------------------------------------------------
def grid_key(level, idx):
    u = (np.asarray(idx, np.int64) + GRID_BIAS).astype(np.uint64).reshape(-1, 3)
    return ((U64(level) << U64(GRID_SHIFTS[0])) | (u[:, 0] << U64(GRID_SHIFTS[1])) | (u[:, 1] << U64(GRID_SHIFTS[2]))
            | u[:, 2])


def grid_home(key, cap):
    return mix64(key).astype(np.uint32) & np.uint32(cap - 1)


def radius_cell(r):
    """Cell size and host-rounded reciprocal of radius_outliers' grid (float32, left to right)."""
    c = np.float32(np.float32(r) * np.float32(RADIUS_CELL_MULT)) * np.float32(RADIUS_CELL_SLACK)
    return np.float32(c), np.float32(np.float32(1.0) / np.float32(c))


def nb_cell(r):
    """Cell size and reciprocal of the grid of estimate_normals_radius, cluster_dbscan and icp."""
    c = np.float32(np.float32(r) * np.float32(NB_CELL_SLACK))
    return c, np.float32(np.float32(1.0) / c)


def cell_recip(pos, inv):
    return np.floor(np.asarray(pos, np.float32) * np.float32(inv)).astype(np.int64)


def cell_div(pos, c):
    return np.floor(np.asarray(pos, np.float32) / np.float32(c)).astype(np.int64)


# ---- fixed-point sums that round on the way to float64 ------------------------------------------------------------
def rounding_sum_values(rng, n, big_lo, big_hi, big_ulp, small, frac_bits):
    """``n`` positive float32 values whose fixed-point sum S = sum(rint(v * 2^frac_bits)) lies above 2^53 and makes
    int64 -> float64 conversion decide the float32 mean.

    ``n - 1`` values lie in [big_lo, big_hi) on a grid of ``big_ulp`` (their fixed-point images are multiples of
    2^16), one equals ``small`` (rint(small * 2^frac_bits) = -1 mod 2^16).  With n = 2^14 the float64 mean is
    float64(S) * 2^-(14 + frac_bits) exactly; S + 1 is made an odd multiple 2^29 (2j + 1) with j odd: rounded to
    nearest, float64(S) is the midpoint between two float32 neighbours and the tie goes to the even one, while a
    conversion toward zero lands below the midpoint and rounds to the odd one."""
    scale = 1 << frac_bits
    q_small = int(np.rint(np.float64(np.float32(small)) * scale))
    assert (q_small + 1) % (1 << 16) == 0
    units = 1 << 16
    m = rng.integers(int(big_lo / big_ulp), int(big_hi / big_ulp), size=n - 1).astype(np.int64)
    assert int(m[0] * big_ulp * scale) % units == 0
    step = int(round(big_ulp * scale / units))                 # fixed-point step of one big value's grid, in 2^16
    assert step == 1
    want = ((3 << 29) - 1 - q_small) % (1 << 31) // units
    delta = (want - int(m.sum())) % (1 << 15)
    m += delta // (n - 1)
    m[:delta % (n - 1)] += 1
    vals = np.concatenate([(m * big_ulp).astype(np.float32), [np.float32(small)]])
    assert vals[:-1].max() < big_hi + 4 * big_ulp
    return vals


def ll2double(s, mode):
    """int -> float64 rounded to nearest even ('rn') or toward zero ('rz')."""
    if mode == "rn":
        return float(s)
    a = abs(s)
    drop = max(a.bit_length() - 53, 0)
    a = (a >> drop) << drop
    return float(a if s >= 0 else -a)


def fixed_mean_model(vals, frac_bits, mode):
    q = [int(v) for v in np.rint(np.asarray(vals, np.float32).astype(np.float64) * (1 << frac_bits))]
    s = sum(q)
    return np.float32(ll2double(s, mode) / len(q) * (1.0 / (1 << frac_bits))), s


# ==== CPU-only guards ============================================================================================
def test_mix64_inverse_round_trips():
    z = np.random.default_rng(0).integers(0, 2**64 - 1, size=100_000, dtype=np.uint64, endpoint=True)
    assert np.array_equal(mix64_inv(mix64(z)), z)
    assert np.array_equal(mix64(mix64_inv(z)), z)
    assert int(mix64(np.uint64(1))) == 0x5692161D100B05E5       # splitmix64's finaliser of 1


def test_same_hash_points_collide():
    rng = np.random.default_rng(1)
    h = (int(rng.integers(0, 2**32)) << 32) | 0xffffffff
    kz = np.float32(rng.uniform(-3.0, 3.0, 200)).view(np.uint32)
    pts = same_hash_points(h, kz)
    assert pts.shape[0] >= 190 and np.isfinite(pts).all()
    assert np.unique(pts.view(np.uint32), axis=0).shape[0] == pts.shape[0]     # distinct points
    hh = dedup_hash(pts)
    assert np.all(hh == U64(h))                                                 # identical 64-bit hashes
    for cap in (1 << 17, 1 << 20, 1 << 22):                                     # the last slot of any table
        assert np.all((hh & U64(cap - 1)) == U64(cap - 1))


def test_voxel_block_model():
    cap = hash_cap(32768)
    rng = np.random.default_rng(2)
    q = rng.integers(-1000, 1000, size=(50_000, 3))
    key = voxel_key(q)
    s = voxel_slot(key, cap)
    assert np.all(s < cap)
    # the four voxels of a 2x2 (x, y) block share a block hash and take distinct places in it
    q0 = np.stack([q[:, 0] & ~1, q[:, 1] & ~1, q[:, 2]], 1)
    for dx, dy in ((0, 0), (1, 0), (0, 1), (1, 1)):
        k = voxel_key(q0 + np.array([dx, dy, 0]))
        assert np.array_equal(voxel_home_block(k, cap), voxel_home_block(voxel_key(q0), cap))
        assert np.all(voxel_sub(k) == U64(dx | (dy << 1)))


def test_rounding_sum_construction_separates_rn_from_rz():
    rng = np.random.default_rng(3)
    for small, lo, hi, ulp, fb in ((1.0 - 2.0**-24, 65024.0, 65500.0, 2.0**-8, 24),
                                   (1.0 - 2.0**-20, 2.0**20 - 1024.0, 2.0**20 - 64.0, 2.0**-4, 20)):
        v = rounding_sum_values(rng, 1 << 14, lo, hi, ulp, small, fb)
        for sign in (1.0, -1.0):
            rn, s = fixed_mean_model(sign * v, fb, "rn")
            rz, _ = fixed_mean_model(sign * v, fb, "rz")
            assert abs(s) > 2**53 and rn != rz


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _body(text, signature):
    i = text.index(signature)
    return text[i:text.index("\n}", i)]


def test_sources_match_the_models():
    """The models' constants are the kernels' constants: a changed hash, key layout or capacity fails here."""
    mix = _body(_src("apc_common.cuh"), "uint64_t mix64(uint64_t z)")
    steps = re.findall(r"z = \(z \^ \(z >> (\d+)\)\) \* (0x[0-9A-Fa-f]+)ull;", mix)
    assert [(int(s), int(m, 16)) for s, m in steps] == list(zip(MIX_SHIFTS[:2], MIX_MULS))
    assert [int(s) for s in re.findall(r"return z \^ \(z >> (\d+)\);", mix)] == [MIX_SHIFTS[2]]

    fe = _src("frontend.cu")
    dh = _body(fe, "uint64_t dedup_hash(float x, float y, float z)")
    m = re.search(r"mix64\(\(\(uint64_t\)kx \| \(\(uint64_t\)ky << 32\)\) \^ mix64\(\(uint64_t\)kz \+ (0x[0-9A-Fa-f]+)ull\)\)", dh)
    assert m and int(m.group(1), 16) == DEDUP_KZ_ADD
    assert "slot[j] = (uint32_t)hash[j] & slot_mask;" in fe               # home slot: the hash's low bits
    assert "((unsigned long long)(h >> 32) << 32) | g" in fe              # fingerprint: its high 32 bits

    vx = _src("voxel.cu")
    vk = _body(vx, "bool voxel_key(float4 p, float vs, uint64_t& key)")
    assert float(re.search(r"const float lim = ([0-9.]+)f;", vk).group(1)) == VOX_POS_LIMIT
    assert float(re.search(r"const float h = ([0-9.]+)f;", vk).group(1)) == VOX_BIAS
    assert set(int(b) for b in re.findall(r"\(int64_t\)q[xyz] \+ (\d+)\)", vk)) == {VOX_BIAS}
    sh = re.search(r"key = \(ux << (\d+)\) \| \(uy << (\d+)\) \| uz;", vk)
    assert (int(sh.group(1)), int(sh.group(2))) == VOX_SHIFTS
    assert "key & ~((1ull << 42) | (1ull << 21))" in vx
    assert "slot = ((((uint32_t)mix64(block)) << 2) & cap_mask) | sub;" in vx
    assert "slot = (slot + 4) & cap_mask;" in vx                         # probing moves block by block

    gk = _body(_src("apc_grid.cuh"), "uint64_t grid_key(uint32_t level, int32_t ix, int32_t iy, int32_t iz)")
    lv = int(re.search(r"\(uint64_t\)level << (\d+)", gk).group(1))
    axes = re.findall(r"\(uint64_t\)\(uint32_t\)\(i[xyz] \+ (\d+)\)(?: << (\d+))?", gk)
    assert (lv,) + tuple(int(s) for _, s in axes[:2]) == GRID_SHIFTS and axes[2][1] == ""
    assert {int(b) for b, _ in axes} == {GRID_BIAS}
    assert "const float h = 262143.0f;" in _src("apc_grid.cuh")
    assert "(uint32_t)mix64(key) & g.cap_mask" in _src("neighbors.cu")

    ctx = _src("ctx.cu")
    m = re.search(r"hash_cap = next_pow2\(\(lf && atoi\(lf\) >= 2 \? \(uint64_t\)atoi\(lf\) : (\d+)ull\) \* M\);", ctx)
    assert m and int(m.group(1)) == SLOTS_PER_POINT
    assert "uint64_t p = 1024;" in _body(ctx, "static uint32_t next_pow2(uint64_t v)")

    nb = _src("neighbors.cu")
    assert "uint64_t want = (uint64_t)levels * M * 4 / 3 + 1024;" in nb
    assert "if (which == 0 && cap < ctx->hash_cap) cap = ctx->hash_cap;" in nb
    assert f"#define KNN_LEVELS {KNN_LEVELS}" in nb
    m = re.search(r"static float radius_cell\(float r32\) \{ return r32 \* ([0-9.]+)f \* ([0-9.]+)f; \}", nb)
    assert float(m.group(1)) == RADIUS_CELL_MULT and m.group(2) == repr(RADIUS_CELL_SLACK)
    assert nb.count(f"r32 * {NB_CELL_SLACK!r}f") >= 3                   # normals radius, DBSCAN, ICP
