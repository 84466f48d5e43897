// Radius and statistical outlier removal with neighbour queries served from a voxel hash.
//
// Replaces Open3D remove_statistical_outliers (pp.py:514-519; SURVEY.md B8) and
// remove_radius_outliers (TODO at pp.py:37; SURVEY.md B9).  Arithmetic contract
// (oracle/outliers.py): d2 = (dx*dx + dy*dy) + dz*dz in float32 unfused; radius test
// d2 <= float32(r)^2 with the query point included; KNN keeps the k smallest d2 (query
// included), averages sqrtf in ascending order sequentially; mu/sigma in float64 with the
// adjacent-pairwise tree reduction.
//
// Structure: a multi-level cell grid in one open-addressing hash table.  Level l has cell
// size c0 * 2^l; the key packs (level:4 | ix:19 | iy:19 | iz:19).  Points are counting-
// sorted per level into cell-contiguous arrays, so a query reads its 27 neighbour cells as
// 27 short contiguous runs.  Queries run in level-0 sorted order so the lanes of a warp
// share cells.  Radius search uses one level with c0 = 2r * (1 + 2^-10); KNN climbs levels
// until the k-th distance is covered by the 27-cell block, and the rare points that never
// are (fewer than k points in range of the coarsest level) fall to an exact brute-force
// kernel.  The table is cleaned by the points that own rank 0 of their cell, not by memset.
#include <cmath>
#include <cstring>
#include "apc_scan.cuh"
#include "apc_grid.cuh"
APC_TRACE_EXPORT(neighbors)

#define KNN_LEVELS 12
#define KNN_KMAX 64           // k_knn_query / k_knn_stragglers; above it the *_wide kernels, up to APC_MAX_NEIGHBORS
#define APC_STRINGIFY2(x) #x
#define APC_STRINGIFY(x) APC_STRINGIFY2(x)

// counters[] slots used by this file (zeroed by k_begin)
#define CTR_CURSOR 0        // [0..KNN_LEVELS) per-level scatter cursors of the KNN grid
#define CTR_STRAGGLERS 12
#define CTR_CURSOR_RADIUS 13  // scatter cursor of the single-level radius / normals grid
#define CTR_BBOX 14         // 6 ordered-int floats: min xyz, max xyz
#define CTR_CURSOR_NORMALS 22  // scatter cursor of the normals stage's grid build (the radius stage of the same
                               // pipeline run has already advanced CTR_CURSOR_RADIUS)

// whole slot in one read-only 128-bit load (the table is not written while a query kernel runs)
__device__ __forceinline__ uint4 grid_load(const GridDev& g, uint32_t s) {
  return __ldg(reinterpret_cast<const uint4*>(&g.slots[s]));
}
__device__ __forceinline__ uint32_t grid_home(const GridDev& g, uint64_t key) { return (uint32_t)mix64(key) & g.cap_mask; }
// Finishes a lookup whose first probe (slot s, contents v) is already in registers: run of the
// cell in [start, start + fill) or false when the cell is empty.
__device__ __forceinline__ bool grid_resolve(const GridDev& g, uint64_t key, uint32_t s, uint4 v, uint32_t& start,
                                             uint32_t& fill) {
  for (uint32_t probe = 0; probe <= g.cap_mask; ++probe) {
    const uint64_t k = (uint64_t)v.x | ((uint64_t)v.y << 32);
    if (k == key) { fill = v.z; start = v.w; return true; }
    if (k == GRID_EMPTY) return false;
    s = (s + 1) & g.cap_mask;
    v = grid_load(g, s);
  }
  return false;
}
__device__ __forceinline__ bool grid_lookup(const GridDev& g, uint64_t key, uint32_t& start, uint32_t& fill) {
  const uint32_t s = grid_home(g, key);
  return grid_resolve(g, key, s, grid_load(g, s), start, fill);
}

// ---- build ------------------------------------------------------------------------------------
// Warp-aggregated: the lanes of a warp that fall into the same cell (neighbouring points do, and at
// the coarse KNN levels nearly all of them) elect a leader that claims / finds the slot and bumps
// the cell's population once for the whole group; the others take consecutive ranks after it.
// At the coarsest levels this replaces hundreds of thousands of atomics on one address by 1/32 of them
// (k_grid_insert over 12 levels of a 586 k-point cloud: 516 -> see profiles/config_times.py).
__global__ void __launch_bounds__(256)
k_grid_insert(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, GridDev g, ApcCtrl* ctrl) {
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t level = blockIdx.y;
  const float c = grid_cell_size(g, level);
  const uint32_t lane = lane_id();
  APC_STAMP(1, 0);
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    int32_t ix = 0, iy = 0, iz = 0;
    bool ok = false;
    if (i < n) {
      p = pts[i];
      ok = grid_coord_g(g, c, p.x, p.y, p.z, ix, iy, iz);
      if (!ok) atomicOr(&ctrl->err, APC_DEVERR_KEY_RANGE);
    }
    const uint32_t vm = __ballot_sync(0xffffffffu, ok);
    uint32_t slot = GRID_NOSLOT, rank = 0;
    if (ok) {
      const uint64_t key = grid_key(level, ix, iy, iz);
      const uint32_t peers = __match_any_sync(vm, key);
      const uint32_t leader = __ffs(peers) - 1u;
      uint32_t first_rank = 0;
      if (lane == leader) {
        uint32_t s = (uint32_t)mix64(key) & g.cap_mask;
        for (uint32_t probe = 0; probe <= g.cap_mask; ++probe) {
          const unsigned long long old = atomicCAS(&g.slots[s].key, GRID_EMPTY, (unsigned long long)key);
          if (old == GRID_EMPTY || old == key) { slot = s; break; }
          s = (s + 1) & g.cap_mask;
        }
        if (slot == GRID_NOSLOT) atomicOr(&ctrl->err, APC_DEVERR_CAPACITY);
        else first_rank = atomicAdd(&g.slots[slot].fill, (uint32_t)__popc(peers));
      }
      slot = __shfl_sync(peers, slot, leader);
      first_rank = __shfl_sync(peers, first_rank, leader);
      rank = first_rank + __popc(peers & ((1u << lane) - 1u));
    }
    if (i < n) {
      g.slot[(size_t)level * n_max + i] = slot;
      g.rank[(size_t)level * n_max + i] = rank;
    }
  }
  APC_STAMP(1, 1);
}

// rank-0 points reserve a contiguous run for their cell (warp-aggregated cursor bump)
__global__ void __launch_bounds__(256)
k_grid_assign(uint32_t n_max, const uint32_t* n_dev, GridDev g, ApcCtrl* ctrl) {
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t level = blockIdx.y;
  const uint32_t lane = lane_id();
  const uint32_t rounds = (n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);
  APC_STAMP(2, 0);
  for (uint32_t r = 0; r < rounds; ++r) {
    const uint32_t i = (r * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x;
    uint32_t slot = GRID_NOSLOT, cnt = 0;
    if (i < n) {
      slot = g.slot[(size_t)level * n_max + i];
      if (slot != GRID_NOSLOT && g.rank[(size_t)level * n_max + i] == 0) cnt = g.slots[slot].fill;
    }
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t base = 0;
    if (lane == 31 && total) {
      base = atomicAdd(&ctrl->counters[g.cursor_base + level], total);
      if (base + total > n_max) atomicOr(&ctrl->err, APC_DEVERR_CAPACITY);   // cursor not reset / corrupt table: never scatter past the array
    }
    base = __shfl_sync(0xffffffffu, base, 31);
    if (cnt) g.slots[slot].start = base + incl - cnt;
  }
  APC_STAMP(2, 1);
}

// The same over the LIST of occupied cells a producer kernel recorded while inserting (GridDev::cells): with
// cells of 2r a voxelised scan occupies ~11 k cells, so this walks 18x fewer entries than the per-point pass.
__global__ void __launch_bounds__(256) k_grid_assign_cells(GridDev g, ApcCtrl* ctrl, uint32_t n_max) {
  pdl_enter();
  const uint32_t nc = min(ctrl->counters[GRID_CTR_CELLS], n_max);
  const uint32_t lane = lane_id();
  for (uint32_t base = blockIdx.x * blockDim.x; base < nc; base += gridDim.x * blockDim.x) {
    const uint32_t i = base + threadIdx.x;
    uint32_t slot = GRID_NOSLOT, cnt = 0;
    if (i < nc) {
      slot = g.cells[i];
      cnt = g.slots[slot].fill;
    }
    uint32_t incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t at = 0;
    if (lane == 31 && total) {
      at = atomicAdd(&ctrl->counters[g.cursor_base], total);
      if (at + total > n_max) atomicOr(&ctrl->err, APC_DEVERR_CAPACITY);
    }
    at = __shfl_sync(0xffffffffu, at, 31);
    if (cnt) g.slots[slot].start = at + incl - cnt;
  }
}

__global__ void __launch_bounds__(256)
k_grid_scatter(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, GridDev g) {
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t level = blockIdx.y;
  APC_STAMP(3, 0);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t slot = g.slot[(size_t)level * n_max + i];
    if (slot == GRID_NOSLOT) continue;
    const float4 p = pts[i];
    const uint32_t pos = g.slots[slot].start + g.rank[(size_t)level * n_max + i];
    if (pos < n_max) g.sorted[(size_t)level * n_max + pos] = make_float4(p.x, p.y, p.z, __uint_as_float(i));
  }
  APC_STAMP(3, 1);
}

__global__ void __launch_bounds__(256) k_grid_clean(uint32_t n_max, const uint32_t* n_dev, GridDev g) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t level = blockIdx.y;
  APC_STAMP(4, 0);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t slot = g.slot[(size_t)level * n_max + i];
    if (slot != GRID_NOSLOT && g.rank[(size_t)level * n_max + i] == 0) {
      g.slots[slot].key = GRID_EMPTY;
      g.slots[slot].fill = 0u;
    }
  }
  APC_STAMP(4, 1);
}

__global__ void k_grid_reset(GridSlot* slots, uint32_t cap) {
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += gridDim.x * blockDim.x) {
    slots[s].key = GRID_EMPTY;
    slots[s].fill = 0u;
    slots[s].start = 0u;
  }
}

__device__ __forceinline__ float d2_f32(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// 27 neighbour cells as dx+1 + 3*(dy+1) + 9*(dz+1), ordered centre, 6 faces, 12 edges, 8 corners
__constant__ int8_t c_cell_order[27] = {13, 4, 10, 12, 14, 16, 22, 1, 3, 5, 7, 9, 11, 15, 17, 19, 21, 23, 25,
                                         0, 2, 6, 8, 18, 20, 24, 26};

// Number of valid records at the front of the level-0 cell-sorted array: the scatter cursor, i.e. the
// points that were actually inserted.  Points that failed grid_coord (non-finite or beyond the key
// range; APC_ERR_KEY_RANGE is raised for them) are never scattered, so the tail of `sorted` beyond
// the cursor holds stale records of an earlier frame whose `orig` may exceed this frame's size: the
// query kernels must not walk it.
__device__ __forceinline__ uint32_t grid_sorted_count(const GridDev& g, const ApcCtrl* ctrl, uint32_t n) {
  return min(n, ctrl->counters[g.cursor_base]);
}

// ---- the warp's 27-cell walk ----------------------------------------------------------------------
// The 27 cells around cell (ix, iy, iz) of `level` as one flat candidate list, for a warp that walks it 32 records
// at a time: lane l < 27 resolves cell l and keeps its run's start in the level's cell-sorted array (cs) and the
// flat index of the run's first record (ps); returns the list's length (all lanes).
__device__ __forceinline__ uint32_t flat27_runs(const GridDev& g, uint32_t level, int32_t ix, int32_t iy, int32_t iz,
                                                uint32_t lane, uint32_t& cs, uint32_t& ps) {
  uint32_t s0 = 0, cf = 0;
  if (lane < 27) {
    const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
    uint32_t b, f;
    if (grid_lookup(g, grid_key(level, ix + dx, iy + dy, iz + dz), b, f)) { s0 = b; cf = f; }
  }
  uint32_t incl = cf;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= (uint32_t)o) incl += v;
  }
  cs = s0;
  ps = incl - cf;
  return __shfl_sync(0xffffffffu, incl, 31);
}
// The same around the level-0 cell of a query taken from the grid (its cell was keyed at insert time).
__device__ __forceinline__ uint32_t flat27_runs(const GridDev& g, float c, float4 q, uint32_t lane, uint32_t& cs, uint32_t& ps) {
  int32_t ix, iy, iz;
  grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
  return flat27_runs(g, 0, ix, iy, iz, lane, cs, ps);
}
// Position in the level's cell-sorted array of record `flat` of that list (called by all lanes of the warp).
__device__ __forceinline__ uint32_t flat27_at(uint32_t cs, uint32_t ps, uint32_t flat) {
  uint32_t run = 0;                                  // largest cell with ps <= flat
#pragma unroll
  for (int step = 16; step > 0; step >>= 1) {
    const uint32_t mid = run + step;
    const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
    if (mid < 27u && v <= flat) run = mid;
  }
  const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
  return rs + (flat - rp);
}
// KNN coverage bound, squared: every point closer to q than `safe` lies inside the 27-cell block around q's cell
// (ix, iy, iz) of edge c.  `safe` is the cell edge plus q's distance to the nearest face of its own cell (1859 against
// 1961 us for the cell edge alone on the C4 scan, profiles/r2x_knn_ab.json), less 0.1 % for the rounding of the
// cell index.
__device__ __forceinline__ float knn_safe2(float4 q, float c, int32_t ix, int32_t iy, int32_t iz) {
  const float fx = fminf(__fsub_rn(q.x, __fmul_rn((float)ix, c)), __fsub_rn(__fmul_rn((float)(ix + 1), c), q.x));
  const float fy = fminf(__fsub_rn(q.y, __fmul_rn((float)iy, c)), __fsub_rn(__fmul_rn((float)(iy + 1), c), q.y));
  const float fz = fminf(__fsub_rn(q.z, __fmul_rn((float)iz, c)), __fsub_rn(__fmul_rn((float)(iz + 1), c), q.z));
  const float safe = __fmul_rn(__fadd_rn(c, fmaxf(0.0f, fminf(fx, fminf(fy, fz)))), 0.999f);
  return __fmul_rn(safe, safe);
}

// ---- radius query -----------------------------------------------------------------------------
// cnt + the neighbours of q within r2 in the run [b, b + f) of the cell-sorted array, stopping at nb_points
// unless the exact count is wanted.
__device__ __forceinline__ uint32_t radius_scan_run(const GridDev& g, uint32_t b, uint32_t f, float4 q, float r2,
                                                    uint32_t nb_points, int need_counts, uint32_t cnt) {
  const uint32_t e = b + f;
  // four points per round: their loads are independent, the exit test runs once per round
  for (uint32_t t = b; t < e && (need_counts || cnt < nb_points); t += 4) {
    float4 p[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) p[u] = g.sorted[min(t + u, e - 1)];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      cnt += (t + u < e && d2_f32(q.x, q.y, q.z, p[u].x, p[u].y, p[u].z) <= r2) ? 1u : 0u;
  }
  return cnt;
}

// Neighbours of q within r2 in the whole 27-cell block, stopping at nb_points unless the exact count is wanted.
__device__ __forceinline__ uint32_t radius_count(const GridDev& g, float c, float4 q, float r2, uint32_t nb_points,
                                                 int need_counts) {
  int32_t ix, iy, iz;
  grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
  uint32_t cnt = 0;
  // own cell first, then faces, edges, corners: when only the keep/drop decision is wanted
  // most points reach nb_points inside their own cell and stop there.  The first probe of the
  // NEXT cell is in flight while the current cell's points are scanned.
  uint64_t key = grid_key(0, ix, iy, iz);
  uint32_t home = grid_home(g, key);
  uint4 first = grid_load(g, home);
  for (int c27 = 0; c27 < 27 && (need_counts || cnt < nb_points); ++c27) {
    const uint64_t key_now = key;
    const uint32_t home_now = home;
    const uint4 first_now = first;
    if (c27 + 1 < 27) {
      const int code = c_cell_order[c27 + 1];
      key = grid_key(0, ix + code % 3 - 1, iy + (code / 3) % 3 - 1, iz + code / 9 - 1);
      home = grid_home(g, key);
      first = grid_load(g, home);
    }
    uint32_t b, f;
    if (!grid_resolve(g, key_now, home_now, first_now, b, f)) continue;
    cnt = radius_scan_run(g, b, f, q, r2, nb_points, need_counts, cnt);
  }
  return cnt;
}

// ---- radius query over cells of 2r: own cell, then only the neighbours the r-ball can reach ------
// With a cell edge of 2r (+ slack) the ball around q reaches, along every axis, at most ONE of the two
// neighbouring cells (the one behind the nearer face), so 1 + 7 cells cover it instead of 27, and a
// neighbour (a face, edge or corner cell) is visited only if the ball reaches its box: sum over the
// offset axes of gap^2 <= r^2, gap = distance from q to that face.  On a voxelised 128-beam scan the
// own cell alone settles 95 % of the keep / drop decisions (cells of r: 75 %), and the others probe
// 3 to 7 cells, not 26 (profiles/r2p_radius_ab.json).  The set of points tested against d2 <= r2 is a
// superset of the ball either way, so counts and decisions are bit-identical to the 27-cell walk.
// Slack: the cell index is floor(fl(x * fl(1/c))) (grid_coord_g), two roundings of 2^-24 each, so a point
// of the cell below has x < ix*c*(1 + 2^-23) and one of the cell above x >= (ix+1)*c*(1 - 2^-23); the
// products, differences and d2 below each carry a relative rounding error of 2^-24.  gap is therefore shortened by 1e-6 * (|q| + c) + 1e-5 * r (8x the worst
// case); if that ever leaves BOTH faces of an axis within reach (coordinates of tens of kilometres) the
// query falls back to the 27-cell walk.
//
// `self` = position of q itself in the cell-sorted array (q = g.sorted[self]).  The own cell is scanned
// OUTWARDS from that position, two records on either side per round: arrival order inside a cell follows
// the order of the input (LiDAR firing order), so the records next to q are its neighbours along the scan
// line and nb_points within r are usually found in the first round or two - scanning the cell from its
// start examined 14 records per query on the 128-beam scan, this examines 5 to 8.
__device__ __forceinline__ uint32_t radius_count_oct(const GridDev& g, float c, float4 q, uint32_t self, float r, float r2,
                                                     uint32_t nb_points, int need_counts) {
  int32_t ix, iy, iz;
  grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
  uint32_t cnt = 0, b, f;
  if (grid_lookup(g, grid_key(0, ix, iy, iz), b, f)) {
    if (need_counts || self < b || self >= b + f) {
      cnt = radius_scan_run(g, b, f, q, r2, nb_points, need_counts, 0u);
    } else {
      const uint32_t e = b + f;
      cnt = 1u;                                   // q itself
      uint32_t up = self + 1, down = self;        // next record above, one past the next record below
      while (cnt < nb_points && (up < e || down > b)) {
        float4 p[4];
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          ok[u] = up + u < e;
          p[u] = g.sorted[ok[u] ? up + u : self];
          ok[2 + u] = down >= b + 1 + u;
          p[2 + u] = g.sorted[ok[2 + u] ? down - 1 - u : self];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) cnt += (ok[u] && d2_f32(q.x, q.y, q.z, p[u].x, p[u].y, p[u].z) <= r2) ? 1u : 0u;
        up = min(up + 2, e);
        down = down >= b + 2 ? down - 2 : b;
      }
    }
  }
  if (!need_counts && cnt >= nb_points) return cnt;
  const float reach = r * 1.00001f;
  const float qa[3] = {q.x, q.y, q.z};
  const int32_t ia[3] = {ix, iy, iz};
  int32_t dir[3];
  float gap2[3];
  bool both = false;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float lo = __fmul_rn((float)ia[a], c), hi = __fmul_rn((float)(ia[a] + 1), c);
    const float slack = 1e-6f * (fabsf(qa[a]) + c) + 1e-5f * r;
    const float gl = fmaxf(0.0f, __fsub_rn(__fsub_rn(qa[a], lo), slack)), gh = fmaxf(0.0f, __fsub_rn(__fsub_rn(hi, qa[a]), slack));
    dir[a] = gl <= gh ? -1 : 1;
    const float gmin = fminf(gl, gh);
    gap2[a] = __fmul_rn(gmin, gmin);
    both |= fmaxf(gl, gh) <= reach;
  }
  if (both) return radius_count(g, c, q, r2, nb_points, need_counts);
  const float reach2 = __fmul_rn(reach, reach);
  // faces, edges, corner: the nearer a box, the likelier it holds the missing neighbours.  One cell at a
  // time: probing the cells of a round together (7 table round trips -> 2) was slower, alone and with all
  // lanes busy (23.5 vs 22.4 us, 65.1 vs 63.8 us/scan) - most walks end at the first or second face.
#pragma unroll 1
  for (int m = 1; m < 8; ++m) {
    const int mask = (0x7653421 >> (4 * (m - 1))) & 7;     // 1, 2, 4, 3, 5, 6, 7
    if (!need_counts && cnt >= nb_points) break;
    const float s2 = ((mask & 1) ? gap2[0] : 0.0f) + ((mask & 2) ? gap2[1] : 0.0f) + ((mask & 4) ? gap2[2] : 0.0f);
    if (s2 > reach2) continue;
    const uint64_t key = grid_key(0, ix + ((mask & 1) ? dir[0] : 0), iy + ((mask & 2) ? dir[1] : 0), iz + ((mask & 4) ? dir[2] : 0));
    if (grid_lookup(g, key, b, f)) cnt = radius_scan_run(g, b, f, q, r2, nb_points, need_counts, cnt);
  }
  return cnt;
}

__global__ void __launch_bounds__(256)
k_radius_query_oct(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r, float r2, uint32_t nb_points, int need_counts,
                   uint8_t* __restrict__ mask, uint32_t* __restrict__ counts, const ApcCtrl* __restrict__ ctrl) {
  pdl_enter();
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  APC_STAMP(0, 0);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    const uint32_t cnt = radius_count_oct(g, c, q, j, r, r2, nb_points, need_counts);
    mask[orig] = cnt >= nb_points ? 1 : 0;
    if (counts) counts[orig] = cnt;
  }
  APC_STAMP(0, 1);
}

// Cell edge of the radius grid: 2r, + 2^-10 slack so that d2 <= r2 never reaches past the neighbouring cell.
// Against cells of r and the 27-cell walk, cells of 2r and the pruned walk above give +6 % saturated
// throughput (profiles/r2p_radius_ab.json).
static float radius_cell(float r32) { return r32 * 2.0f * 1.0009765625f; }

// The radius query over the built grid: keep / drop decisions into `mask`, and the exact counts into `counts`
// when it is not NULL.  For the decision alone one launch of the per-thread walk measured best:
//  - an own-cell pass that lists the points still short of nb_points, then a pass over that list: the first
//    takes 10.6 us, the second still 23 us, saturated throughput does not move (70.5 vs 70.8 us/scan) and the
//    split costs one more launch of latency (profiles/r2g_knobs.json);
//  - the whole warp serving, one after the other, the lanes its own-cell rounds left short: 24.3 vs 21.9 us
//    alone, 67.7 vs 64.8 us/scan with all lanes busy (profiles/r2p_radius_ab.json);
//  - blocks of 64 or 256 threads instead of 128: no difference (profiles/r2ab_fold_lanes.json).
static int radius_query(apc_ctx* ctx, const GridDev& g, uint32_t n_max, const uint32_t* n_dev, float r,
                        uint32_t nb_points, uint8_t* mask, uint32_t* counts, cudaStream_t s) {
  const uint32_t bq = min(apc_div_up(n_max, 128), (uint32_t)APC_SM_COUNT * 16);
  APC_PROF(ctx, "k_radius_query", s);
  apc_klaunch(ctx, k_radius_query_oct, bq, 128, 0, s, n_max, n_dev, g, r, r * r, nb_points, counts ? 1 : 0, mask, counts,
              ctx->ctrl);
  APC_LAUNCH_CHECK(ctx, "k_radius_query_oct");
  return APC_OK;
}

// ---- KNN query ---------------------------------------------------------------------------------
struct TopK {
  float best[KNN_KMAX];
  uint32_t cnt;
  float worst;   // best[k-1] once full, +inf before: candidates are rejected against a register
  __device__ __forceinline__ void reset() { cnt = 0; worst = __int_as_float(0x7f800000); }
  __device__ __forceinline__ void push(float d2, uint32_t k) {
    uint32_t j;
    if (cnt < k) j = cnt++;
    else if (d2 < worst) j = k - 1;
    else return;
    while (j > 0 && best[j - 1] > d2) { best[j] = best[j - 1]; --j; }
    best[j] = d2;
    if (cnt == k) worst = best[k - 1];
  }
  __device__ __forceinline__ float average(uint32_t k) const {  // sequential float32, ascending
    float s = sqrtf(best[0]);
    for (uint32_t j = 1; j < k; ++j) s = __fadd_rn(s, sqrtf(best[j]));
    return __fdiv_rn(s, (float)k);
  }
};

// One WARP per query (the per-thread version - a sorted list in local memory - ran at 7 active lanes
// per instruction and 1750 warp instructions per query: profiles, prof_c4).  Per level:
//   1. the warp's 27-cell walk (flat27_runs) gives the flat candidate list and tells whether the block
//      holds k points at all;
//   2. the lanes stride over the flat list, compute the float32 distances and drop their bit patterns
//      (non-negative floats order like integers) into the warp's shared buffer; longer lists go through
//      the buffer in chunks, each chunk merged with the k best so far;
//   3. the k-th smallest value is found by a 31-step binary search on the bit pattern (each step a
//      strided count + REDUX), the k smallest are compacted in place (ties at the k-th value are
//      interchangeable);
//   4. the level's answer stands if the k-th distance is covered by the block (knn_safe2); then the k
//      values are rank-sorted and summed in ascending order by shuffles - the same sequential float32
//      sum as oracle/outliers.py.
// WarpKeep does steps 2 and 3 for k_knn_query_wide, but in this kernel's place at 32 < k <= 64 it was 20 - 30 %
// slower on the C4 scan (3476 -> 4572 us at k = 33, 4708 -> 5679 us at k = 64; B200 at 1000 W).
#define KNN_CAP 1024
#define KNN_WARPS 4
// newcomers in a batch of 32 above which the batch is sorted and merged instead of inserted one by one
// (2 / 4 / 6 / 10: within 2 %, 32: twice the time; profiles/r2x_knn_ab.json)
#define KNN_MERGE_MIN 6u
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn_query(uint32_t n_max, const uint32_t* n_dev, GridDev g, uint32_t k, float* __restrict__ avg,
            uint32_t* __restrict__ stragglers, ApcCtrl* ctrl) {
  __shared__ uint32_t s_buf[KNN_WARPS][KNN_CAP];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t n_sorted = grid_sorted_count(g, ctrl, n);
  const uint32_t k_eff = min(k, n);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  const uint32_t lt_mask = (1u << lane) - 1u;
  uint32_t* buf = s_buf[w];
  uint32_t* sorted_k = buf + KNN_CAP / 2;          // free once the k best sit at the front (k <= 64)
  for (uint32_t j = blockIdx.x * KNN_WARPS + w; j < n_sorted; j += gridDim.x * KNN_WARPS) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    bool done = false;
    // Always from level 0: starting at the finest level whose own cell already holds 5 / 10 / 16 points
    // examines more candidates than the failed levels cost (2.49 / 2.94 / 3.34 ms against 1.86 ms on the C4
    // scan, profiles/r2x_knn_ab.json).
    for (uint32_t level = 0; level < g.levels && !done; ++level) {
      const float c = g.cell[level];
      int32_t ix, iy, iz;
      if (!grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz)) continue;
      uint32_t cs, ps;
      const uint32_t total = flat27_runs(g, level, ix, iy, iz, lane, cs, ps);
      if (total < k_eff) continue;
      const float4* sp = g.sorted + (size_t)level * n_max;
      const float bound2 = knn_safe2(q, c, ix, iy, iz);
      if (k_eff <= 32u) {
        // 2'. k <= 32 (the reference's default is 20): the k best live in REGISTERS, lane i holding the
        // i-th smallest distance so far.  A batch of 32 candidates is screened with one ballot against
        // the current k-th value; the few that pass are inserted one by one (position by ballot, shift
        // by shuffle) - about 2x fewer instructions per level than the buffer + binary search below.
        const float inf = __int_as_float(0x7f800000);
        float val = inf, kth = inf;
        for (uint32_t base = 0; base < total; base += 32) {
          const uint32_t ci = base + lane;
          const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
          float d2 = inf;
          if (ci < total) {
            const float4 p = sp[at];
            d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
          }
          uint32_t cand = __ballot_sync(0xffffffffu, d2 < kth);
          if ((uint32_t)__popc(cand) > KNN_MERGE_MIN) {
            // many of the batch beat the current k-th value (always the first batch of a pass, often the second):
            // sort the batch across the lanes (bitonic network, 15 shuffle stages) and merge it with the sorted
            // `val` - reversed batch, element-wise minimum = the 32 smallest of the union as a bitonic sequence,
            // 5 more stages put them in order.  ~100 instructions whatever the number of newcomers, against ~14
            // per one-by-one insertion below (the first batch alone used to cost 450).
            float w = d2;
#pragma unroll
            for (uint32_t kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll
              for (uint32_t jj = kk >> 1; jj > 0; jj >>= 1) {
                const float o = __shfl_xor_sync(0xffffffffu, w, jj);
                const bool take_min = ((lane & kk) == 0) == ((lane & jj) == 0);
                w = take_min ? fminf(w, o) : fmaxf(w, o);
              }
            }
            float mrg = fminf(val, __shfl_sync(0xffffffffu, w, 31u - lane));
#pragma unroll
            for (uint32_t jj = 16; jj > 0; jj >>= 1) {
              const float o = __shfl_xor_sync(0xffffffffu, mrg, jj);
              mrg = (lane & jj) == 0 ? fminf(mrg, o) : fmaxf(mrg, o);
            }
            val = mrg;
            kth = __shfl_sync(0xffffffffu, val, k_eff - 1u);
            cand = 0;
          }
          while (cand) {
            const uint32_t b = __ffs(cand) - 1u;
            cand &= cand - 1u;
            const float x = __shfl_sync(0xffffffffu, d2, b);
            if (x < kth) {                                         // (the k-th value shrinks as we insert)
              const uint32_t pos = __popc(__ballot_sync(0xffffffffu, val <= x));
              const float up = __shfl_up_sync(0xffffffffu, val, 1);
              val = lane > pos ? up : (lane == pos ? x : val);
              kth = __shfl_sync(0xffffffffu, val, k_eff - 1u);
            }
          }
        }
        if (kth <= bound2) {
          done = true;
          const float r = sqrtf(val);
          float sum = 0.0f;
          for (uint32_t i = 0; i < k_eff; ++i) {                     // sequential float32 sum, ascending
            const float v = __shfl_sync(0xffffffffu, r, i);
            sum = i == 0 ? v : __fadd_rn(sum, v);
          }
          if (lane == 0) avg[orig] = __fdiv_rn(sum, (float)k_eff);
        }
        continue;
      }
      // 2. + 3. k > 32: candidates through the shared buffer, k best kept at its front
      uint32_t m = 0;
      for (uint32_t c0 = 0; c0 < total;) {
        const uint32_t take = min((uint32_t)KNN_CAP - m, total - c0);
        for (uint32_t base = 0; base < take; base += 32) {
          const uint32_t ci = base + lane;
          const uint32_t at = flat27_at(cs, ps, c0 + min(ci, take - 1u));
          if (ci < take) {
            const float4 p = sp[at];
            buf[m + ci] = __float_as_uint(d2_f32(q.x, q.y, q.z, p.x, p.y, p.z));
          }
        }
        __syncwarp();
        const uint32_t nbuf = m + take;
        c0 += take;
        if (nbuf > k_eff) {
          uint32_t V = 0;                                          // the k-th smallest bit pattern
          for (int bit = 30; bit >= 0; --bit) {
            const uint32_t trial = V | (1u << bit);
            uint32_t below = 0;
            for (uint32_t i = lane; i < nbuf; i += 32) below += buf[i] < trial ? 1u : 0u;
            if (__reduce_add_sync(0xffffffffu, below) < k_eff) V = trial;
          }
          uint32_t below = 0;
          for (uint32_t i = lane; i < nbuf; i += 32) below += buf[i] < V ? 1u : 0u;
          const uint32_t need_eq = k_eff - __reduce_add_sync(0xffffffffu, below);
          uint32_t kept = 0, eq_seen = 0;
          for (uint32_t base = 0; base < nbuf; base += 32) {       // in place: writes never pass the batch being read
            const uint32_t i = base + lane;
            const uint32_t x = i < nbuf ? buf[i] : 0xffffffffu;
            const bool is_eq = i < nbuf && x == V;
            const uint32_t beq = __ballot_sync(0xffffffffu, is_eq);
            const bool keep = (i < nbuf && x < V) || (is_eq && eq_seen + __popc(beq & lt_mask) < need_eq);
            const uint32_t bk = __ballot_sync(0xffffffffu, keep);
            __syncwarp();
            if (keep) buf[kept + __popc(bk & lt_mask)] = x;
            kept += __popc(bk);
            eq_seen += __popc(beq);
            __syncwarp();
          }
          m = k_eff;
        } else {
          m = nbuf;
        }
      }
      // 4. covered by the block?
      uint32_t mx = 0;
      for (uint32_t i = lane; i < k_eff; i += 32) mx = max(mx, buf[i]);
      const float kth = __uint_as_float(__reduce_max_sync(0xffffffffu, mx));
      if (kth <= bound2) done = true;
    }
    if (done && k_eff > 32u) {
      for (uint32_t e = lane; e < k_eff; e += 32) {                 // rank sort (k <= 64)
        const uint32_t x = buf[e];
        uint32_t rank = 0;
        for (uint32_t i = 0; i < k_eff; ++i) {
          const uint32_t y = buf[i];
          rank += (y < x || (y == x && i < e)) ? 1u : 0u;
        }
        sorted_k[rank] = x;
      }
      __syncwarp();
      const float r0 = lane < k_eff ? sqrtf(__uint_as_float(sorted_k[lane])) : 0.0f;
      const float r1 = lane + 32 < k_eff ? sqrtf(__uint_as_float(sorted_k[lane + 32])) : 0.0f;
      float sum = 0.0f;
      for (uint32_t i = 0; i < k_eff; ++i) {                         // sequential float32 sum, ascending
        const float v = __shfl_sync(0xffffffffu, i < 32 ? r0 : r1, i & 31u);
        sum = i == 0 ? v : __fadd_rn(sum, v);
      }
      if (lane == 0) avg[orig] = __fdiv_rn(sum, (float)k_eff);
      __syncwarp();
    } else if (!done && lane == 0) {
      stragglers[atomicAdd(&ctrl->counters[CTR_STRAGGLERS], 1u)] = orig;
    }
  }
}

// Exact brute-force KNN for the few points the grid could not resolve: one CTA per
// straggler, per-thread top-k over a strided scan of all points, then k rounds of
// block-wide minimum extraction.
__global__ void __launch_bounds__(256)
k_knn_stragglers(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, uint32_t k,
                 const uint32_t* __restrict__ stragglers, const ApcCtrl* ctrl, float* __restrict__ avg) {
  __shared__ float s_min[8];
  __shared__ uint32_t s_who[8];
  __shared__ float s_sel[KNN_KMAX];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t k_eff = min(k, n);
  const uint32_t n_str = ctrl->counters[CTR_STRAGGLERS];
  for (uint32_t sidx = blockIdx.x; sidx < n_str; sidx += gridDim.x) {
    const uint32_t orig = stragglers[sidx];
    const float4 q = pts[orig];
    TopK tk;
    tk.reset();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
      const float4 p = pts[i];
      tk.push(d2_f32(q.x, q.y, q.z, p.x, p.y, p.z), k_eff);
    }
    uint32_t head = 0;
    for (uint32_t round = 0; round < k_eff; ++round) {
      float v = head < tk.cnt ? tk.best[head] : __int_as_float(0x7f800000);
      uint32_t who = threadIdx.x;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const uint32_t ow = __shfl_xor_sync(0xffffffffu, who, o);
        if (ov < v || (ov == v && ow < who)) { v = ov; who = ow; }
      }
      if (lane_id() == 0) { s_min[threadIdx.x >> 5] = v; s_who[threadIdx.x >> 5] = who; }
      __syncthreads();
      float bv = s_min[0];
      uint32_t bw = s_who[0];
#pragma unroll
      for (int w = 1; w < 8; ++w)
        if (s_min[w] < bv || (s_min[w] == bv && s_who[w] < bw)) { bv = s_min[w]; bw = s_who[w]; }
      if (threadIdx.x == bw) { ++head; s_sel[round] = bv; }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      float s = sqrtf(s_sel[0]);
      for (uint32_t j = 1; j < k_eff; ++j) s = __fadd_rn(s, sqrtf(s_sel[j]));
      avg[orig] = __fdiv_rn(s, (float)k_eff);
    }
    __syncthreads();
  }
}

// ---- k > 64 (up to APC_MAX_NEIGHBORS; normals: max_nn > 32): per-warp shared candidate buffers -------
// Keys are compared as unsigned integers and have their top bit clear: float32 d2 bit patterns
// (non-negative floats order like integers), or (d2 bits << 32 | index) for the normals.
//
// WarpKeep: a warp streams candidate keys into its buffer (warp-collective add(), one key per lane);
// when the next batch might not fit, the k smallest are found by a binary search on the bit pattern
// (each step a strided count + REDUX) and compacted to the front in place (ties at the k-th value are
// interchangeable: equal keys are equal distances).  From then on the k-th value bounds the batch:
// a key not below it cannot enter the k smallest, so it never takes a buffer slot.  After finish()
// the k smallest (or all, if fewer arrived) sit unordered in buf[0, m).
template <typename K>
struct WarpKeep {
  K* buf;
  uint32_t cap, k, m;   // cap > k + 32: every selection frees room for at least one more batch
  K bound;              // keys >= bound are rejected (all ones before the first selection)
  __device__ __forceinline__ void init(K* b, uint32_t capacity, uint32_t kk) { buf = b; cap = capacity; k = kk; m = 0; bound = ~(K)0; }
  __device__ __forceinline__ void select(uint32_t lane) {
    __syncwarp();
    K V = 0;                                                   // the k-th smallest key
    for (int bit = (int)sizeof(K) * 8 - 2; bit >= 0; --bit) {
      const K trial = V | ((K)1 << bit);
      uint32_t below = 0;
      for (uint32_t i = lane; i < m; i += 32) below += buf[i] < trial ? 1u : 0u;
      if (__reduce_add_sync(0xffffffffu, below) < k) V = trial;
    }
    uint32_t below = 0;
    for (uint32_t i = lane; i < m; i += 32) below += buf[i] < V ? 1u : 0u;
    const uint32_t need_eq = k - __reduce_add_sync(0xffffffffu, below);
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t kept = 0, eq_seen = 0;
    for (uint32_t base = 0; base < m; base += 32) {           // in place: writes never pass the batch being read
      const uint32_t i = base + lane;
      const K x = i < m ? buf[i] : ~(K)0;
      const bool is_eq = i < m && x == V;
      const uint32_t beq = __ballot_sync(0xffffffffu, is_eq);
      const bool keep = (i < m && x < V) || (is_eq && eq_seen + __popc(beq & lt_mask) < need_eq);
      const uint32_t bk = __ballot_sync(0xffffffffu, keep);
      __syncwarp();
      if (keep) buf[kept + __popc(bk & lt_mask)] = x;
      kept += __popc(bk);
      eq_seen += __popc(beq);
      __syncwarp();
    }
    m = k;
    bound = V;
  }
  __device__ __forceinline__ void add(K key, bool valid, uint32_t lane) {
    const bool take = valid && key < bound;
    const uint32_t b = __ballot_sync(0xffffffffu, take);
    if (take) buf[m + __popc(b & ((1u << lane) - 1u))] = key;
    m += __popc(b);
    if (m + 32u > cap) select(lane);
  }
  __device__ __forceinline__ void finish(uint32_t lane) {
    if (m > k) select(lane);
    __syncwarp();
  }
};

// Buffer entries per warp of a WarpKeep: more than k + 32 (a selection always makes room for a batch)
// and at least the power of two warp_sort pads k to.  k = 1024: 1280 entries, 5 KB (KNN) /
// 10 KB (normals) per warp, 20 / 40 KB per block of 4 warps - under the 48 KB of a default launch.
static inline uint32_t wide_cap(uint32_t k) {
  uint32_t pow2 = 1;
  while (pow2 < k) pow2 <<= 1;
  return max(pow2, (k + 31u) / 32u * 32u + 256u);
}

// Ascending bitonic sort of buf[0, n) over the padded power of two (buf must hold it).  Warp-collective.
template <typename K>
__device__ void warp_sort(K* buf, uint32_t n, uint32_t lane) {
  uint32_t len = 1;
  while (len < n) len <<= 1;
  for (uint32_t i = n + lane; i < len; i += 32) buf[i] = ~(K)0;
  __syncwarp();
  for (uint32_t kk = 2; kk <= len; kk <<= 1)
    for (uint32_t jj = kk >> 1; jj > 0; jj >>= 1) {
      for (uint32_t i = lane; i < len; i += 32) {
        const uint32_t p = i ^ jj;
        if (p > i) {
          const K a = buf[i], b = buf[p];
          if ((a > b) == ((i & kk) == 0)) { buf[i] = b; buf[p] = a; }
        }
      }
      __syncwarp();
    }
}

// Mean of sqrtf over the k_eff keys in buf[0, k_eff) (float32 d2 bit patterns, unordered): sorted, then
// the sequential ascending float32 sum of oracle/outliers.py.  Warp-collective; every lane returns the mean.
__device__ float wide_average(uint32_t* buf, uint32_t k_eff, uint32_t lane) {
  warp_sort(buf, k_eff, lane);
  float sum = 0.0f;
  for (uint32_t base = 0; base < k_eff; base += 32) {
    const float r = base + lane < k_eff ? sqrtf(__uint_as_float(buf[base + lane])) : 0.0f;
    const uint32_t cnt = min(32u, k_eff - base);
    for (uint32_t i = 0; i < cnt; ++i) {                          // sequential float32 sum, ascending
      const float v = __shfl_sync(0xffffffffu, r, i);
      sum = base + i == 0 ? v : __fadd_rn(sum, v);
    }
  }
  __syncwarp();
  return __fdiv_rn(sum, (float)k_eff);
}

extern __shared__ __align__(16) unsigned char wide_smem[];

// Selection key of a candidate at float32 distance d2 whose original index is idx: the d2 bit pattern for
// the statistical stage (equal distances are interchangeable there), (d2 bits << 32 | index) for the
// normals (the oracle's total order (d2, index): the neighbourhood itself is exact).
template <typename K> __device__ __forceinline__ K knn_key(float d2, uint32_t idx);
template <> __device__ __forceinline__ uint32_t knn_key<uint32_t>(float d2, uint32_t) { return __float_as_uint(d2); }
template <> __device__ __forceinline__ unsigned long long knn_key<unsigned long long>(float d2, uint32_t idx) {
  return ((unsigned long long)__float_as_uint(d2) << 32) | idx;
}

// The KNN grid's level climb for query q (warp-collective), shared by k_knn_query_wide and k_normals_knn:
// per level, the 27-cell flat candidate list (flat27_runs) streams through a WarpKeep of `cap` keys at buf,
// and the level stands if the k_eff-th distance is covered by the block (knn_safe2).
// Returns true with the k_eff smallest keys in buf[0, k_eff) (unordered); false when no level covers q
// (a straggler).
template <typename K>
__device__ __forceinline__ bool knn_levels(const GridDev& g, uint32_t n_max, float4 q, uint32_t k_eff, K* buf, uint32_t cap,
                                           uint32_t lane) {
  for (uint32_t level = 0; level < g.levels; ++level) {
    const float c = g.cell[level];
    int32_t ix, iy, iz;
    if (!grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz)) continue;
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, level, ix, iy, iz, lane, cs, ps);
    if (total < k_eff) continue;
    const float4* sp = g.sorted + (size_t)level * n_max;
    const float bound2 = knn_safe2(q, c, ix, iy, iz);
    WarpKeep<K> wk;
    wk.init(buf, cap, k_eff);
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
      K key = 0;
      if (ci < total) {
        const float4 p = sp[at];
        key = knn_key<K>(d2_f32(q.x, q.y, q.z, p.x, p.y, p.z), __float_as_uint(p.w));
      }
      wk.add(key, ci < total, lane);
    }
    wk.finish(lane);
    uint32_t mx = 0;                                             // covered by the block? (the d2 bits of the keys)
    for (uint32_t i = lane; i < k_eff; i += 32) mx = max(mx, (uint32_t)(buf[i] >> (8 * sizeof(K) - 32)));
    if (__uint_as_float(__reduce_max_sync(0xffffffffu, mx)) <= bound2) return true;
  }
  return false;
}

// Exact brute force for a query no level covers (warp-collective): every point streams through the
// WarpKeep (after the first selection nearly all are rejected by the bound).  The k_eff smallest keys
// end in buf[0, k_eff), unordered.
template <typename K>
__device__ __forceinline__ void knn_brute(const float4* __restrict__ pts, uint32_t n, float4 q, uint32_t k_eff, K* buf,
                                          uint32_t cap, uint32_t lane) {
  WarpKeep<K> wk;
  wk.init(buf, cap, k_eff);
  for (uint32_t base = 0; base < n; base += 32) {
    const uint32_t i = base + lane;
    K key = 0;
    if (i < n) {
      const float4 p = pts[i];
      key = knn_key<K>(d2_f32(q.x, q.y, q.z, p.x, p.y, p.z), i);
    }
    wk.add(key, i < n, lane);
  }
  wk.finish(lane);
}

// k_knn_query for 64 < k <= APC_MAX_NEIGHBORS: the same level climb, 27-cell flat candidate list and
// coverage test (knn_safe2), the candidates through a WarpKeep of wide_cap(k) entries per warp (dynamic
// shared memory), the accepted level's k distances sorted and summed by wide_average.
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn_query_wide(uint32_t n_max, const uint32_t* n_dev, GridDev g, uint32_t k, uint32_t cap, float* __restrict__ avg,
                 uint32_t* __restrict__ stragglers, ApcCtrl* ctrl) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t n_sorted = grid_sorted_count(g, ctrl, n);
  const uint32_t k_eff = min(k, n);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t* buf = reinterpret_cast<uint32_t*>(wide_smem) + (size_t)w * cap;
  for (uint32_t j = blockIdx.x * KNN_WARPS + w; j < n_sorted; j += gridDim.x * KNN_WARPS) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (knn_levels(g, n_max, q, k_eff, buf, cap, lane)) {
      const float a = wide_average(buf, k_eff, lane);
      if (lane == 0) avg[orig] = a;
    } else if (lane == 0) {
      stragglers[atomicAdd(&ctrl->counters[CTR_STRAGGLERS], 1u)] = orig;
    }
    __syncwarp();
  }
}

// Exact brute force for the points no level of k_knn_query_wide covers: one warp per straggler.
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn_stragglers_wide(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, uint32_t k, uint32_t cap,
                      const uint32_t* __restrict__ stragglers, const ApcCtrl* ctrl, float* __restrict__ avg) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t k_eff = min(k, n);
  const uint32_t n_str = ctrl->counters[CTR_STRAGGLERS];
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t* buf = reinterpret_cast<uint32_t*>(wide_smem) + (size_t)w * cap;
  for (uint32_t sidx = blockIdx.x * KNN_WARPS + w; sidx < n_str; sidx += gridDim.x * KNN_WARPS) {
    const uint32_t orig = stragglers[sidx];
    knn_brute(pts, n, pts[orig], k_eff, buf, cap, lane);
    const float a = wide_average(buf, k_eff, lane);
    if (lane == 0) avg[orig] = a;
  }
}

// ---- float64 adjacent-pairwise tree reductions (mirrors oracle/outliers.py tree_sum) ------------
// in[i] (i < n) -> out[b] = tree sum of the 256 consecutive elements of block b (zero padded).
// mode 0: v = (double)avgf[i]; mode 1: v = ((double)avgf[i] - mu)^2 with mu = stats[0];
// mode 2: v = in[i] (partial sums of a previous level).
__global__ void __launch_bounds__(256)
k_tree_reduce(const float* __restrict__ avgf, const double* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
              uint32_t shift, int mode, const double* __restrict__ stats, double* __restrict__ out) {
  __shared__ double s_w[8];
  // number of valid inputs at this level = ceil(n / 256^shift)
  uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t s = 0; s < shift; ++s) n = (n + 255u) >> 8;
  const uint32_t i = blockIdx.x * 256u + threadIdx.x;
  double v = 0.0;
  if (i < n) {
    if (mode == 2) v = in[i];
    else {
      v = (double)avgf[i];
      if (mode == 1) { const double d = __dsub_rn(v, stats[0]); v = __dmul_rn(d, d); }
    }
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  if (lane_id() == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double a = __dadd_rn(__dadd_rn(s_w[0], s_w[1]), __dadd_rn(s_w[2], s_w[3]));
    const double b = __dadd_rn(__dadd_rn(s_w[4], s_w[5]), __dadd_rn(s_w[6], s_w[7]));
    out[blockIdx.x] = __dadd_rn(a, b);
  }
}

// stats[0]=mu, [1]=sigma, [2]=threshold
__global__ void k_stat_mu(const double* sum, uint32_t n_max, const uint32_t* n_dev, double* stats) {
  const uint32_t n = apc_count(n_dev, n_max);
  stats[0] = n ? __ddiv_rn(sum[0], (double)n) : 0.0;
}
__global__ void k_stat_sigma(const double* sumsq, uint32_t n_max, const uint32_t* n_dev, double std_ratio, double* stats) {
  const uint32_t n = apc_count(n_dev, n_max);
  const double sigma = n > 1 ? sqrt(__ddiv_rn(sumsq[0], (double)(n - 1))) : 0.0;
  stats[1] = sigma;
  stats[2] = __dadd_rn(stats[0], __dmul_rn(std_ratio, sigma));
}
__global__ void k_stat_mask(const float* __restrict__ avg, uint32_t n_max, const uint32_t* n_dev,
                            const double* __restrict__ stats, uint8_t* __restrict__ mask) {
  const uint32_t n = apc_count(n_dev, n_max);
  const double thr = stats[2];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    mask[i] = (n < 2 || (double)avg[i] <= thr) ? 1 : 0;
}

// ---- bounding box -> level-0 cell size -----------------------------------------------------------
__device__ __forceinline__ int32_t f2ord(float f) { const int32_t i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__device__ __forceinline__ float ord2f(int32_t i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__global__ void k_bbox_init(ApcCtrl* ctrl) {
  if (threadIdx.x < 3) ctrl->counters[CTR_BBOX + threadIdx.x] = (uint32_t)0x7fffffff;
  else if (threadIdx.x < 6) ctrl->counters[CTR_BBOX + threadIdx.x] = (uint32_t)0x80000000;
}
__global__ void __launch_bounds__(256) k_bbox(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, ApcCtrl* ctrl) {
  const uint32_t n = apc_count(n_dev, n_max);
  int32_t lo[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, hi[3] = {(int32_t)0x80000000, (int32_t)0x80000000, (int32_t)0x80000000};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    const float v[3] = {p.x, p.y, p.z};
#pragma unroll
    for (int a = 0; a < 3; ++a)
      if (fabsf(v[a]) < 3.0e38f) { lo[a] = min(lo[a], f2ord(v[a])); hi[a] = max(hi[a], f2ord(v[a])); }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    lo[a] = __reduce_min_sync(0xffffffffu, lo[a]);
    hi[a] = __reduce_max_sync(0xffffffffu, hi[a]);
    if (lane_id() == 0) {
      atomicMin(reinterpret_cast<int32_t*>(&ctrl->counters[CTR_BBOX + a]), lo[a]);
      atomicMax(reinterpret_cast<int32_t*>(&ctrl->counters[CTR_BBOX + 3 + a]), hi[a]);
    }
  }
}
// level sizes: c0 = hint if > 0 else max extent / 4096 (>= 1e-4), c_l = c0 * 2^l.  Without a hint c0 is also
// kept large enough for the farthest coordinate to have a level-0 cell index (|index| < 262 143): a small cloud
// far from the origin (a single point at 30 m: extent 0, cells of 1e-4 m) would otherwise fail with
// APC_ERR_KEY_RANGE.  Clouds whose indices stay below 262 000 keep their cell size.
__global__ void k_grid_cells(const ApcCtrl* ctrl, float hint, uint32_t levels, float* cell) {
  float c0 = hint;
  if (!(c0 > 0.0f)) {
    float ext = 0.0f, big = 0.0f;
    for (int a = 0; a < 3; ++a) {
      const float lo = ord2f((int32_t)ctrl->counters[CTR_BBOX + a]), hi = ord2f((int32_t)ctrl->counters[CTR_BBOX + 3 + a]);
      if (hi >= lo) {
        ext = fmaxf(ext, hi - lo);
        big = fmaxf(big, fmaxf(fabsf(lo), fabsf(hi)));
      }
    }
    c0 = fmaxf(fmaxf(ext * (1.0f / 4096.0f), 1.0e-4f), big * (1.0f / 262000.0f));
  }
  for (uint32_t l = 0; l < levels; ++l) { cell[l] = c0; c0 = c0 * 2.0f; }
}

// ---- host side ------------------------------------------------------------------------------------
struct GridHost {
  GridDev d{};
  uint32_t cap = 0, n_alloc = 0;
  uint32_t* cells_buf = nullptr;   // occupied-cell list of the single-level grid (handed out by apc_radius_grid_view)
};

struct NeighborScratch {
  GridHost grid[2];
  uint32_t* stragglers = nullptr;
  double* stats = nullptr;
  double* cov = nullptr;            // [max_points][9] covariances between k_normals_cov and k_normals_eigen
  uint32_t* dbscan_parent = nullptr;   // [max_points] union-find forest of apc_cluster_dbscan's core points
  uint32_t* dbscan_id = nullptr;       // [max_points] cluster id of every root
  uint8_t* dbscan_core = nullptr;      // [max_points] core flags
  double* icp_part = nullptr;          // [ICP_MAX_BLOCKS][32] block partials of k_icp_match's moments
  struct IcpState* icp_state = nullptr;   // apc_icp's T, previous metrics and done flag
  double* gicp_axes[2] = {nullptr, nullptr};   // [max_points][3] regularisation axes of apc_icp_generalized's source, target
  float* spfh = nullptr;               // [max_points][33] SPFH between the two passes of apc_compute_fpfh(_knn)
  unsigned long long* feat_best[2] = {nullptr, nullptr};   // [max_points] (d2 bits, index) minima of the feature search
  int32_t* feat_pairs = nullptr;       // [max_points][2] mutually consistent pairs of apc_correspondences_from_features
  uint32_t* feat_count = nullptr;      // [2] pair counts: all, mutual
  int32_t* fgr_pairs = nullptr;        // [3 * max_points][2] FGR's tuple pairs, or the unused pairs of its feature search
  struct FgrState* fgr_state = nullptr;   // apc_fgr(_from_features)' normalisation, tuple counts and loop outputs
};
// one scratch set per context, owned by the context (created on first use, freed by apc_ctx_destroy)
static NeighborScratch* scratch_of(apc_ctx* ctx) {
  if (!ctx->neighbors) ctx->neighbors = new NeighborScratch();
  return ctx->neighbors;
}

void apc_neighbors_release(apc_ctx* ctx) {
  NeighborScratch* s = ctx->neighbors;
  if (!s) return;
  for (auto& g : s->grid) {
    void* ptrs[] = {g.d.slots, g.d.slot, g.d.rank, g.d.sorted, g.d.cell, g.cells_buf};
    for (void* p : ptrs)
      if (p) cudaFree(p);
  }
  if (s->stragglers) cudaFree(s->stragglers);
  if (s->stats) cudaFree(s->stats);
  if (s->cov) cudaFree(s->cov);
  void* dbscan[] = {s->dbscan_parent, s->dbscan_id, s->dbscan_core};
  for (void* p : dbscan)
    if (p) cudaFree(p);
  void* icp[] = {s->icp_part, s->icp_state, s->gicp_axes[0], s->gicp_axes[1]};
  for (void* p : icp)
    if (p) cudaFree(p);
  void* feat[] = {s->spfh, s->feat_best[0], s->feat_best[1], s->feat_pairs, s->feat_count, s->fgr_pairs, s->fgr_state};
  for (void* p : feat)
    if (p) cudaFree(p);
  delete s;
  ctx->neighbors = nullptr;
}

// Allocates (once) the grid for `levels` levels; must run outside stream capture.
int apc_neighbors_prepare(apc_ctx* ctx, int which) {
  NeighborScratch* sc = scratch_of(ctx);
  GridHost& g = sc->grid[which];
  if (g.d.slots) return APC_OK;
  const uint32_t levels = which == 0 ? 1u : (uint32_t)KNN_LEVELS;
  const size_t M = ctx->max_points;
  uint64_t want = (uint64_t)levels * M * 4 / 3 + 1024;
  uint64_t cap = 1024;
  while (cap < want) cap <<= 1;
  if (which == 0 && cap < ctx->hash_cap) cap = ctx->hash_cap;
  APC_CUDA(ctx, cudaMalloc((void**)&g.d.slots, cap * sizeof(GridSlot)));
  APC_CUDA(ctx, cudaMalloc((void**)&g.d.slot, (size_t)levels * M * sizeof(uint32_t)));
  APC_CUDA(ctx, cudaMalloc((void**)&g.d.rank, (size_t)levels * M * sizeof(uint32_t)));
  APC_CUDA(ctx, cudaMalloc((void**)&g.d.sorted, (size_t)levels * M * sizeof(float4)));
  APC_CUDA(ctx, cudaMalloc((void**)&g.d.cell, 16 * sizeof(float)));
  g.cells_buf = nullptr;
  if (which == 0) APC_CUDA(ctx, cudaMalloc((void**)&g.cells_buf, M * sizeof(uint32_t)));
  g.d.cap_mask = (uint32_t)cap - 1;
  g.d.levels = levels;
  g.d.cursor_base = which == 0 ? CTR_CURSOR_RADIUS : CTR_CURSOR;
  g.cap = (uint32_t)cap;
  k_grid_reset<<<APC_SM_COUNT * 4, 256>>>(g.d.slots, (uint32_t)cap);
  APC_LAUNCH_CHECK(ctx, "k_grid_reset");
  if (!sc->stragglers) APC_CUDA(ctx, cudaMalloc((void**)&sc->stragglers, M * sizeof(uint32_t)));
  if (!sc->stats) APC_CUDA(ctx, cudaMalloc((void**)&sc->stats, 8 * sizeof(double)));
  APC_CUDA(ctx, cudaDeviceSynchronize());
  return APC_OK;
}

int apc_neighbors_reset(apc_ctx* ctx, cudaStream_t s) {
  NeighborScratch* sc = scratch_of(ctx);
  for (auto& g : sc->grid)
    if (g.d.slots) k_grid_reset<<<APC_SM_COUNT * 4, 256, 0, s>>>(g.d.slots, g.cap);
  APC_LAUNCH_CHECK(ctx, "k_grid_reset");
  return APC_OK;
}

static int grid_build(apc_ctx* ctx, GridHost& g, const float4* pts, uint32_t n_max, const uint32_t* n_dev,
                      float cell_hint, bool need_bbox, cudaStream_t s, bool inserted = false, uint32_t cursor_base = 0,
                      bool reciprocal = false) {
  if (g.d.levels == 1) g.d.cursor_base = cursor_base ? cursor_base : CTR_CURSOR_RADIUS;
  const uint32_t bx = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4);
  if (need_bbox) {
    k_bbox_init<<<1, 32, 0, s>>>(ctx->ctrl);
    k_bbox<<<bx, 256, 0, s>>>(pts, n_max, n_dev, ctx->ctrl);
  }
  g.d.cell0 = (g.d.levels == 1 && cell_hint > 0.0f) ? cell_hint : 0.0f;
  g.d.inv0 = (reciprocal && g.d.cell0 > 0.0f) ? 1.0f / g.d.cell0 : 0.0f;
  g.d.cells = inserted ? g.cells_buf : nullptr;
  if (!(g.d.cell0 > 0.0f)) k_grid_cells<<<1, 1, 0, s>>>(ctx->ctrl, cell_hint, g.d.levels, g.d.cell);
  const dim3 grid(bx, g.d.levels);
  if (!inserted) {   // (the pipeline's voxel stage inserts its centroids as it writes them)
    APC_PROF(ctx, "k_grid_insert", s);
    apc_klaunch(ctx, k_grid_insert, grid, 256, 0, s, pts, n_max, n_dev, g.d, ctx->ctrl);
  }
  {
    APC_PROF(ctx, "k_grid_assign", s);
    if (inserted && g.d.cells && g.d.levels == 1)   // the producer listed the occupied cells
      apc_klaunch(ctx, k_grid_assign_cells, min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT), 256, 0, s, g.d, ctx->ctrl, n_max);
    else
      apc_klaunch(ctx, k_grid_assign, grid, 256, 0, s, n_max, n_dev, g.d, ctx->ctrl);
  }
  APC_PROF(ctx, "k_grid_scatter", s);
  apc_klaunch(ctx, k_grid_scatter, grid, 256, 0, s, pts, n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "grid_build");
  return APC_OK;
}

int apc_radius_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int nb_points,
                       double radius, uint8_t* out_mask, uint32_t* out_counts, cudaStream_t s) {
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_mask, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, nb_points >= 1 && radius > 0.0, "nb_points must be >= 1 and radius > 0");
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  GridHost& g = scratch_of(ctx)->grid[0];
  const float r32 = (float)radius;
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  rc = grid_build(ctx, g, pts, n_max, n_dev, radius_cell(r32), false, s, false, 0, true);
  if (rc) return rc;
  rc = radius_query(ctx, g.d, n_max, n_dev, r32, (uint32_t)nb_points, out_mask, out_counts, s);
  if (rc) return rc;
  const dim3 grid(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), 1);
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<grid, 256, 0, s>>>(n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "radius_outliers");
  return APC_OK;
}

// select_by_mask over the radius decision + grid clean-up in one launch (both walk the points in
// original order): keeps the points whose mask is set, in order, and the points that own rank 0
// of their cell reset the cell's slot for the next frame.
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_radius_select(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev, const uint8_t* __restrict__ mask,
                GridDev g, float4* __restrict__ out, uint32_t* out_count, uint64_t* scan_state, const ApcCtrl* ctrl,
                uint32_t n_tiles, const uint32_t* __restrict__ idx_in, uint32_t* __restrict__ out_idx,
                const __grid_constant__ MirrorDev mir) {
  __shared__ uint32_t sm_scan[34];
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t epoch = ctrl->epoch;
  const uint32_t tile = blockIdx.x;
  bool keep[APC_TILE_ITEMS];
  float4 v[APC_TILE_ITEMS];
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    keep[j] = false;
    if (i < n) {
      keep[j] = mask[i] != 0;
      v[j] = in[i];
      const uint32_t slot = g.slot[i];
      if (slot != GRID_NOSLOT && g.rank[i] == 0) {
        g.slots[slot].key = GRID_EMPTY;
        g.slots[slot].fill = 0u;
      }
    }
  }
  uint32_t rank[APC_TILE_ITEMS];
  const uint32_t base = tile_compact_offsets(keep, rank, sm_scan, scan_state, tile, epoch, out_count, n_tiles);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j)
    if (keep[j]) {
      out[base + rank[j]] = v[j];
      mirror_store(mir, base + rank[j], v[j]);
      if (out_idx) {
        const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
        out_idx[base + rank[j]] = idx_in ? idx_in[i] : i;
      }
    }
}

// radius outlier removal + select_by_mask for the pipeline: query, then the fused select/clean
// Device view of the context's radius grid with the cell size of `radius` set: for a producer
// kernel in another file that inserts its output points itself (grid_insert_point) and then calls
// apc_radius_select_nobegin with points_inserted = 1.  Allocates on first use (not under capture).
int apc_radius_grid_view(apc_ctx* ctx, double radius, GridDev* out) {
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  GridHost& g = scratch_of(ctx)->grid[0];
  g.d.cell0 = radius_cell((float)radius);
  g.d.inv0 = 1.0f / g.d.cell0;
  g.d.cells = g.cells_buf;   // the caller inserts: it also lists the occupied cells
  *out = g.d;
  return APC_OK;
}

int apc_radius_select_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int nb_points,
                              double radius, uint8_t* mask_scratch, float* out_xyzi, uint32_t* out_count_dev,
                              int scan_slot, int points_inserted, cudaStream_t s, const uint32_t* idx_in,
                              uint32_t* out_idx, const MirrorDev* mir) {
  APC_REQUIRE(ctx, out_count_dev, "out_count_dev is NULL");
  if (n_max == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_count_dev, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  APC_REQUIRE(ctx, xyzi && mask_scratch && out_xyzi, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, nb_points >= 1 && radius > 0.0, "nb_points must be >= 1 and radius > 0");
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  GridHost& g = scratch_of(ctx)->grid[0];
  const float r32 = (float)radius;
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  rc = grid_build(ctx, g, pts, n_max, n_dev, radius_cell(r32), false, s, points_inserted != 0, 0, true);
  if (rc) return rc;
  rc = radius_query(ctx, g.d, n_max, n_dev, r32, (uint32_t)nb_points, mask_scratch, nullptr, s);
  if (rc) return rc;
  const uint32_t n_tiles = apc_div_up(n_max, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more points than the context was created for");
  APC_PROF(ctx, "k_radius_select", s);
  apc_klaunch(ctx, k_radius_select, n_tiles, APC_TILE_THREADS, 0, s, pts, n_max, n_dev, mask_scratch, g.d, reinterpret_cast<float4*>(out_xyzi),
                                                       out_count_dev, ctx->scan_state[scan_slot], ctx->ctrl, n_tiles,
                                                       idx_in, out_idx, mir ? *mir : MirrorDev{});
  APC_LAUNCH_CHECK(ctx, "radius_select");
  return APC_OK;
}

extern "C" int apc_radius_outliers(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                   int nb_points, double radius, uint8_t* out_mask, uint32_t* out_neighbor_counts,
                                   void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  // points outside the grid's key range (APC_ERR_KEY_RANGE at apc_check) are never queried: defined result
  if (out_mask && n_max) APC_CUDA(ctx, cudaMemsetAsync(out_mask, 0, n_max, s));
  if (out_neighbor_counts && n_max) APC_CUDA(ctx, cudaMemsetAsync(out_neighbor_counts, 0, (size_t)n_max * sizeof(uint32_t), s));
  return apc_radius_nobegin(ctx, xyzi, n_max, n_dev, nb_points, radius, out_mask, out_neighbor_counts, s);
}

int apc_statistical_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int nb_neighbors,
                            double std_ratio, float cell_hint, uint8_t* out_mask, float* out_avg,
                            double* out_stats_dev, cudaStream_t s) {
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_mask, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, nb_neighbors >= 1 && nb_neighbors <= APC_MAX_NEIGHBORS,
              "nb_neighbors must be in 1..APC_MAX_NEIGHBORS (" APC_STRINGIFY(APC_MAX_NEIGHBORS) ")");
  APC_REQUIRE(ctx, std_ratio > 0.0, "std_ratio must be > 0");
  int rc = apc_neighbors_prepare(ctx, 1);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  GridHost& g = sc->grid[1];
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  float* avg = out_avg ? out_avg : ctx->knn_avg;
  double* stats = out_stats_dev ? out_stats_dev : sc->stats;
  rc = grid_build(ctx, g, pts, n_max, n_dev, cell_hint, !(cell_hint > 0.0f), s);
  if (rc) return rc;
  const uint32_t bq = min(apc_div_up(n_max, KNN_WARPS), (uint32_t)APC_SM_COUNT * 16);   // one warp per query, grid-stride
  const uint32_t k = (uint32_t)nb_neighbors;
  if (k <= KNN_KMAX) {
    {
      APC_PROF(ctx, "k_knn_query", s);
      k_knn_query<<<bq, KNN_WARPS * 32, 0, s>>>(n_max, n_dev, g.d, k, avg, sc->stragglers, ctx->ctrl);
    }
    APC_PROF(ctx, "k_knn_stragglers", s);
    k_knn_stragglers<<<APC_SM_COUNT * 2, 256, 0, s>>>(pts, n_max, n_dev, k, sc->stragglers, ctx->ctrl, avg);
  } else {
    const uint32_t cap = wide_cap(k);
    const size_t smem = (size_t)KNN_WARPS * cap * sizeof(uint32_t);
    {
      APC_PROF(ctx, "k_knn_query_wide", s);
      k_knn_query_wide<<<bq, KNN_WARPS * 32, smem, s>>>(n_max, n_dev, g.d, k, cap, avg, sc->stragglers, ctx->ctrl);
    }
    APC_PROF(ctx, "k_knn_stragglers_wide", s);
    k_knn_stragglers_wide<<<APC_SM_COUNT * 2, KNN_WARPS * 32, smem, s>>>(pts, n_max, n_dev, k, cap, sc->stragglers, ctx->ctrl, avg);
  }
  const dim3 gridc(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), g.d.levels);
  {
    APC_PROF(ctx, "k_grid_clean", s);
    k_grid_clean<<<gridc, 256, 0, s>>>(n_max, n_dev, g.d);
  }
  APC_PROF(ctx, "stat_reduce_mask", s);
  // mu: tree over avg (levels of 256), then sigma over squared deviations
  for (int pass = 0; pass < 2; ++pass) {
    uint32_t cnt = n_max, shift = 0;
    const double* in = nullptr;
    double* out = ctx->red_a;
    do {
      const uint32_t blocks = apc_div_up(cnt, 256);
      k_tree_reduce<<<blocks, 256, 0, s>>>(avg, in, n_max, n_dev, shift, shift == 0 ? pass : 2, stats, out);
      in = out;
      out = (out == ctx->red_a) ? ctx->red_b : ctx->red_a;
      cnt = blocks;
      ++shift;
    } while (cnt > 1);
    if (pass == 0) k_stat_mu<<<1, 1, 0, s>>>(in, n_max, n_dev, stats);
    else k_stat_sigma<<<1, 1, 0, s>>>(in, n_max, n_dev, std_ratio, stats);
  }
  const uint32_t bm = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_stat_mask<<<bm, 256, 0, s>>>(avg, n_max, n_dev, stats, out_mask);
  APC_LAUNCH_CHECK(ctx, "statistical_outliers");
  return APC_OK;
}

extern "C" int apc_statistical_outliers(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                        int nb_neighbors, double std_ratio, uint8_t* out_mask, float* out_avg,
                                        double* out_stats_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  return apc_statistical_nobegin(ctx, xyzi, n_max, n_dev, nb_neighbors, std_ratio, 0.0f, out_mask, out_avg,
                                 out_stats_dev, s);
}

// ---- normal estimation (estimate_normals(radius, max_nn), pp.py:521-530; SURVEY.md B11) -------------
// Open3D's tensor EstimateNormals with both arguments set = hybrid search: the max_nn nearest of
// the points with d2 <= float32(r)^2 (query included), covariance of that neighbourhood, eigenvector
// of its smallest eigenvalue by the analytic symmetric 3x3 solver (Eberly, "A Robust Eigensolver for
// 3x3 Symmetric Matrices"), no orientation step; fewer than 3 neighbours -> identity covariance ->
// (0, 0, 1).  The neighbourhood is chosen with the float32 distance of the outlier stages and the
// total order (d2, original index); moments are taken about the query point in float64 (no
// cancellation whatever the coordinates' magnitude).  oracle/normals.py restates the same steps.
__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

// eigenvector of the (well separated) eigenvalue `ev`: the largest cross product of two rows of A - ev I
__device__ void eig_vector0(const double* A, double ev, double* v) {
  const double r0[3] = {A[0] - ev, A[1], A[2]}, r1[3] = {A[1], A[4] - ev, A[5]}, r2[3] = {A[2], A[5], A[8] - ev};
  double c01[3], c02[3], c12[3];
  cross3(r0, r1, c01);
  cross3(r0, r2, c02);
  cross3(r1, r2, c12);
  const double d0 = dot3(c01, c01), d1 = dot3(c02, c02), d2 = dot3(c12, c12);
  const double* best = c01;
  double dmax = d0;
  if (d1 > dmax) { dmax = d1; best = c02; }
  if (d2 > dmax) { dmax = d2; best = c12; }
  const double inv = 1.0 / sqrt(dmax);
  v[0] = best[0] * inv; v[1] = best[1] * inv; v[2] = best[2] * inv;
}

// eigenvector of `ev1` inside the plane orthogonal to the known eigenvector w
__device__ void eig_vector1(const double* A, const double* w, double ev1, double* v) {
  double U[3], V[3];
  if (fabs(w[0]) > fabs(w[1])) {
    const double inv = 1.0 / sqrt(w[0] * w[0] + w[2] * w[2]);
    U[0] = -w[2] * inv; U[1] = 0.0; U[2] = w[0] * inv;
  } else {
    const double inv = 1.0 / sqrt(w[1] * w[1] + w[2] * w[2]);
    U[0] = 0.0; U[1] = w[2] * inv; U[2] = -w[1] * inv;
  }
  cross3(w, U, V);
  const double AU[3] = {A[0] * U[0] + A[1] * U[1] + A[2] * U[2], A[1] * U[0] + A[4] * U[1] + A[5] * U[2],
                        A[2] * U[0] + A[5] * U[1] + A[8] * U[2]};
  const double AV[3] = {A[0] * V[0] + A[1] * V[1] + A[2] * V[2], A[1] * V[0] + A[4] * V[1] + A[5] * V[2],
                        A[2] * V[0] + A[5] * V[1] + A[8] * V[2]};
  double m00 = dot3(U, AU) - ev1, m01 = dot3(U, AV), m11 = dot3(V, AV) - ev1;
  const double a00 = fabs(m00), a01 = fabs(m01), a11 = fabs(m11);
  if (a00 >= a11) {
    if (fmax(a00, a01) > 0.0) {
      if (a00 >= a01) { m01 /= m00; m00 = 1.0 / sqrt(1.0 + m01 * m01); m01 *= m00; }
      else { m00 /= m01; m01 = 1.0 / sqrt(1.0 + m00 * m00); m00 *= m01; }
      for (int k = 0; k < 3; ++k) v[k] = m01 * U[k] - m00 * V[k];
    } else {
      for (int k = 0; k < 3; ++k) v[k] = U[k];
    }
  } else {
    if (fmax(a11, a01) > 0.0) {
      if (a11 >= a01) { m01 /= m11; m11 = 1.0 / sqrt(1.0 + m01 * m01); m01 *= m11; }
      else { m11 /= m01; m01 = 1.0 / sqrt(1.0 + m11 * m11); m11 *= m01; }
      for (int k = 0; k < 3; ++k) v[k] = m11 * U[k] - m01 * V[k];
    } else {
      for (int k = 0; k < 3; ++k) v[k] = U[k];
    }
  }
}

// normal = eigenvector of the smallest eigenvalue of the symmetric covariance C (row-major 3x3)
__device__ void normal_from_covariance(const double* C, double* nrm) {
  double mx = C[0];
  for (int k = 1; k < 9; ++k) mx = C[k] > mx ? C[k] : mx;
  if (mx == 0.0) { nrm[0] = nrm[1] = nrm[2] = 0.0; return; }
  double A[9];
  for (int k = 0; k < 9; ++k) A[k] = C[k] / mx;
  const double norm = A[1] * A[1] + A[2] * A[2] + A[5] * A[5];
  if (!(norm > 0.0)) {   // diagonal: the axis of the smallest entry
    nrm[0] = nrm[1] = nrm[2] = 0.0;
    if (C[0] < C[4] && C[0] < C[8]) nrm[0] = 1.0;
    else if (C[4] < C[0] && C[4] < C[8]) nrm[1] = 1.0;
    else nrm[2] = 1.0;
    return;
  }
  const double q = (A[0] + A[4] + A[8]) / 3.0;
  const double b00 = A[0] - q, b11 = A[4] - q, b22 = A[8] - q;
  const double p = sqrt((b00 * b00 + b11 * b11 + b22 * b22 + norm * 2.0) / 6.0);
  const double c00 = b11 * b22 - A[5] * A[5], c01 = A[1] * b22 - A[5] * A[2], c02 = A[1] * A[5] - b11 * A[2];
  const double det = (b00 * c00 - A[1] * c01 + A[2] * c02) / (p * p * p);
  const double half_det = fmin(fmax(det * 0.5, -1.0), 1.0);
  const double angle = acos(half_det) / 3.0;
  const double beta2 = cos(angle) * 2.0, beta0 = cos(angle + 2.09439510239319549) * 2.0, beta1 = -(beta0 + beta2);
  const double e0 = q + p * beta0, e1 = q + p * beta1, e2 = q + p * beta2;
  double v0[3], v1[3], v2[3];
  if (half_det >= 0.0) {
    eig_vector0(A, e2, v2);
    if (e2 < e0 && e2 < e1) { nrm[0] = v2[0]; nrm[1] = v2[1]; nrm[2] = v2[2]; return; }
    eig_vector1(A, v2, e1, v1);
    if (e1 < e0 && e1 < e2) { nrm[0] = v1[0]; nrm[1] = v1[1]; nrm[2] = v1[2]; return; }
    cross3(v1, v2, nrm);
  } else {
    eig_vector0(A, e0, v0);
    if (e0 < e1 && e0 < e2) { nrm[0] = v0[0]; nrm[1] = v0[1]; nrm[2] = v0[2]; return; }
    eig_vector1(A, v0, e1, v1);
    if (e1 < e0 && e1 < e2) { nrm[0] = v1[0]; nrm[1] = v1[1]; nrm[2] = v1[2]; return; }
    cross3(v0, v1, nrm);
  }
}

// Covariance of a neighbourhood of n_sel points from float64 moments about the query point that the lanes hold in
// parts (v: sums of x, y, z, xx, xy, xz, yy, yz, zz): the warp adds them up (warp-collective), lanes 0..8 store cov9
// of point orig, lane 0 the count.  Fewer than 3 neighbours: identity.
__device__ __forceinline__ void normals_cov_store(double (&v)[9], uint32_t n_sel, uint32_t orig, uint32_t lane,
                                                  uint32_t* __restrict__ counts, double* __restrict__ cov9) {
  double C[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
  if (n_sel >= 3) {
#pragma unroll
    for (int k = 0; k < 9; ++k)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    const double inv = 1.0 / (double)n_sel;
    const double s0 = v[0] * inv, s1 = v[1] * inv, s2 = v[2] * inv;
    C[0] = v[3] * inv - s0 * s0;
    C[1] = C[3] = v[4] * inv - s0 * s1;
    C[2] = C[6] = v[5] * inv - s0 * s2;
    C[4] = v[6] * inv - s1 * s1;
    C[5] = C[7] = v[7] * inv - s1 * s2;
    C[8] = v[8] * inv - s2 * s2;
  }
  double mine = C[0];                                            // C[lane] without a local-memory array
#pragma unroll
  for (int k = 1; k < 9; ++k) mine = lane == (uint32_t)k ? C[k] : mine;
  if (lane < 9) cov9[9 * (size_t)orig + lane] = mine;
  if (lane == 0 && counts) counts[orig] = n_sel;
}

// max_nn <= 32 (the reference's default is 30): one WARP per query, as in k_knn_query.  The lanes stride over
// the 27-cell flat candidate list; the max_nn nearest in-radius neighbours by (d2, original index) live in
// registers, lane i holding the i-th smallest key and the neighbour's position; every lane then contributes its
// neighbour's moments about the query point and normals_cov_store adds them up in float64.  The eigenvector is
// computed by k_normals_eigen, one THREAD per point (a serial float64 solve would idle 31 lanes of the warp here).
__global__ void __launch_bounds__(128)
k_normals_cov(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t max_nn, uint32_t* __restrict__ counts,
              double* __restrict__ cov9, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);   // >= 1: the query's own cell holds the query
    unsigned long long kv = ~0ull, kth = ~0ull;                   // lane i: i-th smallest key so far / the max_nn-th
    uint32_t pv = 0, in_radius = 0;
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t pos = flat27_at(cs, ps, min(ci, total - 1u));
      // key = (d2 bits : 32 | original index : 26 | tag : 6), ordered by (d2, index) like the oracle; the tag (the
      // lane that holds the entry's sorted position) only rides along through the sorting network below
      unsigned long long key = ~0ull;
      if (ci < total) {
        const float4 p = g.sorted[pos];
        const float d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
        if (d2 <= r2) key = ((unsigned long long)__float_as_uint(d2) << 32) | ((unsigned long long)__float_as_uint(p.w) << 6) | lane;
      }
      in_radius += __popc(__ballot_sync(0xffffffffu, key != ~0ull));
      uint32_t cand = __ballot_sync(0xffffffffu, key < kth);
      if ((uint32_t)__popc(cand) > 6u) {
        // many newcomers (dense clouds: the reference's default 0.01 m voxels leave 10 - 30 points within 0.1 m):
        // sort the batch across the lanes (bitonic network on the 64-bit keys) and merge it with the sorted `kv`,
        // ~160 instructions whatever their number against ~25 per one-by-one insertion - 55 % of this kernel's
        // instructions were that insertion loop (profiles/r2y_normals_ab.json).  Same order, same bits.
        unsigned long long w = key;
#pragma unroll
        for (uint32_t kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll
          for (uint32_t jj = kk >> 1; jj > 0; jj >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xffffffffu, w, jj);
            const bool take_min = ((lane & kk) == 0) == ((lane & jj) == 0);
            w = (take_min == (o < w)) ? o : w;
          }
        }
        const unsigned long long old = (kv & ~63ull) | (32u + lane);       // entries of kv: tag = 32 + their lane
        const unsigned long long wr = __shfl_sync(0xffffffffu, w, 31u - lane);
        unsigned long long mrg = wr < old ? wr : old;
#pragma unroll
        for (uint32_t jj = 16; jj > 0; jj >>= 1) {
          const unsigned long long o = __shfl_xor_sync(0xffffffffu, mrg, jj);
          mrg = (((lane & jj) == 0) == (o < mrg)) ? o : mrg;
        }
        const uint32_t tag = (uint32_t)mrg & 63u;
        const uint32_t from_new = __shfl_sync(0xffffffffu, pos, tag & 31u), from_old = __shfl_sync(0xffffffffu, pv, tag & 31u);
        pv = tag < 32u ? from_new : from_old;
        kv = mrg;
        kth = __shfl_sync(0xffffffffu, kv, max_nn - 1u);
        cand = 0;
      }
      while (cand) {
        const uint32_t b = __ffs(cand) - 1u;
        cand &= cand - 1u;
        const unsigned long long x = __shfl_sync(0xffffffffu, key, b);
        const uint32_t xp = __shfl_sync(0xffffffffu, pos, b);
        if (x < kth) {
          const uint32_t at = __popc(__ballot_sync(0xffffffffu, kv <= x));
          const unsigned long long up_k = __shfl_up_sync(0xffffffffu, kv, 1);
          const uint32_t up_p = __shfl_up_sync(0xffffffffu, pv, 1);
          if (lane > at) { kv = up_k; pv = up_p; }
          else if (lane == at) { kv = x; pv = xp; }
          kth = __shfl_sync(0xffffffffu, kv, max_nn - 1u);
        }
      }
    }
    const uint32_t n_sel = min(in_radius, max_nn);
    double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (n_sel >= 3 && lane < n_sel) {
      const float4 p = g.sorted[pv];
      const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
      v[0] = x; v[1] = y; v[2] = z;
      v[3] = x * x; v[4] = x * y; v[5] = x * z; v[6] = y * y; v[7] = y * z; v[8] = z * z;
    }
    normals_cov_store(v, n_sel, orig, lane, counts, cov9);
  }
}

// Covariance of a kept neighbourhood (warp-collective): buf[0, n_sel) holds the neighbours' 64-bit keys (d2 bits
// << 32 | original index), unordered.  The float64 moments about q are summed in key order, the same on every run
// (the keys arrive in the grid's in-cell order, which the build's atomics decide), by normals_cov_store.
__device__ __forceinline__ void normals_cov_of_keys(unsigned long long* buf, uint32_t n_sel, const float4* __restrict__ pts,
                                                    float4 q, uint32_t orig, uint32_t lane, uint32_t* __restrict__ counts,
                                                    double* __restrict__ cov9) {
  double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (n_sel >= 3) {
    warp_sort(buf, n_sel, lane);
    for (uint32_t i = lane; i < n_sel; i += 32) {
      const float4 p = pts[(uint32_t)buf[i]];
      const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
      v[0] += x; v[1] += y; v[2] += z;
      v[3] += x * x; v[4] += x * y; v[5] += x * z; v[6] += y * y; v[7] += y * z; v[8] += z * z;
    }
  }
  normals_cov_store(v, n_sel, orig, lane, counts, cov9);
}

// Hybrid search around a query taken from the grid (warp-collective): the 27-cell walk, every in-radius candidate's
// 64-bit key (d2 bits << 32 | original index: the oracle's total order, so the neighbourhood is exact) through a
// WarpKeep of `cap` entries at buf.  Returns min(in-radius count, max_nn), the number of keys left in buf (unordered).
__device__ __forceinline__ uint32_t hybrid_keep(const GridDev& g, float c, float4 q, float r2, uint32_t max_nn,
                                                unsigned long long* buf, uint32_t cap, uint32_t lane) {
  uint32_t cs, ps;
  const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);
  WarpKeep<unsigned long long> wk;
  wk.init(buf, cap, max_nn);
  uint32_t in_radius = 0;
  for (uint32_t base = 0; base < total; base += 32) {
    const uint32_t ci = base + lane;
    const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
    unsigned long long key = 0;
    bool inside = false;
    if (ci < total) {
      const float4 p = g.sorted[at];
      const float d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
      inside = d2 <= r2;
      key = knn_key<unsigned long long>(d2, __float_as_uint(p.w));
    }
    in_radius += __popc(__ballot_sync(0xffffffffu, inside));
    wk.add(key, inside, lane);
  }
  wk.finish(lane);
  return min(in_radius, max_nn);                                 // == wk.m
}

// 32 < max_nn <= APC_MAX_NEIGHBORS: one warp per query; hybrid_keep keeps the neighbourhood in a WarpKeep of
// wide_cap(max_nn) entries per warp, and normals_cov_of_keys sorts the kept keys, reads the neighbours by original
// index from the input and adds up their float64 moments about the query point.  k_normals_eigen turns cov9 into
// normals.
__global__ void __launch_bounds__(128)
k_normals_wide(uint32_t n_max, const uint32_t* n_dev, GridDev g, const float4* __restrict__ pts, float r2, uint32_t max_nn,
               uint32_t cap, uint32_t* __restrict__ counts, double* __restrict__ cov9, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)(threadIdx.x >> 5) * cap;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    normals_cov_of_keys(buf, hybrid_keep(g, c, q, r2, max_nn, buf, cap, lane), pts, q, orig, lane, counts, cov9);
    __syncwarp();                                                  // buf is reused by the next query
  }
}

// KNN search (Open3D estimate_normals with max_nn only): the max_nn nearest points by (d2, original index),
// no distance bound.  One warp per query climbs the levels of the KNN grid like k_knn_query_wide, with the
// 64-bit keys of k_normals_wide; the queries no level covers go to k_normals_knn_stragglers.
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_normals_knn(uint32_t n_max, const uint32_t* n_dev, GridDev g, const float4* __restrict__ pts, uint32_t k, uint32_t cap,
              uint32_t* __restrict__ counts, double* __restrict__ cov9, uint32_t* __restrict__ stragglers, ApcCtrl* ctrl) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t n_sorted = grid_sorted_count(g, ctrl, n);
  const uint32_t k_eff = min(k, n);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)w * cap;
  for (uint32_t j = blockIdx.x * KNN_WARPS + w; j < n_sorted; j += gridDim.x * KNN_WARPS) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (knn_levels(g, n_max, q, k_eff, buf, cap, lane)) normals_cov_of_keys(buf, k_eff, pts, q, orig, lane, counts, cov9);
    else if (lane == 0) stragglers[atomicAdd(&ctrl->counters[CTR_STRAGGLERS], 1u)] = orig;
    __syncwarp();
  }
}

__global__ void __launch_bounds__(KNN_WARPS * 32)
k_normals_knn_stragglers(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, uint32_t k, uint32_t cap,
                         const uint32_t* __restrict__ stragglers, const ApcCtrl* ctrl, uint32_t* __restrict__ counts,
                         double* __restrict__ cov9) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t k_eff = min(k, n);
  const uint32_t n_str = ctrl->counters[CTR_STRAGGLERS];
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)w * cap;
  for (uint32_t sidx = blockIdx.x * KNN_WARPS + w; sidx < n_str; sidx += gridDim.x * KNN_WARPS) {
    const uint32_t orig = stragglers[sidx];
    const float4 q = pts[orig];
    knn_brute(pts, n, q, k_eff, buf, cap, lane);
    normals_cov_of_keys(buf, k_eff, pts, q, orig, lane, counts, cov9);
    __syncwarp();
  }
}

// Radius search (Open3D estimate_normals with radius only): every point with d2 <= float32(r)^2, no cap on the
// count.  One warp per query over the 27-cell flat candidate list (flat27_runs), nothing kept: each
// in-radius neighbour adds its moments about the query in fixed point, rint(d * 2^40 / r) for the 3 first and
// rint(d d' * 2^40 / r^2) for the 6 second moments, in int64.  Integer sums do not depend on the order the
// grid's atomics leave inside a cell, so the covariance is bit-identical across runs and input permutations.
// Every term is at most ~2^40 and a context holds at most 2^22 points: the sums stay below 2^62.
#define NRM_FIX_ONE 1099511627776.0   // 2^40
__global__ void __launch_bounds__(128)
k_normals_radius(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r, float r2, uint32_t* __restrict__ counts,
                 double* __restrict__ cov9, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  const double s1 = NRM_FIX_ONE / (double)r, s2 = NRM_FIX_ONE / ((double)r * (double)r);
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);
    long long m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t cnt = 0;
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
      bool inside = false;
      if (ci < total) {
        const float4 p = g.sorted[at];
        inside = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z) <= r2;
        if (inside) {
          const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
          m[0] += __double2ll_rn(x * s1); m[1] += __double2ll_rn(y * s1); m[2] += __double2ll_rn(z * s1);
          m[3] += __double2ll_rn(x * x * s2); m[4] += __double2ll_rn(x * y * s2); m[5] += __double2ll_rn(x * z * s2);
          m[6] += __double2ll_rn(y * y * s2); m[7] += __double2ll_rn(y * z * s2); m[8] += __double2ll_rn(z * z * s2);
        }
      }
      cnt += __popc(__ballot_sync(0xffffffffu, inside));
    }
    double C[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};   // fewer than 3 neighbours: identity
    if (cnt >= 3) {
#pragma unroll
      for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m[k] += __shfl_xor_sync(0xffffffffu, m[k], o);
      const double inv = 1.0 / (double)cnt;
      const double u1 = (double)r / NRM_FIX_ONE, u2 = (double)r * (double)r / NRM_FIX_ONE;
      const double a0 = (double)m[0] * u1 * inv, a1 = (double)m[1] * u1 * inv, a2 = (double)m[2] * u1 * inv;
      C[0] = (double)m[3] * u2 * inv - a0 * a0;
      C[1] = C[3] = (double)m[4] * u2 * inv - a0 * a1;
      C[2] = C[6] = (double)m[5] * u2 * inv - a0 * a2;
      C[4] = (double)m[6] * u2 * inv - a1 * a1;
      C[5] = C[7] = (double)m[7] * u2 * inv - a1 * a2;
      C[8] = (double)m[8] * u2 * inv - a2 * a2;
    }
    double mine = C[0];                                            // C[lane] without a local-memory array
#pragma unroll
    for (int k = 1; k < 9; ++k) mine = lane == (uint32_t)k ? C[k] : mine;
    if (lane < 9) cov9[9 * (size_t)orig + lane] = mine;
    if (lane == 0 && counts) counts[orig] = cnt;
  }
}

__global__ void __launch_bounds__(256)
k_normals_eigen(uint32_t n_max, const uint32_t* n_dev, const double* __restrict__ cov9, float* __restrict__ normals) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double C[9], nrm[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) C[k] = cov9[9 * (size_t)i + k];
    normal_from_covariance(C, nrm);
    normals[3 * (size_t)i + 0] = (float)nrm[0];
    normals[3 * (size_t)i + 1] = (float)nrm[1];
    normals[3 * (size_t)i + 2] = (float)nrm[2];
  }
}

// Allocations of the normals stage (grid + covariance scratch): must run outside stream capture.
int apc_normals_prepare(apc_ctx* ctx) {
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  if (!sc->cov) APC_CUDA(ctx, cudaMalloc((void**)&sc->cov, (size_t)ctx->max_points * 9 * sizeof(double)));
  return APC_OK;
}

int apc_normals_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int max_nn, double radius,
                        float* out_normals, uint32_t* out_counts, double* out_cov, cudaStream_t s) {
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_normals, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, max_nn >= 1 && max_nn <= APC_MAX_NEIGHBORS && radius > 0.0,
              "max_nn must be in 1..APC_MAX_NEIGHBORS (" APC_STRINGIFY(APC_MAX_NEIGHBORS) ") and radius > 0");
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  GridHost& g = sc->grid[0];
  const float r32 = (float)radius;
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  // cells of r * (1 + 2^-8) indexed by one multiply with the host-rounded reciprocal (grid_coord_g): the three IEEE
  // divisions per lookup were 9 % of k_normals_cov's instructions.  Two points within r of each other have
  // quotients less than 1 - 2^-8 + 2^-22 |x| / c apart, i.e. fall into the same or adjacent cells for |x| < 16384 r -
  // the range the division with its 2^-10 margin guaranteed.
  rc = grid_build(ctx, g, pts, n_max, n_dev, r32 * 1.00390625f, false, s, false, CTR_CURSOR_NORMALS, true);
  if (rc) return rc;
  // warp per query -> covariances (caller's buffer or context scratch), then thread per point -> eigenvector
  double* cov = out_cov;
  if (!cov) {
    if (!sc->cov) APC_CUDA(ctx, cudaMalloc((void**)&sc->cov, (size_t)ctx->max_points * 9 * sizeof(double)));
    cov = sc->cov;
  }
  const uint32_t bq = min(apc_div_up(n_max, 4), (uint32_t)APC_SM_COUNT * 16);
  if (max_nn <= 32) {
    APC_PROF(ctx, "k_normals_cov", s);
    k_normals_cov<<<bq, 128, 0, s>>>(n_max, n_dev, g.d, r32 * r32, (uint32_t)max_nn, out_counts, cov, ctx->ctrl);
  } else {
    const uint32_t cap = wide_cap((uint32_t)max_nn);
    APC_PROF(ctx, "k_normals_wide", s);
    k_normals_wide<<<bq, 128, (size_t)4 * cap * sizeof(unsigned long long), s>>>(n_max, n_dev, g.d, pts, r32 * r32, (uint32_t)max_nn,
                                                                                 cap, out_counts, cov, ctx->ctrl);
  }
  {
    APC_PROF(ctx, "k_normals_eigen", s);
    k_normals_eigen<<<min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, s>>>(n_max, n_dev, cov, out_normals);
  }
  const dim3 grid(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), 1);
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<grid, 256, 0, s>>>(n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "estimate_normals");
  return APC_OK;
}

extern "C" int apc_estimate_normals(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int max_nn,
                                    double radius, float* out_normals, uint32_t* out_neighbor_counts,
                                    double* out_covariances, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  // points outside the grid's key range (APC_ERR_KEY_RANGE at apc_check) are never queried: defined result
  if (out_normals && n_max) APC_CUDA(ctx, cudaMemsetAsync(out_normals, 0, (size_t)n_max * 3 * sizeof(float), s));
  if (out_neighbor_counts && n_max) APC_CUDA(ctx, cudaMemsetAsync(out_neighbor_counts, 0, (size_t)n_max * sizeof(uint32_t), s));
  return apc_normals_nobegin(ctx, xyzi, n_max, n_dev, max_nn, radius, out_normals, out_neighbor_counts, out_covariances, s);
}

// ---- estimate_normals with one search bound: max_nn only (KNN) or radius only ---------------------------------
// Common start of apc_estimate_normals_knn / _radius once the mode's argument is checked: allocates grid `which`
// and the covariance scratch before anything is launched (nothing is allocated between the call's kernels),
// begins the call and zeroes the outputs.  Points the grid cannot key are never queried: their covariance stays
// zero, so k_normals_eigen gives them the normal (0, 0, 0), and their count is 0.
static int normals_search_begin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, int which, float* out_normals,
                                uint32_t* out_counts, double* out_cov, double** cov, cudaStream_t s) {
  APC_REQUIRE(ctx, xyzi && out_normals, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  int rc = apc_neighbors_prepare(ctx, which);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  if (!out_cov && !sc->cov) APC_CUDA(ctx, cudaMalloc((void**)&sc->cov, (size_t)ctx->max_points * 9 * sizeof(double)));
  *cov = out_cov ? out_cov : sc->cov;
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(*cov, 0, (size_t)n_max * 9 * sizeof(double), s));
  APC_CUDA(ctx, cudaMemsetAsync(out_normals, 0, (size_t)n_max * 3 * sizeof(float), s));
  if (out_counts) APC_CUDA(ctx, cudaMemsetAsync(out_counts, 0, (size_t)n_max * sizeof(uint32_t), s));
  return APC_OK;
}

// covariances -> normals, then the grid cleans itself for the next call of any mode
static int normals_search_finish(apc_ctx* ctx, const GridHost& g, uint32_t n_max, const uint32_t* n_dev, const double* cov,
                                 float* out_normals, cudaStream_t s) {
  {
    APC_PROF(ctx, "k_normals_eigen", s);
    k_normals_eigen<<<min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, s>>>(n_max, n_dev, cov, out_normals);
  }
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<dim3(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), g.d.levels), 256, 0, s>>>(n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "estimate_normals");
  return APC_OK;
}

extern "C" int apc_estimate_normals_knn(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, int max_nn,
                                        float* out_normals, uint32_t* out_neighbor_counts, double* out_covariances,
                                        void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, max_nn >= 1 && max_nn <= APC_MAX_NEIGHBORS,
              "max_nn must be in 1..APC_MAX_NEIGHBORS (" APC_STRINGIFY(APC_MAX_NEIGHBORS) ")");
  if (n_max == 0) return APC_OK;
  cudaStream_t s = (cudaStream_t)stream;
  double* cov = nullptr;
  int rc = normals_search_begin(ctx, xyzi, n_max, 1, out_normals, out_neighbor_counts, out_covariances, &cov, s);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  GridHost& g = sc->grid[1];
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  rc = grid_build(ctx, g, pts, n_max, n_dev, 0.0f, true, s);
  if (rc) return rc;
  const uint32_t cap = wide_cap((uint32_t)max_nn);
  const size_t smem = (size_t)KNN_WARPS * cap * sizeof(unsigned long long);
  const uint32_t bq = min(apc_div_up(n_max, KNN_WARPS), (uint32_t)APC_SM_COUNT * 16);   // one warp per query, grid-stride
  {
    APC_PROF(ctx, "k_normals_knn", s);
    k_normals_knn<<<bq, KNN_WARPS * 32, smem, s>>>(n_max, n_dev, g.d, pts, (uint32_t)max_nn, cap, out_neighbor_counts, cov,
                                                   sc->stragglers, ctx->ctrl);
  }
  {
    APC_PROF(ctx, "k_normals_knn_stragglers", s);
    k_normals_knn_stragglers<<<APC_SM_COUNT * 2, KNN_WARPS * 32, smem, s>>>(pts, n_max, n_dev, (uint32_t)max_nn, cap,
                                                                            sc->stragglers, ctx->ctrl, out_neighbor_counts, cov);
  }
  return normals_search_finish(ctx, g, n_max, n_dev, cov, out_normals, s);
}

extern "C" int apc_estimate_normals_radius(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                           double radius, float* out_normals, uint32_t* out_neighbor_counts,
                                           double* out_covariances, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  const float r32 = (float)radius;
  APC_REQUIRE(ctx, radius > 0.0 && r32 > 0.0f && std::isfinite(r32 * r32), "radius must be finite and > 0");
  if (n_max == 0) return APC_OK;
  cudaStream_t s = (cudaStream_t)stream;
  double* cov = nullptr;
  int rc = normals_search_begin(ctx, xyzi, n_max, 0, out_normals, out_neighbor_counts, out_covariances, &cov, s);
  if (rc) return rc;
  GridHost& g = scratch_of(ctx)->grid[0];
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  // the grid of the hybrid search (apc_normals_nobegin): cells of r * (1 + 2^-8), reciprocal indexing
  rc = grid_build(ctx, g, pts, n_max, n_dev, r32 * 1.00390625f, false, s, false, CTR_CURSOR_NORMALS, true);
  if (rc) return rc;
  {
    APC_PROF(ctx, "k_normals_radius", s);
    k_normals_radius<<<min(apc_div_up(n_max, 4), (uint32_t)APC_SM_COUNT * 16), 128, 0, s>>>(n_max, n_dev, g.d, r32, r32 * r32,
                                                                                        out_neighbor_counts, cov, ctx->ctrl);
  }
  return normals_search_finish(ctx, g, n_max, n_dev, cov, out_normals, s);
}

// ---- cluster_dbscan(eps, min_points) (Open3D PointCloud::ClusterDBSCAN) ----------------------------------------
// Contract (oracle/dbscan.py): N(i) = {j : d2 <= float32(eps)^2}, i included; core iff |N(i)| >= min_points;
// clusters = connected components of the core points linked by N; ids 0, 1, ... in the order of each component's
// lowest core index; a core point gets its component's id, a non-core point the smallest id among the components
// of the core points in N(i), else -1.
//   k_dbscan_core    |N(i)| (stops at min_points when the counts are not wanted) -> core flag, parent[i] = i
//   k_dbscan_union   every core point unions itself with its lower-indexed core neighbours
//   k_dbscan_roots   points every core point at its root, ranks the roots in index order -> ids, n_clusters
//   k_dbscan_label   core: id[root]; non-core: id of the lowest root among its core neighbours, or -1
// The union-find is lock-free over original indices: a union always hooks the larger root under the smaller one
// (atomicCAS on the root's own entry), so every tree's root is its minimum index whatever the thread schedule,
// and the output does not depend on the order the grid's atomics leave inside a cell.  Finds halve paths with
// relaxed stores: every value stored is an ancestor, so the trees stay the same whichever store lands last.
// Points the grid cannot key (APC_ERR_KEY_RANGE) are never in the cell-sorted array: they are in no one's N,
// stay non-core and keep the label -1.

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t uf_find(uint32_t* parent, uint32_t x) {
  uint32_t p = ld_relaxed_u32(&parent[x]);
  while (p != x) {
    const uint32_t gp = ld_relaxed_u32(&parent[p]);
    if (gp == p) return p;
    st_relaxed_u32(&parent[x], gp);                  // path halving
    x = gp;
    p = ld_relaxed_u32(&parent[x]);
  }
  return x;
}
__device__ __forceinline__ void uf_union(uint32_t* parent, uint32_t a, uint32_t b) {
  a = uf_find(parent, a);
  b = uf_find(parent, b);
  while (a != b) {
    if (a > b) { const uint32_t t = a; a = b; b = t; }
    const uint32_t old = atomicCAS(&parent[b], b, a);   // hook the larger root under the smaller
    if (old == b) return;
    b = uf_find(parent, old);                            // b was hooked meanwhile: go on from its new root
    a = uf_find(parent, a);
  }
}

__global__ void __launch_bounds__(128)
k_dbscan_core(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t min_points, uint32_t* __restrict__ counts,
              uint8_t* __restrict__ core, uint32_t* __restrict__ parent, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);
    uint32_t cnt = 0;
    for (uint32_t base = 0; base < total && (counts || cnt < min_points); base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
      bool inside = false;
      if (ci < total) {
        const float4 p = g.sorted[at];
        inside = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z) <= r2;
      }
      cnt += __popc(__ballot_sync(0xffffffffu, inside));
    }
    if (lane == 0) {
      core[orig] = cnt >= min_points ? 1 : 0;
      parent[orig] = orig;
      if (counts) counts[orig] = cnt;
    }
  }
}

__global__ void __launch_bounds__(128)
k_dbscan_union(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, const uint8_t* __restrict__ core,
               uint32_t* parent, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (!core[orig]) continue;                               // warp-uniform
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
      if (ci < total) {
        const float4 p = g.sorted[at];
        const uint32_t o = __float_as_uint(p.w);
        // each edge once, from its higher end (the predicate is symmetric)
        if (o < orig && d2_f32(q.x, q.y, q.z, p.x, p.y, p.z) <= r2 && core[o]) uf_union(parent, orig, o);
      }
    }
  }
}

// One tile of 1024 points in index order: roots flagged, ranked by the look-back scan of apc_scan.cuh.
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_dbscan_roots(uint32_t n_max, const uint32_t* n_dev, const uint8_t* __restrict__ core, uint32_t* parent,
               uint32_t* __restrict__ id, uint32_t* out_count, uint64_t* scan_state, const ApcCtrl* ctrl, uint32_t n_tiles) {
  __shared__ uint32_t sm_scan[34];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t tile = blockIdx.x;
  bool root[APC_TILE_ITEMS];
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k) {
    const uint32_t i = tile * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x;
    root[k] = false;
    if (i < n && core[i]) {
      uint32_t r = i, p = ld_relaxed_u32(&parent[i]);
      while (p != r) {                                      // no halving here: the only store is parent[i] = root
        r = p;
        p = ld_relaxed_u32(&parent[r]);
      }
      st_relaxed_u32(&parent[i], r);
      root[k] = r == i;
    }
  }
  uint32_t rank[APC_TILE_ITEMS];
  const uint32_t base = tile_compact_offsets(root, rank, sm_scan, scan_state, tile, ctrl->epoch, out_count, n_tiles);
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k)
    if (root[k]) id[tile * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x] = base + rank[k];
}

__global__ void __launch_bounds__(128)
k_dbscan_label(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, const uint8_t* __restrict__ core,
               const uint32_t* __restrict__ parent, const uint32_t* __restrict__ id, int32_t* __restrict__ labels,
               const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (core[orig]) {                                       // warp-uniform
      if (lane == 0) labels[orig] = (int32_t)id[parent[orig]];
      continue;
    }
    uint32_t cs, ps;
    const uint32_t total = flat27_runs(g, c, q, lane, cs, ps);
    uint32_t low = 0xffffffffu;                             // lowest root among the core neighbours
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
      if (ci < total) {
        const float4 p = g.sorted[at];
        const uint32_t o = __float_as_uint(p.w);
        if (d2_f32(q.x, q.y, q.z, p.x, p.y, p.z) <= r2 && core[o]) low = min(low, parent[o]);
      }
    }
    low = __reduce_min_sync(0xffffffffu, low);
    if (lane == 0) labels[orig] = low == 0xffffffffu ? -1 : (int32_t)id[low];
  }
}

extern "C" int apc_cluster_dbscan(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, double eps,
                                  int min_points, int32_t* out_labels, uint32_t* out_cluster_count_dev,
                                  uint32_t* out_neighbor_counts, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  const float r32 = (float)eps;
  APC_REQUIRE(ctx, eps > 0.0 && r32 > 0.0f && std::isfinite(r32 * r32), "eps must be finite and > 0");
  APC_REQUIRE(ctx, min_points >= 0, "min_points must be >= 0");
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_labels, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  const uint32_t n_tiles = apc_div_up(n_max, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more points than the context was created for");
  // everything is allocated before the first launch
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  const size_t M = ctx->max_points;
  if (!sc->dbscan_parent) APC_CUDA(ctx, cudaMalloc((void**)&sc->dbscan_parent, M * sizeof(uint32_t)));
  if (!sc->dbscan_id) APC_CUDA(ctx, cudaMalloc((void**)&sc->dbscan_id, M * sizeof(uint32_t)));
  if (!sc->dbscan_core) APC_CUDA(ctx, cudaMalloc((void**)&sc->dbscan_core, M));
  cudaStream_t s = (cudaStream_t)stream;
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(out_labels, 0xff, (size_t)n_max * sizeof(int32_t), s));
  APC_CUDA(ctx, cudaMemsetAsync(sc->dbscan_core, 0, n_max, s));
  if (out_neighbor_counts) APC_CUDA(ctx, cudaMemsetAsync(out_neighbor_counts, 0, (size_t)n_max * sizeof(uint32_t), s));
  GridHost& g = sc->grid[0];
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  const float r2 = r32 * r32;
  // the grid of the normals radius search (apc_estimate_normals_radius): cells of eps * (1 + 2^-8), reciprocal indexing
  rc = grid_build(ctx, g, pts, n_max, n_dev, r32 * 1.00390625f, false, s, false, CTR_CURSOR_NORMALS, true);
  if (rc) return rc;
  const uint32_t bq = min(apc_div_up(n_max, 4), (uint32_t)APC_SM_COUNT * 16);   // one warp per query, grid-stride
  {
    APC_PROF(ctx, "k_dbscan_core", s);
    k_dbscan_core<<<bq, 128, 0, s>>>(n_max, n_dev, g.d, r2, (uint32_t)min_points, out_neighbor_counts, sc->dbscan_core,
                                     sc->dbscan_parent, ctx->ctrl);
  }
  {
    APC_PROF(ctx, "k_dbscan_union", s);
    k_dbscan_union<<<bq, 128, 0, s>>>(n_max, n_dev, g.d, r2, sc->dbscan_core, sc->dbscan_parent, ctx->ctrl);
  }
  {
    APC_PROF(ctx, "k_dbscan_roots", s);
    k_dbscan_roots<<<n_tiles, APC_TILE_THREADS, 0, s>>>(n_max, n_dev, sc->dbscan_core, sc->dbscan_parent, sc->dbscan_id,
                                                        out_cluster_count_dev, ctx->scan_state[0], ctx->ctrl, n_tiles);
  }
  {
    APC_PROF(ctx, "k_dbscan_label", s);
    k_dbscan_label<<<bq, 128, 0, s>>>(n_max, n_dev, g.d, r2, sc->dbscan_core, sc->dbscan_parent, sc->dbscan_id,
                                      out_labels, ctx->ctrl);
  }
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<dim3(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), 1), 256, 0, s>>>(n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "cluster_dbscan");
  return APC_OK;
}

// ---- ICP registration (Open3D t::pipelines::registration::ICP / EvaluateRegistration) -------------------------
// Contract (oracle/registration.py): s' = float32(T s) with every coordinate ((T[r,0]*x + T[r,1]*y) + T[r,2]*z)
// + T[r,3] in float64, unfused, from the ORIGINAL source; the correspondence of s' is the target point with the
// smallest (d2, index) among those with d2_f32 <= float32(r)^2, else -1.
//   k_icp_init    T = init (a kernel argument), zero metrics, clears the done flag
//   k_icp_match   one warp per source point in index order, grid-stride: transform, 27-cell walk over the target's
//                 grid (the grid of apc_cluster_dbscan, cells of r * (1 + 2^-8)), 64-bit (d2 bits, index) warp
//                 minimum -> correspondence; lane k accumulates moment k of the estimation in float64 over the
//                 warp's queries, and the block writes one row of 32 partials
//   k_icp_solve   one block: the partials reduced in a fixed order -> fitness, rmse, the convergence test, the
//                 update (Horn's quaternion for point-to-point, Cholesky for point-to-plane) and T = update T
// apc_icp launches max_iteration (match, solve) pairs up front; both kernels return at once when the loop has
// stopped (done flag), so the call needs no host synchronisation.  The launch configuration depends on n_max
// only, and every sum has a fixed order: results are bit-identical from run to run.
#define ICP_MAX_BLOCKS (APC_SM_COUNT * 16)
#define ICP_PIVOT_REL 1e-12     // Cholesky pivot floor relative to its diagonal entry (oracle PIVOT_REL)

struct IcpState {
  double T[16];
  double prev_f, prev_r;
  uint32_t done;
  uint32_t iterations;
};
struct IcpT16 {
  double v[16];
};

// Lane k accumulates v[a] * v[b] with (a, b) = c_icp_pairs[method][k] (a | b << 4).  v[0..6] depend on the method,
// v[7] = 1, v[8] = d2, v[9] = 0.  Lanes 0 and 1 are n_corr and sum d2 for both methods.
//   point-to-point: v = (s', t); sum s' (2-4), sum t (5-7), sum s'_i t_j (8-16)
//   point-to-plane: v = (J = [s' x n, n], r = (s' - t) . n); J^T J upper triangle (2-22), J^T r (23-28)
__constant__ uint8_t c_icp_pairs[2][32] = {
    {0x77, 0x78, 0x70, 0x71, 0x72, 0x73, 0x74, 0x75, 0x30, 0x40, 0x50, 0x31, 0x41, 0x51, 0x32, 0x42,
     0x52, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99, 0x99},
    {0x77, 0x78, 0x00, 0x10, 0x20, 0x30, 0x40, 0x50, 0x11, 0x21, 0x31, 0x41, 0x51, 0x22, 0x32, 0x42,
     0x52, 0x33, 0x43, 0x53, 0x44, 0x54, 0x55, 0x60, 0x61, 0x62, 0x63, 0x64, 0x65, 0x99, 0x99, 0x99}};

__device__ __forceinline__ double icp_pick(const double (&v)[10], uint32_t a) {
  double x = v[0];
#pragma unroll
  for (uint32_t k = 1; k < 10; ++k) x = a == k ? v[k] : x;
  return x;
}
__device__ __forceinline__ float icp_row(const double (&T)[12], int r, double x, double y, double z) {
  return __double2float_rn(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(T[4 * r], x), __dmul_rn(T[4 * r + 1], y)),
                                               __dmul_rn(T[4 * r + 2], z)), T[4 * r + 3]));
}
// flat27_runs for a query that was not inserted into the grid: a point whose cell cannot be keyed (beyond the
// key range or not finite) has an empty list.  Warp-uniform.
__device__ __forceinline__ uint32_t flat27_runs_outside(const GridDev& g, float c, float4 q, uint32_t lane, uint32_t& cs,
                                                        uint32_t& ps) {
  int32_t ix, iy, iz;
  cs = ps = 0;
  if (!grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz)) return 0;
  return flat27_runs(g, 0, ix, iy, iz, lane, cs, ps);
}
// warp minimum of a 64-bit key: high words, then the low words of the lanes that hold the high minimum
__device__ __forceinline__ uint64_t warp_min_u64(uint64_t k) {
  const uint32_t hi = __reduce_min_sync(0xffffffffu, (uint32_t)(k >> 32));
  const uint32_t lo = __reduce_min_sync(0xffffffffu, (uint32_t)(k >> 32) == hi ? (uint32_t)k : 0xffffffffu);
  return ((uint64_t)hi << 32) | lo;
}
// ICP's correspondence search for the transformed source point q (warp-collective): the smallest (d2 bits << 32 |
// index) key over the target points with d2 <= r2 in the 27 cells around q, the same in every lane; all ones when
// there is none.
__device__ __forceinline__ uint64_t icp_best(const GridDev& g, float c, float4 q, float r2, uint32_t lane) {
  uint32_t cs, ps;
  const uint32_t total = flat27_runs_outside(g, c, q, lane, cs, ps);
  uint64_t best = ~0ull;
  for (uint32_t base = 0; base < total; base += 32) {
    const uint32_t ci = base + lane;
    const uint32_t at = flat27_at(cs, ps, min(ci, total - 1u));
    if (ci < total) {
      const float4 t = g.sorted[at];
      const float d2 = d2_f32(q.x, q.y, q.z, t.x, t.y, t.z);
      if (d2 <= r2) best = min(best, ((uint64_t)__float_as_uint(d2) << 32) | __float_as_uint(t.w));
    }
  }
  return warp_min_u64(best);
}

__global__ void k_icp_init(IcpT16 init, IcpState* __restrict__ st, double* __restrict__ out_T, double* __restrict__ out_stats,
                           int32_t* __restrict__ out_info, int32_t status) {
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    st->T[k] = init.v[k];
    if (out_T) out_T[k] = init.v[k];
  }
  st->prev_f = st->prev_r = 0.0;
  st->done = status != APC_ICP_OK;
  st->iterations = 0;
  out_stats[0] = out_stats[1] = 0.0;
  if (out_info) {
    out_info[0] = out_info[1] = out_info[3] = 0;
    out_info[2] = status;
  }
}

__global__ void __launch_bounds__(128)
k_icp_match(const float4* __restrict__ src, uint32_t n_max, const uint32_t* n_dev, const float4* __restrict__ tgt,
            const float* __restrict__ tgt_normals, GridDev g, float r2, int method, const IcpState* __restrict__ st,
            int32_t* __restrict__ corr_out, float* __restrict__ d2_out, double* __restrict__ partials) {
  if (st->done) return;                                     // the loop has stopped: block-uniform
  __shared__ double sm[4][32];
  const uint32_t n = apc_count(n_dev, n_max);
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t pair = c_icp_pairs[method][lane], pa = pair & 15u, pb = pair >> 4;
  double T[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) T[k] = st->T[k];
  double acc = 0.0;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += (gridDim.x * blockDim.x) >> 5) {
    const float4 p = src[i];
    const double x = p.x, y = p.y, z = p.z;
    const float4 q = make_float4(icp_row(T, 0, x, y, z), icp_row(T, 1, x, y, z), icp_row(T, 2, x, y, z), 0.0f);
    const uint64_t best = icp_best(g, c, q, r2, lane);
    const bool found = best != ~0ull;                       // warp-uniform
    const uint32_t j = (uint32_t)best;
    const float d2 = __uint_as_float((uint32_t)(best >> 32));
    if (found) {
      const float4 t = tgt[j];
      double v[10];
      const double sx = q.x, sy = q.y, sz = q.z, tx = t.x, ty = t.y, tz = t.z;
      if (method == APC_ICP_POINT_TO_PLANE) {
        const double nx = tgt_normals[3 * (size_t)j], ny = tgt_normals[3 * (size_t)j + 1], nz = tgt_normals[3 * (size_t)j + 2];
        v[0] = sy * nz - sz * ny; v[1] = sz * nx - sx * nz; v[2] = sx * ny - sy * nx;
        v[3] = nx; v[4] = ny; v[5] = nz;
        v[6] = ((sx - tx) * nx + (sy - ty) * ny) + (sz - tz) * nz;
      } else {
        v[0] = sx; v[1] = sy; v[2] = sz; v[3] = tx; v[4] = ty; v[5] = tz; v[6] = 0.0;
      }
      v[7] = 1.0; v[8] = d2; v[9] = 0.0;
      acc += icp_pick(v, pa) * icp_pick(v, pb);
    }
    if (lane == 0) {
      if (corr_out) corr_out[i] = found ? (int32_t)j : -1;
      if (d2_out) d2_out[i] = found ? d2 : 0.0f;
    }
  }
  sm[warp][lane] = acc;
  __syncthreads();
  if (threadIdx.x < 32) partials[32 * (size_t)blockIdx.x + lane] = ((sm[0][lane] + sm[1][lane]) + sm[2][lane]) + sm[3][lane];
}

// The serial solve of k_icp_solve (one thread) keeps its matrices in shared memory: as local arrays they spilled.
struct IcpWork {
  double N[4][4], V[4][4];    // point-to-point: Horn's matrix and its Jacobi rotations
  double L[6][6];             // point-to-plane: the normal equations, overwritten by their Cholesky factor
};

// Largest-eigenvalue eigenvector of the symmetric 4x4 N (cyclic Jacobi)
__device__ __forceinline__ void icp_top_eigvec4(double (&N)[4][4], double (&V)[4][4], double (&q)[4]) {
  for (int a = 0; a < 4; ++a)
    for (int b = 0; b < 4; ++b) V[a][b] = a == b ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 30; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int a = 0; a < 4; ++a) {
      diag += N[a][a] * N[a][a];
      for (int b = a + 1; b < 4; ++b) off += N[a][b] * N[a][b];
    }
    if (!(off > 1e-36 * diag)) break;
    for (int a = 0; a < 3; ++a)
      for (int b = a + 1; b < 4; ++b) {
        if (N[a][b] == 0.0) continue;
        const double theta = (N[b][b] - N[a][a]) / (2.0 * N[a][b]);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < 4; ++k) {                        // N = J^T N J, columns then rows
          const double x = N[k][a], y = N[k][b];
          N[k][a] = cs * x - sn * y;
          N[k][b] = sn * x + cs * y;
        }
        for (int k = 0; k < 4; ++k) {
          const double x = N[a][k], y = N[b][k];
          N[a][k] = cs * x - sn * y;
          N[b][k] = sn * x + cs * y;
        }
        for (int k = 0; k < 4; ++k) {
          const double x = V[k][a], y = V[k][b];
          V[k][a] = cs * x - sn * y;
          V[k][b] = sn * x + cs * y;
        }
      }
  }
  int m = 0;
  for (int a = 1; a < 4; ++a)
    if (N[a][a] > N[m][m]) m = a;
  for (int k = 0; k < 4; ++k) q[k] = V[k][m];
}

// Kabsch from the raw moments: H = sum s' t^T - sum s' sum t^T / n; the proper rotation maximising tr(R^T H) is
// the quaternion of the largest eigenvalue of Horn's matrix (the SVD solution with its reflection fix).
__device__ __forceinline__ void icp_point_to_point(const double* M, IcpWork& wk, double (&U)[16]) {
  const double n = M[0];
  const double ms[3] = {M[2] / n, M[3] / n, M[4] / n}, mt[3] = {M[5] / n, M[6] / n, M[7] / n};
  double H[3][3];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) H[a][b] = M[8 + 3 * a + b] - n * ms[a] * mt[b];   // lane 8 + 3a + b: sum s'_a t_b
  const double Sxx = H[0][0], Sxy = H[0][1], Sxz = H[0][2], Syx = H[1][0], Syy = H[1][1], Syz = H[1][2], Szx = H[2][0],
               Szy = H[2][1], Szz = H[2][2];
  const double N[4][4] = {{Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx},
                          {Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz},
                          {Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy},
                          {Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz}};
  for (int a = 0; a < 4; ++a)
    for (int b = 0; b < 4; ++b) wk.N[a][b] = N[a][b];
  double q[4];
  icp_top_eigvec4(wk.N, wk.V, q);
  const double nq = sqrt(((q[0] * q[0] + q[1] * q[1]) + q[2] * q[2]) + q[3] * q[3]);
  const double w = q[0] / nq, x = q[1] / nq, y = q[2] / nq, z = q[3] / nq;
  const double R[3][3] = {{w * w + x * x - y * y - z * z, 2.0 * (x * y - w * z), 2.0 * (x * z + w * y)},
                          {2.0 * (x * y + w * z), w * w - x * x + y * y - z * z, 2.0 * (y * z - w * x)},
                          {2.0 * (x * z - w * y), 2.0 * (y * z + w * x), w * w - x * x - y * y + z * z}};
  for (int a = 0; a < 3; ++a) {
    for (int b = 0; b < 3; ++b) U[4 * a + b] = R[a][b];
    U[4 * a + 3] = mt[a] - ((R[a][0] * ms[0] + R[a][1] * ms[1]) + R[a][2] * ms[2]);
  }
  U[12] = U[13] = U[14] = 0.0;
  U[15] = 1.0;
}

// One Gauss-Newton step: (sum J^T J) x = -(sum J^T r) by Cholesky; false when a pivot is not above ICP_PIVOT_REL
// times its diagonal entry.  x = (alpha, beta, gamma, tx, ty, tz) -> Rz(gamma) Ry(beta) Rx(alpha) (Open3D's
// PoseToTransformation).
__device__ __forceinline__ bool icp_point_to_plane(const double* M, IcpWork& wk, double (&U)[16]) {
  double (&L)[6][6] = wk.L;
  int k = 2;
  for (int c = 0; c < 6; ++c)
    for (int r = c; r < 6; ++r) L[r][c] = M[k++];          // lower triangle of sum J^T J
  for (int j = 0; j < 6; ++j) {
    const double ajj = L[j][j];
    double d = ajj;
    for (int m = 0; m < j; ++m) d -= L[j][m] * L[j][m];
    if (!(isfinite(d) && d > ICP_PIVOT_REL * ajj)) return false;
    L[j][j] = sqrt(d);
    for (int i = j + 1; i < 6; ++i) {
      double e = L[i][j];
      for (int m = 0; m < j; ++m) e -= L[i][m] * L[j][m];
      L[i][j] = e / L[j][j];
    }
  }
  double y[6], x[6];
  for (int i = 0; i < 6; ++i) {
    double e = -M[23 + i];
    for (int m = 0; m < i; ++m) e -= L[i][m] * y[m];
    y[i] = e / L[i][i];
  }
  for (int i = 5; i >= 0; --i) {
    double e = y[i];
    for (int m = i + 1; m < 6; ++m) e -= L[m][i] * x[m];
    x[i] = e / L[i][i];
  }
  double sa, ca, sb, cb, sg, cg;
  sincos(x[0], &sa, &ca);
  sincos(x[1], &sb, &cb);
  sincos(x[2], &sg, &cg);
  U[0] = cg * cb;  U[1] = -sg * ca + cg * sb * sa;  U[2] = sg * sa + cg * sb * ca;   U[3] = x[3];
  U[4] = sg * cb;  U[5] = cg * ca + sg * sb * sa;   U[6] = -cg * sa + sg * sb * ca;  U[7] = x[4];
  U[8] = -sb;      U[9] = cb * sa;                  U[10] = cb * ca;                 U[11] = x[5];
  U[12] = 0.0;     U[13] = 0.0;                     U[14] = 0.0;                     U[15] = 1.0;
  return true;
}

// method < 0: evaluate_registration, metrics only.
// 8 warps reduce the partials; one thread solves.  __maxnreg__: with the default budget of a 256-thread block the
// serial solve spilled (64 registers); it needs 90.
#define ICP_SOLVE_WARPS 8
__global__ void __maxnreg__(128)
k_icp_solve(const double* __restrict__ partials, uint32_t n_parts, uint32_t n_max, const uint32_t* n_dev, int method,
            int iteration, double relative_fitness, double relative_rmse, IcpState* __restrict__ st,
            double* __restrict__ out_T, double* __restrict__ out_stats, int32_t* __restrict__ out_info) {
  if (st->done) return;                                     // block-uniform
  __shared__ double sm[ICP_SOLVE_WARPS][32];
  __shared__ IcpWork wk;
  const uint32_t m = threadIdx.x & 31u, w = threadIdx.x >> 5;
  // thread (w, m): moment m of blocks w, w + 8, ..., in four independent chains (the loads overlap)
  double part[4] = {0.0, 0.0, 0.0, 0.0};
  uint32_t b = w;
  for (; b + 3 * ICP_SOLVE_WARPS < n_parts; b += 4 * ICP_SOLVE_WARPS)
#pragma unroll
    for (int u = 0; u < 4; ++u) part[u] += partials[32 * (size_t)(b + u * ICP_SOLVE_WARPS) + m];
  for (; b < n_parts; b += ICP_SOLVE_WARPS) part[0] += partials[32 * (size_t)b + m];
  sm[w][m] = (part[0] + part[1]) + (part[2] + part[3]);
  __syncthreads();
  if (w != 0) return;
  double tot = 0.0;
#pragma unroll
  for (int k = 0; k < ICP_SOLVE_WARPS; ++k) tot += sm[k][m];
  __syncwarp();
  sm[0][m] = tot;
  __syncwarp();
  if (m != 0) return;
  const double* M = sm[0];
  const double n_corr = M[0];
  const uint32_t n = apc_count(n_dev, n_max);
  const double fitness = n_corr > 0.0 ? n_corr / (double)n : 0.0, rmse = n_corr > 0.0 ? sqrt(M[1] / n_corr) : 0.0;
  out_stats[0] = fitness;
  out_stats[1] = rmse;
  if (method < 0) return;
  int32_t status = APC_ICP_OK;
  double U[16];
  if (n_corr == 0.0) status = APC_ICP_NO_CORRESPONDENCE;
  else if (method == APC_ICP_POINT_TO_POINT) icp_point_to_point(M, wk, U);
  else if (!icp_point_to_plane(M, wk, U)) status = APC_ICP_DEGENERATE;
  int32_t converged = 0;
  if (status == APC_ICP_OK) {
    double T[16];
    for (int r = 0; r < 4; ++r)
      for (int c = 0; c < 4; ++c)
        T[4 * r + c] = ((U[4 * r] * st->T[c] + U[4 * r + 1] * st->T[4 + c]) + U[4 * r + 2] * st->T[8 + c]) +
                       U[4 * r + 3] * st->T[12 + c];
    for (int k = 0; k < 16; ++k) st->T[k] = out_T[k] = T[k];
    st->iterations = iteration + 1;
    converged = iteration > 0 && fabs(st->prev_f - fitness) < relative_fitness && fabs(st->prev_r - rmse) < relative_rmse;
    st->prev_f = fitness;
    st->prev_r = rmse;
  }
  st->done = status != APC_ICP_OK || converged;
  out_info[0] = (int32_t)st->iterations;
  out_info[1] = converged;
  out_info[2] = status;
  out_info[3] = 0;
}

// Checks, scratch (allocated before the first launch), the call's begin, output initialisation and the target's
// grid.  *empty: one cloud has no points, nothing more to launch.
static int icp_begin(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const float* tgt_xyzi, uint32_t n_tgt,
                     const uint32_t* n_tgt_dev, double r, const double* T16_host, double* out_stats, int32_t* out_corr, float* out_d2,
                     double* out_T, int32_t* out_info, int32_t empty_status, bool* empty, cudaStream_t s) {
  APC_REQUIRE(ctx, src_xyzi && tgt_xyzi && T16_host && out_stats, "NULL pointer");
  APC_REQUIRE(ctx, n_src <= ctx->max_points && n_tgt <= ctx->max_points, "more points than the context was created for");
  const float r32 = (float)r;
  APC_REQUIRE(ctx, r > 0.0 && r32 > 0.0f && std::isfinite(r32 * r32), "max_correspondence_distance must be finite and > 0");
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  if (!sc->icp_part) APC_CUDA(ctx, cudaMalloc((void**)&sc->icp_part, (size_t)ICP_MAX_BLOCKS * 32 * sizeof(double)));
  if (!sc->icp_state) APC_CUDA(ctx, cudaMalloc((void**)&sc->icp_state, sizeof(IcpState)));
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  if (out_corr && n_src) APC_CUDA(ctx, cudaMemsetAsync(out_corr, 0xff, (size_t)n_src * sizeof(int32_t), s));
  if (out_d2 && n_src) APC_CUDA(ctx, cudaMemsetAsync(out_d2, 0, (size_t)n_src * sizeof(float), s));
  *empty = n_src == 0 || n_tgt == 0;
  IcpT16 init;
  memcpy(init.v, T16_host, sizeof(init.v));
  k_icp_init<<<1, 1, 0, s>>>(init, sc->icp_state, out_T, out_stats, out_info, *empty ? empty_status : APC_ICP_OK);
  APC_LAUNCH_CHECK(ctx, "k_icp_init");
  if (*empty) return APC_OK;
  // the grid of apc_cluster_dbscan / apc_estimate_normals_radius: cells of r * (1 + 2^-8), reciprocal indexing
  return grid_build(ctx, sc->grid[0], reinterpret_cast<const float4*>(tgt_xyzi), n_tgt, n_tgt_dev, r32 * 1.00390625f,
                    false, s, false, CTR_CURSOR_NORMALS, true);
}

static int icp_finish(apc_ctx* ctx, uint32_t n_tgt, const uint32_t* n_tgt_dev, cudaStream_t s) {
  const GridHost& g = scratch_of(ctx)->grid[0];
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<dim3(min(apc_div_up(n_tgt, 256), (uint32_t)APC_SM_COUNT * 4), 1), 256, 0, s>>>(n_tgt, n_tgt_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "icp");
  return APC_OK;
}

static uint32_t icp_blocks(uint32_t n_src) { return min(apc_div_up(n_src, 4), (uint32_t)ICP_MAX_BLOCKS); }

extern "C" int apc_evaluate_registration(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                                         const float* tgt_xyzi, uint32_t n_tgt, const uint32_t* n_tgt_dev,
                                         double max_correspondence_distance, const double* T16_host,
                                         int32_t* out_correspondences, float* out_d2, double* out_stats_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  bool empty = false;
  int rc = icp_begin(ctx, src_xyzi, n_src, tgt_xyzi, n_tgt, n_tgt_dev, max_correspondence_distance, T16_host, out_stats_dev,
                     out_correspondences, out_d2, nullptr, nullptr, APC_ICP_OK, &empty, s);
  if (rc || empty) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  const float r32 = (float)max_correspondence_distance;
  const uint32_t bq = icp_blocks(n_src);
  {
    APC_PROF(ctx, "k_icp_match", s);
    k_icp_match<<<bq, 128, 0, s>>>(reinterpret_cast<const float4*>(src_xyzi), n_src, n_src_dev,
                                   reinterpret_cast<const float4*>(tgt_xyzi), nullptr, sc->grid[0].d, r32 * r32,
                                   APC_ICP_POINT_TO_POINT, sc->icp_state, out_correspondences, out_d2, sc->icp_part);
  }
  {
    APC_PROF(ctx, "k_icp_solve", s);
    k_icp_solve<<<1, ICP_SOLVE_WARPS * 32, 0, s>>>(sc->icp_part, bq, n_src, n_src_dev, -1, 0, 0.0, 0.0, sc->icp_state, nullptr,
                                   out_stats_dev, nullptr);
  }
  return icp_finish(ctx, n_tgt, n_tgt_dev, s);
}

extern "C" int apc_icp(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                       const float* tgt_xyzi, const float* tgt_normals, uint32_t n_tgt, const uint32_t* n_tgt_dev,
                       double max_correspondence_distance, const double* init_T16_host, int method, int max_iteration,
                       double relative_fitness, double relative_rmse, double* out_T16_dev, double* out_stats_dev,
                       int32_t* out_info_dev, int32_t* out_correspondences, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, out_T16_dev && out_info_dev, "NULL pointer");
  APC_REQUIRE(ctx, max_iteration >= 0, "max_iteration must be >= 0");
  APC_REQUIRE(ctx, method == APC_ICP_POINT_TO_POINT || method == APC_ICP_POINT_TO_PLANE, "unknown ICP method");
  APC_REQUIRE(ctx, method != APC_ICP_POINT_TO_PLANE || tgt_normals, "point-to-plane ICP needs the target's normals");
  cudaStream_t s = (cudaStream_t)stream;
  bool empty = false;
  int rc = icp_begin(ctx, src_xyzi, n_src, tgt_xyzi, n_tgt, n_tgt_dev, max_correspondence_distance, init_T16_host, out_stats_dev,
                     out_correspondences, nullptr, out_T16_dev, out_info_dev,
                     max_iteration > 0 ? APC_ICP_NO_CORRESPONDENCE : APC_ICP_OK, &empty, s);
  if (rc || empty) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  const float r32 = (float)max_correspondence_distance;
  const uint32_t bq = icp_blocks(n_src);
  for (int j = 0; j < max_iteration; ++j) {
    {
      APC_PROF(ctx, "k_icp_match", s);
      k_icp_match<<<bq, 128, 0, s>>>(reinterpret_cast<const float4*>(src_xyzi), n_src, n_src_dev,
                                     reinterpret_cast<const float4*>(tgt_xyzi), tgt_normals, sc->grid[0].d, r32 * r32,
                                     method, sc->icp_state, out_correspondences, nullptr, sc->icp_part);
    }
    APC_PROF(ctx, "k_icp_solve", s);
    k_icp_solve<<<1, ICP_SOLVE_WARPS * 32, 0, s>>>(sc->icp_part, bq, n_src, n_src_dev, method, j, relative_fitness, relative_rmse,
                                   sc->icp_state, out_T16_dev, out_stats_dev, out_info_dev);
  }
  APC_LAUNCH_CHECK(ctx, "icp");
  return icp_finish(ctx, n_tgt, n_tgt_dev, s);
}

// ---- Generalized ICP (Open3D t::pipelines::registration::TransformationEstimationForGeneralizedICP) ------------
// Contract (oracle/gicp.py): matching, metrics, the loop and the solve are those of point-to-plane; only
// the per-correspondence system differs.  Every point's covariance gives one regularisation axis a (the
// eigenvector of its smallest eigenvalue, normal_from_covariance; NaN when an entry is not finite), and Segal's
// regularised covariance U diag(1, 1, eps) U^T is I - (1 - eps) a a^T.  For s' matched to t:
//   m = R a_s (R the upper-left 3x3 of the accumulated T), M = 2I - (1 - eps)(m m^T + a_t a_t^T), W = M^-1,
//   e = s' - t, J = [-[s']x | I]; H = sum J^T W J, b = sum J^T W e, then H x = -b as in point-to-plane.
//   k_gicp_prep       one thread per point of both clouds, once per call: covariance -> axis (context scratch)
//   k_icp_match_gicp  the matching of k_icp_match; lane k accumulates entry k of (n, sum d2, H, b) in
//                     point-to-plane's layout (c_icp_pairs[APC_ICP_POINT_TO_PLANE]), from s', m, a_t and e
//   k_icp_solve       unchanged, launched as point-to-plane
__global__ void __launch_bounds__(256)
k_gicp_prep(const float* __restrict__ src_cov, uint32_t n_src_max, const uint32_t* n_src_dev,
            const float* __restrict__ tgt_cov, uint32_t n_tgt_max, const uint32_t* n_tgt_dev, double* __restrict__ src_axes,
            double* __restrict__ tgt_axes, double* __restrict__ out_src_axes, double* __restrict__ out_tgt_axes) {
  const uint32_t ns = apc_count(n_src_dev, n_src_max), nt = apc_count(n_tgt_dev, n_tgt_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ns + nt; i += gridDim.x * blockDim.x) {
    const bool is_src = i < ns;
    const size_t k = is_src ? i : i - ns;
    const float* cov = (is_src ? src_cov : tgt_cov) + 9 * k;
    double C[9], a[3];
    bool finite = true;
#pragma unroll
    for (int u = 0; u < 9; ++u) {
      C[u] = cov[u];
      finite = finite && isfinite(C[u]);
    }
    if (finite) normal_from_covariance(C, a);
    else a[0] = a[1] = a[2] = __longlong_as_double(0x7ff8000000000000ll);
    double* axes = is_src ? src_axes : tgt_axes;
    double* out = is_src ? out_src_axes : out_tgt_axes;
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      axes[3 * k + u] = a[u];
      if (out) out[3 * k + u] = a[u];
    }
  }
}

__global__ void __launch_bounds__(128)
k_icp_match_gicp(const float4* __restrict__ src, uint32_t n_max, const uint32_t* n_dev, const float4* __restrict__ tgt,
                 const double* __restrict__ src_axes, const double* __restrict__ tgt_axes, GridDev g, float r2,
                 double one_minus_eps, const IcpState* __restrict__ st, int32_t* __restrict__ corr_out,
                 double* __restrict__ partials) {
  if (st->done) return;                                     // the loop has stopped: block-uniform
  __shared__ double sm[4][32];
  const uint32_t n = apc_count(n_dev, n_max);
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  // lane k: J_pa . W V_pb with V_b = J_b (b < 6) or e (b = 6); pa 7: n, pa 8: sum d2, pa 9: unused lanes
  const uint32_t pair = c_icp_pairs[APC_ICP_POINT_TO_PLANE][lane], pa = pair & 15u, pb = pair >> 4;
  double T[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) T[k] = st->T[k];
  double acc = 0.0;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += (gridDim.x * blockDim.x) >> 5) {
    const float4 p = src[i];
    const double x = p.x, y = p.y, z = p.z;
    const float4 q = make_float4(icp_row(T, 0, x, y, z), icp_row(T, 1, x, y, z), icp_row(T, 2, x, y, z), 0.0f);
    const uint64_t best = icp_best(g, c, q, r2, lane);
    const bool found = best != ~0ull;                       // warp-uniform
    const uint32_t j = (uint32_t)best;
    if (found) {
      const float4 t = tgt[j];
      const double sx = q.x, sy = q.y, sz = q.z;
      const double ex = sx - t.x, ey = sy - t.y, ez = sz - t.z;
      const double as0 = src_axes[3 * (size_t)i], as1 = src_axes[3 * (size_t)i + 1], as2 = src_axes[3 * (size_t)i + 2];
      const double a0 = tgt_axes[3 * (size_t)j], a1 = tgt_axes[3 * (size_t)j + 1], a2 = tgt_axes[3 * (size_t)j + 2];
      const double m0 = (T[0] * as0 + T[1] * as1) + T[2] * as2, m1 = (T[4] * as0 + T[5] * as1) + T[6] * as2,
                   m2 = (T[8] * as0 + T[9] * as1) + T[10] * as2;
      const double k = one_minus_eps;
      const double M00 = 2.0 - k * (m0 * m0 + a0 * a0), M11 = 2.0 - k * (m1 * m1 + a1 * a1),
                   M22 = 2.0 - k * (m2 * m2 + a2 * a2), M01 = -k * (m0 * m1 + a0 * a1), M02 = -k * (m0 * m2 + a0 * a2),
                   M12 = -k * (m1 * m2 + a1 * a2);
      // W = adj(M) / det(M)
      const double A00 = M11 * M22 - M12 * M12, A01 = M02 * M12 - M01 * M22, A02 = M01 * M12 - M02 * M11;
      const double inv = 1.0 / ((M00 * A00 + M01 * A01) + M02 * A02);
      const double W00 = A00 * inv, W01 = A01 * inv, W02 = A02 * inv, W11 = (M00 * M22 - M02 * M02) * inv,
                   W12 = (M01 * M02 - M00 * M12) * inv, W22 = (M00 * M11 - M01 * M01) * inv;
      // V_pb: J_b = e_b x s' (b < 3), the unit vector e_(b-3) (3 <= b < 6), or e (b = 6)
      const double vx = pb == 6 ? ex : pb == 3 ? 1.0 : pb == 1 ? sz : pb == 2 ? -sy : 0.0;
      const double vy = pb == 6 ? ey : pb == 4 ? 1.0 : pb == 0 ? -sz : pb == 2 ? sx : 0.0;
      const double vz = pb == 6 ? ez : pb == 5 ? 1.0 : pb == 0 ? sy : pb == 1 ? -sx : 0.0;
      const double wx = (W00 * vx + W01 * vy) + W02 * vz, wy = (W01 * vx + W11 * vy) + W12 * vz,
                   wz = (W02 * vx + W12 * vy) + W22 * vz;
      // J_a . w: (e_a x s') . w = (s' x w)_a for a < 3, w_(a-3) otherwise
      double val = pa == 0 ? sy * wz - sz * wy : pa == 1 ? sz * wx - sx * wz : pa == 2 ? sx * wy - sy * wx
                 : pa == 3 ? wx : pa == 4 ? wy : wz;
      val = pa == 7 ? 1.0 : pa == 8 ? (double)__uint_as_float((uint32_t)(best >> 32)) : pa == 9 ? 0.0 : val;
      acc += val;
    }
    if (lane == 0 && corr_out) corr_out[i] = found ? (int32_t)j : -1;
  }
  sm[warp][lane] = acc;
  __syncthreads();
  if (threadIdx.x < 32) partials[32 * (size_t)blockIdx.x + lane] = ((sm[0][lane] + sm[1][lane]) + sm[2][lane]) + sm[3][lane];
}

extern "C" int apc_icp_generalized(apc_ctx* ctx, const float* src_xyzi, const float* src_cov, uint32_t n_src,
                                   const uint32_t* n_src_dev, const float* tgt_xyzi, const float* tgt_cov, uint32_t n_tgt,
                                   const uint32_t* n_tgt_dev, double max_correspondence_distance,
                                   const double* init_T16_host, double epsilon, int max_iteration, double relative_fitness,
                                   double relative_rmse, double* out_T16_dev, double* out_stats_dev, int32_t* out_info_dev,
                                   int32_t* out_correspondences, double* out_src_axes_dev, double* out_tgt_axes_dev,
                                   void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, out_T16_dev && out_info_dev, "NULL pointer");
  APC_REQUIRE(ctx, max_iteration >= 0, "max_iteration must be >= 0");
  APC_REQUIRE(ctx, src_cov && tgt_cov, "generalized ICP needs the covariances of both clouds");
  APC_REQUIRE(ctx, std::isfinite(epsilon) && epsilon > 0.0, "epsilon must be finite and > 0");
  NeighborScratch* sc = scratch_of(ctx);
  for (double*& axes : sc->gicp_axes)       // before the first launch: the call can be captured in a graph
    if (!axes) APC_CUDA(ctx, cudaMalloc((void**)&axes, (size_t)ctx->max_points * 3 * sizeof(double)));
  cudaStream_t s = (cudaStream_t)stream;
  bool empty = false;
  int rc = icp_begin(ctx, src_xyzi, n_src, tgt_xyzi, n_tgt, n_tgt_dev, max_correspondence_distance, init_T16_host,
                     out_stats_dev, out_correspondences, nullptr, out_T16_dev, out_info_dev,
                     max_iteration > 0 ? APC_ICP_NO_CORRESPONDENCE : APC_ICP_OK, &empty, s);
  if (rc) return rc;
  if (out_src_axes_dev && n_src) APC_CUDA(ctx, cudaMemsetAsync(out_src_axes_dev, 0, (size_t)n_src * 3 * sizeof(double), s));
  if (out_tgt_axes_dev && n_tgt) APC_CUDA(ctx, cudaMemsetAsync(out_tgt_axes_dev, 0, (size_t)n_tgt * 3 * sizeof(double), s));
  if (empty) return APC_OK;
  {
    APC_PROF(ctx, "k_gicp_prep", s);
    k_gicp_prep<<<min(apc_div_up(n_src + n_tgt, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, s>>>(
        src_cov, n_src, n_src_dev, tgt_cov, n_tgt, n_tgt_dev, sc->gicp_axes[0], sc->gicp_axes[1], out_src_axes_dev,
        out_tgt_axes_dev);
  }
  const float r32 = (float)max_correspondence_distance;
  const uint32_t bq = icp_blocks(n_src);
  for (int j = 0; j < max_iteration; ++j) {
    {
      APC_PROF(ctx, "k_icp_match_gicp", s);
      k_icp_match_gicp<<<bq, 128, 0, s>>>(reinterpret_cast<const float4*>(src_xyzi), n_src, n_src_dev,
                                          reinterpret_cast<const float4*>(tgt_xyzi), sc->gicp_axes[0], sc->gicp_axes[1],
                                          sc->grid[0].d, r32 * r32, 1.0 - epsilon, sc->icp_state, out_correspondences,
                                          sc->icp_part);
    }
    APC_PROF(ctx, "k_icp_solve", s);
    k_icp_solve<<<1, ICP_SOLVE_WARPS * 32, 0, s>>>(sc->icp_part, bq, n_src, n_src_dev, APC_ICP_POINT_TO_PLANE, j,
                                                   relative_fitness, relative_rmse, sc->icp_state, out_T16_dev,
                                                   out_stats_dev, out_info_dev);
  }
  APC_LAUNCH_CHECK(ctx, "icp_generalized");
  return icp_finish(ctx, n_tgt, n_tgt_dev, s);
}

// ---- FPFH features (Open3D t::pipelines::registration::ComputeFPFHFeature) -----------------------------------
// Contract (oracle/features.py).  Neighbourhoods are those of the normals stage: hybrid (the max_nn nearest within
// float32(r)^2, k_normals_wide's walk) or KNN (the max_nn nearest, k_normals_knn's level climb + stragglers), kept
// through a WarpKeep of (d2 bits << 32 | index) keys and sorted, so entry 0 is at d2 = 0 (the query or a duplicate).
//   pass 0  the pair features (float64) of the query with entries 1..m-1 -> 33 bin counts in per-warp shared
//           counters (integer: order-free) -> SPFH = count * (100 / (m - 1)), float32
//   pass 1  the same search again (cheaper than storing n * max_nn lists); lane j sums spfh[k][j] / d2_k over the
//           entries with d2 > 0 in key order (float64), each group of 11 is scaled by 100 / its sum (the group sum
//           taken sequentially over the 11 bin totals), spfh[i] is added, float32
// One warp per query.  Points the grid cannot key are never queried: their SPFH, feature and count stay 0.
#define FPFH_BINS 33
#define FPFH_PI 3.141592653589793
#define FPFH_2PI 6.283185307179586

// Bins of Open3D's ComputePairFeatures(p1, n1, p2, n2) (float64); false when a feature is not finite (no bin).
// The swap test is |a1| < |a2| (Open3D: acos|a1| > acos|a2|, equal except where acos rounds two values together).
__device__ __forceinline__ bool fpfh_pair_bins(float4 p1, const double (&n1)[3], float4 p2, const double (&n2)[3],
                                               uint32_t& b0, uint32_t& b1, uint32_t& b2) {
  const double dx = (double)p2.x - (double)p1.x, dy = (double)p2.y - (double)p1.y, dz = (double)p2.z - (double)p1.z;
  const double d = sqrt((dx * dx + dy * dy) + dz * dz);
  double f0 = 0.0, f1 = 0.0, f2 = 0.0;
  if (d != 0.0) {
    const double a1 = ((n1[0] * dx + n1[1] * dy) + n1[2] * dz) / d;
    const double a2 = ((n2[0] * dx + n2[1] * dy) + n2[2] * dz) / d;
    const bool swap = fabs(a1) < fabs(a2);
    const double u0 = swap ? n2[0] : n1[0], u1 = swap ? n2[1] : n1[1], u2 = swap ? n2[2] : n1[2];
    const double t0 = swap ? n1[0] : n2[0], t1 = swap ? n1[1] : n2[1], t2 = swap ? n1[2] : n2[2];
    const double e0 = swap ? -dx : dx, e1 = swap ? -dy : dy, e2 = swap ? -dz : dz;
    double v0 = e1 * u2 - e2 * u1, v1 = e2 * u0 - e0 * u2, v2 = e0 * u1 - e1 * u0;
    const double vn = sqrt((v0 * v0 + v1 * v1) + v2 * v2);
    if (vn != 0.0) {
      f2 = swap ? -a2 : a1;
      v0 = v0 / vn; v1 = v1 / vn; v2 = v2 / vn;
      const double w0 = u1 * v2 - u2 * v1, w1 = u2 * v0 - u0 * v2, w2 = u0 * v1 - u1 * v0;
      f1 = (v0 * t0 + v1 * t1) + v2 * t2;
      f0 = atan2((w0 * t0 + w1 * t1) + w2 * t2, (u0 * t0 + u1 * t1) + u2 * t2);
    }
  }
  if (!(isfinite(f0) && isfinite(f1) && isfinite(f2))) return false;
  b0 = (uint32_t)fmin(fmax(floor((11.0 * (f0 + FPFH_PI)) / FPFH_2PI), 0.0), 10.0);
  b1 = (uint32_t)fmin(fmax(floor((11.0 * (f1 + 1.0)) * 0.5), 0.0), 10.0);
  b2 = (uint32_t)fmin(fmax(floor((11.0 * (f2 + 1.0)) * 0.5), 0.0), 10.0);
  return true;
}

// One query's pass over its sorted neighbourhood buf[0, m) (warp-collective).  cnt: this warp's 33 shared counters.
template <int PASS>
__device__ __forceinline__ void fpfh_of_keys(const unsigned long long* buf, uint32_t m, const float4* __restrict__ pts,
                                             const float* __restrict__ normals, float4 q, uint32_t orig, uint32_t lane,
                                             uint32_t* cnt, float* __restrict__ spfh, float* __restrict__ feat,
                                             uint32_t* __restrict__ counts) {
  if (PASS == 0) {
    cnt[lane] = 0u;
    if (lane == 0) cnt[32] = 0u;
    __syncwarp();
    const double n1[3] = {(double)normals[3 * (size_t)orig], (double)normals[3 * (size_t)orig + 1],
                          (double)normals[3 * (size_t)orig + 2]};
    for (uint32_t i = 1 + lane; i < m; i += 32) {
      const uint32_t k = (uint32_t)buf[i];
      const double n2[3] = {(double)normals[3 * (size_t)k], (double)normals[3 * (size_t)k + 1],
                            (double)normals[3 * (size_t)k + 2]};
      uint32_t b0, b1, b2;
      if (fpfh_pair_bins(q, n1, pts[k], n2, b0, b1, b2)) {
        atomicAdd(&cnt[b0], 1u);
        atomicAdd(&cnt[11u + b1], 1u);
        atomicAdd(&cnt[22u + b2], 1u);
      }
    }
    __syncwarp();
    const double incr = m > 1 ? 100.0 / (double)(m - 1) : 0.0;
    spfh[(size_t)FPFH_BINS * orig + lane] = (float)((double)cnt[lane] * incr);
    if (lane == 0) {
      spfh[(size_t)FPFH_BINS * orig + 32] = (float)((double)cnt[32] * incr);
      if (counts) counts[orig] = m;
    }
    __syncwarp();
  } else {
    double acc = 0.0, acc32 = 0.0;                               // lane j: bin j; lane 0 also bin 32
    for (uint32_t i = 1; i < m; ++i) {
      const unsigned long long key = buf[i];
      const float d2 = __uint_as_float((uint32_t)(key >> 32));
      if (d2 > 0.0f) {
        const float* row = spfh + (size_t)FPFH_BINS * (uint32_t)key;
        acc = acc + (double)row[lane] / (double)d2;
        if (lane == 0) acc32 = acc32 + (double)row[32] / (double)d2;
      }
    }
    double scale[3];
#pragma unroll
    for (int gidx = 0; gidx < 3; ++gidx) {
      double sum = __shfl_sync(0xffffffffu, acc, 11 * gidx);
      for (int t = 1; t < 11; ++t) {
        const int j = 11 * gidx + t;
        const double v = j < 32 ? __shfl_sync(0xffffffffu, acc, j) : __shfl_sync(0xffffffffu, acc32, 0);
        sum = sum + v;
      }
      scale[gidx] = sum != 0.0 ? 100.0 / sum : 0.0;
    }
    const float* own = spfh + (size_t)FPFH_BINS * orig;
    const double sl = lane < 11 ? scale[0] : lane < 22 ? scale[1] : scale[2];
    feat[(size_t)FPFH_BINS * orig + lane] = (float)(acc * sl + (double)own[lane]);
    if (lane == 0) feat[(size_t)FPFH_BINS * orig + 32] = (float)(acc32 * scale[2] + (double)own[32]);
  }
}

// Hybrid search: k_normals_wide's hybrid_keep, the kept keys sorted.
template <int PASS>
__global__ void __launch_bounds__(128)
k_fpfh_hybrid(uint32_t n_max, const uint32_t* n_dev, GridDev g, const float4* __restrict__ pts,
              const float* __restrict__ normals, float r2, uint32_t max_nn, uint32_t cap, float* __restrict__ spfh,
              float* __restrict__ feat, uint32_t* __restrict__ counts, const ApcCtrl* __restrict__ ctrl) {
  __shared__ uint32_t s_cnt[4][FPFH_BINS];
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)w * cap;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    const uint32_t m = hybrid_keep(g, c, q, r2, max_nn, buf, cap, lane);
    warp_sort(buf, m, lane);
    fpfh_of_keys<PASS>(buf, m, pts, normals, q, orig, lane, s_cnt[w], spfh, feat, counts);
    __syncwarp();                                                  // buf is reused by the next query
  }
}

// KNN search: k_normals_knn's level climb; pass 0 lists the queries no level covers, pass 1 reuses that list.
template <int PASS>
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_fpfh_knn(uint32_t n_max, const uint32_t* n_dev, GridDev g, const float4* __restrict__ pts, const float* __restrict__ normals,
           uint32_t k, uint32_t cap, float* __restrict__ spfh, float* __restrict__ feat, uint32_t* __restrict__ counts,
           uint32_t* __restrict__ stragglers, ApcCtrl* ctrl) {
  __shared__ uint32_t s_cnt[KNN_WARPS][FPFH_BINS];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t n_sorted = grid_sorted_count(g, ctrl, n);
  const uint32_t k_eff = min(k, n);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)w * cap;
  for (uint32_t j = blockIdx.x * KNN_WARPS + w; j < n_sorted; j += gridDim.x * KNN_WARPS) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (knn_levels(g, n_max, q, k_eff, buf, cap, lane)) {
      warp_sort(buf, k_eff, lane);
      fpfh_of_keys<PASS>(buf, k_eff, pts, normals, q, orig, lane, s_cnt[w], spfh, feat, counts);
    } else if (PASS == 0 && lane == 0) {
      stragglers[atomicAdd(&ctrl->counters[CTR_STRAGGLERS], 1u)] = orig;
    }
    __syncwarp();
  }
}

template <int PASS>
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_fpfh_knn_stragglers(const float4* __restrict__ pts, const float* __restrict__ normals, uint32_t n_max, const uint32_t* n_dev,
                      uint32_t k, uint32_t cap, const uint32_t* __restrict__ stragglers, const ApcCtrl* ctrl,
                      float* __restrict__ spfh, float* __restrict__ feat, uint32_t* __restrict__ counts) {
  __shared__ uint32_t s_cnt[KNN_WARPS][FPFH_BINS];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t k_eff = min(k, n);
  const uint32_t n_str = ctrl->counters[CTR_STRAGGLERS];
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(wide_smem) + (size_t)w * cap;
  for (uint32_t sidx = blockIdx.x * KNN_WARPS + w; sidx < n_str; sidx += gridDim.x * KNN_WARPS) {
    const uint32_t orig = stragglers[sidx];
    const float4 q = pts[orig];
    knn_brute(pts, n, q, k_eff, buf, cap, lane);
    warp_sort(buf, k_eff, lane);
    fpfh_of_keys<PASS>(buf, k_eff, pts, normals, q, orig, lane, s_cnt[w], spfh, feat, counts);
    __syncwarp();
  }
}

static int fpfh_run(apc_ctx* ctx, const float* xyzi, const float* normals, uint32_t n_max, const uint32_t* n_dev,
                    int max_nn, double radius, bool knn, float* out_features, float* out_spfh, uint32_t* out_counts,
                    cudaStream_t s) {
  APC_REQUIRE(ctx, max_nn >= 1 && max_nn <= APC_MAX_NEIGHBORS,
              "max_nn must be in 1..APC_MAX_NEIGHBORS (" APC_STRINGIFY(APC_MAX_NEIGHBORS) ")");
  const float r32 = (float)radius;
  if (!knn) APC_REQUIRE(ctx, radius > 0.0 && r32 > 0.0f && std::isfinite(r32 * r32), "radius must be finite and > 0");
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && normals && out_features, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  // everything is allocated before the first launch
  const int which = knn ? 1 : 0;
  int rc = apc_neighbors_prepare(ctx, which);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  if (!out_spfh && !sc->spfh) APC_CUDA(ctx, cudaMalloc((void**)&sc->spfh, (size_t)ctx->max_points * FPFH_BINS * sizeof(float)));
  float* spfh = out_spfh ? out_spfh : sc->spfh;
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(out_features, 0, (size_t)n_max * FPFH_BINS * sizeof(float), s));
  APC_CUDA(ctx, cudaMemsetAsync(spfh, 0, (size_t)n_max * FPFH_BINS * sizeof(float), s));
  if (out_counts) APC_CUDA(ctx, cudaMemsetAsync(out_counts, 0, (size_t)n_max * sizeof(uint32_t), s));
  GridHost& g = sc->grid[which];
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  if (knn) rc = grid_build(ctx, g, pts, n_max, n_dev, 0.0f, true, s);
  else rc = grid_build(ctx, g, pts, n_max, n_dev, r32 * 1.00390625f, false, s, false, CTR_CURSOR_NORMALS, true);
  if (rc) return rc;
  const uint32_t cap = wide_cap((uint32_t)max_nn);
  const size_t smem = (size_t)4 * cap * sizeof(unsigned long long);
  const uint32_t bq = min(apc_div_up(n_max, 4), (uint32_t)APC_SM_COUNT * 16);   // one warp per query, grid-stride
  if (knn) {
    {
      APC_PROF(ctx, "k_fpfh_knn_spfh", s);
      k_fpfh_knn<0><<<bq, KNN_WARPS * 32, smem, s>>>(n_max, n_dev, g.d, pts, normals, (uint32_t)max_nn, cap, spfh,
                                                     out_features, out_counts, sc->stragglers, ctx->ctrl);
    }
    {
      APC_PROF(ctx, "k_fpfh_knn_stragglers_spfh", s);
      k_fpfh_knn_stragglers<0><<<APC_SM_COUNT * 2, KNN_WARPS * 32, smem, s>>>(
          pts, normals, n_max, n_dev, (uint32_t)max_nn, cap, sc->stragglers, ctx->ctrl, spfh, out_features, out_counts);
    }
    {
      APC_PROF(ctx, "k_fpfh_knn", s);
      k_fpfh_knn<1><<<bq, KNN_WARPS * 32, smem, s>>>(n_max, n_dev, g.d, pts, normals, (uint32_t)max_nn, cap, spfh,
                                                     out_features, out_counts, sc->stragglers, ctx->ctrl);
    }
    {
      APC_PROF(ctx, "k_fpfh_knn_stragglers", s);
      k_fpfh_knn_stragglers<1><<<APC_SM_COUNT * 2, KNN_WARPS * 32, smem, s>>>(
          pts, normals, n_max, n_dev, (uint32_t)max_nn, cap, sc->stragglers, ctx->ctrl, spfh, out_features, out_counts);
    }
  } else {
    {
      APC_PROF(ctx, "k_fpfh_hybrid_spfh", s);
      k_fpfh_hybrid<0><<<bq, 128, smem, s>>>(n_max, n_dev, g.d, pts, normals, r32 * r32, (uint32_t)max_nn, cap, spfh,
                                             out_features, out_counts, ctx->ctrl);
    }
    {
      APC_PROF(ctx, "k_fpfh_hybrid", s);
      k_fpfh_hybrid<1><<<bq, 128, smem, s>>>(n_max, n_dev, g.d, pts, normals, r32 * r32, (uint32_t)max_nn, cap, spfh,
                                             out_features, out_counts, ctx->ctrl);
    }
  }
  APC_PROF(ctx, "k_grid_clean", s);
  k_grid_clean<<<dim3(min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 4), g.d.levels), 256, 0, s>>>(n_max, n_dev, g.d);
  APC_LAUNCH_CHECK(ctx, "compute_fpfh");
  return APC_OK;
}

extern "C" int apc_compute_fpfh(apc_ctx* ctx, const float* xyzi, const float* normals, uint32_t n_max, const uint32_t* n_dev,
                                int max_nn, double radius, float* out_features, float* out_spfh,
                                uint32_t* out_neighbor_counts, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  return fpfh_run(ctx, xyzi, normals, n_max, n_dev, max_nn, radius, false, out_features, out_spfh, out_neighbor_counts,
                  (cudaStream_t)stream);
}

extern "C" int apc_compute_fpfh_knn(apc_ctx* ctx, const float* xyzi, const float* normals, uint32_t n_max,
                                    const uint32_t* n_dev, int max_nn, float* out_features, float* out_spfh,
                                    uint32_t* out_neighbor_counts, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  return fpfh_run(ctx, xyzi, normals, n_max, n_dev, max_nn, 0.0, true, out_features, out_spfh, out_neighbor_counts,
                  (cudaStream_t)stream);
}

// ---- correspondences_from_features (Open3D t::pipelines::registration::CorrespondencesFromFeatures) ------------
// Contract (oracle/features.py): d2 = sum_j (a_j - b_j)^2 in float32, increasing j, unfused; a row's match is the
// other set's row with the smallest (d2, index) among the finite d2, none when no d2 is finite.  Brute force,
// O(n_a * n_b * dim) like Open3D's CUDA KNN:
//   k_feat_nn      one thread per query row (held in registers), the other set's rows through shared-memory tiles;
//                  the rows are split across blockIdx.y and the splits combine by a 64-bit atomicMin on
//                  (d2 bits << 32 | index), a total order, so the result does not depend on the schedule
//   k_feat_pairs   tiles of 1024 source rows in index order: the pairs (i, nn_st[i]) of the rows with a match and,
//                  with the mutual filter, of those with nn_ts[nn_st[i]] == i, compacted in order (apc_scan.cuh)
//   k_feat_select  the mutual set when it has more than ratio * n_src pairs, else the unfiltered set (fell_back)
#define FEAT_THREADS 128
#define FEAT_TILE 64

template <int DMAX>
__global__ void __launch_bounds__(FEAT_THREADS)
k_feat_nn(const float* __restrict__ a, uint32_t na_max, const uint32_t* na_dev, const float* __restrict__ b, uint32_t nb_max,
          const uint32_t* nb_dev, uint32_t dim, uint32_t rows_per_split, unsigned long long* __restrict__ best) {
  __shared__ float s_b[FEAT_TILE * DMAX];
  const uint32_t na = apc_count(na_dev, na_max), nb = apc_count(nb_dev, nb_max);
  const uint32_t i = blockIdx.x * FEAT_THREADS + threadIdx.x;
  const uint32_t t0 = blockIdx.y * rows_per_split, t1 = min(t0 + rows_per_split, nb);
  if (blockIdx.x * FEAT_THREADS >= na || t0 >= t1) return;       // block-uniform
  float q[DMAX];
#pragma unroll
  for (uint32_t d = 0; d < DMAX; ++d) q[d] = (i < na && d < dim) ? a[(size_t)i * dim + d] : 0.0f;
  unsigned long long key = ~0ull;
  for (uint32_t tb = t0; tb < t1; tb += FEAT_TILE) {
    const uint32_t rows = min((uint32_t)FEAT_TILE, t1 - tb);
    __syncthreads();
    for (uint32_t e = threadIdx.x; e < rows * dim; e += FEAT_THREADS) s_b[e] = b[(size_t)tb * dim + e];
    __syncthreads();
    for (uint32_t r = 0; r < rows; ++r) {
      const float* row = s_b + r * dim;
      float d2 = 0.0f;
#pragma unroll
      for (uint32_t d = 0; d < DMAX; ++d)
        if (d < dim) {
          const float x = __fsub_rn(q[d], row[d]);
          d2 = __fadd_rn(d2, __fmul_rn(x, x));
        }
      if (d2 <= 3.402823466e38f) key = min(key, ((unsigned long long)__float_as_uint(d2) << 32) | (tb + r));   // NaN, inf: never
    }
  }
  if (i < na && key != ~0ull) atomicMin(&best[i], key);
}

__global__ void __launch_bounds__(APC_TILE_THREADS)
k_feat_pairs(uint32_t n_max, const uint32_t* n_dev, const unsigned long long* __restrict__ best_st,
             const unsigned long long* __restrict__ best_ts, int32_t* __restrict__ nearest, int32_t* __restrict__ pairs_all,
             int32_t* __restrict__ pairs_mut, uint32_t* count2, uint64_t* state_all, uint64_t* state_mut,
             const ApcCtrl* ctrl, uint32_t n_tiles) {
  __shared__ uint32_t sm_all[34], sm_mut[34];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t tile = blockIdx.x;
  bool keep[APC_TILE_ITEMS], mut[APC_TILE_ITEMS];
  int32_t nn[APC_TILE_ITEMS];
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k) {
    const uint32_t i = tile * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x;
    nn[k] = (i < n && best_st[i] != ~0ull) ? (int32_t)(uint32_t)best_st[i] : -1;
    keep[k] = nn[k] >= 0;
    mut[k] = keep[k] && best_ts && best_ts[nn[k]] != ~0ull && (uint32_t)best_ts[nn[k]] == i;
    if (nearest && i < n_max) nearest[i] = nn[k];
  }
  uint32_t rank[APC_TILE_ITEMS];
  uint32_t base = tile_compact_offsets(keep, rank, sm_all, state_all, tile, ctrl->epoch, &count2[0], n_tiles);
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k)
    if (keep[k]) {
      pairs_all[2 * (size_t)(base + rank[k])] = (int32_t)(tile * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x);
      pairs_all[2 * (size_t)(base + rank[k]) + 1] = nn[k];
    }
  if (best_ts) {                                                   // block-uniform
    base = tile_compact_offsets(mut, rank, sm_mut, state_mut, tile, ctrl->epoch, &count2[1], n_tiles);
#pragma unroll
    for (int k = 0; k < APC_TILE_ITEMS; ++k)
      if (mut[k]) {
        pairs_mut[2 * (size_t)(base + rank[k])] = (int32_t)(tile * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x);
        pairs_mut[2 * (size_t)(base + rank[k]) + 1] = nn[k];
      }
  }
}

// Open3D keeps the mutual set when it has more than ratio * n_src pairs and otherwise warns and falls back.
__global__ void __launch_bounds__(256)
k_feat_select(uint32_t n_max, const uint32_t* n_dev, const uint32_t* __restrict__ count2, int mutual, double ratio,
              const int32_t* __restrict__ pairs_mut, int32_t* __restrict__ pairs, uint32_t* __restrict__ info) {
  const uint32_t n = apc_count(n_dev, n_max);
  const bool use_mut = mutual && (double)count2[1] > ratio * (double)n;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    info[0] = use_mut ? count2[1] : count2[0];
    info[1] = (mutual && !use_mut) ? 1u : 0u;
  }
  if (!use_mut) return;
  const uint32_t e_end = 2u * count2[1];
  for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < e_end; e += gridDim.x * blockDim.x) pairs[e] = pairs_mut[e];
}

static int feat_search(apc_ctx* ctx, const float* a, uint32_t na, const uint32_t* na_dev, const float* b, uint32_t nb,
                       const uint32_t* nb_dev, uint32_t dim, unsigned long long* best, cudaStream_t s) {
  APC_CUDA(ctx, cudaMemsetAsync(best, 0xff, (size_t)na * sizeof(unsigned long long), s));
  if (nb == 0) return APC_OK;
  const uint32_t blocks_a = apc_div_up(na, FEAT_THREADS), tiles_b = apc_div_up(nb, FEAT_TILE);
  const uint32_t splits = max(1u, min(apc_div_up(APC_SM_COUNT * 4, blocks_a), tiles_b));   // >= 4 blocks per SM
  const uint32_t rows_per_split = apc_div_up(tiles_b, splits) * FEAT_TILE;
  const dim3 grid(blocks_a, apc_div_up(nb, rows_per_split));
  APC_PROF(ctx, "k_feat_nn", s);
  if (dim <= 33) k_feat_nn<33><<<grid, FEAT_THREADS, 0, s>>>(a, na, na_dev, b, nb, nb_dev, dim, rows_per_split, best);
  else k_feat_nn<64><<<grid, FEAT_THREADS, 0, s>>>(a, na, na_dev, b, nb, nb_dev, dim, rows_per_split, best);
  return APC_OK;
}

extern "C" int apc_correspondences_from_features(apc_ctx* ctx, const float* src, uint32_t n_src, const uint32_t* n_src_dev,
                                                 const float* tgt, uint32_t n_tgt, const uint32_t* n_tgt_dev, int dim,
                                                 int mutual_filter, double ratio, int32_t* out_pairs,
                                                 int32_t* out_nearest, uint32_t* out_info_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, (src || !n_src) && (tgt || !n_tgt) && out_pairs && out_info_dev, "NULL pointer");   // empty: may be NULL
  APC_REQUIRE(ctx, dim >= 1 && dim <= 64, "dim must be in 1..64");
  APC_REQUIRE(ctx, std::isfinite(ratio) && ratio >= 0.0, "mutual_consistency_ratio must be finite and >= 0");
  APC_REQUIRE(ctx, n_src <= ctx->max_points && n_tgt <= ctx->max_points, "more rows than the context was created for");
  const uint32_t n_tiles = apc_div_up(n_src, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more rows than the context was created for");
  // everything is allocated before the first launch
  NeighborScratch* sc = scratch_of(ctx);
  const size_t M = ctx->max_points;
  for (auto& p : sc->feat_best)
    if (!p) APC_CUDA(ctx, cudaMalloc((void**)&p, M * sizeof(unsigned long long)));
  if (!sc->feat_pairs) APC_CUDA(ctx, cudaMalloc((void**)&sc->feat_pairs, M * 2 * sizeof(int32_t)));
  if (!sc->feat_count) APC_CUDA(ctx, cudaMalloc((void**)&sc->feat_count, 2 * sizeof(uint32_t)));
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(out_info_dev, 0, 2 * sizeof(uint32_t), s));
  if (n_src == 0) return APC_OK;
  // rows no pair reaches (source rows without a match) read as -1 rather than as whatever the buffer held
  APC_CUDA(ctx, cudaMemsetAsync(out_pairs, 0xff, (size_t)n_src * 2 * sizeof(int32_t), s));
  rc = feat_search(ctx, src, n_src, n_src_dev, tgt, n_tgt, n_tgt_dev, (uint32_t)dim, sc->feat_best[0], s);
  if (rc) return rc;
  const bool mutual = mutual_filter != 0;
  if (mutual && n_tgt) {
    rc = feat_search(ctx, tgt, n_tgt, n_tgt_dev, src, n_src, n_src_dev, (uint32_t)dim, sc->feat_best[1], s);
    if (rc) return rc;
  }
  {
    APC_PROF(ctx, "k_feat_pairs", s);
    k_feat_pairs<<<n_tiles, APC_TILE_THREADS, 0, s>>>(n_src, n_src_dev, sc->feat_best[0],
                                                      (mutual && n_tgt) ? sc->feat_best[1] : nullptr, out_nearest,
                                                      out_pairs, sc->feat_pairs, sc->feat_count, ctx->scan_state[0],
                                                      ctx->scan_state[1], ctx->ctrl, n_tiles);
  }
  if (mutual && !n_tgt) APC_CUDA(ctx, cudaMemsetAsync(sc->feat_count + 1, 0, sizeof(uint32_t), s));
  APC_PROF(ctx, "k_feat_select", s);
  k_feat_select<<<min(apc_div_up(2 * n_src, 256), (uint32_t)APC_SM_COUNT * 4), 256, 0, s>>>(
      n_src, n_src_dev, sc->feat_count, mutual ? 1 : 0, ratio, sc->feat_pairs, out_pairs, out_info_dev);
  APC_LAUNCH_CHECK(ctx, "correspondences_from_features");
  return APC_OK;
}

// ---- Fast Global Registration (Open3D pipelines::registration::FastGlobalRegistration) ---------------------------
// Contract (oracle/fgr.py): the pairs (the mutual set of the feature search, or the caller's in-range pairs), the
// tuple test on a counter-based stream, normalisation by the means of both clouds and the largest centred norm D,
// then iteration_number Gauss-Newton steps of sum s |p - T q|^2 with s = (par / (|r|^2 + par))^2 and the
// graduated par, and finally the inverse of T in metres.
//   k_fgr_pairs    (apc_fgr) tiles of 1024 input pairs in order: the pairs with both indices inside their clouds,
//                  compacted in order (apc_scan.cuh); the others are dropped
//   k_fgr_tuples   tiles of `steps` x 1024 trials in trial order: each trial draws its three pairs (splitmix64_dev)
//                  and tests the edge ratios in float64; the tile's accept ballots stay in shared memory while one
//                  cross-tile scan places the tile, then the first maximum_tuple_count accepted tuples are written
//   k_fgr_norm     one block: means and D of both clouds in a fixed order, par, T = I, TOO_FEW
//   k_fgr_accum    one warp per pair, grid-stride: q' = T q, r, s; lane k accumulates moment k of the three axes'
//                  rows in point-to-plane's layout (c_icp_pairs[APC_ICP_POINT_TO_PLANE]); block rows of 32 partials
//   k_icp_solve    unchanged, launched as point-to-plane without a convergence test: T = update T, or DEGENERATE
//   k_fgr_final    the inverse in metres and the info
// iteration_number (accum, solve) pairs are launched up front and return at once after a DEGENERATE step, so the call
// makes no host synchronisation.  Launch configurations depend on host sizes only and every sum has a fixed order.
#define FGR_TRIALS_PER_PAIR 100u
#define FGR_MIN_PAIRS 10u
#define FGR_TUPLE_MAX_STEPS 128u   // a tile of tuple trials holds at most 128 x 1024 (16 KB of ballots)

struct FgrState {
  double mu_s[3], mu_t[3];
  double g, par0;
  uint32_t used, accepted, trials;
  double icp_T[16], icp_stats[2];   // outputs of k_icp_solve
  int32_t icp_info[4];
};

__global__ void __launch_bounds__(APC_TILE_THREADS)
k_fgr_pairs(const int32_t* __restrict__ in, uint32_t n_max, const uint32_t* n_dev, uint32_t n_src_max,
            const uint32_t* n_src_dev, uint32_t n_tgt_max, const uint32_t* n_tgt_dev, int32_t* __restrict__ out,
            uint32_t* count, uint64_t* state, const ApcCtrl* ctrl, uint32_t n_tiles) {
  __shared__ uint32_t sm[34];
  const uint32_t n = apc_count(n_dev, n_max), ns = apc_count(n_src_dev, n_src_max), nt = apc_count(n_tgt_dev, n_tgt_max);
  bool keep[APC_TILE_ITEMS];
  int32_t a[APC_TILE_ITEMS], b[APC_TILE_ITEMS];
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k) {
    const uint32_t e = blockIdx.x * APC_TILE_POINTS + k * APC_TILE_THREADS + threadIdx.x;
    a[k] = b[k] = -1;
    if (e < n) {
      a[k] = in[2 * (size_t)e];
      b[k] = in[2 * (size_t)e + 1];
    }
    keep[k] = a[k] >= 0 && (uint32_t)a[k] < ns && b[k] >= 0 && (uint32_t)b[k] < nt;
  }
  uint32_t rank[APC_TILE_ITEMS];
  const uint32_t base = tile_compact_offsets(keep, rank, sm, state, blockIdx.x, ctrl->epoch, count, n_tiles);
#pragma unroll
  for (int k = 0; k < APC_TILE_ITEMS; ++k)
    if (keep[k]) {
      out[2 * (size_t)(base + rank[k])] = a[k];
      out[2 * (size_t)(base + rank[k]) + 1] = b[k];
    }
}

__device__ __forceinline__ uint32_t fgr_draw(uint64_t seed, uint32_t t, uint32_t k, uint32_t K) {
  const uint64_t z = splitmix64_dev(seed + ((uint64_t)t << 32) + k);
  return (uint32_t)(((z >> 32) * (uint64_t)K) >> 32);
}
// sqrt((dx*dx + dy*dy) + dz*dz) in float64, unfused
__device__ __forceinline__ double fgr_len(float4 a, float4 b) {
  const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y), dz = __dsub_rn(a.z, b.z);
  return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}
__device__ __forceinline__ bool fgr_accept(const float4* __restrict__ src, const float4* __restrict__ tgt,
                                           const int32_t* __restrict__ pairs, uint64_t seed, uint32_t t, uint32_t K,
                                           double scale) {
  float4 p[3], q[3];
#pragma unroll
  for (uint32_t k = 0; k < 3; ++k) {
    const uint32_t c = fgr_draw(seed, t, k, K);
    p[k] = src[pairs[2 * (size_t)c]];
    q[k] = tgt[pairs[2 * (size_t)c + 1]];
  }
  bool ok = true;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const double li = fgr_len(p[e], p[(e + 1) % 3]), lj = fgr_len(q[e], q[(e + 1) % 3]);
    ok = ok && __dmul_rn(li, scale) < lj && lj < __ddiv_rn(li, scale);
  }
  return ok;
}

// Trial t of tile b is item j (0..3) of thread x at step u: t = (b * steps + u) * 1024 + j * 256 + x, so ballot word
// w = u * 32 + j * 8 + warp holds the trials w * 32 + lane of the tile, and word order is trial order.
__global__ void __launch_bounds__(256)
k_fgr_tuples(const float4* __restrict__ src, const float4* __restrict__ tgt, const int32_t* __restrict__ pairs,
             const uint32_t* K_dev, uint32_t K_max, uint32_t steps, uint64_t seed, double scale, uint32_t max_count,
             int32_t* __restrict__ out, FgrState* __restrict__ fst, uint64_t* state, const ApcCtrl* ctrl, uint32_t n_tiles) {
  __shared__ uint32_t bits[FGR_TUPLE_MAX_STEPS * 32], before[FGR_TUPLE_MAX_STEPS * 32];
  __shared__ uint32_t sm_total, sm_scan;
  const uint32_t K = apc_count(K_dev, K_max), n_trials = FGR_TRIALS_PER_PAIR * K;
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, words = steps * 32u;
  const uint32_t t0 = blockIdx.x * steps * 1024u;
  for (uint32_t u = 0; u < steps; ++u)
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) {
      const uint32_t t = t0 + u * 1024u + j * 256u + threadIdx.x;
      const uint32_t b = __ballot_sync(0xffffffffu, t < n_trials && fgr_accept(src, tgt, pairs, seed, t, K, scale));
      if (lane == 0) bits[u * 32u + j * 8u + warp] = b;
    }
  __syncthreads();
  if (warp == 0) {                                  // exclusive prefix of the words' counts, in word order
    uint32_t carry = 0;
    for (uint32_t w0 = 0; w0 < words; w0 += 32) {
      const uint32_t c = __popc(bits[w0 + lane]);
      uint32_t incl = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += v;
      }
      before[w0 + lane] = carry + incl - c;
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) sm_total = carry;
  }
  __syncthreads();
  const uint32_t total = sm_total;
  const uint32_t excl = scan_two_level(state, blockIdx.x, n_tiles, ctrl->epoch, total, &sm_scan);
  if (blockIdx.x == n_tiles - 1 && threadIdx.x == 0) fst->accepted = excl + total;
  if (excl >= max_count) return;                    // block-uniform
  for (uint32_t u = 0; u < steps; ++u)
    for (uint32_t j = 0; j < 4; ++j) {
      const uint32_t w = u * 32u + j * 8u + warp, word = bits[w];
      if (!((word >> lane) & 1u)) continue;
      const uint32_t rank = excl + before[w] + __popc(word & ((1u << lane) - 1u));
      if (rank >= max_count) continue;
      const uint32_t t = t0 + u * 1024u + j * 256u + threadIdx.x;
      for (uint32_t k = 0; k < 3; ++k) {
        const uint32_t c = fgr_draw(seed, t, k, K);
        out[2 * (3 * (size_t)rank + k)] = pairs[2 * (size_t)c];
        out[2 * (3 * (size_t)rank + k) + 1] = pairs[2 * (size_t)c + 1];
      }
      if (rank == max_count - 1) fst->trials = t + 1;
    }
}

// block-wide reductions of k_fgr_norm (1024 threads) in a fixed order; the max propagates NaN
__device__ __forceinline__ double fgr_max_nan(double a, double b) { return (b > a || b != b) ? b : a; }
template <bool MAX>
__device__ __forceinline__ double fgr_block_reduce(double v, double* sm) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const double x = __shfl_down_sync(0xffffffffu, v, o);
    v = MAX ? fgr_max_nan(v, x) : v + x;
  }
  __syncthreads();                                  // sm is reused by the next reduction
  if (lane == 0) sm[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = sm[lane];
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const double x = __shfl_down_sync(0xffffffffu, v, o);
      v = MAX ? fgr_max_nan(v, x) : v + x;
    }
    if (lane == 0) sm[32] = v;
  }
  __syncthreads();
  return sm[32];
}

__global__ void __launch_bounds__(1024)
k_fgr_norm(const float4* __restrict__ src, uint32_t n_src_max, const uint32_t* n_src_dev, const float4* __restrict__ tgt,
           uint32_t n_tgt_max, const uint32_t* n_tgt_dev, const uint32_t* K_dev, uint32_t K_max, int tuple_test,
           uint32_t max_count, int absolute, FgrState* __restrict__ fst, IcpState* __restrict__ ist) {
  __shared__ double sm[33];
  const float4* pts[2] = {src, tgt};
  const uint32_t n[2] = {apc_count(n_src_dev, n_src_max), apc_count(n_tgt_dev, n_tgt_max)};
  double mu[2][3], dmax = 0.0;
  for (int c = 0; c < 2; ++c) {
    double sx = 0.0, sy = 0.0, sz = 0.0;
    for (uint32_t i = threadIdx.x; i < n[c]; i += blockDim.x) {
      const float4 p = pts[c][i];
      sx += p.x; sy += p.y; sz += p.z;
    }
    mu[c][0] = fgr_block_reduce<false>(sx, sm) / (double)n[c];
    mu[c][1] = fgr_block_reduce<false>(sy, sm) / (double)n[c];
    mu[c][2] = fgr_block_reduce<false>(sz, sm) / (double)n[c];
    for (uint32_t i = threadIdx.x; i < n[c]; i += blockDim.x) {
      const float4 p = pts[c][i];
      const double dx = p.x - mu[c][0], dy = p.y - mu[c][1], dz = p.z - mu[c][2];
      dmax = fgr_max_nan(dmax, sqrt((dx * dx + dy * dy) + dz * dz));
    }
  }
  const double D = fgr_block_reduce<true>(dmax, sm);
  if (threadIdx.x) return;
  const uint32_t K = apc_count(K_dev, K_max);
  const uint32_t used = tuple_test ? 3u * min(fst->accepted, max_count) : K;
  for (int k = 0; k < 3; ++k) {
    fst->mu_s[k] = mu[0][k];
    fst->mu_t[k] = mu[1][k];
  }
  fst->g = absolute ? 1.0 : D;
  fst->par0 = absolute ? D : 1.0;
  fst->used = used;
  for (int k = 0; k < 16; ++k) ist->T[k] = (k % 5 == 0) ? 1.0 : 0.0;
  ist->prev_f = ist->prev_r = 0.0;
  ist->done = used < FGR_MIN_PAIRS;
  ist->iterations = 0;
}

__global__ void __launch_bounds__(128)
k_fgr_accum(const float4* __restrict__ src, const float4* __restrict__ tgt, const int32_t* __restrict__ pairs,
            const FgrState* __restrict__ fst, const IcpState* __restrict__ ist, int iteration, int decrease_mu,
            double max_corr, double division_factor, double* __restrict__ partials) {
  if (ist->done) return;                                    // block-uniform
  __shared__ double sm[4][32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t pair = c_icp_pairs[APC_ICP_POINT_TO_PLANE][lane], pa = pair & 15u, pb = pair >> 4;
  double par = fst->par0;                                   // the schedule's steps at 0, 4, 8, ... <= iteration
  if (decrease_mu)
    for (int j = 0; j <= iteration && par > max_corr; j += 4) par /= division_factor;
  const double g = fst->g;
  const double ms[3] = {fst->mu_s[0], fst->mu_s[1], fst->mu_s[2]}, mt[3] = {fst->mu_t[0], fst->mu_t[1], fst->mu_t[2]};
  double T[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) T[k] = ist->T[k];
  const uint32_t n = fst->used;
  double acc = 0.0;
  for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += (gridDim.x * blockDim.x) >> 5) {
    const float4 ps = src[pairs[2 * (size_t)i]], pt = tgt[pairs[2 * (size_t)i + 1]];
    const double p[3] = {(ps.x - ms[0]) / g, (ps.y - ms[1]) / g, (ps.z - ms[2]) / g};
    const double q[3] = {(pt.x - mt[0]) / g, (pt.y - mt[1]) / g, (pt.z - mt[2]) / g};
    double qt[3], r[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      qt[a] = ((T[4 * a] * q[0] + T[4 * a + 1] * q[1]) + T[4 * a + 2] * q[2]) + T[4 * a + 3];
      r[a] = p[a] - qt[a];
    }
    double s = par / (((r[0] * r[0] + r[1] * r[1]) + r[2] * r[2]) + par);
    s = s * s;
    const double w = lane == 0 ? 1.0 : s;                   // lane 0 counts the pairs
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      double v[10] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, r[a], 1.0, 0.0, 0.0};
      if (a == 0) { v[1] = -qt[2]; v[2] = qt[1]; v[3] = -1.0; }
      if (a == 1) { v[0] = qt[2]; v[2] = -qt[0]; v[4] = -1.0; }
      if (a == 2) { v[0] = -qt[1]; v[1] = qt[0]; v[5] = -1.0; }
      acc += w * (icp_pick(v, pa) * icp_pick(v, pb));
    }
  }
  sm[warp][lane] = acc;
  __syncthreads();
  if (threadIdx.x < 32) partials[32 * (size_t)blockIdx.x + lane] = ((sm[0][lane] + sm[1][lane]) + sm[2][lane]) + sm[3][lane];
}

// rotation R^T, translation mu_t - R^T mu_s - g R^T t of the normalised T = [R | t]
__global__ void k_fgr_final(const FgrState* __restrict__ fst, const IcpState* __restrict__ ist, const uint32_t* in_dev,
                            uint32_t in_max, const uint32_t* K_dev, uint32_t K_max, int tuple_test, uint32_t max_count,
                            double* __restrict__ out_T, int32_t* __restrict__ out_info) {
  const uint32_t K = apc_count(K_dev, K_max), in = apc_count(in_dev, in_max);
  const bool too_few = fst->used < FGR_MIN_PAIRS;
  const double* T = ist->T;
  double R[3][3], t[3];
  for (int a = 0; a < 3; ++a) {
    for (int b = 0; b < 3; ++b) R[a][b] = too_few ? (a == b ? 1.0 : 0.0) : T[4 * b + a];     // R^T
    t[a] = T[4 * a + 3];
  }
  for (int a = 0; a < 3; ++a) {
    const double rs = (R[a][0] * fst->mu_s[0] + R[a][1] * fst->mu_s[1]) + R[a][2] * fst->mu_s[2];
    const double rt = (R[a][0] * t[0] + R[a][1] * t[1]) + R[a][2] * t[2];
    for (int b = 0; b < 3; ++b) out_T[4 * a + b] = R[a][b];
    out_T[4 * a + 3] = too_few ? 0.0 : (fst->mu_t[a] - rs) - fst->g * rt;
    out_T[12 + a] = 0.0;
  }
  out_T[15] = 1.0;
  out_info[0] = too_few ? 0 : (int32_t)ist->iterations;
  out_info[1] = (int32_t)in;
  out_info[2] = (int32_t)fst->used;
  out_info[3] = too_few ? APC_FGR_TOO_FEW : (fst->icp_info[2] == APC_ICP_DEGENERATE ? APC_FGR_DEGENERATE : APC_FGR_OK);
  out_info[4] = !tuple_test ? 0 : (int32_t)(fst->accepted >= max_count ? fst->trials : FGR_TRIALS_PER_PAIR * K);
  out_info[5] = (int32_t)(in - K);
}

static int fgr_check(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const float* tgt_xyzi, uint32_t n_tgt,
                     double division_factor, double max_corr, int iteration_number, double* out_T16_dev,
                     int32_t* out_info_dev) {
  APC_REQUIRE(ctx, (src_xyzi || !n_src) && (tgt_xyzi || !n_tgt) && out_T16_dev && out_info_dev, "NULL pointer");
  APC_REQUIRE(ctx, n_src <= ctx->max_points && n_tgt <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, std::isfinite(division_factor) && division_factor > 1.0, "division_factor must be finite and > 1");
  APC_REQUIRE(ctx, std::isfinite(max_corr) && max_corr > 0.0, "maximum_correspondence_distance must be finite and > 0");
  APC_REQUIRE(ctx, iteration_number >= 0, "iteration_number must be >= 0");
  return APC_OK;
}

// Scratch (allocated before the first launch): the pairs of the feature search, the used pairs, the loop's state.
static int fgr_scratch(apc_ctx* ctx) {
  NeighborScratch* sc = scratch_of(ctx);
  const size_t M = ctx->max_points;
  if (!sc->feat_pairs) APC_CUDA(ctx, cudaMalloc((void**)&sc->feat_pairs, M * 2 * sizeof(int32_t)));
  if (!sc->feat_count) APC_CUDA(ctx, cudaMalloc((void**)&sc->feat_count, 2 * sizeof(uint32_t)));
  if (!sc->fgr_pairs) APC_CUDA(ctx, cudaMalloc((void**)&sc->fgr_pairs, 3 * M * 2 * sizeof(int32_t)));
  if (!sc->fgr_state) APC_CUDA(ctx, cudaMalloc((void**)&sc->fgr_state, sizeof(FgrState)));
  if (!sc->icp_part) APC_CUDA(ctx, cudaMalloc((void**)&sc->icp_part, (size_t)ICP_MAX_BLOCKS * 32 * sizeof(double)));
  if (!sc->icp_state) APC_CUDA(ctx, cudaMalloc((void**)&sc->icp_state, sizeof(IcpState)));
  return APC_OK;
}

// Everything after the pairs: sc->feat_pairs holds K = feat_count[1] (<= K_max) pairs, in = the pairs before
// dropping.  The tuple test runs when max_count > 0.
static int fgr_run(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev, const float* tgt_xyzi,
                   uint32_t n_tgt, const uint32_t* n_tgt_dev, uint32_t K_max, const uint32_t* in_dev, uint32_t in_max,
                   double division_factor, int absolute, int decrease_mu, double max_corr, int iteration_number,
                   double tuple_scale, uint32_t max_count, uint64_t seed, double* out_T16_dev, int32_t* out_info_dev,
                   int32_t* out_pairs_used, cudaStream_t s) {
  NeighborScratch* sc = scratch_of(ctx);
  FgrState* fst = sc->fgr_state;
  const float4* src = reinterpret_cast<const float4*>(src_xyzi);
  const float4* tgt = reinterpret_cast<const float4*>(tgt_xyzi);
  const uint32_t* K_dev = sc->feat_count + 1;
  const bool tuple_test = max_count > 0;
  const int32_t* used = sc->feat_pairs;
  uint32_t used_max = K_max;
  if (tuple_test) {
    int32_t* out = out_pairs_used ? out_pairs_used : sc->fgr_pairs;
    const uint64_t trials = (uint64_t)FGR_TRIALS_PER_PAIR * K_max;
    uint32_t steps = 1;
    while ((trials + steps * 1024ull - 1) / (steps * 1024ull) > ctx->max_tiles) steps *= 2;
    APC_REQUIRE(ctx, steps <= FGR_TUPLE_MAX_STEPS, "more pairs than the context can test");
    const uint32_t n_tiles = (uint32_t)((trials + steps * 1024ull - 1) / (steps * 1024ull));
    if (n_tiles) {
      APC_PROF(ctx, "k_fgr_tuples", s);
      k_fgr_tuples<<<n_tiles, 256, 0, s>>>(src, tgt, sc->feat_pairs, K_dev, K_max, steps, seed, tuple_scale, max_count,
                                           out, fst, ctx->scan_state[2], ctx->ctrl, n_tiles);
    }
    used = out;
    used_max = 3 * max_count;
  } else if (out_pairs_used && K_max) {
    APC_CUDA(ctx, cudaMemcpyAsync(out_pairs_used, sc->feat_pairs, (size_t)K_max * 2 * sizeof(int32_t),
                                  cudaMemcpyDeviceToDevice, s));
  }
  {
    APC_PROF(ctx, "k_fgr_norm", s);
    k_fgr_norm<<<1, 1024, 0, s>>>(src, n_src, n_src_dev, tgt, n_tgt, n_tgt_dev, K_dev, K_max, tuple_test ? 1 : 0,
                                  max_count, absolute, fst, sc->icp_state);
  }
  const uint32_t bq = min(apc_div_up(used_max, 4), (uint32_t)ICP_MAX_BLOCKS);
  for (int j = 0; bq && j < iteration_number; ++j) {
    {
      APC_PROF(ctx, "k_fgr_accum", s);
      k_fgr_accum<<<bq, 128, 0, s>>>(src, tgt, used, fst, sc->icp_state, j, decrease_mu, max_corr, division_factor,
                                     sc->icp_part);
    }
    APC_PROF(ctx, "k_icp_solve", s);
    k_icp_solve<<<1, ICP_SOLVE_WARPS * 32, 0, s>>>(sc->icp_part, bq, 1, nullptr, APC_ICP_POINT_TO_PLANE, j, -1.0, -1.0,
                                                   sc->icp_state, fst->icp_T, fst->icp_stats, fst->icp_info);
  }
  APC_PROF(ctx, "k_fgr_final", s);
  k_fgr_final<<<1, 1, 0, s>>>(fst, sc->icp_state, in_dev, in_max, K_dev, K_max, tuple_test ? 1 : 0, max_count,
                              out_T16_dev, out_info_dev);
  APC_LAUNCH_CHECK(ctx, "fgr");
  return APC_OK;
}

extern "C" int apc_fgr_from_features(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                                     const float* tgt_xyzi, uint32_t n_tgt, const uint32_t* n_tgt_dev,
                                     const float* src_feat, const float* tgt_feat, int dim, double division_factor,
                                     int use_absolute_scale, int decrease_mu, double maximum_correspondence_distance,
                                     int iteration_number, double tuple_scale, int maximum_tuple_count, int tuple_test,
                                     uint64_t seed, double* out_T16_dev, int32_t* out_info_dev,
                                     int32_t* out_pairs_used, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  int rc = fgr_check(ctx, src_xyzi, n_src, tgt_xyzi, n_tgt, division_factor, maximum_correspondence_distance,
                     iteration_number, out_T16_dev, out_info_dev);
  if (rc) return rc;
  APC_REQUIRE(ctx, (src_feat || !n_src) && (tgt_feat || !n_tgt), "NULL pointer");
  APC_REQUIRE(ctx, dim >= 1 && dim <= 64, "dim must be in 1..64");
  APC_REQUIRE(ctx, tuple_scale > 0.0 && tuple_scale <= 1.0, "tuple_scale must be in (0, 1]");
  APC_REQUIRE(ctx, maximum_tuple_count >= 1 && (uint32_t)maximum_tuple_count <= ctx->max_points,
              "maximum_tuple_count must be in 1..max_points");
  const uint32_t n_tiles = apc_div_up(n_src, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more rows than the context was created for");
  NeighborScratch* sc = scratch_of(ctx);
  for (auto& p : sc->feat_best)
    if (!p) APC_CUDA(ctx, cudaMalloc((void**)&p, (size_t)ctx->max_points * sizeof(unsigned long long)));
  rc = fgr_scratch(ctx);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(sc->fgr_state, 0, sizeof(FgrState), s));
  APC_CUDA(ctx, cudaMemsetAsync(sc->feat_count, 0, 2 * sizeof(uint32_t), s));
  if (n_src && n_tgt) {
    rc = feat_search(ctx, src_feat, n_src, n_src_dev, tgt_feat, n_tgt, n_tgt_dev, (uint32_t)dim, sc->feat_best[0], s);
    if (!rc) rc = feat_search(ctx, tgt_feat, n_tgt, n_tgt_dev, src_feat, n_src, n_src_dev, (uint32_t)dim, sc->feat_best[1], s);
    if (rc) return rc;
    APC_PROF(ctx, "k_feat_pairs", s);
    k_feat_pairs<<<n_tiles, APC_TILE_THREADS, 0, s>>>(n_src, n_src_dev, sc->feat_best[0], sc->feat_best[1], nullptr,
                                                      sc->fgr_pairs, sc->feat_pairs, sc->feat_count, ctx->scan_state[0],
                                                      ctx->scan_state[1], ctx->ctrl, n_tiles);
  }
  const uint32_t K_max = n_tgt ? n_src : 0;
  return fgr_run(ctx, src_xyzi, n_src, n_src_dev, tgt_xyzi, n_tgt, n_tgt_dev, K_max, sc->feat_count + 1, K_max,
                 division_factor, use_absolute_scale ? 1 : 0, decrease_mu ? 1 : 0, maximum_correspondence_distance,
                 iteration_number, tuple_scale, tuple_test ? (uint32_t)maximum_tuple_count : 0u, seed, out_T16_dev,
                 out_info_dev, out_pairs_used, s);
}

extern "C" int apc_fgr(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                       const float* tgt_xyzi, uint32_t n_tgt, const uint32_t* n_tgt_dev, const int32_t* pairs,
                       uint32_t n_pairs, const uint32_t* n_pairs_dev, double division_factor, int use_absolute_scale,
                       int decrease_mu, double maximum_correspondence_distance, int iteration_number,
                       double* out_T16_dev, int32_t* out_info_dev, int32_t* out_pairs_used, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  int rc = fgr_check(ctx, src_xyzi, n_src, tgt_xyzi, n_tgt, division_factor, maximum_correspondence_distance,
                     iteration_number, out_T16_dev, out_info_dev);
  if (rc) return rc;
  APC_REQUIRE(ctx, pairs || !n_pairs, "NULL pointer");
  APC_REQUIRE(ctx, n_pairs <= ctx->max_points, "more pairs than the context was created for");
  const uint32_t n_tiles = apc_div_up(n_pairs, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more pairs than the context was created for");
  rc = fgr_scratch(ctx);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  cudaStream_t s = (cudaStream_t)stream;
  rc = apc_begin(ctx, s);
  if (rc) return rc;
  APC_CUDA(ctx, cudaMemsetAsync(sc->fgr_state, 0, sizeof(FgrState), s));
  APC_CUDA(ctx, cudaMemsetAsync(sc->feat_count, 0, 2 * sizeof(uint32_t), s));
  if (n_tiles) {
    APC_PROF(ctx, "k_fgr_pairs", s);
    k_fgr_pairs<<<n_tiles, APC_TILE_THREADS, 0, s>>>(pairs, n_pairs, n_pairs_dev, n_src, n_src_dev, n_tgt, n_tgt_dev,
                                                     sc->feat_pairs, sc->feat_count + 1, ctx->scan_state[0], ctx->ctrl,
                                                     n_tiles);
  }
  return fgr_run(ctx, src_xyzi, n_src, n_src_dev, tgt_xyzi, n_tgt, n_tgt_dev, n_pairs, n_pairs_dev, n_pairs,
                 division_factor, use_absolute_scale ? 1 : 0, decrease_mu ? 1 : 0, maximum_correspondence_distance,
                 iteration_number, 1.0, 0u, 0, out_T16_dev, out_info_dev, out_pairs_used, s);
}
