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
// share cells.  Radius search uses one level with c0 = r * (1 + 2^-10); KNN climbs levels
// until the k-th distance is covered by the 27-cell block, and the rare points that never
// are (fewer than k points in range of the coarsest level) fall to an exact brute-force
// kernel.  The table is cleaned by the points that own rank 0 of their cell, not by memset.
#include <cmath>
#include <cstdlib>
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

// ---- radius query -----------------------------------------------------------------------------
// Neighbours of q within r2 among the first `n_cells` cells of the centre-first order (1 = own cell
// only, 27 = the whole block), stopping at nb_points unless the exact count is wanted.
__device__ __forceinline__ uint32_t radius_count(const GridDev& g, float c, float4 q, float r2, uint32_t nb_points,
                                                 int need_counts, int n_cells) {
  int32_t ix, iy, iz;
  grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
  uint32_t cnt = 0;
  // own cell first, then faces, edges, corners: when only the keep/drop decision is wanted
  // most points reach nb_points inside their own cell and stop there.  The first probe of the
  // NEXT cell is in flight while the current cell's points are scanned.
  uint64_t key = grid_key(0, ix, iy, iz);
  uint32_t home = grid_home(g, key);
  uint4 first = grid_load(g, home);
  for (int c27 = 0; c27 < n_cells && (need_counts || cnt < nb_points); ++c27) {
    const uint64_t key_now = key;
    const uint32_t home_now = home;
    const uint4 first_now = first;
    if (c27 + 1 < n_cells) {
      const int code = c_cell_order[c27 + 1];
      key = grid_key(0, ix + code % 3 - 1, iy + (code / 3) % 3 - 1, iz + code / 9 - 1);
      home = grid_home(g, key);
      first = grid_load(g, home);
    }
    uint32_t b, f;
    if (!grid_resolve(g, key_now, home_now, first_now, b, f)) continue;
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
  }
  return cnt;
}

__global__ void __launch_bounds__(128)
k_radius_query(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t nb_points, int need_counts,
               uint8_t* __restrict__ mask, uint32_t* __restrict__ counts, const ApcCtrl* __restrict__ ctrl) {
  pdl_enter();
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  APC_STAMP(0, 0);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    const uint32_t cnt = radius_count(g, c, q, r2, nb_points, need_counts, 27);
    mask[orig] = cnt >= nb_points ? 1 : 0;
    if (counts) counts[orig] = cnt;
  }
  APC_STAMP(0, 1);
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
  if (both) return radius_count(g, c, q, r2, nb_points, need_counts, 27);
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

// Decision-only variant (keep iff >= nb_points within r) - an A/B knob that lost, see radius_decide.  The per-thread walk above
// costs what its SLOWEST lane costs: two thirds of its warp instructions were the own-cell loop running on for
// the one or two lanes of a warp that do not find nb_points near themselves (profiles/r2v_ncu_full.csv,
// hot_lines).  Here every lane scans outwards for at most `own_rounds` rounds (8 records); the lanes still
// short of nb_points are then served by the WHOLE WARP, one after the other: the rest of the lane's own cell
// 32 records at a time (ballot + popc), then lanes 1..7 resolve the <= 7 box-pruned neighbour cells in one
// round trip and the warp walks their runs as one flat list.  A warp with more than `coop_max` such lanes
// (a sparse region: everybody is short) lets them walk alone as before - there the per-thread walk keeps all
// lanes busy.  Counts may overshoot nb_points (whole batches are counted); the decision is the same.
__global__ void __launch_bounds__(128)
k_radius_decide_oct(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r, float r2, uint32_t nb_points,
                    uint8_t* __restrict__ mask, const ApcCtrl* __restrict__ ctrl, uint32_t own_rounds, uint32_t coop_max) {
  pdl_enter();
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = lane_id();
  const float reach = r * 1.00001f, reach2 = __fmul_rn(reach, reach);
  APC_STAMP(0, 0);
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const uint32_t j = base + threadIdx.x;
    const bool live = j < n;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
    int32_t ix = 0, iy = 0, iz = 0;
    uint32_t cnt = 0, b = 0, e = 0, up = 0, down = 0;
    bool pending = false;
    if (live) {
      q = g.sorted[j];
      grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
      uint32_t f;
      if (grid_lookup(g, grid_key(0, ix, iy, iz), b, f) && j >= b && j < b + f) {
        e = b + f;
        cnt = 1u;                                   // q itself
        up = j + 1;
        down = j;
        for (uint32_t round = 0; round < own_rounds && cnt < nb_points && (up < e || down > b); ++round) {
          float4 p[4];
          bool ok[4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            ok[u] = up + u < e;
            p[u] = g.sorted[ok[u] ? up + u : j];
            ok[2 + u] = down >= b + 1 + u;
            p[2 + u] = g.sorted[ok[2 + u] ? down - 1 - u : j];
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) cnt += (ok[u] && d2_f32(q.x, q.y, q.z, p[u].x, p[u].y, p[u].z) <= r2) ? 1u : 0u;
          up = min(up + 2, e);
          down = down >= b + 2 ? down - 2 : b;
        }
        pending = cnt < nb_points;
      } else {
        cnt = radius_count_oct(g, c, q, j, r, r2, nb_points, 0);   // (a record outside its own cell's run: not reachable)
      }
    }
    uint32_t bal = __ballot_sync(0xffffffffu, pending);
    if (bal && (uint32_t)__popc(bal) <= coop_max) {
      while (bal) {
        const uint32_t L = __ffs(bal) - 1u;
        bal &= bal - 1u;
        const float qx = __shfl_sync(0xffffffffu, q.x, L), qy = __shfl_sync(0xffffffffu, q.y, L), qz = __shfl_sync(0xffffffffu, q.z, L);
        uint32_t cL = __shfl_sync(0xffffffffu, cnt, L);
        const uint32_t bL = __shfl_sync(0xffffffffu, b, L), eL = __shfl_sync(0xffffffffu, e, L);
        const uint32_t upL = __shfl_sync(0xffffffffu, up, L), downL = __shfl_sync(0xffffffffu, down, L);
        const int32_t ixL = __shfl_sync(0xffffffffu, ix, L), iyL = __shfl_sync(0xffffffffu, iy, L), izL = __shfl_sync(0xffffffffu, iz, L);
        // 1. what is left of the own cell: [bL, downL) and [upL, eL)
        const uint32_t lo_n = downL - bL, tot = lo_n + (eL - upL);
        for (uint32_t t0 = 0; t0 < tot && cL < nb_points; t0 += 32) {
          const uint32_t t = t0 + lane;
          bool hit = false;
          if (t < tot) {
            const float4 p = g.sorted[t < lo_n ? bL + t : upL + (t - lo_n)];
            hit = d2_f32(qx, qy, qz, p.x, p.y, p.z) <= r2;
          }
          cL += __popc(__ballot_sync(0xffffffffu, hit));
        }
        if (cL < nb_points) {
          // 2. the neighbour cells the ball reaches (same pruning as radius_count_oct)
          const float qa[3] = {qx, qy, qz};
          const int32_t ia[3] = {ixL, iyL, izL};
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
          if (both) {                                 // slack not small against r: the lane walks all 27 cells itself
            uint32_t full = 0;
            if (lane == L) full = radius_count(g, c, q, r2, nb_points, 0, 27);
            cL = __shfl_sync(0xffffffffu, full, L);
          } else {
            uint32_t ns = 0, nf = 0;
            if (lane >= 1u && lane < 8u) {
              const float s2 = ((lane & 1u) ? gap2[0] : 0.0f) + ((lane & 2u) ? gap2[1] : 0.0f) + ((lane & 4u) ? gap2[2] : 0.0f);
              if (s2 <= reach2) {
                const uint64_t key = grid_key(0, ixL + ((lane & 1u) ? dir[0] : 0), iyL + ((lane & 2u) ? dir[1] : 0),
                                              izL + ((lane & 4u) ? dir[2] : 0));
                uint32_t bb, ff;
                if (grid_lookup(g, key, bb, ff)) { ns = bb; nf = ff; }
              }
            }
            uint32_t incl = nf;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
              const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
              if (lane >= (uint32_t)o) incl += v;
            }
            const uint32_t ps = incl - nf;                       // first flat index of lane's run
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 7);
            for (uint32_t t0 = 0; t0 < total && cL < nb_points; t0 += 32) {
              const uint32_t t = t0 + lane;
              const uint32_t flat = min(t, total - 1u);
              uint32_t run = 0;                                  // largest m in 1..7 with ps[m] <= flat
#pragma unroll
              for (int step = 4; step > 0; step >>= 1) {
                const uint32_t mid = run + step;
                const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
                if (mid < 8u && v <= flat) run = mid;
              }
              const uint32_t rs = __shfl_sync(0xffffffffu, ns, run), rp = __shfl_sync(0xffffffffu, ps, run);
              bool hit = false;
              if (t < total) {
                const float4 p = g.sorted[rs + (flat - rp)];
                hit = d2_f32(qx, qy, qz, p.x, p.y, p.z) <= r2;
              }
              cL += __popc(__ballot_sync(0xffffffffu, hit));
            }
          }
        }
        if (lane == L) cnt = cL;
      }
    } else if (pending) {
      cnt = radius_count_oct(g, c, q, j, r, r2, nb_points, 0);
    }
    if (live) mask[__float_as_uint(q.w)] = cnt >= nb_points ? 1 : 0;
  }
  APC_STAMP(0, 1);
}

// Cell edge of the radius grid in units of r (+ 2^-10 slack so that d2 <= r2 never reaches past the
// neighbouring cell): >= 2 = the pruned 8-cell walk above (default 2), 1 = the 27-cell walk (APC_RADIUS_CELL).
static float radius_cell_mult() {
  static const float m = []() {
    const char* e = getenv("APC_RADIUS_CELL");
    const float v = e ? (float)atof(e) : 2.0f;
    return v >= 2.0f ? v : 1.0f;
  }();
  return m;
}
static float radius_cell(float r32) { return r32 * radius_cell_mult() * 1.0009765625f; }

// The keep / drop decision in two launches (the exact counts are not wanted):
//   fast  every point against its OWN cell only - one probe, one or two rounds of loads, every thread
//         done within the same few microseconds; the few that did not reach nb_points there are
//         appended (warp-aggregated) to a pending list;
//   slow  the pending points against the whole 27-cell block.
// Idea: one launch doing both keeps ALL threads' registers resident until the slowest walker of each CTA
// is through its 27 dependent probes.  Measured (APC_RADIUS_SPLIT=1, profiles/r2g_knobs.json): the own-cell
// pass takes 10.6 us, but the pending pass still takes 23 us (its walkers are the whole cost) and saturated
// throughput does not move (70.5 vs 70.8 us/scan), for one more launch of latency: OFF by default.
#define CTR_RADIUS_PENDING 23
__global__ void __launch_bounds__(128)
k_radius_fast(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t nb_points, uint8_t* __restrict__ mask,
              uint32_t* __restrict__ pending, ApcCtrl* ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = lane_id();
  for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
    const uint32_t j = base + threadIdx.x;
    bool open = false;
    if (j < n) {
      const float4 q = g.sorted[j];
      const uint32_t cnt = radius_count(g, c, q, r2, nb_points, 0, 1);
      open = cnt < nb_points;
      if (!open) mask[__float_as_uint(q.w)] = 1;
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, open);
    if (bal) {
      uint32_t at = 0;
      if (lane == 0) at = atomicAdd(&ctrl->counters[CTR_RADIUS_PENDING], (uint32_t)__popc(bal));
      at = __shfl_sync(0xffffffffu, at, 0);
      if (open) pending[at + __popc(bal & ((1u << lane) - 1u))] = j;
    }
  }
}
__global__ void __launch_bounds__(128)
k_radius_slow(GridDev g, float r2, uint32_t nb_points, uint8_t* __restrict__ mask, const uint32_t* __restrict__ pending,
              const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = ctrl->counters[CTR_RADIUS_PENDING];
  const float c = grid_cell_size(g, 0);
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) {
    const float4 q = g.sorted[pending[k]];
    const uint32_t cnt = radius_count(g, c, q, r2, nb_points, 0, 27);
    mask[__float_as_uint(q.w)] = cnt >= nb_points ? 1 : 0;
  }
}

// decision-only radius query: the single launch (default) or the split (APC_RADIUS_SPLIT=1)
static int radius_decide(apc_ctx* ctx, const GridDev& g, uint32_t n_max, const uint32_t* n_dev, float r, float r2,
                         uint32_t nb_points, uint8_t* mask, cudaStream_t s) {
  static const bool split = []() { const char* e = getenv("APC_RADIUS_SPLIT"); return e && atoi(e) != 0; }();
  const uint32_t bq = min(apc_div_up(n_max, 128), (uint32_t)APC_SM_COUNT * 16);
  if (radius_cell_mult() >= 2.0f) {
    // APC_RADIUS_COOP = "own_rounds,coop_max": warp-cooperative service of the lanes left short (k_radius_decide_oct).
    // Default coop_max = 0 = the per-thread walk k_radius_query_oct: the cooperative variant LOST the A/B (24.3 vs
    // 21.9 us alone, 67.7 vs 64.8 us/scan with all lanes busy at 2,8; 33.4 us at 2,32; profiles/r2p_radius_ab.json)
    static const uint32_t own_rounds = []() { const char* e = getenv("APC_RADIUS_COOP"); return e ? (uint32_t)atoi(e) : 2u; }();
    static const uint32_t coop_max = []() {
      const char* e = getenv("APC_RADIUS_COOP");
      const char* comma = e ? strchr(e, ',') : nullptr;
      return comma ? (uint32_t)atoi(comma + 1) : 0u;
    }();
    APC_PROF(ctx, "k_radius_query", s);
    if (coop_max)
      apc_klaunch(ctx, k_radius_decide_oct, bq, 128, 0, s, n_max, n_dev, g, r, r2, nb_points, mask, ctx->ctrl, own_rounds, coop_max);
    else {
      static const uint32_t blk = []() { const char* e = getenv("APC_RADIUS_BLOCK"); const int v = e ? atoi(e) : 128; return (uint32_t)((v == 64 || v == 256) ? v : 128); }();
      const uint32_t bqb = min(apc_div_up(n_max, blk), (uint32_t)APC_SM_COUNT * (2048u / blk));
      apc_klaunch(ctx, k_radius_query_oct, bqb, blk, 0, s, n_max, n_dev, g, r, r2, nb_points, 0, mask, nullptr, ctx->ctrl);
    }
    APC_LAUNCH_CHECK(ctx, "k_radius_query_oct");
    return APC_OK;
  }
  if (!split) {
    APC_PROF(ctx, "k_radius_query", s);
    apc_klaunch(ctx, k_radius_query, bq, 128, 0, s, n_max, n_dev, g, r2, nb_points, 0, mask, nullptr, ctx->ctrl);
    APC_LAUNCH_CHECK(ctx, "k_radius_query");
    return APC_OK;
  }
  {
    APC_PROF(ctx, "k_radius_fast", s);
    k_radius_fast<<<bq, 128, 0, s>>>(n_max, n_dev, g, r2, nb_points, mask, ctx->nb_count, ctx->ctrl);
  }
  APC_PROF(ctx, "k_radius_slow", s);
  k_radius_slow<<<min(bq, (uint32_t)APC_SM_COUNT * 4), 128, 0, s>>>(g, r2, nb_points, mask, ctx->nb_count, ctx->ctrl);
  APC_LAUNCH_CHECK(ctx, "k_radius_fast/slow");
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
//   1. lanes 0..26 resolve the 27 neighbour cells in parallel; a warp scan of the run lengths gives
//      the flat candidate list and tells whether the block holds k points at all;
//   2. the lanes stride over the flat list (run found by a 5-step shuffle search), compute the
//      float32 distances and drop their bit patterns (non-negative floats order like integers)
//      into the warp's shared buffer; longer lists go through the buffer in chunks, each chunk
//      merged with the k best so far;
//   3. the k-th smallest value is found by a 31-step binary search on the bit pattern (each step a
//      strided count + REDUX), the k smallest are compacted in place (ties at the k-th value are
//      interchangeable);
//   4. the level's answer stands if the k-th distance is covered by the block (same test as before);
//      then the k values are rank-sorted and summed in ascending order by shuffles - the same
//      sequential float32 sum as oracle/outliers.py.
#define KNN_CAP 1024
#define KNN_WARPS 4
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn_query(uint32_t n_max, const uint32_t* n_dev, GridDev g, uint32_t k, float* __restrict__ avg,
            uint32_t* __restrict__ stragglers, ApcCtrl* ctrl, uint32_t start_fill, int exact_margin, uint32_t merge_min) {
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
    // Optional starting level (start_fill > 0, an A/B knob that lost): the finest level whose OWN cell already
    // holds start_fill points (lane l reads the population of the query's cell at level l through the slot
    // recorded at insert time: two dependent loads for all levels at once).
    uint32_t level0 = 0;
    if (start_fill) {
      uint32_t fill = 0;
      if (lane < g.levels) {
        const uint32_t sl = g.slot[(size_t)lane * n_max + orig];
        if (sl != GRID_NOSLOT) fill = g.slots[sl].fill;
      }
      const uint32_t okm = __ballot_sync(0xffffffffu, fill >= start_fill);
      level0 = okm ? (uint32_t)__ffs(okm) - 1u : g.levels - 1u;
    }
    for (uint32_t level = level0; level < g.levels && !done; ++level) {
      const float c = g.cell[level];
      int32_t ix, iy, iz;
      if (!grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz)) continue;
      // 1. the 27 cells, one per lane
      uint32_t cs = 0, cf = 0;
      if (lane < 27) {
        const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
        uint32_t b, f;
        if (grid_lookup(g, grid_key(level, ix + dx, iy + dy, iz + dz), b, f)) { cs = b; cf = f; }
      }
      uint32_t incl = cf;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (uint32_t)o) incl += v;
      }
      const uint32_t ps = incl - cf;                               // first flat index of this lane's run
      const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
      if (total < k_eff) continue;
      const float4* sp = g.sorted + (size_t)level * n_max;
      // every point closer than `safe` lies inside the 27-cell block: the cell edge plus (exact_margin) the
      // query's distance to the nearest face of its own cell, less 0.1 % for the rounding of the cell index
      float safe = c;
      if (exact_margin) {
        const float mx = fminf(__fsub_rn(q.x, __fmul_rn((float)ix, c)), __fsub_rn(__fmul_rn((float)(ix + 1), c), q.x));
        const float my = fminf(__fsub_rn(q.y, __fmul_rn((float)iy, c)), __fsub_rn(__fmul_rn((float)(iy + 1), c), q.y));
        const float mz = fminf(__fsub_rn(q.z, __fmul_rn((float)iz, c)), __fsub_rn(__fmul_rn((float)(iz + 1), c), q.z));
        safe = __fadd_rn(c, fmaxf(0.0f, fminf(mx, fminf(my, mz))));
      }
      safe = __fmul_rn(safe, 0.999f);
      if (k_eff <= 32u) {
        // 2'. k <= 32 (the reference's default is 20): the k best live in REGISTERS, lane i holding the
        // i-th smallest distance so far.  A batch of 32 candidates is screened with one ballot against
        // the current k-th value; the few that pass are inserted one by one (position by ballot, shift
        // by shuffle) - about 2x fewer instructions per level than the buffer + binary search below.
        const float inf = __int_as_float(0x7f800000);
        float val = inf, kth = inf;
        for (uint32_t base = 0; base < total; base += 32) {
          const uint32_t ci = base + lane;
          const uint32_t flat = min(ci, total - 1u);
          uint32_t run = 0;                                        // largest t with ps[t] <= flat
#pragma unroll
          for (int step = 16; step > 0; step >>= 1) {
            const uint32_t mid = run + step;
            const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
            if (mid < 27u && v <= flat) run = mid;
          }
          const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
          float d2 = inf;
          if (ci < total) {
            const float4 p = sp[rs + (flat - rp)];
            d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
          }
          uint32_t cand = __ballot_sync(0xffffffffu, d2 < kth);
          if ((uint32_t)__popc(cand) > merge_min) {
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
        if (kth <= __fmul_rn(safe, safe)) {
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
          const uint32_t flat = c0 + min(ci, take - 1u);
          uint32_t run = 0;                                        // largest t with ps[t] <= flat
#pragma unroll
          for (int step = 16; step > 0; step >>= 1) {
            const uint32_t mid = run + step;
            const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
            if (mid < 27u && v <= flat) run = mid;
          }
          const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
          if (ci < take) {
            const float4 p = sp[rs + (flat - rp)];
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
      if (kth <= __fmul_rn(safe, safe)) done = true;
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

// ---- k > 64 (up to APC_MAX_NEIGHBORS): per-warp shared candidate buffers ---------------------------
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

// Buffer entries per warp for k > 64: more than k + 32 (a selection always makes room for a batch)
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
// per level, lanes 0..26 resolve the 27 cells, the flat candidate list streams through a WarpKeep of `cap`
// keys at buf, and the level stands if the k_eff-th distance is covered by the block (`safe`, exact_margin).
// Returns true with the k_eff smallest keys in buf[0, k_eff) (unordered); false when no level covers q
// (a straggler).
template <typename K>
__device__ __forceinline__ bool knn_levels(const GridDev& g, uint32_t n_max, float4 q, uint32_t k_eff, K* buf, uint32_t cap,
                                           int exact_margin, uint32_t lane) {
  for (uint32_t level = 0; level < g.levels; ++level) {
    const float c = g.cell[level];
    int32_t ix, iy, iz;
    if (!grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz)) continue;
    uint32_t cs = 0, cf = 0;
    if (lane < 27) {
      const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
      uint32_t b, f;
      if (grid_lookup(g, grid_key(level, ix + dx, iy + dy, iz + dz), b, f)) { cs = b; cf = f; }
    }
    uint32_t incl = cf;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t ps = incl - cf;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    if (total < k_eff) continue;
    const float4* sp = g.sorted + (size_t)level * n_max;
    float safe = c;
    if (exact_margin) {
      const float mx = fminf(__fsub_rn(q.x, __fmul_rn((float)ix, c)), __fsub_rn(__fmul_rn((float)(ix + 1), c), q.x));
      const float my = fminf(__fsub_rn(q.y, __fmul_rn((float)iy, c)), __fsub_rn(__fmul_rn((float)(iy + 1), c), q.y));
      const float mz = fminf(__fsub_rn(q.z, __fmul_rn((float)iz, c)), __fsub_rn(__fmul_rn((float)(iz + 1), c), q.z));
      safe = __fadd_rn(c, fmaxf(0.0f, fminf(mx, fminf(my, mz))));
    }
    safe = __fmul_rn(safe, 0.999f);
    WarpKeep<K> wk;
    wk.init(buf, cap, k_eff);
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t flat = min(ci, total - 1u);
      uint32_t run = 0;                                          // largest t with ps[t] <= flat
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t mid = run + step;
        const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
        if (mid < 27u && v <= flat) run = mid;
      }
      const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
      K key = 0;
      if (ci < total) {
        const float4 p = sp[rs + (flat - rp)];
        key = knn_key<K>(d2_f32(q.x, q.y, q.z, p.x, p.y, p.z), __float_as_uint(p.w));
      }
      wk.add(key, ci < total, lane);
    }
    wk.finish(lane);
    uint32_t mx = 0;                                             // covered by the block? (the d2 bits of the keys)
    for (uint32_t i = lane; i < k_eff; i += 32) mx = max(mx, (uint32_t)(buf[i] >> (8 * sizeof(K) - 32)));
    if (__uint_as_float(__reduce_max_sync(0xffffffffu, mx)) <= __fmul_rn(safe, safe)) return true;
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
// coverage test (`safe`, exact_margin), the candidates through a WarpKeep of wide_cap(k) entries per
// warp (dynamic shared memory), the accepted level's k distances sorted and summed by wide_average.
__global__ void __launch_bounds__(KNN_WARPS * 32)
k_knn_query_wide(uint32_t n_max, const uint32_t* n_dev, GridDev g, uint32_t k, uint32_t cap, float* __restrict__ avg,
                 uint32_t* __restrict__ stragglers, ApcCtrl* ctrl, int exact_margin) {
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t n_sorted = grid_sorted_count(g, ctrl, n);
  const uint32_t k_eff = min(k, n);
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t* buf = reinterpret_cast<uint32_t*>(wide_smem) + (size_t)w * cap;
  for (uint32_t j = blockIdx.x * KNN_WARPS + w; j < n_sorted; j += gridDim.x * KNN_WARPS) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    if (knn_levels(g, n_max, q, k_eff, buf, cap, exact_margin, lane)) {
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
  static const bool cell_list = getenv("APC_NO_CELL_LIST") == nullptr;   // A/B knob
  g.d.cells = (inserted && cell_list) ? g.cells_buf : nullptr;
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
  const float r2 = r32 * r32;                       // float32(r)^2, rounded once
  // cells of r (+ slack, so that d2 <= r2 never reaches 2 cells away); measured alternatives at
  // 200k points: cells of 2r 37 us, one warp per cell group with shuffled broadcasts 85 us,
  // neighbour-cell lookups issued in rounds of 6-13 32-50 us, this per-thread walk 29-32 us
  const float cell = radius_cell(r32);
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  rc = grid_build(ctx, g, pts, n_max, n_dev, cell, false, s, false, 0, radius_cell_mult() >= 2.0f);
  if (rc) return rc;
  if (out_counts) {
    const uint32_t bq = min(apc_div_up(n_max, 128), (uint32_t)APC_SM_COUNT * 16);
    APC_PROF(ctx, "k_radius_query", s);
    if (radius_cell_mult() >= 2.0f)
      apc_klaunch(ctx, k_radius_query_oct, bq, 128, 0, s, n_max, n_dev, g.d, r32, r2, (uint32_t)nb_points, 1, out_mask, out_counts, ctx->ctrl);
    else
      apc_klaunch(ctx, k_radius_query, bq, 128, 0, s, n_max, n_dev, g.d, r2, (uint32_t)nb_points, 1, out_mask, out_counts, ctx->ctrl);
  } else {
    rc = radius_decide(ctx, g.d, n_max, n_dev, r32, r2, (uint32_t)nb_points, out_mask, s);
    if (rc) return rc;
  }
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
  g.d.inv0 = radius_cell_mult() >= 2.0f ? 1.0f / g.d.cell0 : 0.0f;
  g.d.cells = getenv("APC_NO_CELL_LIST") ? nullptr : g.cells_buf;   // the caller inserts: it also lists the occupied cells
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
  rc = grid_build(ctx, g, pts, n_max, n_dev, radius_cell(r32), false, s, points_inserted != 0, 0, radius_cell_mult() >= 2.0f);
  if (rc) return rc;
  rc = radius_decide(ctx, g.d, n_max, n_dev, r32, r32 * r32, (uint32_t)nb_points, mask_scratch, s);
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
  static const int margin_env = []() { const char* e = getenv("APC_KNN_MARGIN"); return e ? atoi(e) : 1; }();
  if (nb_neighbors > KNN_KMAX) {
    const uint32_t cap = wide_cap((uint32_t)nb_neighbors);
    const size_t smem = (size_t)KNN_WARPS * cap * sizeof(uint32_t);
    {
      APC_PROF(ctx, "k_knn_query_wide", s);
      k_knn_query_wide<<<bq, KNN_WARPS * 32, smem, s>>>(n_max, n_dev, g.d, (uint32_t)nb_neighbors, cap, avg, sc->stragglers,
                                                        ctx->ctrl, margin_env);
    }
    {
      APC_PROF(ctx, "k_knn_stragglers_wide", s);
      k_knn_stragglers_wide<<<APC_SM_COUNT * 2, KNN_WARPS * 32, smem, s>>>(pts, n_max, n_dev, (uint32_t)nb_neighbors, cap,
                                                                           sc->stragglers, ctx->ctrl, avg);
    }
  } else {
    {
      APC_PROF(ctx, "k_knn_query", s);
      // APC_KNN_START_FILL: own-cell population that selects the starting level (default 0 = always level 0: skipping
      // fine levels by this estimate examines more candidates than the failed passes cost - 2.49 / 2.94 / 3.34 ms
      // against 1.86 ms for a population of 5 / 10 / 16 on the C4 scan);
      // APC_KNN_MARGIN=0: guaranteed radius = the cell edge only (profiles/r2x_knn_ab.json)
      static const int fill_env = []() { const char* e = getenv("APC_KNN_START_FILL"); return e ? atoi(e) : -1; }();
      const uint32_t start_fill = fill_env > 0 ? (uint32_t)fill_env : 0u;
      // newcomers in a batch of 32 above which the batch is sorted and merged instead of inserted one by one
      static const uint32_t merge_min = []() { const char* e = getenv("APC_KNN_MERGE_MIN"); return e ? (uint32_t)atoi(e) : 6u; }();
      k_knn_query<<<bq, KNN_WARPS * 32, 0, s>>>(n_max, n_dev, g.d, (uint32_t)nb_neighbors, avg, sc->stragglers, ctx->ctrl,
                                                start_fill, margin_env, merge_min);
    }
    {
      APC_PROF(ctx, "k_knn_stragglers", s);
      k_knn_stragglers<<<APC_SM_COUNT * 2, 256, 0, s>>>(pts, n_max, n_dev, (uint32_t)nb_neighbors, sc->stragglers, ctx->ctrl, avg);
    }
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
#define NRM_KMAX 64

struct NearList {
  unsigned long long key[NRM_KMAX];   // d2 bits << 32 | original index: d2 >= 0, so integer order = (d2, index) order
  uint32_t pos[NRM_KMAX];             // position of the neighbour in the cell-sorted array
  uint32_t cnt, worst;
  __device__ __forceinline__ void find_worst(uint32_t k) {
    worst = 0;
    for (uint32_t j = 1; j < k; ++j)
      if (key[j] > key[worst]) worst = j;
  }
  __device__ __forceinline__ void push(unsigned long long kk, uint32_t p, uint32_t k) {
    if (cnt < k) {
      key[cnt] = kk;
      pos[cnt] = p;
      if (++cnt == k) find_worst(k);
    } else if (kk < key[worst]) {
      key[worst] = kk;
      pos[worst] = p;
      find_worst(k);
    }
  }
};

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

__global__ void __launch_bounds__(128)
k_normals_query(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t max_nn, float* __restrict__ normals,
                uint32_t* __restrict__ counts, double* __restrict__ covariances, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    int32_t ix, iy, iz;
    grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
    NearList nl;
    nl.cnt = 0;
    nl.worst = 0;
    for (int c27 = 0; c27 < 27; ++c27) {
      const int dx = c27 % 3 - 1, dy = (c27 / 3) % 3 - 1, dz = c27 / 9 - 1;
      uint32_t b, f;
      if (!grid_lookup(g, grid_key(0, ix + dx, iy + dy, iz + dz), b, f)) continue;
      const uint32_t e = b + f;
      for (uint32_t t = b; t < e; ++t) {
        const float4 p = g.sorted[t];
        const float d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
        if (d2 <= r2)
          nl.push(((unsigned long long)__float_as_uint(d2) << 32) | __float_as_uint(p.w), t, max_nn);
      }
    }
    double C[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};   // fewer than 3 neighbours: identity
    if (nl.cnt >= 3) {
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, m00 = 0.0, m01 = 0.0, m02 = 0.0, m11 = 0.0, m12 = 0.0, m22 = 0.0;
      for (uint32_t k = 0; k < nl.cnt; ++k) {
        const float4 p = g.sorted[nl.pos[k]];
        const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
        s0 += x; s1 += y; s2 += z;
        m00 += x * x; m01 += x * y; m02 += x * z; m11 += y * y; m12 += y * z; m22 += z * z;
      }
      const double inv = 1.0 / (double)nl.cnt;
      s0 *= inv; s1 *= inv; s2 *= inv;
      C[0] = m00 * inv - s0 * s0;
      C[1] = C[3] = m01 * inv - s0 * s1;
      C[2] = C[6] = m02 * inv - s0 * s2;
      C[4] = m11 * inv - s1 * s1;
      C[5] = C[7] = m12 * inv - s1 * s2;
      C[8] = m22 * inv - s2 * s2;
    }
    double nrm[3];
    normal_from_covariance(C, nrm);
    normals[3 * (size_t)orig + 0] = (float)nrm[0];
    normals[3 * (size_t)orig + 1] = (float)nrm[1];
    normals[3 * (size_t)orig + 2] = (float)nrm[2];
    if (counts) counts[orig] = nl.cnt;
    if (covariances)
      for (int k = 0; k < 9; ++k) covariances[9 * (size_t)orig + k] = C[k];
  }
}

// max_nn <= 32 (the reference's default is 30): one WARP per query, as in k_knn_query.  Lanes 0..26
// resolve the 27 cells; the lanes stride over the flat candidate list; the max_nn nearest in-radius
// neighbours by (d2, original index) live in registers, lane i holding the i-th smallest key and the
// neighbour's position; every lane then contributes its neighbour's moments about the query point
// and a shuffle tree adds them up in float64.  The eigenvector is computed by k_normals_eigen, one
// THREAD per point (a serial float64 solve would idle 31 lanes of the warp here).
__global__ void __launch_bounds__(128)
k_normals_cov(uint32_t n_max, const uint32_t* n_dev, GridDev g, float r2, uint32_t max_nn, uint32_t* __restrict__ counts,
              double* __restrict__ cov9, const ApcCtrl* __restrict__ ctrl) {
  const uint32_t n = grid_sorted_count(g, ctrl, apc_count(n_dev, n_max));
  const float c = grid_cell_size(g, 0);
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += (gridDim.x * blockDim.x) >> 5) {
    const float4 q = g.sorted[j];
    const uint32_t orig = __float_as_uint(q.w);
    int32_t ix, iy, iz;
    grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
    uint32_t cs = 0, cf = 0;
    if (lane < 27) {
      const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
      uint32_t b, f;
      if (grid_lookup(g, grid_key(0, ix + dx, iy + dy, iz + dz), b, f)) { cs = b; cf = f; }
    }
    uint32_t incl = cf;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t ps = incl - cf;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);   // >= 1: the query's own cell holds the query
    unsigned long long kv = ~0ull, kth = ~0ull;                   // lane i: i-th smallest key so far / the max_nn-th
    uint32_t pv = 0, in_radius = 0;
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t flat = min(ci, total - 1u);
      uint32_t run = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t mid = run + step;
        const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
        if (mid < 27u && v <= flat) run = mid;
      }
      const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
      const uint32_t pos = rs + (flat - rp);
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
    double C[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};   // fewer than 3 neighbours: identity
    if (n_sel >= 3) {
      double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      if (lane < n_sel) {
        const float4 p = g.sorted[pv];
        const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
        v[0] = x; v[1] = y; v[2] = z;
        v[3] = x * x; v[4] = x * y; v[5] = x * z; v[6] = y * y; v[7] = y * z; v[8] = z * z;
      }
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
    if (lane < 9) cov9[9 * (size_t)orig + lane] = C[lane];
    if (lane == 0 && counts) counts[orig] = n_sel;
  }
}

// Covariance of a kept neighbourhood (warp-collective): buf[0, n_sel) holds the neighbours' 64-bit keys (d2 bits
// << 32 | original index), unordered.  The float64 moments about q are summed in key order, the same on every run
// (the keys arrive in the grid's in-cell order, which the build's atomics decide); lanes 0..8 write cov9 of point
// orig, lane 0 the count.  Fewer than 3 neighbours: identity.
__device__ __forceinline__ void normals_cov_of_keys(unsigned long long* buf, uint32_t n_sel, const float4* __restrict__ pts,
                                                    float4 q, uint32_t orig, uint32_t lane, uint32_t* __restrict__ counts,
                                                    double* __restrict__ cov9) {
  double C[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
  if (n_sel >= 3) {
    warp_sort(buf, n_sel, lane);
    double v[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (uint32_t i = lane; i < n_sel; i += 32) {
      const float4 p = pts[(uint32_t)buf[i]];
      const double x = (double)p.x - (double)q.x, y = (double)p.y - (double)q.y, z = (double)p.z - (double)q.z;
      v[0] += x; v[1] += y; v[2] += z;
      v[3] += x * x; v[4] += x * y; v[5] += x * z; v[6] += y * y; v[7] += y * z; v[8] += z * z;
    }
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

// 64 < max_nn <= APC_MAX_NEIGHBORS: one warp per query over the same 27-cell flat candidate list as
// k_normals_cov; the in-radius candidates stream through a WarpKeep of 64-bit keys (d2 bits << 32 |
// original index: the oracle's total order, so the neighbourhood is exact) of wide_cap(max_nn) entries per
// warp; the kept keys are sorted, and the lanes read the neighbours by original index from the input and add up
// their float64 moments about the query point.  k_normals_eigen turns cov9 into normals.
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
    int32_t ix, iy, iz;
    grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
    uint32_t cs = 0, cf = 0;
    if (lane < 27) {
      const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
      uint32_t b, f;
      if (grid_lookup(g, grid_key(0, ix + dx, iy + dy, iz + dz), b, f)) { cs = b; cf = f; }
    }
    uint32_t incl = cf;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t ps = incl - cf;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    WarpKeep<unsigned long long> wk;
    wk.init(buf, cap, max_nn);
    uint32_t in_radius = 0;
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t flat = min(ci, total - 1u);
      uint32_t run = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t mid = run + step;
        const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
        if (mid < 27u && v <= flat) run = mid;
      }
      const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
      unsigned long long key = 0;
      bool inside = false;
      if (ci < total) {
        const float4 p = g.sorted[rs + (flat - rp)];
        const float d2 = d2_f32(q.x, q.y, q.z, p.x, p.y, p.z);
        inside = d2 <= r2;
        key = ((unsigned long long)__float_as_uint(d2) << 32) | __float_as_uint(p.w);
      }
      in_radius += __popc(__ballot_sync(0xffffffffu, inside));
      wk.add(key, inside, lane);
    }
    wk.finish(lane);
    normals_cov_of_keys(buf, min(in_radius, max_nn), pts, q, orig, lane, counts, cov9);   // n_sel == wk.m
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
    if (knn_levels(g, n_max, q, k_eff, buf, cap, 1, lane)) normals_cov_of_keys(buf, k_eff, pts, q, orig, lane, counts, cov9);
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
// count.  One warp per query over the 27-cell flat candidate list of k_normals_wide, nothing kept: each
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
    int32_t ix, iy, iz;
    grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
    uint32_t cs = 0, cf = 0;
    if (lane < 27) {
      const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
      uint32_t b, f;
      if (grid_lookup(g, grid_key(0, ix + dx, iy + dy, iz + dz), b, f)) { cs = b; cf = f; }
    }
    uint32_t incl = cf;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += v;
    }
    const uint32_t ps = incl - cf;
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    long long m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    uint32_t cnt = 0;
    for (uint32_t base = 0; base < total; base += 32) {
      const uint32_t ci = base + lane;
      const uint32_t flat = min(ci, total - 1u);
      uint32_t run = 0;
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const uint32_t mid = run + step;
        const uint32_t v = __shfl_sync(0xffffffffu, ps, mid & 31u);
        if (mid < 27u && v <= flat) run = mid;
      }
      const uint32_t rs = __shfl_sync(0xffffffffu, cs, run), rp = __shfl_sync(0xffffffffu, ps, run);
      bool inside = false;
      if (ci < total) {
        const float4 p = g.sorted[rs + (flat - rp)];
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
int apc_normals_prepare(apc_ctx* ctx, int max_nn) {
  int rc = apc_neighbors_prepare(ctx, 0);
  if (rc) return rc;
  NeighborScratch* sc = scratch_of(ctx);
  // k_normals_cov (max_nn <= 32) and k_normals_wide (max_nn > 64) hand their covariances to k_normals_eigen
  const bool via_cov = max_nn <= 32 || max_nn > NRM_KMAX;
  if (via_cov && !sc->cov) APC_CUDA(ctx, cudaMalloc((void**)&sc->cov, (size_t)ctx->max_points * 9 * sizeof(double)));
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
  GridHost& g = scratch_of(ctx)->grid[0];
  const float r32 = (float)radius;
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  // cells of r * (1 + 2^-8) indexed by one multiply with the host-rounded reciprocal (grid_coord_g): the three IEEE
  // divisions per lookup were 9 % of k_normals_cov's instructions.  Two points within r of each other have
  // quotients less than 1 - 2^-8 + 2^-22 |x| / c apart, i.e. fall into the same or adjacent cells for |x| < 16384 r -
  // the range the division with its 2^-10 margin guaranteed.
  rc = grid_build(ctx, g, pts, n_max, n_dev, r32 * 1.00390625f, false, s, false, CTR_CURSOR_NORMALS, true);
  if (rc) return rc;
  if (max_nn <= 32 || max_nn > NRM_KMAX) {
    // warp per query -> covariances (caller's buffer or context scratch), then thread per point -> eigenvector
    NeighborScratch* sc = scratch_of(ctx);
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
    APC_PROF(ctx, "k_normals_eigen", s);
    k_normals_eigen<<<min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, s>>>(n_max, n_dev, cov, out_normals);
  } else {
    const uint32_t bq = min(apc_div_up(n_max, 128), (uint32_t)APC_SM_COUNT * 16);
    APC_PROF(ctx, "k_normals_query", s);
    k_normals_query<<<bq, 128, 0, s>>>(n_max, n_dev, g.d, r32 * r32, (uint32_t)max_nn, out_normals, out_counts, out_cov, ctx->ctrl);
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

// The 27 cells around q as one flat candidate list, for a warp that walks it 32 records at a time: lane l < 27
// resolves cell l and keeps its run's start in the cell-sorted array (cs) and the flat index of the run's first
// record (ps); returns the list's length (all lanes).  This is k_normals_radius's walk; that kernel keeps its inline
// copy because calling these helpers changes its instruction schedule.
__device__ __forceinline__ uint32_t flat27_runs(const GridDev& g, float c, float4 q, uint32_t lane, uint32_t& cs, uint32_t& ps) {
  int32_t ix, iy, iz;
  grid_coord_g(g, c, q.x, q.y, q.z, ix, iy, iz);  // succeeded at insert time
  uint32_t s0 = 0, cf = 0;
  if (lane < 27) {
    const int dx = (int)(lane % 3u) - 1, dy = (int)((lane / 3u) % 3u) - 1, dz = (int)(lane / 9u) - 1;
    uint32_t b, f;
    if (grid_lookup(g, grid_key(0, ix + dx, iy + dy, iz + dz), b, f)) { s0 = b; cf = f; }
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
// Position in g.sorted of record `flat` of that list (called by all lanes of the warp).
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
