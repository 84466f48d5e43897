// Fused front end: PointCloud2 unpack + read_points NaN skip + duplicate removal +
// non-finite filter + float32 transforms + ROI crop + order-preserving compaction, over up
// to 8 sensors in one launch (multi-LiDAR concatenation), plus the stand-alone mask /
// select / gather kernels behind the Open3D-like carrier methods.
//
// Reference call sites replaced: utils.py:206-211 (read_points), utils.py:102-121
// (positions / intensity casts), utils.py:509-546 (remove_duplicates, open3d back end),
// pp.py:469 (remove_non_finite_points), pp.py:482,487,490 (transform), utils.py:240-301
// (crop_pointcloud), utils.py:271,297 + pp.py:542 (select_by_mask / select_by_index),
// pointcloud_concatenator.py:1-5 (merge N sensors into one cloud in a target frame).

#include "apc_load.cuh"
APC_TRACE_EXPORT(frontend)

struct FrontendParams {
  SegDev seg[APC_MAX_CLOUDS];
  uint32_t n_seg;
  uint32_t n_tiles;
  uint32_t skip_nans, dedup, remove_nan, remove_inf;
  uint32_t n_T;
  float T[APC_MAX_TRANSFORMS][16];
  uint32_t crop_enable, crop_mode, crop_invert;
  double lo[3], hi[3];
  float lo32[3], hi32[3];
  // dedup table
  unsigned long long* slots;
  uint32_t slot_mask;
  uint32_t* p2slot;
  // outputs
  float4* out_xyzi;
  uint32_t* out_src;
  uint8_t* out_stage;
  uint32_t* out_count;
  uint64_t* scan_state;
  ApcCtrl* ctrl;
};

// ---- duplicate removal: 64-bit open-addressing slots {fingerprint:32 | lowest point index:32} -----
// The 96-bit key (bit patterns of x, y, z) does not fit an atomic word, so a slot holds a 32-bit
// fingerprint of the key next to the representative's index; a fingerprint hit is confirmed by
// reading the representative's coordinates back from the input (only real duplicates and 2^-32
// fingerprint collisions get there).  Equal keys then lower the index with atomicMin (same
// fingerprint in the high half, so the minimum is the lower index).
// Probing: compare-and-swap first, linear, all the items of a thread in lockstep so that their
// atomic round trips overlap (a thread's latency is the longest of its probe chains, not their
// sum).  Measured at 262k points (eager, CUDA events): 8 us with no table access at all, 10 us for
// one CAS per point, 16 us for this kernel; a variant that first read a 4-slot bucket with
// ld.global.cg and then CASed the first free slot took 33 us - concurrent inserts see the same
// free slot and lose the race, and the re-read can be served a stale copy.
#define DEDUP_EMPTY 0xffffffffffffffffull

__device__ __forceinline__ uint64_t dedup_hash(float x, float y, float z) {
  const uint32_t kx = __float_as_uint(x), ky = __float_as_uint(y), kz = __float_as_uint(z);
  return mix64(((uint64_t)kx | ((uint64_t)ky << 32)) ^ mix64((uint64_t)kz + 0x9E3779B97F4A7C15ull));
}
__device__ __forceinline__ unsigned long long dedup_word(uint64_t h, uint32_t g) {
  return ((unsigned long long)(h >> 32) << 32) | g;   // never all ones: g is a valid point index
}

// Inserts ITEMS points per thread.  `same(j, rep)` tells whether point `rep` has item j's x/y/z
// bit patterns (called on fingerprint hits only).
template <int ITEMS, typename SameFn>
__device__ __forceinline__ void dedup_insert_items(unsigned long long* slots, uint32_t slot_mask, uint32_t* p2slot,
                                                   ApcCtrl* ctrl, const uint64_t (&hash)[ITEMS],
                                                   const unsigned long long (&word)[ITEMS], bool (&act)[ITEMS], SameFn same) {
  uint32_t slot[ITEMS];
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) slot[j] = (uint32_t)hash[j] & slot_mask;
  for (uint32_t probe = 0; probe <= slot_mask; ++probe) {
    unsigned long long old[ITEMS];
#pragma unroll
    for (int j = 0; j < ITEMS; ++j)   // issue every unfinished item's CAS before looking at any result
      old[j] = act[j] ? atomicCAS(&slots[slot[j]], DEDUP_EMPTY, word[j]) : 0ull;
    bool any = false;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
      if (!act[j]) continue;
      bool done = old[j] == DEDUP_EMPTY;
      if (!done && (old[j] >> 32) == (word[j] >> 32) && same(j, (uint32_t)old[j])) {
        if ((uint32_t)word[j] < (uint32_t)old[j]) atomicMin(&slots[slot[j]], word[j]);   // a later point got here first
        done = true;
      }
      if (done) {
        p2slot[(uint32_t)word[j]] = slot[j];
        act[j] = false;
      } else {
        slot[j] = (slot[j] + 1) & slot_mask;
        any = true;
      }
    }
    if (!any) return;
  }
#pragma unroll
  for (int j = 0; j < ITEMS; ++j)
    if (act[j]) {
      atomicOr(&ctrl->err, APC_DEVERR_CAPACITY);
      p2slot[(uint32_t)word[j]] = 0;
    }
}

// x/y/z of point `g` of the launch, straight from the byte records (the confirm step above)
template <bool GENERIC, typename P>
__device__ __forceinline__ void load_xyz_global(const P& prm, uint32_t g, float& x, float& y, float& z) {
  uint32_t si = 0;
#pragma unroll
  for (uint32_t k = 1; k < APC_MAX_CLOUDS; ++k)
    if (k < prm.n_seg && g >= prm.seg[k].point_begin) si = k;
  const SegDev& s = prm.seg[si];
  if (!GENERIC) {   // FAST16: x, y, z are the first three floats of a 16-byte record
    const float4 v = __ldg(reinterpret_cast<const float4*>(s.data) + (g - s.point_begin));
    x = v.x; y = v.y; z = v.z;
    return;
  }
  const uint8_t* rec = s.data + (size_t)(g - s.point_begin) * s.step;
  x = field_as_f32(rec + s.off[0], s.dt[0]);
  y = field_as_f32(rec + s.off[1], s.dt[1]);
  z = field_as_f32(rec + s.off[2], s.dt[2]);
}

template <bool GENERIC>
__device__ __noinline__ bool dedup_same_record(const FrontendParams& prm, uint32_t rep, uint32_t kx, uint32_t ky, uint32_t kz) {
  float rx, ry, rz;
  load_xyz_global<GENERIC>(prm, rep, rx, ry, rz);
  return __float_as_uint(rx) == kx && __float_as_uint(ry) == ky && __float_as_uint(rz) == kz;
}

// Pass 1 of duplicate removal over the raw byte buffers.
template <bool GENERIC>
__global__ void __launch_bounds__(APC_TILE_THREADS) k_dedup_insert(const __grid_constant__ FrontendParams prm) {
  extern __shared__ __align__(16) uint8_t stage[];
  __shared__ __align__(8) uint64_t bar;
  pdl_enter();
  const uint32_t tile = blockIdx.x;
  const uint32_t si = find_segment(prm, tile);
  const SegDev& s = prm.seg[si];
  TilePoint pt[APC_TILE_ITEMS];
  APC_STAMP(0, 0);
  load_tile<GENERIC>(s, tile - s.tile_begin, prm.skip_nans != 0, stage, &bar, pt);
  if (pt[0].x == 123456.f) APC_STAMP(0, 3);   // data dependence: the stamp below follows the loads
  APC_STAMP(0, 1);
  uint64_t hash[APC_TILE_ITEMS];
  unsigned long long word[APC_TILE_ITEMS];
  bool act[APC_TILE_ITEMS];
  const uint32_t g0 = s.point_begin + (tile - s.tile_begin) * APC_TILE_POINTS + threadIdx.x;
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    act[j] = pt[j].valid && pt[j].no_nan;
    hash[j] = dedup_hash(pt[j].x, pt[j].y, pt[j].z);
    word[j] = dedup_word(hash[j], g0 + j * APC_TILE_THREADS);
  }
  // fingerprint hits are confirmed out of line (rare; keeps the probe loop small: inlined into
  // every probe the byte-record decoder made this kernel 190 KB of SASS)
  dedup_insert_items<APC_TILE_ITEMS>(prm.slots, prm.slot_mask, prm.p2slot, prm.ctrl, hash, word, act,
                                     [&](int j, uint32_t rep) {
    return dedup_same_record<GENERIC>(prm, rep, __float_as_uint(pt[j].x), __float_as_uint(pt[j].y), __float_as_uint(pt[j].z));
  });
  APC_STAMP(0, 2);
}

__device__ __forceinline__ bool crop_keep(const FrontendParams& prm, float x, float y, float z) {
  bool in_all, out_any;
  if (prm.crop_mode == APC_CROP_NUMPY) {
    const double px = (double)x, py = (double)y, pz = (double)z;
    in_all = (px >= prm.lo[0]) & (px <= prm.hi[0]) & (py >= prm.lo[1]) & (py <= prm.hi[1]) &
             (pz >= prm.lo[2]) & (pz <= prm.hi[2]);
    out_any = (px <= prm.lo[0]) | (px >= prm.hi[0]) | (py <= prm.lo[1]) | (py >= prm.hi[1]) |
              (pz <= prm.lo[2]) | (pz >= prm.hi[2]);
  } else {
    in_all = (x >= prm.lo32[0]) & (x <= prm.hi32[0]) & (y >= prm.lo32[1]) & (y <= prm.hi32[1]) &
             (z >= prm.lo32[2]) & (z <= prm.hi32[2]);
    out_any = (x <= prm.lo32[0]) | (x >= prm.hi32[0]) | (y <= prm.lo32[1]) | (y >= prm.hi32[1]) |
              (z <= prm.lo32[2]) | (z >= prm.hi32[2]);
  }
  if (!prm.crop_invert) return in_all;
  return prm.crop_mode == APC_CROP_OPEN3D ? !in_all : out_any;
}

template <bool GENERIC>
__global__ void __launch_bounds__(APC_TILE_THREADS) k_frontend(const __grid_constant__ FrontendParams prm) {
  extern __shared__ __align__(16) uint8_t stage[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t sm_scan[34];
  pdl_enter();
  const uint32_t tile = blockIdx.x;
  const uint32_t si = find_segment(prm, tile);
  const SegDev& s = prm.seg[si];
  const uint32_t epoch = prm.ctrl->epoch;
  TilePoint pt[APC_TILE_ITEMS];
  APC_STAMP(1, 0);
  load_tile<GENERIC>(s, tile - s.tile_begin, prm.skip_nans != 0, stage, &bar, pt);

  bool keep[APC_TILE_ITEMS];
  uint32_t gidx[APC_TILE_ITEMS];
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t g = s.point_begin + (tile - s.tile_begin) * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    gidx[j] = g;
    bool alive = pt[j].valid && pt[j].no_nan;
    uint32_t st = alive ? APC_STAGE_NANSKIP : 0u;
    if (prm.dedup && alive) {
      const uint32_t sl = prm.p2slot[g];
      alive = ((uint32_t)prm.slots[sl] == g);
      // the surviving representative resets its slot: the table is clean for the next frame
      if (alive) prm.slots[sl] = DEDUP_EMPTY;
    }
    if (alive) st |= APC_STAGE_DEDUP;
    float x = pt[j].x, y = pt[j].y, z = pt[j].z;
    if (prm.remove_nan && (is_nan_f(x) || is_nan_f(y) || is_nan_f(z))) alive = false;
    if (prm.remove_inf && (is_inf_f(x) || is_inf_f(y) || is_inf_f(z))) alive = false;
    if (alive) st |= APC_STAGE_FINITE;
    if (s.has_T) xform_f32(s.T, x, y, z);
    for (uint32_t k = 0; k < prm.n_T; ++k) xform_f32(prm.T[k], x, y, z);
    if (prm.crop_enable && alive) alive = crop_keep(prm, x, y, z);
    if (alive) st |= APC_STAGE_CROP;
    pt[j].x = x; pt[j].y = y; pt[j].z = z;
    keep[j] = alive;
    if (prm.out_stage && pt[j].valid) prm.out_stage[g] = (uint8_t)st;
  }
  uint32_t rank[APC_TILE_ITEMS];
  APC_STAMP(1, 1);
  const uint32_t base = tile_compact_offsets(keep, rank, sm_scan, prm.scan_state, tile, epoch,
                                             prm.out_count, prm.n_tiles);
  APC_STAMP(1, 2);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    if (keep[j]) {
      const uint32_t o = base + rank[j];
      prm.out_xyzi[o] = make_float4(pt[j].x, pt[j].y, pt[j].z, pt[j].w);
      if (prm.out_src) prm.out_src[o] = gidx[j];
    }
  }
  APC_STAMP(1, 3);
}

// Second half of the front end for the sorted duplicate-removal back ends (numpy / torch,
// utils.py:520-542): the rows to keep arrive as an index list into the NaN-skipped cloud (sorted
// first occurrences, or torch's inverse map), so the load is a gather; non-finite filter,
// transforms, crop and the ordered compaction are the same as in k_frontend.
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_frontend_gather(const __grid_constant__ FrontendParams prm, const float4* __restrict__ src,
                  const uint32_t* __restrict__ idx, const uint32_t* __restrict__ src_orig, uint32_t n_max,
                  const uint32_t* n_dev) {
  __shared__ uint32_t sm_scan[34];
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t epoch = prm.ctrl->epoch;
  const uint32_t tile = blockIdx.x;
  bool keep[APC_TILE_ITEMS];
  float4 v[APC_TILE_ITEMS];
  uint32_t g[APC_TILE_ITEMS];
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    keep[j] = false;
    g[j] = 0u;
    if (i < n) {
      g[j] = idx[i];
      const float4 p = src[g[j]];
      float x = p.x, y = p.y, z = p.z;
      bool alive = true;
      if (prm.remove_nan && (is_nan_f(x) || is_nan_f(y) || is_nan_f(z))) alive = false;
      if (prm.remove_inf && (is_inf_f(x) || is_inf_f(y) || is_inf_f(z))) alive = false;
      for (uint32_t k = 0; k < prm.n_T; ++k) xform_f32(prm.T[k], x, y, z);
      if (prm.crop_enable && alive) alive = crop_keep(prm, x, y, z);
      v[j] = make_float4(x, y, z, p.w);
      keep[j] = alive;
    }
  }
  uint32_t rank[APC_TILE_ITEMS];
  const uint32_t base = tile_compact_offsets(keep, rank, sm_scan, prm.scan_state, tile, epoch, prm.out_count, prm.n_tiles);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    if (keep[j]) {
      const uint32_t o = base + rank[j];
      prm.out_xyzi[o] = v[j];
      if (prm.out_src) prm.out_src[o] = src_orig ? src_orig[g[j]] : g[j];
    }
  }
}

// ---- generic fill (hash-table clears) -----------------------------------------------------
__global__ void k_fill_u32(uint32_t* p, uint32_t v, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
  for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    if (i + 3 < n) {
      *reinterpret_cast<uint4*>(p + i) = make_uint4(v, v, v, v);
    } else {
      for (size_t k = i; k < n; ++k) p[k] = v;
    }
  }
}
int apc_fill_u32(apc_ctx* ctx, void* p, uint32_t v, size_t n_words, cudaStream_t s) {
  if (n_words == 0) return APC_OK;
  const uint32_t blocks = (uint32_t)min((size_t)APC_SM_COUNT * 8, (n_words / 4 + 255) / 256 + 1);
  k_fill_u32<<<blocks, 256, 0, s>>>(reinterpret_cast<uint32_t*>(p), v, n_words);
  APC_LAUNCH_CHECK(ctx, "k_fill_u32");
  return APC_OK;
}

// ---- host side ------------------------------------------------------------------------------
static bool is_fast16(const apc_cloud_desc& c, uint8_t* nan_words) {
  if (c.point_step != 16 || (((uintptr_t)c.data_dev) & 15u)) return false;
  if (c.x.datatype != APC_FLOAT32 || c.y.datatype != APC_FLOAT32 || c.z.datatype != APC_FLOAT32) return false;
  if (c.x.offset != 0 || c.y.offset != 4 || c.z.offset != 8) return false;
  if (c.intensity.datatype != 0 && (c.intensity.datatype != APC_FLOAT32 || c.intensity.offset != 12)) return false;
  uint8_t w = 0;
  for (uint32_t f = 0; f < c.n_nan_fields; ++f) {
    const apc_field& nf = c.nan_fields[f];
    if (nf.datatype == APC_FLOAT32) {
      if (nf.offset & 3) return false;
      w |= (uint8_t)(1u << (nf.offset >> 2));
    } else if (nf.datatype == APC_FLOAT64) {
      return false;
    }  // integer fields are never NaN
  }
  *nan_words = w;
  return true;
}

static int field_size(int dt) {
  switch (dt) {
    case APC_INT8: case APC_UINT8: return 1;
    case APC_INT16: case APC_UINT16: return 2;
    case APC_INT32: case APC_UINT32: case APC_FLOAT32: return 4;
    case APC_FLOAT64: return 8;
    default: return 0;
  }
}

static int build_params(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                        const apc_filter_cfg* cfg, FrontendParams& prm, uint32_t* total_points,
                        uint32_t* smem_bytes) {
  APC_REQUIRE(ctx, clouds && n_clouds >= 1 && n_clouds <= APC_MAX_CLOUDS, "n_clouds out of range");
  memset(&prm, 0, sizeof(prm));
  uint32_t tiles = 0, points = 0, smem = 0;
  for (uint32_t i = 0; i < n_clouds; ++i) {
    const apc_cloud_desc& c = clouds[i];
    SegDev& s = prm.seg[i];
    APC_REQUIRE(ctx, c.n_points == 0 || c.data_dev, "cloud data pointer is NULL");
    APC_REQUIRE(ctx, c.point_step >= 1 && c.point_step <= 192, "point_step must be 1..192");
    APC_REQUIRE(ctx, c.n_nan_fields <= APC_MAX_FIELDS, "too many NaN-tested fields");
    const apc_field* f4[4] = {&c.x, &c.y, &c.z, &c.intensity};
    for (int k = 0; k < 4; ++k) {
      const int sz = field_size(f4[k]->datatype);
      APC_REQUIRE(ctx, (k == 3 && f4[k]->datatype == 0) || sz > 0, "x/y/z datatype invalid");
      APC_REQUIRE(ctx, f4[k]->offset >= 0 && (uint32_t)(f4[k]->offset + sz) <= c.point_step, "field outside the record");
      s.off[k] = (int16_t)f4[k]->offset;
      s.dt[k] = (uint8_t)f4[k]->datatype;
    }
    for (uint32_t f = 0; f < c.n_nan_fields; ++f) {
      const int sz = field_size(c.nan_fields[f].datatype);
      APC_REQUIRE(ctx, sz > 0 && c.nan_fields[f].offset >= 0 &&
                           (uint32_t)(c.nan_fields[f].offset + sz) <= c.point_step, "NaN field outside the record");
      s.nan_off[f] = (uint16_t)c.nan_fields[f].offset;
      s.nan_dt[f] = (uint8_t)c.nan_fields[f].datatype;
    }
    s.n_nan = (uint8_t)c.n_nan_fields;
    s.data = reinterpret_cast<const uint8_t*>(c.data_dev);
    s.n = c.n_points;
    s.step = c.point_step;
    s.tile_begin = tiles;
    s.point_begin = points;
    s.has_T = c.has_transform ? 1 : 0;
    memcpy(s.T, c.transform, sizeof(s.T));
    uint8_t nw = 0;
    s.fast16 = is_fast16(c, &nw) ? 1 : 0;
    s.nan_words = nw;
    if (!s.fast16) smem = max(smem, APC_TILE_POINTS * c.point_step);
    tiles += apc_div_up(c.n_points, APC_TILE_POINTS);
    APC_REQUIRE(ctx, (uint64_t)points + c.n_points <= ctx->max_points, "more points than the context was created for");
    points += c.n_points;
  }
  prm.n_seg = n_clouds;
  prm.n_tiles = tiles;
  if (cfg) {
    APC_REQUIRE(ctx, cfg->n_transforms <= APC_MAX_TRANSFORMS, "too many transforms");
    APC_REQUIRE(ctx, cfg->crop_mode >= 0 && cfg->crop_mode <= 2, "bad crop mode");
    APC_REQUIRE(ctx, cfg->dedup_mode >= APC_DEDUP_OFF && cfg->dedup_mode <= APC_DEDUP_TORCH_COMPAT, "bad dedup mode");
    prm.skip_nans = cfg->skip_nans != 0;
    prm.dedup = cfg->dedup_mode == APC_DEDUP_OPEN3D;
    prm.remove_nan = cfg->remove_nan != 0;
    prm.remove_inf = cfg->remove_inf != 0;
    prm.n_T = cfg->n_transforms;
    memcpy(prm.T, cfg->transforms, sizeof(prm.T));
    prm.crop_enable = cfg->crop_enable != 0;
    prm.crop_mode = (uint32_t)cfg->crop_mode;
    prm.crop_invert = cfg->crop_invert != 0;
    for (int k = 0; k < 3; ++k) {
      prm.lo[k] = cfg->roi_min[k];
      prm.hi[k] = cfg->roi_max[k];
      prm.lo32[k] = (float)cfg->roi_min[k];
      prm.hi32[k] = (float)cfg->roi_max[k];
    }
  }
  prm.slots = ctx->dedup_slots;
  // the whole duplicate table (one point in four slots): using half of it (load 0.5, half the 32-byte
  // sectors touched per scan) was slower, 69.7 vs 68.1 us/scan
  prm.slot_mask = ctx->hash_cap - 1;
  prm.p2slot = ctx->p2slot;
  prm.ctrl = ctx->ctrl;
  *total_points = points;
  *smem_bytes = smem;
  return APC_OK;
}

static int set_smem(apc_ctx* ctx, uint32_t smem) {
  // the attribute is per device: opt in once on every device a context lives on (both kernels share
  // the limit); static shared memory counts against the 48 KB default too, so opt in well below it
  static bool configured[64] = {};
  const int dev = ctx->device >= 0 && ctx->device < 64 ? ctx->device : 0;
  if (smem > 32 * 1024 && !configured[dev]) {
    APC_CUDA(ctx, cudaFuncSetAttribute(k_frontend<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 192 * 1024));
    APC_CUDA(ctx, cudaFuncSetAttribute(k_dedup_insert<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 192 * 1024));
    configured[dev] = true;
  }
  return APC_OK;
}

int apc_unique_rows_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, uint32_t*, uint32_t*, uint32_t*, int,
                            cudaStream_t);
int apc_sort_prepare(apc_ctx*);
int apc_frontend_nobegin(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                         const apc_filter_cfg* cfg, float* out_xyzi, uint32_t* out_src_idx,
                         uint8_t* out_stage_mask, uint32_t* out_count_dev, int scan_slot, cudaStream_t s);

// Front end with the numpy / torch duplicate-removal back ends: those return the rows in sorted
// order (utils.py:532-542), so the chain is NaN skip (k_frontend, everything else off) ->
// sorted unique rows (sort.cu) -> gather + remaining filters (k_frontend_gather).
static int frontend_sorted_dedup(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                 const apc_filter_cfg* cfg, float* out_xyzi, uint32_t* out_src_idx,
                                 uint8_t* out_stage_mask, uint32_t* out_count_dev, int scan_slot, cudaStream_t s) {
  APC_REQUIRE(ctx, !out_stage_mask, "per-point stage masks are not defined for the sorted duplicate-removal back ends");
  APC_REQUIRE(ctx, ctx->sort_a, "sort scratch not prepared");
  uint32_t n_total = 0;
  for (uint32_t i = 0; i < n_clouds && i < APC_MAX_CLOUDS; ++i) {
    APC_REQUIRE(ctx, !clouds[i].has_transform, "per-sensor transforms cannot be combined with the sorted duplicate-removal back ends");
    n_total += clouds[i].n_points;
  }
  apc_filter_cfg first;
  memset(&first, 0, sizeof(first));
  first.skip_nans = cfg->skip_nans;
  uint32_t* dc = ctx->dev_counts;
  float* stage_xyzi = reinterpret_cast<float*>(ctx->sorted_pts);
  int rc = apc_frontend_nobegin(ctx, clouds, n_clouds, &first, stage_xyzi, out_src_idx ? ctx->idx_a : nullptr, nullptr,
                                dc + 14, scan_slot, s);
  if (rc) return rc;
  if (n_total == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_count_dev, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  const bool numpy_mode = cfg->dedup_mode == APC_DEDUP_NUMPY;
  rc = apc_unique_rows_nobegin(ctx, stage_xyzi, n_total, dc + 14, numpy_mode ? ctx->sort_idx : nullptr,
                               numpy_mode ? nullptr : ctx->sort_idx, dc + 13, 5, s);
  if (rc) return rc;
  FrontendParams prm;
  uint32_t total = 0, smem = 0;
  rc = build_params(ctx, clouds, n_clouds, cfg, prm, &total, &smem);
  if (rc) return rc;
  prm.out_xyzi = reinterpret_cast<float4*>(out_xyzi);
  prm.out_src = out_src_idx;
  prm.out_count = out_count_dev;
  prm.scan_state = ctx->scan_state[6];
  prm.n_tiles = apc_div_up(n_total, APC_TILE_POINTS);
  APC_PROF(ctx, "k_frontend_gather", s);
  // numpy: one row per unique group; torch as written in the reference: one row per input row
  k_frontend_gather<<<prm.n_tiles, APC_TILE_THREADS, 0, s>>>(prm, ctx->sorted_pts, ctx->sort_idx,
                                                             out_src_idx ? ctx->idx_a : nullptr, n_total,
                                                             numpy_mode ? dc + 13 : dc + 14);
  APC_LAUNCH_CHECK(ctx, "k_frontend_gather");
  return APC_OK;
}

// Internal: front end without the epoch bump (the pipeline bumps once per run).
int apc_frontend_nobegin(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                         const apc_filter_cfg* cfg, float* out_xyzi, uint32_t* out_src_idx,
                         uint8_t* out_stage_mask, uint32_t* out_count_dev, int scan_slot, cudaStream_t s) {
  APC_REQUIRE(ctx, out_xyzi && out_count_dev, "output pointer is NULL");
  if (cfg && (cfg->dedup_mode == APC_DEDUP_NUMPY || cfg->dedup_mode == APC_DEDUP_TORCH_COMPAT))
    return frontend_sorted_dedup(ctx, clouds, n_clouds, cfg, out_xyzi, out_src_idx, out_stage_mask, out_count_dev,
                                 scan_slot, s);
  FrontendParams prm;
  uint32_t total = 0, smem = 0;
  int rc = build_params(ctx, clouds, n_clouds, cfg, prm, &total, &smem);
  if (rc) return rc;
  prm.out_xyzi = reinterpret_cast<float4*>(out_xyzi);
  prm.out_src = out_src_idx;
  prm.out_stage = out_stage_mask;
  prm.out_count = out_count_dev;
  prm.scan_state = ctx->scan_state[scan_slot];
  if (prm.n_tiles == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_count_dev, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  APC_REQUIRE(ctx, prm.n_tiles <= ctx->max_tiles, "too many tiles for this context");
  rc = set_smem(ctx, smem);
  if (rc) return rc;
  const bool generic = smem != 0;   // some segment needs the byte-record decoder
  if (prm.dedup) {
    APC_PROF(ctx, "k_dedup_insert", s);
    if (generic) apc_klaunch(ctx, k_dedup_insert<true>, prm.n_tiles, APC_TILE_THREADS, smem, s, prm);
    else apc_klaunch(ctx, k_dedup_insert<false>, prm.n_tiles, APC_TILE_THREADS, 0, s, prm);
    APC_LAUNCH_CHECK(ctx, "k_dedup_insert");
  }
  APC_PROF(ctx, "k_frontend", s);
  if (generic) apc_klaunch(ctx, k_frontend<true>, prm.n_tiles, APC_TILE_THREADS, smem, s, prm);
  else apc_klaunch(ctx, k_frontend<false>, prm.n_tiles, APC_TILE_THREADS, 0, s, prm);
  APC_LAUNCH_CHECK(ctx, "k_frontend");
  return APC_OK;
}

int apc_dedup_reset(apc_ctx* ctx, cudaStream_t s) {
  return apc_fill_u32(ctx, ctx->dedup_slots, 0xffffffffu, (size_t)ctx->hash_cap * 2, s);
}

extern "C" int apc_frontend(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                            const apc_filter_cfg* cfg, float* out_xyzi, uint32_t* out_src_idx,
                            uint8_t* out_stage_mask, uint32_t* out_count_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = APC_OK;
  if (cfg && cfg->dedup_mode >= APC_DEDUP_NUMPY) rc = apc_sort_prepare(ctx);
  if (!rc) rc = apc_begin(ctx, s);
  if (rc) return rc;
  return apc_frontend_nobegin(ctx, clouds, n_clouds, cfg, out_xyzi, out_src_idx, out_stage_mask,
                              out_count_dev, 0, s);
}

extern "C" int apc_unpack(apc_ctx* ctx, const apc_cloud_desc* cloud, float* out_xyzi, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  apc_cloud_desc c = *cloud;
  c.has_transform = 0;
  return apc_frontend_nobegin(ctx, &c, 1, nullptr, out_xyzi, nullptr, nullptr, ctx->dev_counts + 15, 0, s);
}

// ---- SoA stand-alone kernels ------------------------------------------------------------------
struct F16 { float v[16]; };

__global__ void k_transform(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
                            const __grid_constant__ F16 T, float4* __restrict__ out) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float4 p = in[i];
    xform_f32(T.v, p.x, p.y, p.z);
    out[i] = p;
  }
}

extern "C" int apc_transform(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                             const float* T16_host, float* out_xyzi, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, T16_host && (n_max == 0 || (xyzi && out_xyzi)), "NULL pointer");
  if (n_max == 0) return APC_OK;
  F16 T;
  memcpy(T.v, T16_host, sizeof(T.v));
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_transform<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(xyzi), n_max, n_dev, T,
                                                        reinterpret_cast<float4*>(out_xyzi));
  APC_LAUNCH_CHECK(ctx, "k_transform");
  return APC_OK;
}

struct CropPrm {
  uint32_t crop_mode, crop_invert;
  double lo[3], hi[3];
  float lo32[3], hi32[3];
};

__global__ void k_crop_mask(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
                            const __grid_constant__ CropPrm c, uint8_t* __restrict__ mask) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    bool in_all, out_any;
    if (c.crop_mode == APC_CROP_NUMPY) {
      const double px = p.x, py = p.y, pz = p.z;
      in_all = (px >= c.lo[0]) & (px <= c.hi[0]) & (py >= c.lo[1]) & (py <= c.hi[1]) & (pz >= c.lo[2]) & (pz <= c.hi[2]);
      out_any = (px <= c.lo[0]) | (px >= c.hi[0]) | (py <= c.lo[1]) | (py >= c.hi[1]) | (pz <= c.lo[2]) | (pz >= c.hi[2]);
    } else {
      in_all = (p.x >= c.lo32[0]) & (p.x <= c.hi32[0]) & (p.y >= c.lo32[1]) & (p.y <= c.hi32[1]) &
               (p.z >= c.lo32[2]) & (p.z <= c.hi32[2]);
      out_any = (p.x <= c.lo32[0]) | (p.x >= c.hi32[0]) | (p.y <= c.lo32[1]) | (p.y >= c.hi32[1]) |
                (p.z <= c.lo32[2]) | (p.z >= c.hi32[2]);
    }
    bool k = in_all;
    if (c.crop_invert) k = (c.crop_mode == APC_CROP_OPEN3D) ? !in_all : out_any;
    mask[i] = k ? 1 : 0;
  }
}

extern "C" int apc_crop_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                             const double* roi_min, const double* roi_max, int mode, int invert,
                             uint8_t* out_mask, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, roi_min && roi_max && mode >= 0 && mode <= 2, "bad crop arguments");
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_mask, "NULL pointer");
  CropPrm c;
  c.crop_mode = (uint32_t)mode;
  c.crop_invert = invert != 0;
  for (int k = 0; k < 3; ++k) {
    c.lo[k] = roi_min[k]; c.hi[k] = roi_max[k];
    c.lo32[k] = (float)roi_min[k]; c.hi32[k] = (float)roi_max[k];
  }
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_crop_mask<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(xyzi), n_max, n_dev, c, out_mask);
  APC_LAUNCH_CHECK(ctx, "k_crop_mask");
  return APC_OK;
}

__global__ void k_non_finite_mask(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
                                  int rm_nan, int rm_inf, uint8_t* __restrict__ mask) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    bool k = true;
    if (rm_nan && (is_nan_f(p.x) || is_nan_f(p.y) || is_nan_f(p.z))) k = false;
    if (rm_inf && (is_inf_f(p.x) || is_inf_f(p.y) || is_inf_f(p.z))) k = false;
    mask[i] = k ? 1 : 0;
  }
}

extern "C" int apc_non_finite_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                   int remove_nan, int remove_inf, uint8_t* out_mask, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_mask, "NULL pointer");
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_non_finite_mask<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(xyzi), n_max, n_dev,
                                                              remove_nan, remove_inf, out_mask);
  APC_LAUNCH_CHECK(ctx, "k_non_finite_mask");
  return APC_OK;
}

__global__ void k_dup_insert_soa(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
                                 unsigned long long* slots, uint32_t mask, uint32_t* p2slot, ApcCtrl* ctrl) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    const uint64_t hash[1] = {dedup_hash(p.x, p.y, p.z)};
    const unsigned long long word[1] = {dedup_word(hash[0], i)};
    bool act[1] = {true};
    dedup_insert_items<1>(slots, mask, p2slot, ctrl, hash, word, act, [&](int, uint32_t rep) {
      const float4 r = in[rep];
      return __float_as_uint(r.x) == __float_as_uint(p.x) && __float_as_uint(r.y) == __float_as_uint(p.y) &&
             __float_as_uint(r.z) == __float_as_uint(p.z);
    });
  }
}
__global__ void k_dup_mask_soa(uint32_t n_max, const uint32_t* n_dev, unsigned long long* __restrict__ slots,
                               const uint32_t* __restrict__ p2slot, uint8_t* __restrict__ mask) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t sl = p2slot[i];
    const bool win = (uint32_t)slots[sl] == i;
    mask[i] = win ? 1 : 0;
    if (win) slots[sl] = DEDUP_EMPTY;  // self-clean
  }
}

extern "C" int apc_duplicate_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                  uint8_t* out_mask, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_mask, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_dup_insert_soa<<<blocks, 256, 0, s>>>(reinterpret_cast<const float4*>(xyzi), n_max, n_dev, ctx->dedup_slots,
                                          ctx->hash_cap - 1, ctx->p2slot, ctx->ctrl);
  APC_LAUNCH_CHECK(ctx, "k_dup_insert_soa");
  k_dup_mask_soa<<<blocks, 256, 0, s>>>(n_max, n_dev, ctx->dedup_slots, ctx->p2slot, out_mask);
  APC_LAUNCH_CHECK(ctx, "k_dup_mask_soa");
  return APC_OK;
}

// order-preserving select_by_mask over an SoA cloud
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_select_by_mask(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev, const uint8_t* __restrict__ mask,
                 int invert, float4* __restrict__ out, uint32_t* __restrict__ out_idx, uint32_t* out_count,
                 uint64_t* scan_state, const ApcCtrl* ctrl, uint32_t n_tiles, const uint32_t* __restrict__ idx_in,
                 const __grid_constant__ MirrorDev mir) {
  __shared__ uint32_t sm_scan[34];
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t epoch = ctrl->epoch;
  const uint32_t tile = blockIdx.x;
  bool keep[APC_TILE_ITEMS];
  float4 v[APC_TILE_ITEMS];
  APC_STAMP(2, 0);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    keep[j] = false;
    if (i < n) {
      keep[j] = (mask[i] != 0) != (invert != 0);
      if (in) v[j] = in[i];
    }
  }
  uint32_t rank[APC_TILE_ITEMS];
  APC_STAMP(2, 1);
  const uint32_t base = tile_compact_offsets(keep, rank, sm_scan, scan_state, tile, epoch, out_count, n_tiles);
  APC_STAMP(2, 2);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    if (keep[j]) {
      const uint32_t o = base + rank[j];
      if (out) out[o] = v[j];
      mirror_store(mir, o, v[j]);
      if (out_idx) {   // index of the survivor in this stage's input, or (idx_in) in an earlier stage's
        const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
        out_idx[o] = idx_in ? idx_in[i] : i;
      }
    }
  }
  APC_STAMP(2, 3);
}

int apc_select_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                       const uint8_t* mask, int invert, float* out_xyzi, uint32_t* out_idx,
                       uint32_t* out_count_dev, int scan_slot, cudaStream_t s, const uint32_t* idx_in,
                       const MirrorDev* mir) {
  APC_REQUIRE(ctx, out_count_dev, "out_count_dev is NULL");
  APC_REQUIRE(ctx, !mir || mir->n == 0 || xyzi, "mirrored output needs the point rows");
  if (n_max == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_count_dev, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  APC_REQUIRE(ctx, mask, "mask is NULL");
  const uint32_t n_tiles = apc_div_up(n_max, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more points than the context was created for");
  APC_PROF(ctx, "k_select_by_mask", s);
  apc_klaunch(ctx, k_select_by_mask, n_tiles, APC_TILE_THREADS, 0, s, reinterpret_cast<const float4*>(xyzi), n_max, n_dev, mask, invert,
                                                        reinterpret_cast<float4*>(out_xyzi), out_idx, out_count_dev,
                                                        ctx->scan_state[scan_slot], ctx->ctrl, n_tiles, idx_in,
                                                        mir ? *mir : MirrorDev{});
  APC_LAUNCH_CHECK(ctx, "k_select_by_mask");
  return APC_OK;
}

extern "C" int apc_select_by_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                  const uint8_t* mask, int invert, float* out_xyzi, uint32_t* out_idx,
                                  uint32_t* out_count_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  return apc_select_nobegin(ctx, xyzi, n_max, n_dev, mask, invert, out_xyzi, out_idx, out_count_dev, 0, s, nullptr, nullptr);
}

template <typename T>
__global__ void k_gather(const T* __restrict__ src, const uint32_t* __restrict__ idx, uint32_t n_max,
                         const uint32_t* n_dev, T* __restrict__ out) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = src[idx[i]];
}
struct B12 { uint32_t a, b, c; };

extern "C" int apc_gather(apc_ctx* ctx, const void* src, uint32_t elem_size, const uint32_t* idx,
                          uint32_t n_max, const uint32_t* n_dev, void* out, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, src && idx && out, "NULL pointer");
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  switch (elem_size) {
    case 1: k_gather<uint8_t><<<blocks, 256, 0, s>>>((const uint8_t*)src, idx, n_max, n_dev, (uint8_t*)out); break;
    case 2: k_gather<uint16_t><<<blocks, 256, 0, s>>>((const uint16_t*)src, idx, n_max, n_dev, (uint16_t*)out); break;
    case 4: k_gather<uint32_t><<<blocks, 256, 0, s>>>((const uint32_t*)src, idx, n_max, n_dev, (uint32_t*)out); break;
    case 8: k_gather<uint64_t><<<blocks, 256, 0, s>>>((const uint64_t*)src, idx, n_max, n_dev, (uint64_t*)out); break;
    case 12: k_gather<B12><<<blocks, 256, 0, s>>>((const B12*)src, idx, n_max, n_dev, (B12*)out); break;
    case 16: k_gather<uint4><<<blocks, 256, 0, s>>>((const uint4*)src, idx, n_max, n_dev, (uint4*)out); break;
    default: return apc_set_error(ctx, APC_ERR_BAD_ARG, "elem_size must be 1,2,4,8,12 or 16");
  }
  APC_LAUNCH_CHECK(ctx, "k_gather");
  return APC_OK;
}

// ---- carrier layout glue: positions float32[N,3] (+ intensity float32[N]) <-> SoA float4 -------
// The Open3D-style carrier keeps `positions` as N x 3 (utils.py:102-104, pp.py:426) while every
// kernel works on float4 records; these two kernels convert without touching the host.
__global__ void k_pack_xyzi(const float* __restrict__ pos3, const float* __restrict__ inten, uint32_t n,
                            float4* __restrict__ out) {
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = make_float4(pos3[3 * (size_t)i], pos3[3 * (size_t)i + 1], pos3[3 * (size_t)i + 2], inten ? inten[i] : 0.0f);
}
__global__ void k_split_xyzi(const float4* __restrict__ in, uint32_t n_max, const uint32_t* n_dev,
                             float* __restrict__ pos3, float* __restrict__ inten) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = in[i];
    pos3[3 * (size_t)i] = p.x; pos3[3 * (size_t)i + 1] = p.y; pos3[3 * (size_t)i + 2] = p.z;
    if (inten) inten[i] = p.w;
  }
}

extern "C" int apc_pack_xyzi(apc_ctx* ctx, const float* pos3, const float* intensity, uint32_t n, float* out_xyzi,
                             void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n == 0) return APC_OK;
  APC_REQUIRE(ctx, pos3 && out_xyzi, "NULL pointer");
  k_pack_xyzi<<<min(apc_div_up(n, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, (cudaStream_t)stream>>>(
      pos3, intensity, n, reinterpret_cast<float4*>(out_xyzi));
  APC_LAUNCH_CHECK(ctx, "k_pack_xyzi");
  return APC_OK;
}

extern "C" int apc_split_xyzi(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, float* out_pos3,
                              float* out_intensity, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, xyzi && out_pos3, "NULL pointer");
  k_split_xyzi<<<min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(xyzi), n_max, n_dev, out_pos3, out_intensity);
  APC_LAUNCH_CHECK(ctx, "k_split_xyzi");
  return APC_OK;
}
