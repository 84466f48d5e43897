// Voxel-grid mean downsampling on packed 63-bit voxel keys.
//
// Replaces Open3D t.PointCloud.voxel_down_sample (pp.py:509-512; SURVEY.md B7).
//   key       = floor(float32(x) / float32(voxel_size)) per axis, 21 bits each (+2^20 bias)
//   table     = open addressing, 64-bit atomicCAS on the key word of a 16-byte hot slot; the four voxels
//               of a 2x2 (x, y) block share one 64-byte burst, probing moves block by block (see VoxSlot)
//   centroid  = order-independent fixed-point sums (rint(x*2^24), 64-bit integer atomics) so
//               the result is deterministic and bit-identical to oracle/voxel.py
//               centroids_fixed whatever order the atomics land in; the point that claims a
//               slot adds nothing atomically (see VoxSlot)
//   order     = first-occurrence: a point is "first" when it holds the lowest index of its
//               slot; an order-preserving scan over the first-flags numbers the voxels
// The table is self-cleaning: the thread that finalises a voxel resets its slot, so no
// per-frame memset of the (capacity x 64 B) table sits on the critical path.
#include "apc_scan.cuh"
#include "apc_grid.cuh"
APC_TRACE_EXPORT(voxel)

#define VOX_EMPTY 0xffffffffffffffffull
#define VOX_NOSLOT 0xffffffffu

__device__ __forceinline__ bool voxel_key(float4 p, float vs, uint64_t& key) {
  const float lim = 65536.0f;
  if (!(fabsf(p.x) < lim && fabsf(p.y) < lim && fabsf(p.z) < lim)) return false;  // also rejects NaN
  const float qx = floorf(__fdiv_rn(p.x, vs)), qy = floorf(__fdiv_rn(p.y, vs)), qz = floorf(__fdiv_rn(p.z, vs));
  const float h = 1048576.0f;
  if (!(qx >= -h && qx < h && qy >= -h && qy < h && qz >= -h && qz < h)) return false;
  const uint64_t ux = (uint64_t)((int64_t)qx + 1048576), uy = (uint64_t)((int64_t)qy + 1048576),
                 uz = (uint64_t)((int64_t)qz + 1048576);
  key = (ux << 42) | (uy << 21) | uz;
  return true;
}

// rint(v * 2^24) / rint(w * 2^20): exact product in float64, round-half-even like numpy.rint
__device__ __forceinline__ unsigned long long fixed_xyz(float v) {
  return (unsigned long long)__double2ll_rn((double)v * 16777216.0);
}
__device__ __forceinline__ unsigned long long fixed_intensity(float w, ApcCtrl* ctrl) {
  if (fabsf(w) < 1048576.0f) return (unsigned long long)__double2ll_rn((double)w * 1048576.0);
  atomicOr(&ctrl->err, APC_DEVERR_KEY_RANGE);
  return 0ull;
}

// One point per thread: the key CAS, the probes when the slot holds another voxel, then a joiner's
// accumulations.  Four points per thread with their atomics issued in lockstep was slower both alone
// (23.5 vs 15.7 us: more resident warps hide the dependent atomic chain) and with eight lanes sharing the GPU
// (70.5 vs 68.9 us/scan, profiles/r2g_knobs.json) although it held half the registers: the atomic round
// trips, not the register file, set this kernel's cost.
__global__ void __launch_bounds__(256)
k_voxel_insert(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, float vs,
               VoxSlot* __restrict__ slots, VoxAcc* __restrict__ accs, uint32_t cap_mask, uint32_t* __restrict__ p2slot,
               ApcCtrl* ctrl) {
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  APC_STAMP(0, 0);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float4 p = pts[i];
    uint64_t key = 0;
    if (!voxel_key(p, vs, key)) {
      atomicOr(&ctrl->err, APC_DEVERR_KEY_RANGE);
      p2slot[i] = VOX_NOSLOT;
      continue;
    }
    // block = the voxel's 2x2 neighbourhood in x, y (bit 0 of either index cleared); sub = its place in it
    const uint64_t block = key & ~((1ull << 42) | (1ull << 21));
    const uint32_t sub = (uint32_t)((key >> 42) & 1ull) | ((uint32_t)((key >> 21) & 1ull) << 1);
    uint32_t slot = ((((uint32_t)mix64(block)) << 2) & cap_mask) | sub;
    unsigned long long old = atomicCAS(&slots[slot].key, VOX_EMPTY, (unsigned long long)key);
    for (uint32_t probe = 1; old != VOX_EMPTY && old != key && probe <= (cap_mask >> 2); ++probe) {  // next block, same place
      slot = (slot + 4) & cap_mask;
      old = atomicCAS(&slots[slot].key, VOX_EMPTY, (unsigned long long)key);
    }
    VoxSlot* s = &slots[slot];
    if (old == VOX_EMPTY) {          // owner: nothing to accumulate yet
      s->owner = i;
      p2slot[i] = slot;
    } else if (old == key) {         // joins an existing voxel
      p2slot[i] = slot;
      atomicMin(&s->first, i);
      VoxAcc* a = &accs[slot];
      atomicAdd(&a->cnt, 1u);
      atomicAdd(&a->acc[0], fixed_xyz(p.x));
      atomicAdd(&a->acc[1], fixed_xyz(p.y));
      atomicAdd(&a->acc[2], fixed_xyz(p.z));
      atomicAdd(&a->acc[3], fixed_intensity(p.w, ctrl));
    } else {
      atomicOr(&ctrl->err, APC_DEVERR_CAPACITY);
      p2slot[i] = VOX_NOSLOT;
    }
  }
  APC_STAMP(0, 1);
}

__device__ __forceinline__ float fixed_mean(unsigned long long sum, double cnt, double inv_scale) {
  return __double2float_rn(__dmul_rn(__ddiv_rn(__ll2double_rn((long long)sum), cnt), inv_scale));
}

// A point is its voxel's FIRST when it holds the lowest index of the voxel (owner or joiner); the
// order-preserving scan over the first-flags numbers the voxels in first-occurrence order.  The
// centroid (owner's coordinates + the joiners' sums, exact integers, one float64 divide) is
// computed BEFORE the cross-tile scan so that the slot and owner loads overlap the scan's wait;
// after the scan only stores remain.
// GRID: the pipeline's next stage is radius outlier removal - every centroid is inserted into the
// neighbour grid right here (cell claim + arrival rank, whose atomics also overlap the scan's wait)
// and the stand-alone k_grid_insert pass over the centroids is not launched.
template <bool GRID>
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_voxel_finalize(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, const uint32_t* __restrict__ p2slot,
                 VoxSlot* __restrict__ slots, VoxAcc* __restrict__ accs, uint32_t* __restrict__ rank_of_slot,
                 float4* __restrict__ out, uint32_t* __restrict__ out_counts, uint32_t* out_count,
                 uint64_t* scan_state, ApcCtrl* ctrl, uint32_t n_tiles, const __grid_constant__ GridDev grid) {
  __shared__ uint32_t sm_scan[34];
  pdl_enter();
  const uint32_t n = apc_count(n_dev, n_max);
  const uint32_t epoch = ctrl->epoch;
  const uint32_t tile = blockIdx.x;
  bool is_first[APC_TILE_ITEMS];
  uint32_t slot[APC_TILE_ITEMS];
  uint4 head[APC_TILE_ITEMS];
  APC_STAMP(1, 0);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    slot[j] = i < n ? p2slot[i] : VOX_NOSLOT;
  }
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j)     // the whole hot slot {key lo, key hi, first, owner} in one load: all in flight
    head[j] = slot[j] != VOX_NOSLOT ? ld_relaxed_u4(&slots[slot[j]]) : make_uint4(0u, 0u, 0u, 0u);
  float4 cen[APC_TILE_ITEMS];
  uint32_t npts[APC_TILE_ITEMS];
  uint32_t gslot[APC_TILE_ITEMS], grank[APC_TILE_ITEMS];
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = tile * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    // a slot whose key already reads empty was finalised (and cleaned) by an earlier tile: this
    // point is then certainly not the first of its voxel
    is_first[j] = slot[j] != VOX_NOSLOT && !(head[j].x == 0xffffffffu && head[j].y == 0xffffffffu) &&
                  i == min(head[j].z, head[j].w);
    npts[j] = 1u;
    if (is_first[j]) {
      const float4 po = pts[head[j].w];   // the owner - mostly i itself: 3 voxels in 4 hold one point
      ulonglong2 a01 = make_ulonglong2(0ull, 0ull), a23 = make_ulonglong2(0ull, 0ull);
      if (head[j].z != 0xffffffffu) {     // somebody joined: sums and their count live in the cold record
        const uint4* raw = reinterpret_cast<const uint4*>(&accs[slot[j]]);
        a01 = *reinterpret_cast<const ulonglong2*>(&raw[0]);
        a23 = *reinterpret_cast<const ulonglong2*>(&raw[1]);
        npts[j] = raw[2].x + 1u;
      }
      const double dc = (double)npts[j];
      cen[j] = make_float4(fixed_mean(a01.x + fixed_xyz(po.x), dc, 1.0 / 16777216.0),
                           fixed_mean(a01.y + fixed_xyz(po.y), dc, 1.0 / 16777216.0),
                           fixed_mean(a23.x + fixed_xyz(po.z), dc, 1.0 / 16777216.0),
                           fixed_mean(a23.y + fixed_intensity(po.w, ctrl), dc, 1.0 / 1048576.0));
    }
  }
  uint32_t rank[APC_TILE_ITEMS];
  APC_STAMP(1, 1);
  // ranks inside the tile, publish the tile's total, THEN the grid atomics (the successors' wait
  // does not include them), then collect the predecessors' totals
  const uint32_t total = tile_ranks(is_first, rank, sm_scan);
  if (threadIdx.x == 0) scan_publish(scan_state, tile, epoch, total);
  if (GRID) grid_insert_items<APC_TILE_ITEMS>(grid, 0, is_first, cen, grid.cell0, ctrl, gslot, grank);
  const uint32_t base = scan_two_level_impl<true>(scan_state, tile, n_tiles, epoch, total, &sm_scan[33]);
  if (threadIdx.x == 0 && tile == n_tiles - 1 && out_count) *out_count = base + total;
  APC_STAMP(1, 2);
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    if (is_first[j]) {
      const uint32_t s = slot[j];
      const uint32_t r = base + rank[j];
      out[r] = cen[j];
      if (GRID) {
        grid.slot[r] = gslot[j];
        grid.rank[r] = grank[j];
      }
      if (out_counts) out_counts[r] = npts[j];
      if (rank_of_slot) rank_of_slot[s] = r;   // only the point->voxel map needs it (a scattered 4-byte store per voxel)
      // self-clean the slot for the next frame: {key = empty, first = none, owner = 0}; the cold record
      // only where it was written
      st_relaxed_u4(&slots[s], make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0u));
      if (npts[j] > 1u) {
        uint4* raw = reinterpret_cast<uint4*>(&accs[s]);
        raw[0] = make_uint4(0u, 0u, 0u, 0u);
        raw[1] = make_uint4(0u, 0u, 0u, 0u);
        raw[2] = make_uint4(0u, 0u, 0u, 0u);
      }
    }
  }
  APC_STAMP(1, 3);
}

__global__ void k_voxel_p2v(uint32_t n_max, const uint32_t* n_dev, const uint32_t* __restrict__ p2slot,
                            const uint32_t* __restrict__ rank_of_slot, int32_t* __restrict__ p2v) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = p2slot[i];
    p2v[i] = (s == VOX_NOSLOT) ? -1 : (int32_t)rank_of_slot[s];
  }
}

// Whole-table reset (context creation and error recovery only).
__global__ void k_voxel_reset(VoxSlot* slots, VoxAcc* accs, uint32_t cap) {
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += gridDim.x * blockDim.x) {
    *reinterpret_cast<uint4*>(&slots[s]) = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0u);
    uint4* acc = reinterpret_cast<uint4*>(&accs[s]);
    acc[0] = make_uint4(0u, 0u, 0u, 0u);
    acc[1] = make_uint4(0u, 0u, 0u, 0u);
    acc[2] = make_uint4(0u, 0u, 0u, 0u);
  }
}

int apc_voxel_reset(apc_ctx* ctx, cudaStream_t s) {
  k_voxel_reset<<<APC_SM_COUNT * 4, 256, 0, s>>>(ctx->vox_slots, ctx->vox_acc, ctx->hash_cap);
  APC_LAUNCH_CHECK(ctx, "k_voxel_reset");
  return APC_OK;
}

// `radius_grid`: when non-NULL the centroids are also inserted into that neighbour grid (see GRID above).
int apc_voxel_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, float voxel_size,
                      float* out_xyzi, int32_t* out_p2v, uint32_t* out_voxel_counts, uint32_t* out_count_dev,
                      int scan_slot, const GridDev* radius_grid, cudaStream_t s) {
  APC_REQUIRE(ctx, out_count_dev, "out_count_dev is NULL");
  APC_REQUIRE(ctx, voxel_size > 0.0f, "voxel_size must be > 0");
  if (n_max == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_count_dev, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  APC_REQUIRE(ctx, xyzi && out_xyzi, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  {
    APC_PROF(ctx, "k_voxel_insert", s);
    apc_klaunch(ctx, k_voxel_insert, blocks, 256, 0, s, reinterpret_cast<const float4*>(xyzi), n_max, n_dev, voxel_size, ctx->vox_slots,
                ctx->vox_acc, ctx->hash_cap - 1, ctx->p2slot, ctx->ctrl);
  }
  APC_LAUNCH_CHECK(ctx, "k_voxel_insert");
  const uint32_t n_tiles = apc_div_up(n_max, APC_TILE_POINTS);
  APC_PROF(ctx, "k_voxel_finalize", s);
  if (radius_grid)
    apc_klaunch(ctx, k_voxel_finalize<true>, n_tiles, APC_TILE_THREADS, 0, s,
        reinterpret_cast<const float4*>(xyzi), n_max, n_dev, ctx->p2slot, ctx->vox_slots, ctx->vox_acc, out_p2v ? ctx->vox_rank : nullptr,
        reinterpret_cast<float4*>(out_xyzi), out_voxel_counts, out_count_dev, ctx->scan_state[scan_slot], ctx->ctrl,
        n_tiles, *radius_grid);
  else
    apc_klaunch(ctx, k_voxel_finalize<false>, n_tiles, APC_TILE_THREADS, 0, s,
        reinterpret_cast<const float4*>(xyzi), n_max, n_dev, ctx->p2slot, ctx->vox_slots, ctx->vox_acc, out_p2v ? ctx->vox_rank : nullptr,
        reinterpret_cast<float4*>(out_xyzi), out_voxel_counts, out_count_dev, ctx->scan_state[scan_slot], ctx->ctrl,
        n_tiles, GridDev{});
  APC_LAUNCH_CHECK(ctx, "k_voxel_finalize");
  if (out_p2v) {
    k_voxel_p2v<<<blocks, 256, 0, s>>>(n_max, n_dev, ctx->p2slot, ctx->vox_rank, out_p2v);
    APC_LAUNCH_CHECK(ctx, "k_voxel_p2v");
  }
  return APC_OK;
}

extern "C" int apc_voxel_downsample(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                    float voxel_size, float* out_xyzi, int32_t* out_p2v,
                                    uint32_t* out_voxel_counts, uint32_t* out_count_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  return apc_voxel_nobegin(ctx, xyzi, n_max, n_dev, voxel_size, out_xyzi, out_p2v, out_voxel_counts, out_count_dev, 1,
                           nullptr, s);
}

// Per-attribute voxel mean (Open3D: attr.to(float32) -> index_add -> sum / count, SURVEY.md B7), made
// ORDER-INDEPENDENT like the positions: every value is accumulated as the integer rint(v * 2^frac_bits)
// (64-bit atomics), the mean is one float64 divide rounded to float32.  Deterministic whatever order the
// atomics land in, bit-equal to oracle/voxel.py centroids_fixed(scale = 2^frac_bits); for integer-valued
// attributes (ring, return_type, integer time stamps: frac_bits = 0) the sums are exact, which is also what
// Open3D's float32 serial sum gives while it stays below 2^24.  |v * 2^frac_bits| must be < 2^40.
struct AttrAcc {
  long long sum;
  uint32_t cnt;
  uint32_t pad;
};
static_assert(sizeof(AttrAcc) == 16, "AttrAcc aliases the float4 scratch");
__global__ void k_attr_zero(uint32_t n_max, const uint32_t* n_vox, AttrAcc* acc) {
  const uint32_t n = apc_count(n_vox, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    *reinterpret_cast<uint4*>(&acc[i]) = make_uint4(0u, 0u, 0u, 0u);
}
__global__ void k_attr_add(const float* __restrict__ attr, const int32_t* __restrict__ p2v, uint32_t n_max,
                           const uint32_t* n_dev, double scale, AttrAcc* acc, ApcCtrl* ctrl) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int32_t v = p2v[i];
    if (v < 0) continue;
    const double q = __dmul_rn((double)attr[i], scale);
    if (!(fabs(q) < 1099511627776.0)) {          // 2^40 (also rejects NaN / inf)
      atomicOr(&ctrl->err, APC_DEVERR_KEY_RANGE);
      continue;
    }
    atomicAdd(reinterpret_cast<unsigned long long*>(&acc[v].sum), (unsigned long long)__double2ll_rn(q));
    atomicAdd(&acc[v].cnt, 1u);
  }
}
__global__ void k_attr_div(uint32_t n_max, const uint32_t* n_vox, const AttrAcc* __restrict__ acc, double inv_scale,
                           float* __restrict__ out) {
  const uint32_t n = apc_count(n_vox, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    out[i] = __double2float_rn(__dmul_rn(__ddiv_rn(__ll2double_rn(acc[i].sum), (double)acc[i].cnt), inv_scale));
}

extern "C" int apc_voxel_mean_attr(apc_ctx* ctx, const float* attr, const int32_t* p2v, uint32_t n_max,
                                   const uint32_t* n_dev, const uint32_t* n_voxels_dev, int32_t frac_bits,
                                   float* out_attr, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  if (n_max == 0) return APC_OK;
  APC_REQUIRE(ctx, attr && p2v && out_attr, "NULL pointer");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  APC_REQUIRE(ctx, frac_bits >= 0 && frac_bits <= 30, "frac_bits must be in 0..30");
  cudaStream_t s = (cudaStream_t)stream;
  AttrAcc* acc = reinterpret_cast<AttrAcc*>(ctx->sorted_pts);   // scratch reuse: [max_points] x 16 bytes
  const double scale = (double)(1u << frac_bits);
  const uint32_t blocks = min(apc_div_up(n_max, 256), (uint32_t)APC_SM_COUNT * 8);
  k_attr_zero<<<blocks, 256, 0, s>>>(n_max, n_voxels_dev, acc);
  k_attr_add<<<blocks, 256, 0, s>>>(attr, p2v, n_max, n_dev, scale, acc, ctx->ctrl);
  k_attr_div<<<blocks, 256, 0, s>>>(n_max, n_voxels_dev, acc, 1.0 / scale, out_attr);
  APC_LAUNCH_CHECK(ctx, "k_attr_*");
  return APC_OK;
}
