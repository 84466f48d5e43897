// PointCloud2 byte-record loader: AoS bytes (arbitrary point_step / field offsets / datatypes)
// -> per-thread (x, y, z, intensity) float registers.
//
// Two paths, chosen per sensor segment on the host:
//   FAST16  - point_step == 16, x/y/z(/intensity) float32 at 0/4/8/12, 16-byte aligned base:
//             one coalesced 128-bit streaming load per point, no staging.
//   GENERIC - the tile's bytes are staged into shared memory with one TMA bulk copy
//             (cp.async.bulk, completion on an mbarrier) so HBM sees full-line sequential
//             reads whatever the record stride; fields are then picked out of shared memory.
#pragma once
#include "apc_scan.cuh"

// Compact per-segment descriptor passed by value in kernel parameters.
struct SegDev {
  const uint8_t* data;
  uint32_t n;            // points in this segment
  uint32_t step;         // point_step
  uint32_t tile_begin;   // first tile of this segment in the launch
  uint32_t point_begin;  // global index of its first point
  int16_t off[4];        // x, y, z, intensity byte offsets
  uint8_t dt[4];         // datatypes (0 = absent)
  uint8_t n_nan;         // number of NaN-tested fields (generic path)
  uint8_t has_T;
  uint8_t fast16;        // 1 -> FAST16 path
  uint8_t nan_words;     // FAST16: bit w set -> 32-bit word w of the record is NaN-tested
  uint16_t nan_off[APC_MAX_FIELDS];
  uint8_t nan_dt[APC_MAX_FIELDS];
  float T[16];
};

// ---- mbarrier / TMA bulk-copy PTX wrappers (sm_90+; SASS: UBLKCP / SYNCS) ---------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                             uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- unaligned little-endian field reads (shared or global) ------------------------------
__device__ __forceinline__ uint32_t ld_u16_any(const uint8_t* p) {
  if ((((uintptr_t)p) & 1u) == 0) return *reinterpret_cast<const uint16_t*>(p);
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8);
}
__device__ __forceinline__ uint32_t ld_u32_any(const uint8_t* p) {
  const uintptr_t a = (uintptr_t)p;
  if ((a & 3u) == 0) return *reinterpret_cast<const uint32_t*>(p);
  if ((a & 1u) == 0)
    return (uint32_t) * reinterpret_cast<const uint16_t*>(p) |
           ((uint32_t) * reinterpret_cast<const uint16_t*>(p + 2) << 16);
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ uint64_t ld_u64_any(const uint8_t* p) {
  return (uint64_t)ld_u32_any(p) | ((uint64_t)ld_u32_any(p + 4) << 32);
}

// numpy ``.astype(np.float32)`` of one field (utils.py:102-104,121)
__device__ __forceinline__ float field_as_f32(const uint8_t* p, uint32_t dt) {
  switch (dt) {
    case APC_FLOAT32: return __uint_as_float(ld_u32_any(p));
    case APC_FLOAT64: return __double2float_rn(__longlong_as_double((long long)ld_u64_any(p)));
    case APC_INT8: return (float)(int8_t)p[0];
    case APC_UINT8: return (float)p[0];
    case APC_INT16: return (float)(int16_t)ld_u16_any(p);
    case APC_UINT16: return (float)ld_u16_any(p);
    case APC_INT32: return __int2float_rn((int32_t)ld_u32_any(p));
    case APC_UINT32: return __uint2float_rn(ld_u32_any(p));
    default: return 0.0f;
  }
}
__device__ __forceinline__ bool field_is_nan(const uint8_t* p, uint32_t dt) {
  if (dt == APC_FLOAT32) {
    const uint32_t b = ld_u32_any(p);
    return (b & 0x7fffffffu) > 0x7f800000u;
  }
  if (dt == APC_FLOAT64) {
    const uint64_t b = ld_u64_any(p);
    return (b & 0x7fffffffffffffffull) > 0x7ff0000000000000ull;
  }
  return false;
}

struct TilePoint {
  float x, y, z, w;
  bool valid;   // inside the segment
  bool no_nan;  // passes the read_points NaN test (true when nothing is tested)
};

// Loads the striped tile `tile_local` of segment `s`: item j of thread t is point
// tile_local*1024 + j*256 + t.  `stage` is dynamic shared memory (>= 1024*step bytes,
// 16-byte aligned) used only by the generic path; `bar` a shared mbarrier.
// GENERIC = false compiles the FAST16 path only (the host launches that instantiation when every
// segment qualifies): the byte-record decoder is a lot of code, and keeping it out of the common
// kernel keeps the hot loop inside the instruction cache.
template <bool GENERIC>
__device__ __forceinline__ void load_tile(const SegDev& s, uint32_t tile_local, bool test_nan,
                                          uint8_t* stage, uint64_t* bar,
                                          TilePoint (&pt)[APC_TILE_ITEMS]) {
  const uint32_t first = tile_local * APC_TILE_POINTS;
  const uint32_t in_tile = min(APC_TILE_POINTS, s.n - first);
  if (!GENERIC || s.fast16) {
    const float4* src = reinterpret_cast<const float4*>(s.data) + first;
#pragma unroll
    for (int j = 0; j < APC_TILE_ITEMS; ++j) {
      const uint32_t e = j * APC_TILE_THREADS + threadIdx.x;
      pt[j].valid = e < in_tile;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pt[j].valid) v = ld_stream_f4(src + e);
      bool nn = true;
      if (test_nan) {
        if ((s.nan_words & 1u) && is_nan_f(v.x)) nn = false;
        if ((s.nan_words & 2u) && is_nan_f(v.y)) nn = false;
        if ((s.nan_words & 4u) && is_nan_f(v.z)) nn = false;
        if ((s.nan_words & 8u) && is_nan_f(v.w)) nn = false;
      }
      pt[j].x = v.x; pt[j].y = v.y; pt[j].z = v.z;
      pt[j].w = s.dt[3] ? v.w : 0.0f;
      pt[j].no_nan = nn;
    }
    return;
  }
  if (!GENERIC) return;
  // ---- generic: stage the tile's bytes in shared memory --------------------------------
  const uint8_t* gsrc = s.data + (size_t)first * s.step;
  const uint32_t bytes = in_tile * s.step;
  const bool aligned = ((((uintptr_t)s.data) & 15u) == 0);  // tile offsets are multiples of 16
  const uint32_t bulk = aligned ? (bytes & ~15u) : 0u;
  if (bulk) {
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
      mbar_arrive_expect_tx(bar, bulk);
      tma_bulk_g2s(stage, gsrc, bulk, bar);
    }
  }
  for (uint32_t b = bulk + threadIdx.x; b < bytes; b += APC_TILE_THREADS) stage[b] = gsrc[b];
  if (bulk) mbar_wait(bar, 0);
  __syncthreads();
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t e = j * APC_TILE_THREADS + threadIdx.x;
    pt[j].valid = e < in_tile;
    pt[j].x = pt[j].y = pt[j].z = pt[j].w = 0.0f;
    pt[j].no_nan = true;
    if (pt[j].valid) {
      const uint8_t* rec = stage + (size_t)e * s.step;
      pt[j].x = field_as_f32(rec + s.off[0], s.dt[0]);
      pt[j].y = field_as_f32(rec + s.off[1], s.dt[1]);
      pt[j].z = field_as_f32(rec + s.off[2], s.dt[2]);
      if (s.dt[3]) pt[j].w = field_as_f32(rec + s.off[3], s.dt[3]);
      if (test_nan) {
        bool nn = true;
        for (uint32_t f = 0; f < s.n_nan; ++f)
          if (field_is_nan(rec + s.nan_off[f], s.nan_dt[f])) nn = false;
        pt[j].no_nan = nn;
      }
    }
  }
}

// segment lookup by tile index (<= 8 segments, linear)
template <typename P>
__device__ __forceinline__ uint32_t find_segment(const P& prm, uint32_t tile) {
  uint32_t s = 0;
#pragma unroll
  for (uint32_t k = 1; k < APC_MAX_CLOUDS; ++k)
    if (k < prm.n_seg && tile >= prm.seg[k].tile_begin) s = k;
  return s;
}
