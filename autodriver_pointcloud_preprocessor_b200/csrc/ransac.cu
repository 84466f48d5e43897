// RANSAC ground-plane segmentation with batched hypothesis scoring.
//
// Replaces Open3D segment_plane (pp.py:533-543; SURVEY.md B10), float64 like the legacy
// implementation the tensor API converts to.  Contract shared with oracle/ransac.py:
//   - hypotheses from the counter-based splitmix64 stream (or an explicit sample table),
//     fitted with the "fast plane fit" in a fixed operation order (bit-exact vs the oracle);
//   - the hypotheses are generated and fitted ONCE (k_rs_hypotheses, one thread each);
//   - one scoring pass scores all of them: each CTA stages a chunk of 16 or 20 planes in shared
//     memory and streams tiles of points past them; inlier-ness is the float64 decision
//     dist < thr; the error term (a tie-breaker between hypotheses with equal inlier counts
//     only, a DEFINED deviation from Open3D's float64 rmse: DESIGN.md section 5) is the integer
//     rint(d32^2 * float32(2^16/thr^2)) with d32 the float32 FMA distance; both are
//     order-independent, so warp reductions + per-CTA rows give deterministic totals;
//   - the last CTA to retire applies Open3D's sequential selection / early-stop rule;
//   - final pass: inlier mask against the winning hypothesis + moment sums for the
//     least-squares refit, reduced in a fixed order.
#include <cmath>
#include "apc_scan.cuh"
APC_TRACE_EXPORT(ransac)

#define RS_CHUNK 16
#define RS_MAX_N 16

__device__ __forceinline__ void plane_from_moments(double cx, double cy, double cz, double xx, double xy, double xz,
                                                   double yy, double yz, double zz, double* out) {
  const double det_x = __dsub_rn(__dmul_rn(yy, zz), __dmul_rn(yz, yz));
  const double det_y = __dsub_rn(__dmul_rn(xx, zz), __dmul_rn(xz, xz));
  const double det_z = __dsub_rn(__dmul_rn(xx, yy), __dmul_rn(xy, xy));
  double nx, ny, nz;
  if (det_x >= det_y && det_x >= det_z) {
    nx = det_x;
    ny = __dsub_rn(__dmul_rn(xz, yz), __dmul_rn(xy, zz));
    nz = __dsub_rn(__dmul_rn(xy, yz), __dmul_rn(xz, yy));
  } else if (det_y >= det_z) {
    nx = __dsub_rn(__dmul_rn(xz, yz), __dmul_rn(xy, zz));
    ny = det_y;
    nz = __dsub_rn(__dmul_rn(xy, xz), __dmul_rn(yz, xx));
  } else {
    nx = __dsub_rn(__dmul_rn(xy, yz), __dmul_rn(xz, yy));
    ny = __dsub_rn(__dmul_rn(xy, xz), __dmul_rn(yz, xx));
    nz = det_z;
  }
  const double norm = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
  if (!(norm > 0.0)) { out[0] = out[1] = out[2] = out[3] = 0.0; return; }
  nx = __ddiv_rn(nx, norm); ny = __ddiv_rn(ny, norm); nz = __ddiv_rn(nz, norm);
  out[0] = nx; out[1] = ny; out[2] = nz;
  out[3] = -__dadd_rn(__dadd_rn(__dmul_rn(nx, cx), __dmul_rn(ny, cy)), __dmul_rn(nz, cz));
}

// ---- packed float32x2 arithmetic (Blackwell FMUL2 / FFMA2: two IEEE-rn results per issue slot) ----
// ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even under --fmad=false, so the
// float32 distance is DEFINED with fused multiply-adds, written out explicitly here and emulated
// exactly (single rounding) by oracle/ransac.py:fma32 - nothing is left to the compiler's choice.
__device__ __forceinline__ unsigned long long pk2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long mul2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

// acc += bits(v) if c, as ONE predicated integer add (the compiler's own choice for the C form
// is a SEL of the value or zero followed by an add)
__device__ __forceinline__ void add_if(uint32_t& acc, bool c, float v) {
  asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p add.u32 %0, %0, %2;\n\t}"
      : "+r"(acc) : "r"((uint32_t)c), "r"(__float_as_uint(v)));
}

// One hypothesis from its sample points (s[0..n), staged in shared memory): plane through three
// points, or the least-squares "fast plane fit" - same operation order as oracle/ransac.py.
__device__ void rs_fit(const float4* s, uint32_t n, double* out) {
  if (n == 3) {
    const float4 a = s[0], b = s[1], c = s[2];
    const double e1x = __dsub_rn((double)b.x, (double)a.x), e1y = __dsub_rn((double)b.y, (double)a.y), e1z = __dsub_rn((double)b.z, (double)a.z);
    const double e2x = __dsub_rn((double)c.x, (double)a.x), e2y = __dsub_rn((double)c.y, (double)a.y), e2z = __dsub_rn((double)c.z, (double)a.z);
    double nx = __dsub_rn(__dmul_rn(e1y, e2z), __dmul_rn(e1z, e2y));
    double ny = __dsub_rn(__dmul_rn(e1z, e2x), __dmul_rn(e1x, e2z));
    double nz = __dsub_rn(__dmul_rn(e1x, e2y), __dmul_rn(e1y, e2x));
    const double norm = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
    if (!(norm > 0.0)) { out[0] = out[1] = out[2] = out[3] = 0.0; return; }
    nx = __ddiv_rn(nx, norm); ny = __ddiv_rn(ny, norm); nz = __ddiv_rn(nz, norm);
    out[0] = nx; out[1] = ny; out[2] = nz;
    out[3] = -__dadd_rn(__dadd_rn(__dmul_rn(nx, (double)a.x), __dmul_rn(ny, (double)a.y)), __dmul_rn(nz, (double)a.z));
    return;
  }
  double cx = 0.0, cy = 0.0, cz = 0.0;
  for (uint32_t j = 0; j < n; ++j) {
    const float4 p = s[j];
    cx = __dadd_rn(cx, (double)p.x); cy = __dadd_rn(cy, (double)p.y); cz = __dadd_rn(cz, (double)p.z);
  }
  const double dn = (double)n;
  cx = __ddiv_rn(cx, dn); cy = __ddiv_rn(cy, dn); cz = __ddiv_rn(cz, dn);
  double xx = 0, xy = 0, xz = 0, yy = 0, yz = 0, zz = 0;
  for (uint32_t j = 0; j < n; ++j) {
    const float4 p = s[j];
    const double rx = __dsub_rn((double)p.x, cx), ry = __dsub_rn((double)p.y, cy), rz = __dsub_rn((double)p.z, cz);
    xx = __dadd_rn(xx, __dmul_rn(rx, rx)); xy = __dadd_rn(xy, __dmul_rn(rx, ry)); xz = __dadd_rn(xz, __dmul_rn(rx, rz));
    yy = __dadd_rn(yy, __dmul_rn(ry, ry)); yz = __dadd_rn(yz, __dmul_rn(ry, rz)); zz = __dadd_rn(zz, __dmul_rn(rz, rz));
  }
  plane_from_moments(cx, cy, cz, xx, xy, xz, yy, yz, zz, out);
}

__device__ __forceinline__ double plane_dist(const double* pl, double x, double y, double z) {
  return fabs(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(pl[0], x), __dmul_rn(pl[1], y)), __dmul_rn(pl[2], z)), pl[3]));
}

#define RS_EPS 5.0e-7f          // relative slack of the float32 pre-test (see k_rs_score)
#define RS_MAGIC 8388608.0f     // 2^23: (u + 2^23) has rint(u) in its low mantissa bits for 0 <= u < 2^23
#define RS_MAGIC_BITS 0x4B000000u
#define RS_FLUSH_TILES 32       // the packed per-thread accumulators hold at most 128 points (see k_rs_score)
#define CTR_RS_SCORE_TICKET 21  // ctrl->counters slot: chunk columns of k_rs_score whose tallies are summed
__device__ __noinline__ void rs_select_cta(const double* __restrict__ planes, const unsigned long long* scores,
                                           uint32_t P, uint32_t ransac_n, uint32_t iters, double log1mp,
                                           double* __restrict__ plane8, uint32_t* __restrict__ info);

// Scoring + selection in one launch (the hypotheses come from k_rs_hypotheses).
// grid = (persistent CTAs striding over point tiles, chunks of CH hypotheses).
//   prologue  the CTA requests its first tile of points, then stages its chunk's planes (float64
//             and packed float32 pairs) in shared memory while those loads are in flight.
//   scoring   a thread streams 4 points per tile past the CH planes.  The signed distance is
//             evaluated in float32 for TWO hypotheses per instruction (FMUL2/FADD2) and compared
//             with thr -/+ a rigorous bound on |d32 - d64|: below -> inlier, above -> outlier,
//             in between (a few points per million) -> the thread re-decides those in float64,
//             so the inlier set is exactly the float64 one of oracle/ransac.py.  The error term
//             rint(d32^2 * 2^16/thr^2) comes out of the same packed pipeline: one FFMA2 adds the
//             2^23 magic number, leaving the integer in the mantissa (no F2I); summed as integers.
//   epilogue  warp REDUX -> per-warp rows in shared memory -> one row of per-CTA tallies in
//             global memory (no atomics); the last CTA of each chunk column (a ticket per column)
//             adds that column's rows up into scores_copy, and the last column to finish applies
//             Open3D's sequential selection rule.
#define RS_QCAP 128
// Exact re-decision of one queued point against hypotheses h_first, h_first + h_step, ...: the
// evaluations whose float32 distance lies inside the rounding band [lo, hi) are decided by the
// float64 distance and, when inliers, added to the CTA's exact tallies (shared-memory atomics).
template <int CH>
__device__ __forceinline__ void rs_exact_point(float4 pt, float hm, double thr, float thr32, float scale32,
                                               const double (*s_pl)[4], const float (*s_pk)[8],
                                               unsigned long long* s_cnt, unsigned long long* s_err, int h_first,
                                               int h_step) {
  const float x = pt.x, y = pt.y, z = pt.z;
  const float m = RS_EPS * (fabsf(x) + fabsf(y) + fabsf(z)) + hm;   // same expression as the scoring loop
  const float lo = thr32 - m, hi = thr32 + m;
  for (int h = h_first; h < CH; h += h_step) {
    const float* pk = &s_pk[h >> 1][h & 1];
    const float d = __fmaf_rn(pk[4], z, __fmaf_rn(pk[2], y, __fmaf_rn(pk[0], x, pk[6])));
    if (fabsf(d) < hi && !(fabsf(d) < lo) && plane_dist(s_pl[h], (double)x, (double)y, (double)z) < thr) {
      const float v = __fmaf_rn(__fmul_rn(d, d), scale32, RS_MAGIC);
      atomicAdd(&s_cnt[h], 1ull);
      atomicAdd(&s_err[h], (unsigned long long)(__float_as_uint(v) - RS_MAGIC_BITS));
    }
  }
}

#ifdef RS_TRACE
__device__ unsigned long long g_rs_trace[1024 * 8];
__device__ unsigned long long g_rs_trace2[1024 * 32];
extern "C" int apc_debug_rs_trace2(unsigned long long* out_host) {
  return (int)cudaMemcpyFromSymbol(out_host, g_rs_trace2, sizeof(g_rs_trace2));
}
extern "C" int apc_debug_rs_trace(unsigned long long* out_host) {
  return (int)cudaMemcpyFromSymbol(out_host, g_rs_trace, sizeof(g_rs_trace));
}
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define RS_STAMP(k) do { if (threadIdx.x == 0) g_rs_trace[(blockIdx.y * gridDim.x + blockIdx.x) * 8 + (k)] = gtime(); } while (0)
#else
#define RS_STAMP(k) do { } while (0)
#endif


// Hypothesis generation: ONE thread per hypothesis (counter-based sampling with rejection of
// repeats, or the caller's sample table), sample points staged through shared memory, float64
// fit.  A separate small launch so that the scoring CTAs (one per SM, half a register file each)
// do not all repeat it: in round 1 each of the 29 CTAs of a chunk column spent 3.5 us of its
// 15 us on the same 20 fits (profiles/r2a_rs_trace_before.txt).
#define RS_HYP_THREADS 64
__global__ void __launch_bounds__(RS_HYP_THREADS)
k_rs_hypotheses(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, uint32_t ransac_n, uint32_t iters,
                uint64_t seed, const int32_t* __restrict__ table, double* __restrict__ planes,
                uint32_t* __restrict__ col_tickets) {
  __shared__ uint32_t s_idx[RS_HYP_THREADS][RS_MAX_N + 1];   // +1: rows on different banks
  __shared__ float4 s_sp[RS_HYP_THREADS][RS_MAX_N];
  pdl_enter();
  const uint32_t P = apc_count(n_dev, n_max);
  const uint32_t tid = threadIdx.x;
  const uint32_t it = blockIdx.x * RS_HYP_THREADS + tid;
  const bool live = it < iters && P >= ransac_n;
  if (live) {
    if (table) {
      for (uint32_t j = 0; j < ransac_n; ++j) s_idx[tid][j] = min((uint32_t)table[(size_t)it * ransac_n + j], P - 1);
    } else {
      uint32_t got = 0;
      for (uint64_t c = 0; got < ransac_n; ++c) {
        const uint64_t z = splitmix64_dev(seed + ((uint64_t)it << 32) + c);
        const uint32_t cand = (uint32_t)(((z >> 32) * (uint64_t)P) >> 32);
        bool dup = false;
        for (uint32_t j = 0; j < got; ++j) dup |= (s_idx[tid][j] == cand);
        if (!dup) s_idx[tid][got++] = cand;
      }
    }
    for (uint32_t j = 0; j < ransac_n; ++j) s_sp[tid][j] = pts[s_idx[tid][j]];   // independent loads, all in flight
  }
  if (it < iters) {
    col_tickets[it] = 0;   // k_rs_score's chunk columns (fewer than iters), counted from zero on every call
    double pl[4] = {0.0, 0.0, 0.0, 0.0};
    if (live) rs_fit(s_sp[tid], ransac_n, pl);
#pragma unroll
    for (int k = 0; k < 4; ++k) planes[4 * (size_t)it + k] = pl[k];
  }
}

template <int CH>
__global__ void __launch_bounds__(APC_TILE_THREADS, 1)
k_rs_score(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, uint32_t ransac_n, uint32_t iters,
           const double* __restrict__ planes, double thr,
           unsigned long long* scores, double log1mp, double* __restrict__ plane8, uint32_t* __restrict__ info,
           unsigned long long* __restrict__ scores_copy, uint32_t* __restrict__ col_tickets, ApcCtrl* ctrl) {
  static_assert(CH % 2 == 0, "hypotheses are scored in pairs");
  __shared__ double s_pl[CH][4];
  __shared__ __align__(16) float s_pk[CH / 2][8];   // {a0,a1, b0,b1, c0,c1, d0,d1} of a pair, float32
  __shared__ unsigned long long s_cnt[CH], s_err[CH];   // float64-decided evaluations (rare, smem atomics)
  __shared__ uint32_t s_wcnt[APC_TILE_THREADS / 32][CH];       // per-warp totals: each warp owns its row, no atomics
  __shared__ unsigned long long s_werr[APC_TILE_THREADS / 32][CH];
  __shared__ float s_hm;                            // hypothesis part of the float32 error bound (chunk max)
  __shared__ float4 s_q[RS_QCAP];                   // points waiting for the exact float64 decision
  __shared__ uint32_t s_qn;
  pdl_enter();
  const uint32_t P = apc_count(n_dev, n_max);
  const uint32_t h0 = blockIdx.y * CH;
  const uint32_t nh = min((uint32_t)CH, iters - h0);
  const uint32_t tid = threadIdx.x;
  RS_STAMP(0);
  APC_STAMP(0, 0);
#ifdef RS_TRACE
  if (threadIdx.x == 0) {
    uint32_t sm;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
    unsigned long long* t = &g_rs_trace[(blockIdx.y * gridDim.x + blockIdx.x) * 8];
    t[7] = sm;
    t[5] = t[6] = 0;   // written by the column's last CTA / the selecting CTA only
  }
#endif
  // ---- prologue: the first tile's points are requested before anything else; the chunk's planes
  // (k_rs_hypotheses) are staged in shared memory while those loads are in flight ---------------
  float4 nxt[APC_TILE_ITEMS];
  {
    const uint32_t first = blockIdx.x * APC_TILE_POINTS;
#pragma unroll
    for (int j = 0; j < APC_TILE_ITEMS; ++j) {
      const uint32_t i = first + j * APC_TILE_THREADS + tid;
      nxt[j] = i < P ? pts[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  for (uint32_t t = tid; t < (APC_TILE_THREADS / 32) * CH; t += APC_TILE_THREADS) {
    (&s_wcnt[0][0])[t] = 0;
    (&s_werr[0][0])[t] = 0;
  }
  if (tid == 0) s_qn = 0;
  if (tid < CH) {
    s_cnt[tid] = 0; s_err[tid] = 0;
    double pl[4] = {0.0, 0.0, 0.0, 0.0};
    if (tid < nh) {
      const double2 ab = *reinterpret_cast<const double2*>(planes + 4 * (size_t)(h0 + tid));
      const double2 cd = *reinterpret_cast<const double2*>(planes + 4 * (size_t)(h0 + tid) + 2);
      pl[0] = ab.x; pl[1] = ab.y; pl[2] = cd.x; pl[3] = cd.y;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      s_pl[tid][k] = pl[k];
      s_pk[tid >> 1][2 * k + (tid & 1)] = (float)pl[k];
    }
  }
  __syncthreads();
  if (tid < 32) {
    // |d32 - d64| <= ~4 * 2^-24 * (|a||x|+|b||y|+|c||z|+|d|), |a|,|b|,|c| <= 1 (unit normal):
    // RS_EPS = 5e-7 is 2x that; "+ thr + 1" covers the rounding of the threshold and of the bound
    float m = 0.0f;
    for (uint32_t h = tid; h < CH; h += 32) m = fmaxf(m, fabsf((float)s_pl[h][3]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (tid == 0) s_hm = RS_EPS * (m + (float)thr + 1.0f);
  }
  __syncthreads();
  RS_STAMP(1);
  // ---- scoring ------------------------------------------------------------------------------
  const float thr32 = (float)thr;
  const float scale32 = (float)(65536.0 / (thr * thr));
  const unsigned long long SC2 = pk2(scale32, scale32), MG2 = pk2(RS_MAGIC, RS_MAGIC);
  const float hm = s_hm;
  // acc[h] += bits(u + 2^23) = 0x4B000000 + rint(u) per sure inlier.  Over a window of at most
  // 128 points, sum rint(u) < 2^24 stays in the low 24 bits and the inlier count k sits in the
  // top byte as k * 0x4B mod 256 (0x4B is odd, so k = top * 99 mod 256): ONE 32-bit accumulator
  // per hypothesis carries both the count and the error sum.
  uint32_t acc[CH];
#pragma unroll
  for (int h = 0; h < CH; ++h) acc[h] = 0;
  uint32_t tiles_done = 0;
  auto flush = [&]() {         // warp totals (REDUX) -> this warp's row in shared memory
    const uint32_t w = tid >> 5;
#pragma unroll
    for (int h = 0; h < CH; ++h) {
      const uint32_t k = ((acc[h] >> 24) * 99u) & 255u, e = acc[h] & 0xffffffu;
      const uint32_t c = __reduce_add_sync(0xffffffffu, k), es = __reduce_add_sync(0xffffffffu, e);
      if (lane_id() == 0) {
        s_wcnt[w][h] += c;
        s_werr[w][h] += es;
      }
      acc[h] = 0;
    }
  };
  for (uint32_t first = blockIdx.x * APC_TILE_POINTS; first < P; first += gridDim.x * APC_TILE_POINTS) {
    float4 p[APC_TILE_ITEMS];
#pragma unroll
    for (int j = 0; j < APC_TILE_ITEMS; ++j) p[j] = nxt[j];
    {                                              // the next tile's loads fly under this tile's math
      const uint32_t nfirst = first + gridDim.x * APC_TILE_POINTS;
#pragma unroll
      for (int j = 0; j < APC_TILE_ITEMS; ++j) {
        const uint32_t i = nfirst + j * APC_TILE_THREADS + tid;
        nxt[j] = (nfirst < P && i < P) ? pts[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float lo[APC_TILE_ITEMS], hi[APC_TILE_ITEMS];
    bool amb = false;            // one of this thread's evaluations of the tile lies inside the rounding band
#pragma unroll
    for (int j = 0; j < APC_TILE_ITEMS; ++j) {
      const uint32_t i = first + j * APC_TILE_THREADS + tid;
      const float m = RS_EPS * (fabsf(p[j].x) + fabsf(p[j].y) + fabsf(p[j].z)) + hm;   // = rs_exact_point's
      lo[j] = i < P ? thr32 - m : -1.0f;     // past the end: neither inlier nor ambiguous
      hi[j] = i < P ? thr32 + m : -1.0f;
    }
#pragma unroll
    for (int hp = 0; hp < CH / 2; ++hp) {
      const ulonglong2 ab = *reinterpret_cast<const ulonglong2*>(&s_pk[hp][0]);
      const ulonglong2 cd = *reinterpret_cast<const ulonglong2*>(&s_pk[hp][4]);
#pragma unroll
      for (int j = 0; j < APC_TILE_ITEMS; ++j) {
        const unsigned long long X = pk2(p[j].x, p[j].x), Y = pk2(p[j].y, p[j].y), Z = pk2(p[j].z, p[j].z);
        const unsigned long long d2 = fma2(cd.x, Z, fma2(ab.y, Y, fma2(ab.x, X, cd.y)));   // c*z + (b*y + (a*x + d))
        const unsigned long long v2 = fma2(mul2(d2, d2), SC2, MG2);
        float d0, d1, v0, v1;
        upk2(d2, d0, d1);
        upk2(v2, v0, v1);
        const bool in0 = fabsf(d0) < lo[j], in1 = fabsf(d1) < lo[j];
        amb = amb | (in0 != (fabsf(d0) < hi[j])) | (in1 != (fabsf(d1) < hi[j]));
        add_if(acc[2 * hp], in0, v0);
        add_if(acc[2 * hp + 1], in1, v1);
      }
    }
    // an evaluation inside the rounding band (a few per million): the thread queues its points of
    // this tile; the whole CTA re-decides queued points in float64 after the scoring loop, CH
    // threads per point (re-deciding a point with no in-band evaluation is a no-op)
    if (amb) {
      const uint32_t q = atomicAdd(&s_qn, (uint32_t)APC_TILE_ITEMS);
#pragma unroll
      for (int j = 0; j < APC_TILE_ITEMS; ++j) {
        // past the end of the cloud: an all-infinite point is never in band (no-op entry)
        const float inf = __int_as_float(0x7f800000);
        const float4 e = first + j * APC_TILE_THREADS + tid < P ? p[j] : make_float4(inf, inf, inf, 0.f);
        if (q + j < RS_QCAP) s_q[q + j] = e;
        else rs_exact_point<CH>(e, hm, thr, thr32, scale32, s_pl, s_pk, s_cnt, s_err, 0, 1);   // queue full: inline
      }
    }
    if (++tiles_done == RS_FLUSH_TILES) { flush(); tiles_done = 0; }
  }
  RS_STAMP(2);
  flush();
  __syncthreads();
  {
    const uint32_t nq = min(s_qn, (uint32_t)RS_QCAP);
    for (uint32_t e = tid; e < nq * CH; e += APC_TILE_THREADS)
      rs_exact_point<CH>(s_q[e / CH], hm, thr, thr32, scale32, s_pl, s_pk, s_cnt, s_err, e % CH, CH);
    if (nq) __syncthreads();   // nq is CTA-uniform
  }
  RS_STAMP(3);
  // per-CTA partial tallies {count, error}, plain stores: row blockIdx.x of the column's [gridDim.x][CH]
  // block, the blocks of the columns one after the other (thousands of same-line global atomics from 260
  // CTAs cost ~17 us of serialisation in L2)
  ulonglong2* col = reinterpret_cast<ulonglong2*>(scores) + (size_t)blockIdx.y * gridDim.x * CH;
  if (tid < nh) {
    unsigned long long c = s_cnt[tid], e = s_err[tid];
#pragma unroll
    for (int w = 0; w < APC_TILE_THREADS / 32; ++w) { c += s_wcnt[w][tid]; e += s_werr[w][tid]; }
    col[blockIdx.x * CH + tid] = make_ulonglong2(c, e);
  }
  // the last CTA of the column (ticket) sums the column's rows; the last column to be summed runs the
  // selection: one launch and one inter-kernel dependency less on the per-scan critical path.  Barrier,
  // then ONE thread takes each ticket with an acq_rel atomic (see ticket_acq_rel).
  __shared__ bool s_last;
  __syncthreads();
  if (tid == 0) s_last = (ticket_acq_rel(&col_tickets[blockIdx.y]) == gridDim.x - 1);
  __syncthreads();
  RS_STAMP(4);
  APC_STAMP(0, 1);
  if (!s_last) return;
  {
    // G groups of CH threads add every G-th row (integer sums: the order is immaterial)
    constexpr uint32_t G = APC_TILE_THREADS / CH;
    __shared__ ulonglong2 s_col[G][CH];
    const uint32_t h = tid % CH, g = tid / CH;
    if (g < G) {
      unsigned long long c = 0, e = 0;
      if (h < nh)
        for (uint32_t r = g; r < gridDim.x; r += G) {
          const ulonglong2 v = __ldcg(col + r * CH + h);
          c += v.x;
          e += v.y;
        }
      s_col[g][h] = make_ulonglong2(c, e);
    }
    __syncthreads();
    if (tid < nh) {
      unsigned long long c = 0, e = 0;
#pragma unroll
      for (uint32_t k = 0; k < G; ++k) { c += s_col[k][tid].x; e += s_col[k][tid].y; }
      reinterpret_cast<ulonglong2*>(scores_copy)[h0 + tid] = make_ulonglong2(c, e);
    }
  }
  __syncthreads();
  if (tid == 0) s_last = (ticket_acq_rel(&ctrl->counters[CTR_RS_SCORE_TICKET]) == gridDim.y - 1);
  __syncthreads();
  RS_STAMP(5);
  if (!s_last) return;
  rs_select_cta(planes, scores_copy, P, ransac_n, iters, log1mp, plane8, info);
  RS_STAMP(6);
  APC_STAMP(0, 2);
}

// Open3D's sequential selection + early-stop rule over the batched scores, run by one CTA.
// Sequential semantics (oracle/ransac.py:select): hypotheses are visited in order, one replaces
// the best when it has more inliers, or as many and a smaller error; every replacement moves the
// early-stop bound, and once an iteration lies beyond the bound all later ones do too.  So only
// the PREFIX RECORDS of the sequence can ever be selected: the CTA finds them with a parallel
// prefix-max over a sortable key, and one thread walks that short list (a handful of entries,
// one log() each) instead of all num_iterations hypotheses.
// info = {best iteration | 0xffffffff, n_inliers (filled later), 0, 0}; plane8[4..7] = winner.
// scores = {inliers, error} of every hypothesis, summed over the points by the column CTAs.
__device__ __noinline__ void rs_select_cta(const double* __restrict__ planes_in, const unsigned long long* scores,
                                           uint32_t P, uint32_t ransac_n, uint32_t iters, double log1mp,
                                           double* __restrict__ plane8, uint32_t* __restrict__ info) {
  const double* planes = planes_in;                 // written by k_rs_hypotheses, the previous launch
  __shared__ unsigned long long s_wmax[APC_TILE_THREADS / 32];
  __shared__ unsigned long long s_carry;             // best key of all earlier chunks
  __shared__ uint32_t s_rec_it[APC_TILE_THREADS];    // prefix records of the current chunk, in order
  __shared__ double s_rec_break[APC_TILE_THREADS];   // early-stop bound each record would set
  __shared__ uint32_t s_nrec;
  __shared__ uint32_t sb_it;
  __shared__ double sb_break;
  __shared__ bool sb_stop;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) { s_carry = 0; sb_it = 0xffffffffu; sb_break = (double)iters; sb_stop = false; }
  __syncthreads();
  for (uint32_t c0 = 0; c0 < iters; c0 += APC_TILE_THREADS) {
    // a chunk of 256 hypotheses, one per thread
    const uint32_t it = c0 + tid;
    unsigned long long key = 0, inl = 0;
    if (it < iters) {
      const ulonglong2 v = __ldcg(reinterpret_cast<const ulonglong2*>(scores) + it);
      inl = v.x;
      const unsigned long long err = v.y;
      const double* pl = planes + 4 * (size_t)it;
      const bool valid = !(pl[0] == 0.0 && pl[1] == 0.0 && pl[2] == 0.0 && pl[3] == 0.0);
      // more inliers first, then the smaller error: inl < 2^23, err < 2^40 (4M points x 2^16)
      if (valid && inl > 0) key = (inl << 40) | (0xffffffffffull - (err < 0xffffffffffull ? err : 0xffffffffffull));
    }
    // exclusive prefix max over the chunk (+ carry): warp scan, then the warp totals
    unsigned long long incl = key;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o && v > incl) incl = v;
    }
    unsigned long long excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 0;
    if (lane == 31) s_wmax[warp] = incl;
    if (tid == 0) s_nrec = 0;
    __syncthreads();
    unsigned long long before = s_carry;
    for (uint32_t w = 0; w < warp; ++w) before = s_wmax[w] > before ? s_wmax[w] : before;
    if (excl > before) before = excl;
    const bool record = key > before;                 // strictly better than everything earlier
    // ordered list of the records: ballot ranks inside the warp, warp offsets through smem
    const uint32_t bal = __ballot_sync(0xffffffffu, record);
    __shared__ uint32_t s_wrec[APC_TILE_THREADS / 32];
    if (lane == 0) s_wrec[warp] = __popc(bal);
    __syncthreads();
    uint32_t off = 0;
    for (uint32_t w = 0; w < warp; ++w) off += s_wrec[w];
    if (record) {
      // the bound this hypothesis sets if it becomes the best (log() evaluated by all records in
      // parallel, not one after the other by the walking thread)
      double brk = 0.0;
      if (inl < P) {
        const double fitness = __ddiv_rn((double)inl, (double)P);
        double fn = fitness;
        for (uint32_t j = 1; j < ransac_n; ++j) fn = __dmul_rn(fn, fitness);
        const double denom = log(__dsub_rn(1.0, fn));
        const double cand = (denom == 0.0) ? __longlong_as_double(0x7ff0000000000000ll) : __ddiv_rn(log1mp, denom);
        brk = cand < (double)iters ? cand : (double)iters;
      }
      const uint32_t r = off + __popc(bal & ((1u << lane) - 1u));
      s_rec_it[r] = it;
      s_rec_break[r] = brk;
    }
    if (tid == APC_TILE_THREADS - 1) {
      s_nrec = off + __popc(bal);
      const unsigned long long m = key > before ? key : before;
      s_carry = m;                                    // the last thread's inclusive max = chunk max
    }
    __syncthreads();
    if (tid == 0 && !sb_stop) {
      double break_it = sb_break;
      uint32_t best_it = sb_it;
      for (uint32_t r = 0; r < s_nrec; ++r) {
        const uint32_t rit = s_rec_it[r];
        if ((double)rit > break_it) { sb_stop = true; break; }   // beyond the bound: so is everything later
        best_it = rit;
        break_it = s_rec_break[r];
      }
      sb_it = best_it;
      sb_break = break_it;
    }
    __syncthreads();
  }
  if (tid == 0) { info[0] = sb_it; info[1] = 0; info[2] = 0; info[3] = 0; }
  if (tid < 4) plane8[4 + tid] = sb_it == 0xffffffffu ? 0.0 : planes[4 * (size_t)sb_it + tid];
}

#define CTR_RS_TICKET 20  // ctrl->counters slot: CTAs of k_rs_final that have published their partials

// Final inliers against the winning hypothesis + moment sums for the least-squares refit.
// Each CTA (1024 points) writes one partial; the last CTA to finish (ticket counter) sums the
// partials in index order - a fixed reduction order, so the refit is deterministic - and
// solves for the plane.  With `keep_out` the kernel also performs pp.py:542
// select_by_index(inliers, invert=True) itself: the non-inliers are compacted in order
// (ballot ranks + decoupled look-back) straight into the output cloud, so the pipeline needs no
// separate select_by_mask launch (and no second read of the points).
__global__ void __launch_bounds__(APC_TILE_THREADS)
k_rs_final(const float4* __restrict__ pts, uint32_t n_max, const uint32_t* n_dev, double* __restrict__ plane8,
           uint32_t* __restrict__ info, double thr, uint8_t* __restrict__ mask, double* __restrict__ partials,
           float4* __restrict__ keep_out, uint32_t* keep_count, uint64_t* scan_state, uint32_t n_tiles, ApcCtrl* ctrl,
           const uint32_t* __restrict__ keep_idx_in, uint32_t* __restrict__ keep_idx_out,
           const __grid_constant__ MirrorDev mir, const float* __restrict__ nrm_in, float* __restrict__ nrm_out) {
  __shared__ double s_red[8][10];
  __shared__ bool s_last;
  __shared__ uint32_t sm_scan[34];
  pdl_enter();
  const uint32_t P = apc_count(n_dev, n_max);
  APC_STAMP(1, 0);
  const bool have = info[0] != 0xffffffffu;
  const double pl[4] = {plane8[4], plane8[5], plane8[6], plane8[7]};
  double acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = 0.0;
  float4 p[APC_TILE_ITEMS];
  bool keep[APC_TILE_ITEMS];
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = blockIdx.x * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    p[j] = i < P ? pts[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  }
#pragma unroll
  for (int j = 0; j < APC_TILE_ITEMS; ++j) {
    const uint32_t i = blockIdx.x * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
    keep[j] = false;
    if (i < P) {
      const double x = p[j].x, y = p[j].y, z = p[j].z;
      const bool inl = have && plane_dist(pl, x, y, z) < thr;
      if (mask) mask[i] = inl ? 1 : 0;
      keep[j] = !inl;
      if (inl) {
        acc[0] += 1.0; acc[1] += x; acc[2] += y; acc[3] += z;
        acc[4] += x * x; acc[5] += x * y; acc[6] += x * z; acc[7] += y * y; acc[8] += y * z; acc[9] += z * z;
      }
    }
  }
  if (keep_out) {
    uint32_t rank[APC_TILE_ITEMS];
    const uint32_t base = tile_compact_offsets(keep, rank, sm_scan, scan_state, blockIdx.x, ctrl->epoch, keep_count, n_tiles);
#pragma unroll
    for (int j = 0; j < APC_TILE_ITEMS; ++j)
      if (keep[j]) {
        keep_out[base + rank[j]] = p[j];
        mirror_store(mir, base + rank[j], p[j]);
        if (nrm_out) {     // the normals travel through select_by_index(inliers, invert=True) like every attribute (pp.py:542)
          const uint32_t i = blockIdx.x * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
          const size_t o = base + rank[j];
          nrm_out[3 * o] = nrm_in[3 * (size_t)i];
          nrm_out[3 * o + 1] = nrm_in[3 * (size_t)i + 1];
          nrm_out[3 * o + 2] = nrm_in[3 * (size_t)i + 2];
        }
        if (keep_idx_out) {
          const uint32_t i = blockIdx.x * APC_TILE_POINTS + j * APC_TILE_THREADS + threadIdx.x;
          keep_idx_out[base + rank[j]] = keep_idx_in ? keep_idx_in[i] : i;
        }
      }
  }
  // tiles past the device-side count hold no points: no partial row (the last CTA reads only the
  // rows of the tiles in use - adding their zeros would not change a bit of the sums)
  const uint32_t used_tiles = min(gridDim.x, (P + APC_TILE_POINTS - 1) / APC_TILE_POINTS);
  if (blockIdx.x < used_tiles) {
#pragma unroll
    for (int k = 0; k < 10; ++k) {
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      if (lane_id() == 0) s_red[threadIdx.x >> 5][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < 10) {
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += s_red[w][threadIdx.x];
      partials[(size_t)blockIdx.x * 10 + threadIdx.x] = s;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) s_last = (ticket_acq_rel(&ctrl->counters[CTR_RS_TICKET]) == gridDim.x - 1);
  __syncthreads();
  APC_STAMP(1, 1);
  if (!s_last) return;
  // last CTA: stage 256 partial rows at a time in shared memory (parallel, coalesced loads),
  // then thread k < 10 adds moment k in CTA order
  __shared__ double s_part[256 * 10];
  __shared__ double s_tot[10];
  double run = 0.0;
  const volatile double* vp = partials;
  for (uint32_t b0 = 0; b0 < used_tiles; b0 += 256) {
    const uint32_t rows = min(256u, used_tiles - b0);
    __syncthreads();
    for (uint32_t e = threadIdx.x; e < rows * 10; e += blockDim.x) s_part[e] = vp[(size_t)b0 * 10 + e];
    __syncthreads();
    if (threadIdx.x < 10)
      for (uint32_t b = 0; b < rows; ++b) run += s_part[b * 10 + threadIdx.x];
  }
  if (threadIdx.x < 10) s_tot[threadIdx.x] = run;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double n = s_tot[0];
    info[1] = (uint32_t)n;
    if (n < 1.0) { plane8[0] = plane8[1] = plane8[2] = plane8[3] = 0.0; return; }
    const double cx = s_tot[1] / n, cy = s_tot[2] / n, cz = s_tot[3] / n;
    const double xx = s_tot[4] - n * cx * cx, xy = s_tot[5] - n * cx * cy, xz = s_tot[6] - n * cx * cz;
    const double yy = s_tot[7] - n * cy * cy, yz = s_tot[8] - n * cy * cz, zz = s_tot[9] - n * cz * cz;
    plane_from_moments(cx, cy, cz, xx, xy, xz, yy, yz, zz, plane8);
  }
  APC_STAMP(1, 2);
}

int apc_segment_plane_nobegin(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev, double thr,
                              int ransac_n, int iters, double prob, uint64_t seed, const int32_t* table,
                              double* out_plane, uint8_t* out_mask, uint32_t* out_info, float* out_keep_xyzi,
                              uint32_t* out_keep_count, int scan_slot, cudaStream_t s, const uint32_t* keep_idx_in,
                              uint32_t* keep_idx_out, const MirrorDev* mir, const float* nrm_in, float* nrm_out) {
  APC_REQUIRE(ctx, out_plane && out_info && (out_mask || out_keep_xyzi), "NULL output pointer");
  APC_REQUIRE(ctx, !out_keep_xyzi || out_keep_count, "out_keep_count is NULL");
  APC_REQUIRE(ctx, prob > 0.0 && prob <= 1.0, "probability must be in (0, 1]");
  APC_REQUIRE(ctx, ransac_n >= 3 && ransac_n <= RS_MAX_N, "ransac_n must be in 3..16");
  APC_REQUIRE(ctx, iters >= 1 && (uint32_t)iters <= ctx->rs_max_iters, "num_iterations must be in 1..4096");
  APC_REQUIRE(ctx, thr > 0.0, "distance_threshold must be > 0");
  APC_REQUIRE(ctx, n_max <= ctx->max_points, "more points than the context was created for");
  if (!n_dev && n_max < (uint32_t)ransac_n) return apc_set_error(ctx, APC_ERR_TOO_FEW, "fewer points than ransac_n");
  if (n_max == 0) {
    APC_CUDA(ctx, cudaMemsetAsync(out_plane, 0, 8 * sizeof(double), s));
    APC_CUDA(ctx, cudaMemsetAsync(out_info, 0xff, sizeof(uint32_t), s));
    APC_CUDA(ctx, cudaMemsetAsync(out_info + 1, 0, 3 * sizeof(uint32_t), s));
    if (out_keep_count) APC_CUDA(ctx, cudaMemsetAsync(out_keep_count, 0, sizeof(uint32_t), s));
    return APC_OK;
  }
  APC_REQUIRE(ctx, xyzi, "NULL pointer");
  const float4* pts = reinterpret_cast<const float4*>(xyzi);
  const uint32_t n_tiles = apc_div_up(n_max, APC_TILE_POINTS);
  APC_REQUIRE(ctx, n_tiles <= ctx->max_tiles, "more points than the context was created for");
  // hypotheses per CTA (CH) = 20 or 16, with ONE CTA per SM.  Half the chunk (10 / 8) with TWO CTAs per SM does
  // the same arithmetic per SM, but the two co-resident CTAs share the issue slots, so a CTA's scoring phase
  // does not shrink (8.6 vs 8.2 us), the kernel ends later (19.1 vs 16.1 us) and saturated throughput is the
  // same (70.5 vs 71.2 us/scan, profiles/r2g_rs_trace_ch10.txt): the larger chunk stays.
  const uint32_t pad16 = apc_div_up(iters, 16) * 16, pad20 = apc_div_up(iters, 20) * 20;
  const uint32_t ch = pad20 < pad16 ? 20u : 16u;   // whichever pads num_iterations less (100 = 5 x 20)
  const uint32_t n_chunks = apc_div_up(iters, ch);
  // every CTA strides over the same number of point tiles
  const uint32_t gx0 = min(n_tiles, max(1u, (uint32_t)APC_SM_COUNT / n_chunks));
  const uint32_t gx = apc_div_up(n_tiles, apc_div_up(n_tiles, gx0));
  const dim3 grid(gx, n_chunks);
  const double log1mp = prob < 1.0 ? log(1.0 - prob) : -INFINITY;
  {
    APC_PROF(ctx, "k_rs_hypotheses", s);
    apc_klaunch(ctx, k_rs_hypotheses, apc_div_up(iters, RS_HYP_THREADS), RS_HYP_THREADS, 0, s, pts, n_max, n_dev, ransac_n, iters, seed, table,
                                                                              ctx->rs_planes, ctx->rs_col_tickets);
  }
  {
    APC_PROF(ctx, "k_rs_score", s);
#define RS_LAUNCH(CHV)                                                                                              \
  apc_klaunch(ctx, k_rs_score<CHV>, grid, APC_TILE_THREADS, 0, s, pts, n_max, n_dev, ransac_n, iters, ctx->rs_planes, thr, ctx->rs_scores, \
                                                    log1mp, out_plane, out_info, ctx->rs_scores_copy, ctx->rs_col_tickets, ctx->ctrl)
    if (ch == 20) RS_LAUNCH(20);
    else RS_LAUNCH(16);
#undef RS_LAUNCH
  }
  APC_PROF(ctx, "k_rs_final", s);
  apc_klaunch(ctx, k_rs_final, n_tiles, APC_TILE_THREADS, 0, s, pts, n_max, n_dev, out_plane, out_info, thr, out_mask, ctx->rs_partials,
                                                  reinterpret_cast<float4*>(out_keep_xyzi), out_keep_count,
                                                  ctx->scan_state[scan_slot], n_tiles, ctx->ctrl, keep_idx_in, keep_idx_out,
                                                  mir && out_keep_xyzi ? *mir : MirrorDev{}, nrm_in,
                                                  out_keep_xyzi ? nrm_out : nullptr);
  APC_LAUNCH_CHECK(ctx, "segment_plane");
  return APC_OK;
}

extern "C" int apc_segment_plane(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                 double distance_threshold, int ransac_n, int num_iterations, double probability,
                                 uint64_t seed, const int32_t* sample_table_dev, double* out_plane_dev,
                                 uint8_t* out_inlier_mask, uint32_t* out_info_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, out_inlier_mask, "NULL output pointer");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  return apc_segment_plane_nobegin(ctx, xyzi, n_max, n_dev, distance_threshold, ransac_n, num_iterations, probability,
                                   seed, sample_table_dev, out_plane_dev, out_inlier_mask, out_info_dev, nullptr, nullptr,
                                   4, s, nullptr, nullptr, nullptr, nullptr, nullptr);
}

// Per-hypothesis tallies {inlier count, integer error sum} of the most recent segment_plane call.
extern "C" int apc_segment_plane_scores(apc_ctx* ctx, uint64_t* out_scores_dev, uint32_t num_iterations, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, out_scores_dev && num_iterations <= ctx->rs_max_iters, "bad arguments");
  APC_CUDA(ctx, cudaMemcpyAsync(out_scores_dev, ctx->rs_scores_copy, (size_t)num_iterations * 2 * sizeof(uint64_t),
                                cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return APC_OK;
}
