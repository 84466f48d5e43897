// Shared device/host plumbing for the apc kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "apc.h"

#define APC_SM_COUNT 148  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

// ---- context -----------------------------------------------------------------------------
// Control block living in device memory (one per context).
struct ApcCtrl {
  uint32_t epoch;       // bumped once per public API call; tags decoupled look-back states
  uint32_t err;         // sticky data-dependent error bits (see ERR_* below)
  uint32_t counters[30];
};
enum { APC_DEVERR_KEY_RANGE = 1u, APC_DEVERR_CAPACITY = 2u };

#define APC_NUM_SCAN_STATES 8

// One voxel of the open-addressing table, split in a 16-byte HOT slot and a 48-byte COLD record kept in
// separate arrays.  The hot slot is everything a single-point voxel ever touches (77 % of the voxels of a
// 0.1 m C2 scan): the point whose CAS claims the slot (the "owner") records its index with a plain store
// and its coordinates are added when the voxel is finalised.  Only the points that JOIN an existing voxel
// pay the accumulating atomics (0.7 M per scan instead of 1.8 M), which land in the cold record.
// Placement keeps neighbours together: the slot index is hash(2x2 block of voxels in x, y) * 4 + the
// voxel's position inside the block, so the four voxels of a block share ONE 64-byte DRAM burst (two
// 32-byte sectors) and eight share a 128-byte line - a surface fills 2 to 4 of a block's slots.  Round 1
// used 32-byte hot slots (one sector per voxel, two per burst): the table is random-access traffic, read
// and written back by both the insert and the finalize kernel, and at 1 M points it IS the voxel stage's
// DRAM traffic (178 B per point against 36 B algorithmic, profiles/r2d_voxel_ab_ncu.csv).
struct __align__(16) VoxSlot {
  unsigned long long key;     // packed 63-bit voxel key, all ones = empty
  uint32_t first;             // lowest index among the JOINING points (0xffffffff: none)
  uint32_t owner;             // index of the point that claimed the slot
};
struct __align__(16) VoxAcc {
  unsigned long long acc[4];  // fixed-point sums over the joining points: x, y, z (2^-24 m), intensity (2^-20)
  uint32_t cnt;               // number of joining points (the owner is not counted)
  uint32_t pad[3];
};
static_assert(sizeof(VoxSlot) == 16 && sizeof(VoxAcc) == 48, "voxel table layout");

// Optional per-kernel timing with CUDA events on the launching stream (apc_profile_*).
struct ApcProf {
  bool enabled = false;
  std::vector<cudaEvent_t> ev;       // pairs: start, stop
  std::vector<const char*> names;    // one per pair
  size_t used = 0;                   // pairs in use
};

struct apc_ctx {
  ApcProf prof;
  int device = 0;
  uint32_t max_points = 0;
  std::string err;
  ApcCtrl* ctrl = nullptr;                       // device
  uint64_t* scan_state[APC_NUM_SCAN_STATES] = {};  // device, max_tiles words each
  uint32_t max_tiles = 0;
  // hash tables (capacity = power of two >= 2*max_points)
  uint32_t hash_cap = 0;
  struct VoxSlot* vox_slots = nullptr;  // [hash_cap] hot slots {key, first, owner}
  struct VoxAcc* vox_acc = nullptr;     // [hash_cap] cold records: fixed-point sums + count of the joining points
  uint32_t* vox_rank = nullptr;     // [hash_cap] output row of the slot
  uint32_t* p2slot = nullptr;       // [max_points]
  unsigned long long* dedup_slots = nullptr;  // [hash_cap] {key fingerprint:32 | lowest point index:32}
  float4* sorted_pts = nullptr;     // [max_points] NaN-skipped cloud of the sorted duplicate-removal modes
  float* knn_avg = nullptr;         // [max_points]
  double* red_a = nullptr;          // reduction ping-pong
  double* red_b = nullptr;
  // ransac
  double* rs_planes = nullptr;      // [max_iters*4]
  unsigned long long* rs_scores = nullptr;  // per-CTA tally rows of k_rs_score {inliers, err}, column by column
  unsigned long long* rs_scores_copy = nullptr;  // [max_iters*2] the last call's tallies, summed over the CTAs
  uint32_t* rs_col_tickets = nullptr;  // [max_iters] retired CTAs of each chunk column of k_rs_score
  double* rs_partials = nullptr;    // refit partial sums
  uint32_t rs_max_iters = 0;
  // pipeline ping-pong buffers
  float4* buf_a = nullptr;
  float4* buf_b = nullptr;
  uint8_t* mask_a = nullptr;
  uint32_t* idx_a = nullptr;
  uint32_t* idx_b = nullptr;        // second row-index buffer of the pipeline's index maps
  uint32_t* dev_counts = nullptr;   // [16] intermediate device counters
  // sorted-unique rows (sort.cu), allocated on first use
  uint4* sort_a = nullptr;          // [max_points] {kx, ky, kz, index} ping
  uint4* sort_b = nullptr;          // pong
  uint32_t* sort_hist = nullptr;    // [12][256] digit histograms
  uint64_t* sort_status = nullptr;  // [sort tiles][256] look-back words
  uint32_t* sort_idx = nullptr;     // [max_points] first-index / inverse list of the pipeline's sort modes
  float* nrm_scratch = nullptr;     // [3 * max_points] normals of the cloud entering the ground stage (pipeline), on first use
  struct NeighborScratch* neighbors = nullptr;   // neighbour grids + KNN scratch (neighbors.cu), on first use
  bool low_latency = false;         // apc_ctx_set_low_latency: programmatic dependent launches on the pipeline path
  // profiling probe (APC_LAUNCH_BUDGET=k at context creation, profiles/kernel_marginal.py): only the first k
  // kernels of every public call are launched, so that the cost of the k-th kernel with all lanes busy is
  // the difference between two runs.  -1 = off.
  int launch_budget = -1;
  mutable int launch_seq = 0;       // launches issued since apc_begin
};

// RAII timer around one kernel launch; a no-op unless profiling is enabled on the context.
struct ProfScope {
  apc_ctx* c;
  cudaStream_t s;
  cudaEvent_t stop = nullptr;
  ProfScope(apc_ctx* ctx, const char* name, cudaStream_t stream) : c(ctx), s(stream) {
    if (!c->prof.enabled) return;
    ApcProf& p = c->prof;
    if (p.used * 2 + 2 > p.ev.size()) {
      cudaEvent_t a, b;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
      p.ev.push_back(a);
      p.ev.push_back(b);
      p.names.push_back(name);
    }
    p.names[p.used] = name;
    cudaEventRecord(p.ev[p.used * 2], s);
    stop = p.ev[p.used * 2 + 1];
    ++p.used;
  }
  ~ProfScope() {
    if (stop) cudaEventRecord(stop, s);
  }
};
#define APC_PROF_CAT2(a, b) a##b
#define APC_PROF_CAT(a, b) APC_PROF_CAT2(a, b)
#define APC_PROF(ctx, name, stream) ProfScope APC_PROF_CAT(_prof_, __LINE__)(ctx, name, stream)

int apc_set_error(apc_ctx* ctx, int code, const char* what, cudaError_t ce = cudaSuccess);
// bumps the epoch; every public entry point calls it first
int apc_begin(apc_ctx* ctx, cudaStream_t s);

#define APC_CUDA(ctx, call)                                                \
  do {                                                                     \
    cudaError_t _e = (call);                                               \
    if (_e != cudaSuccess) return apc_set_error((ctx), APC_ERR_CUDA, #call, _e); \
  } while (0)

#define APC_LAUNCH_CHECK(ctx, name)                                        \
  do {                                                                     \
    cudaError_t _e = cudaGetLastError();                                   \
    if (_e != cudaSuccess) return apc_set_error((ctx), APC_ERR_CUDA, name, _e); \
  } while (0)

#define APC_REQUIRE(ctx, cond, msg)                                        \
  do {                                                                     \
    if (!(cond)) return apc_set_error((ctx), APC_ERR_BAD_ARG, msg);        \
  } while (0)

static inline uint32_t apc_div_up(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

// Kernel launch of the per-scan path.  In low-latency mode (one scan in flight: the ROS node, pp.py:1056)
// every launch carries the programmatic-stream-serialization attribute: the next kernel of the chain is
// set up and its CTAs made resident while the current one still runs, and starts computing the moment
// the current one has completed and flushed (griddepcontrol.wait at the top of every such kernel),
// instead of paying a launch latency of ~3 us per stage boundary, 13 times per scan.  Off by default:
// with eight lanes sharing the GPU the pre-launched, waiting CTAs would only take room from the other
// lanes' kernels.  Errors are picked up by the APC_LAUNCH_CHECK that follows the call.
#ifdef __CUDACC__
template <typename... P, typename... A>
static inline void apc_klaunch(const apc_ctx* ctx, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem,
                               cudaStream_t s, A&&... args) {
  if (ctx->launch_budget >= 0 && ctx->launch_seq++ >= ctx->launch_budget) return;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  if (ctx->low_latency) {
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
  }
  cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}
// First statement of every kernel launched through apc_klaunch: wait for the preceding kernel's results
// (a no-op for an ordinary launch), then let the following kernel be set up behind this one.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
#endif

// ---- device helpers ----------------------------------------------------------------------
#ifdef __CUDACC__

// The pipeline's eight output counters (APC_CNT_*), assembled from the stages' device counters by the
// one-thread k_pipeline_counts, the last kernel of every pipeline run.
struct CountsEpilogue {
  const uint32_t* dc;          // the context's dev_counts
  uint32_t* out;               // uint32[8]
  uint32_t n_input, last;
  int has_vox, has_stat, has_rad, has_ground;
  uint32_t n_mir;
  uint32_t* mir[APC_MAX_MIRRORS];   // the peers' copies of this frame's counters (see apc_out_mirror)
};
__device__ __forceinline__ void pipeline_counts_write(const CountsEpilogue& e, const ApcCtrl* ctrl) {
  const volatile uint32_t* dc = e.dc;
  uint32_t c[8];
  c[APC_CNT_INPUT] = e.n_input;
  c[APC_CNT_FILTERED] = dc[1];
  uint32_t cur = dc[1];
  c[APC_CNT_VOXELS] = cur = e.has_vox ? dc[2] : cur;
  c[APC_CNT_AFTER_STAT] = cur = e.has_stat ? dc[3] : cur;
  c[APC_CNT_AFTER_RADIUS] = cur = e.has_rad ? dc[4] : cur;
  c[APC_CNT_GROUND_INLIERS] = e.has_ground ? dc[8 + 1] : 0u;
  c[APC_CNT_OUTPUT] = dc[e.last];
  c[APC_CNT_STATUS] = *reinterpret_cast<const volatile uint32_t*>(&ctrl->err);
#pragma unroll
  for (int k = 0; k < 8; ++k) e.out[k] = c[k];
  for (uint32_t m = 0; m < e.n_mir; ++m)
#pragma unroll
    for (int k = 0; k < 8; ++k) e.mir[m][k] = c[k];
}

__device__ __forceinline__ uint32_t apc_count(const uint32_t* n_dev, uint32_t n_max) {
  uint32_t n = n_dev ? *n_dev : n_max;
  return n < n_max ? n : n_max;
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// Counter-based random stream of RANSAC's hypotheses and FGR's tuples (oracle/ransac.py: splitmix64)
__device__ __forceinline__ uint64_t splitmix64_dev(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
  return __reduce_add_sync(0xffffffffu, v);
}

__device__ __forceinline__ uint64_t ld_volatile_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// 128-bit relaxed accesses at gpu scope: a 16-byte aligned vector access is performed as one transaction,
// and the qualifier keeps the compiler from splitting, caching or re-ordering it against the other CTAs'
// accesses to the same slot (voxel.cu: slots are cleaned by one CTA while others still read them).
__device__ __forceinline__ uint4 ld_relaxed_u4(const void* p) {
  uint4 v;
  asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u4(void* p, uint4 v) {
  asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// "Last CTA" ticket: called by ONE thread after a __syncthreads().  The acq_rel RMW at gpu scope
// releases everything the CTA wrote before the barrier and acquires what the other CTAs released,
// without the sequentially-consistent fence __threadfence() compiles to (MEMBAR.SC: measured
// ~65 ns each and globally serialised, i.e. ~17 us across the 260 CTAs of one RANSAC launch).
__device__ __forceinline__ uint32_t ticket_acq_rel(uint32_t* counter) {
  uint32_t old;
  asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
  return old;
}

// streaming 128-bit load / store (inputs are read once, outputs written once)
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// ---- mirrored output rows (multi-GPU exchange fused into the final stage) ---------------------
// The batched replay configuration ends with "every GPU holds every GPU's output"
// (BASELINE.json north_star; SURVEY.md section 8e).  Instead of gathering finished slabs with
// copy engines or NCCL afterwards, the kernel that writes the final cloud also stores every
// surviving row into the peers' buffers over NVLink (peer-mapped pointers; entry 0 may be an NVLS
// multicast address, written once and replicated by the switch): only real rows travel, there is
// no padding, no staging copy and no second read of the slab.
struct MirrorDev {
  uint32_t n;          // destinations besides the local output (0 = none)
  uint32_t multicast;  // != 0: out[0] is a multicast address (multimem.st)
  float4* out[APC_MAX_MIRRORS];
};
__device__ __forceinline__ void mirror_store(const MirrorDev& m, uint32_t row, float4 v) {
  for (uint32_t k = 0; k < m.n; ++k) {
    if (k == 0 && m.multicast)
      asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(m.out[0] + row), "f"(v.x),
                   "f"(v.y), "f"(v.z), "f"(v.w)
                   : "memory");
    else
      m.out[k][row] = v;
  }
}

// 64-bit mix (splitmix64 finaliser) used as the hash of packed keys
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// float32 rigid/projective transform, unfused, left to right, IEEE divide by w
// (Open3D t.PointCloud.transform; oracle/filters.py:transform)
__device__ __forceinline__ void xform_f32(const float* __restrict__ T, float& x, float& y, float& z) {
  float r0 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[0], x), __fmul_rn(T[1], y)), __fmul_rn(T[2], z)), T[3]);
  float r1 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[4], x), __fmul_rn(T[5], y)), __fmul_rn(T[6], z)), T[7]);
  float r2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[8], x), __fmul_rn(T[9], y)), __fmul_rn(T[10], z)), T[11]);
  float w = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(T[12], x), __fmul_rn(T[13], y)), __fmul_rn(T[14], z)), T[15]);
  x = __fdiv_rn(r0, w);
  y = __fdiv_rn(r1, w);
  z = __fdiv_rn(r2, w);
}

// ---- optional CTA timeline (build with APC_TRACE=1; read with profiles/cta_trace.py) ------------
#ifdef APC_TRACE
static __device__ unsigned long long g_apc_trace[8][2048][4];   // per translation unit: [kernel id][CTA][stamp]
#define APC_TRACE_EXPORT(name)                                                              \
  extern "C" int apc_debug_trace_##name(unsigned long long* out_host) {                     \
    cudaError_t e = cudaMemcpyFromSymbol(out_host, g_apc_trace, sizeof(g_apc_trace));       \
    void* p = nullptr;                                                                      \
    cudaGetSymbolAddress(&p, g_apc_trace);                                                  \
    cudaMemset(p, 0, sizeof(g_apc_trace));                                                  \
    return (int)e;                                                                          \
  }
__device__ __forceinline__ void apc_stamp(int kid, int k) {
  if (threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const uint32_t cta = blockIdx.x + blockIdx.y * gridDim.x;
    if (cta < 2048) g_apc_trace[kid][cta][k] = t;
  }
}
#define APC_STAMP(kid, k) apc_stamp(kid, k)
#else
#define APC_STAMP(kid, k) do { } while (0)
#define APC_TRACE_EXPORT(name)
#endif

__device__ __forceinline__ bool is_nan_f(float v) { return v != v; }
__device__ __forceinline__ bool is_inf_f(float v) { return fabsf(v) == __int_as_float(0x7f800000); }

#endif  // __CUDACC__
