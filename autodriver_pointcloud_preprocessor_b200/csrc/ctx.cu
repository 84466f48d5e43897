// Context lifecycle, scratch sizing, error reporting (apc.h lifecycle section).
// Replaces the reference's per-node device/point-cloud setup (pp.py:272-280, pp.py:309).
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "apc_common.cuh"

static thread_local std::string g_create_error;
APC_TRACE_EXPORT(ctx)



// table resets (context creation and error recovery); defined next to the kernels that own them
int apc_voxel_reset(apc_ctx* ctx, cudaStream_t s);
int apc_dedup_reset(apc_ctx* ctx, cudaStream_t s);
int apc_neighbors_reset(apc_ctx* ctx, cudaStream_t s);
void apc_neighbors_release(apc_ctx* ctx);
void apc_sort_release(apc_ctx* ctx);

static int reset_tables(apc_ctx* ctx, cudaStream_t s) {
  int rc = apc_voxel_reset(ctx, s);
  if (!rc) rc = apc_dedup_reset(ctx, s);
  if (!rc) rc = apc_neighbors_reset(ctx, s);
  return rc;
}

int apc_set_error(apc_ctx* ctx, int code, const char* what, cudaError_t ce) {
  char buf[512];
  if (ce != cudaSuccess)
    snprintf(buf, sizeof(buf), "apc error %d: %s: %s", code, what, cudaGetErrorString(ce));
  else
    snprintf(buf, sizeof(buf), "apc error %d: %s", code, what);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

__global__ void k_begin(ApcCtrl* ctrl) {
  pdl_enter();
  APC_STAMP(0, 0);
  if (threadIdx.x == 0) ctrl->epoch = ctrl->epoch + 1u;
  if (threadIdx.x < 30) ctrl->counters[threadIdx.x] = 0u;
}

int apc_begin(apc_ctx* ctx, cudaStream_t s) {
  int cur = -1;
  if (cudaGetDevice(&cur) == cudaSuccess && cur != ctx->device)
    return apc_set_error(ctx, APC_ERR_BAD_ARG, "the context lives on another device than the calling thread's current one");
  ctx->launch_seq = 0;
  apc_klaunch(ctx, k_begin, 1, 32, 0, s, ctx->ctrl);
  APC_LAUNCH_CHECK(ctx, "k_begin");
  return APC_OK;
}

template <typename T>
static cudaError_t dalloc(T** p, size_t n) {
  return cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T));
}

static uint32_t next_pow2(uint64_t v) {
  uint64_t p = 1024;
  while (p < v) p <<= 1;
  return (uint32_t)p;
}

extern "C" int apc_version(void) { return APC_VERSION; }

extern "C" uint32_t apc_ctx_max_points(const apc_ctx* ctx) { return ctx ? ctx->max_points : 0; }

extern "C" const char* apc_last_error(const apc_ctx* ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int apc_ctx_destroy(apc_ctx* ctx) {
  if (!ctx) return APC_OK;
  cudaSetDevice(ctx->device);
  apc_neighbors_release(ctx);
  apc_sort_release(ctx);
  for (cudaEvent_t e : ctx->prof.ev) cudaEventDestroy(e);
  void* ptrs[] = {ctx->ctrl, ctx->vox_slots, ctx->vox_acc, ctx->vox_rank, ctx->p2slot,
                  ctx->dedup_slots, ctx->sorted_pts, ctx->knn_avg, ctx->red_a,
                  ctx->red_b, ctx->rs_planes, ctx->rs_scores, ctx->rs_scores_copy, ctx->rs_col_tickets, ctx->rs_partials, ctx->buf_a, ctx->buf_b,
                  ctx->mask_a, ctx->idx_a, ctx->idx_b, ctx->dev_counts, ctx->nrm_scratch};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  for (auto* p : ctx->scan_state)
    if (p) cudaFree(p);
  delete ctx;
  return APC_OK;
}

extern "C" int apc_ctx_create(int device, uint32_t max_points, apc_ctx** out) {
  if (!out) return apc_set_error(nullptr, APC_ERR_BAD_ARG, "out is NULL");
  *out = nullptr;
  if (max_points == 0 || max_points > (1u << 22))
    return apc_set_error(nullptr, APC_ERR_BAD_ARG, "max_points must be in 1..4194304");
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return apc_set_error(nullptr, APC_ERR_CUDA, "cudaSetDevice", e);
  apc_ctx* ctx = new apc_ctx();
  ctx->device = device;
  ctx->max_points = max_points;
  if (const char* lb = getenv("APC_LAUNCH_BUDGET")) ctx->launch_budget = atoi(lb);
  const size_t M = max_points;
  // load factor <= 0.25: short probe chains (the warp-wide worst chain sets the latency).
  // APC_HASH_SLOTS_PER_POINT overrides for experiments.
  const char* lf = getenv("APC_HASH_SLOTS_PER_POINT");
  ctx->hash_cap = next_pow2((lf && atoi(lf) >= 2 ? (uint64_t)atoi(lf) : 4ull) * M);
  const size_t C = ctx->hash_cap;
  ctx->max_tiles = apc_div_up((uint32_t)(C > M ? C : M), 1024) + 8;
  ctx->rs_max_iters = 4096;
  const size_t red = C / 256 + 64;
#define A(expr)                                                         \
  if ((e = (expr)) != cudaSuccess) {                                    \
    apc_set_error(nullptr, APC_ERR_CUDA, "cudaMalloc(" #expr ")", e);  \
    apc_ctx_destroy(ctx);                                               \
    return APC_ERR_CUDA;                                                \
  }
  A(dalloc(&ctx->ctrl, 1));
  for (auto& p : ctx->scan_state) A(dalloc(&p, (size_t)ctx->max_tiles + 1024));   // + APC_SCAN_GROUPS group words
  A(dalloc(&ctx->vox_slots, C));
  A(dalloc(&ctx->vox_acc, C));
  A(dalloc(&ctx->vox_rank, C));
  A(dalloc(&ctx->p2slot, M));
  A(dalloc(&ctx->dedup_slots, C));
  A(dalloc(&ctx->sorted_pts, M));
  A(dalloc(&ctx->knn_avg, M));
  A(dalloc(&ctx->red_a, red));
  A(dalloc(&ctx->red_b, red));
  A(dalloc(&ctx->rs_planes, (size_t)ctx->rs_max_iters * 4));
  // per-CTA tally rows of k_rs_score: <= 2 CTAs per SM, 20 hypotheses each, plus one padded row per launch
  A(dalloc(&ctx->rs_scores, (size_t)(APC_SM_COUNT * 2 * 20 + ctx->rs_max_iters + 64) * 2));
  A(dalloc(&ctx->rs_scores_copy, (size_t)ctx->rs_max_iters * 2));
  A(cudaMemset(ctx->rs_scores_copy, 0, (size_t)ctx->rs_max_iters * 2 * sizeof(unsigned long long)));
  A(dalloc(&ctx->rs_col_tickets, ctx->rs_max_iters));
  A(dalloc(&ctx->rs_partials, (size_t)(M / 256 + 64) * 10));
  A(dalloc(&ctx->buf_a, M));
  A(dalloc(&ctx->buf_b, M));
  A(dalloc(&ctx->mask_a, M));
  A(dalloc(&ctx->idx_a, M));
  A(dalloc(&ctx->idx_b, M));
  A(dalloc(&ctx->dev_counts, 16));
  A(cudaMemset(ctx->ctrl, 0, sizeof(ApcCtrl)));
  for (auto& p : ctx->scan_state) A(cudaMemset(p, 0, ((size_t)ctx->max_tiles + 1024) * sizeof(uint64_t)));
  A(cudaMemset(ctx->dev_counts, 0, 16 * sizeof(uint32_t)));
  if (reset_tables(ctx, 0) != APC_OK) {
    g_create_error = ctx->err;
    apc_ctx_destroy(ctx);
    return APC_ERR_CUDA;
  }
  A(cudaDeviceSynchronize());
#undef A
  *out = ctx;
  return APC_OK;
}

extern "C" int apc_ctx_set_low_latency(apc_ctx* ctx, int on) {
  if (!ctx) return APC_ERR_BAD_ARG;
  ctx->low_latency = on != 0;
  return APC_OK;
}

extern "C" int apc_profile_enable(apc_ctx* ctx, int on) {
  if (!ctx) return APC_ERR_BAD_ARG;
  ctx->prof.enabled = on != 0;
  ctx->prof.used = 0;
  return APC_OK;
}

extern "C" int apc_profile_report(apc_ctx* ctx, char* buf, uint32_t buf_len) {
  if (!ctx || !buf || buf_len == 0) return APC_ERR_BAD_ARG;
  APC_CUDA(ctx, cudaDeviceSynchronize());
  ApcProf& p = ctx->prof;
  std::vector<const char*> names;
  std::vector<double> total;
  std::vector<int> count;
  for (size_t i = 0; i < p.used; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.ev[2 * i], p.ev[2 * i + 1]) != cudaSuccess) continue;
    size_t k = 0;
    for (; k < names.size(); ++k)
      if (strcmp(names[k], p.names[i]) == 0) break;
    if (k == names.size()) { names.push_back(p.names[i]); total.push_back(0.0); count.push_back(0); }
    total[k] += ms;
    count[k] += 1;
  }
  p.used = 0;
  std::string out;
  char line[160];
  for (size_t k = 0; k < names.size(); ++k) {
    snprintf(line, sizeof(line), "%s %.6f %d\n", names[k], total[k], count[k]);
    out += line;
  }
  const size_t n = out.size() < (size_t)buf_len - 1 ? out.size() : (size_t)buf_len - 1;
  memcpy(buf, out.data(), n);
  buf[n] = 0;
  return (int)n;
}

extern "C" int apc_check(apc_ctx* ctx, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  APC_CUDA(ctx, cudaStreamSynchronize(s));
  uint32_t err = 0;
  APC_CUDA(ctx, cudaMemcpy(&err, &ctx->ctrl->err, sizeof(err), cudaMemcpyDeviceToHost));
  if (err) {
    APC_CUDA(ctx, cudaMemset(&ctx->ctrl->err, 0, sizeof(uint32_t)));
    // a failed insert may have left the self-cleaning tables dirty: wipe them
    int rc = reset_tables(ctx, s);
    if (rc) return rc;
    APC_CUDA(ctx, cudaStreamSynchronize(s));
    if (err & APC_DEVERR_KEY_RANGE)
      return apc_set_error(ctx, APC_ERR_KEY_RANGE,
                           "voxel index outside +-2^20 or coordinate magnitude >= 2^16 m (non-finite input?)");
    return apc_set_error(ctx, APC_ERR_CAPACITY, "hash table / scratch capacity exceeded");
  }
  return APC_OK;
}
