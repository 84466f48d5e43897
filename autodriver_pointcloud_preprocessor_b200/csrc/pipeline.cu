// preprocess() end to end on the device (pp.py:447-544): front end -> voxel ->
// statistical outliers -> radius outliers -> RANSAC ground removal, chained through device
// counters so that no stage waits for the host, plus CUDA-graph capture / replay of the
// whole chain (one launch per scan).
#include <cmath>

#include "apc_grid.cuh"
APC_TRACE_EXPORT(pipeline)

// stage entry points without the per-call epoch bump (defined in the stage files)
int apc_frontend_nobegin(apc_ctx*, const apc_cloud_desc*, uint32_t, const apc_filter_cfg*, float*, uint32_t*, uint8_t*,
                         uint32_t*, int, cudaStream_t);
int apc_voxel_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, float, float*, int32_t*, uint32_t*, uint32_t*,
                      int, const GridDev*, cudaStream_t);
int apc_radius_grid_view(apc_ctx*, double, GridDev*);
int apc_select_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, const uint8_t*, int, float*, uint32_t*,
                       uint32_t*, int, cudaStream_t, const uint32_t*, const MirrorDev*);
int apc_radius_select_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, int, double, uint8_t*, float*, uint32_t*, int,
                              int, cudaStream_t, const uint32_t*, uint32_t*, const MirrorDev*);
int apc_statistical_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, int, double, float, uint8_t*, float*,
                            double*, cudaStream_t);
int apc_segment_plane_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, double, int, int, double, uint64_t,
                              const int32_t*, double*, uint8_t*, uint32_t*, float*, uint32_t*, int, cudaStream_t,
                              const uint32_t*, uint32_t*, const MirrorDev*, const float*, float*);
int apc_normals_nobegin(apc_ctx*, const float*, uint32_t, const uint32_t*, int, double, float*, uint32_t*, double*, cudaStream_t);
int apc_neighbors_prepare(apc_ctx*, int);
int apc_normals_prepare(apc_ctx*);
int apc_sort_prepare(apc_ctx*);

// dev_counts layout inside the context
enum { DC_FILTERED = 1, DC_VOXELS = 2, DC_STAT = 3, DC_RADIUS = 4, DC_OUT = 6, DC_INFO = 8 /* 4 words */ };   // pipeline_counts_write reads 1, 2, 3, 4, 8 + 1

__global__ void k_pipeline_counts(const __grid_constant__ CountsEpilogue fin, const ApcCtrl* ctrl) {
  pdl_enter();
  pipeline_counts_write(fin, ctrl);
  APC_STAMP(0, 0);
}

__global__ void k_iota(uint32_t* out, uint32_t n_max, const uint32_t* n_dev) {
  const uint32_t n = apc_count(n_dev, n_max);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = i;
}

static int run_pipeline(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds, const apc_pipeline_cfg* cfg,
                        float* out_xyzi, uint32_t* out_counts_dev, double* out_plane_dev, cudaStream_t s,
                        const apc_pipeline_maps* maps = nullptr, const apc_out_mirror* mirror = nullptr) {
  APC_REQUIRE(ctx, clouds && cfg && out_xyzi && out_counts_dev, "NULL pointer");
  MirrorDev mir{};
  CountsEpilogue fin{};
  if (mirror) {
    APC_REQUIRE(ctx, mirror->n_xyzi <= APC_MAX_MIRRORS && mirror->n_counts <= APC_MAX_MIRRORS, "too many mirrors");
    APC_REQUIRE(ctx, mirror->n_xyzi == 0 || cfg->stat_enable || cfg->radius_enable || cfg->ground_enable,
                "mirrored output rows need a selection stage (outlier or ground removal) at the end of the pipeline");
    mir.n = mirror->n_xyzi;
    mir.multicast = mirror->xyzi_multicast != 0;
    for (uint32_t k = 0; k < mir.n; ++k) {
      APC_REQUIRE(ctx, mirror->xyzi_dev[k], "mirror pointer is NULL");
      mir.out[k] = reinterpret_cast<float4*>(mirror->xyzi_dev[k]);
    }
    fin.n_mir = mirror->n_counts;
    for (uint32_t k = 0; k < fin.n_mir; ++k) {
      APC_REQUIRE(ctx, mirror->counts_dev[k], "mirror pointer is NULL");
      fin.mir[k] = mirror->counts_dev[k];
    }
  }
  uint32_t n_total = 0;
  for (uint32_t i = 0; i < n_clouds && i < APC_MAX_CLOUDS; ++i) n_total += clouds[i].n_points;
  const bool has_vox = cfg->voxel_size > 0.0f;
  const bool has_stat = cfg->stat_enable != 0, has_rad = cfg->radius_enable != 0, has_ground = cfg->ground_enable != 0;
  const int n_stages = 1 + has_vox + has_stat + has_rad + has_ground;
  const bool has_normals = cfg->normals_enable != 0;
  APC_REQUIRE(ctx, !has_normals || (maps && maps->normals_dev), "normals_enable needs maps.normals_dev");
  // k_begin and k_pipeline_counts stay launches of their own.  Folding them into k_dedup_insert and k_rs_final
  // (11 launches per C2 scan instead of 13) was slower: interleaved A/B, 8 lanes, two runs each - 64.84 / 64.69
  // us per scan folded against 63.37 / 63.77 with the two one-CTA launches, and the same single-scan latency
  // (0.133 ms): inside a captured graph the tiny launches cost less than what they take off the two big
  // kernels' critical paths (profiles/r2ab_fold_lanes.json).
  int rc = apc_begin(ctx, s);
  if (rc) return rc;
  uint32_t* dc = ctx->dev_counts;
  float* ping = reinterpret_cast<float*>(ctx->buf_a);
  float* pong = reinterpret_cast<float*>(ctx->buf_b);
  int stage = 0;
  auto last_mir = [&](void) -> const MirrorDev* {   // the stage that has just taken dst() == out_xyzi also mirrors
    return (stage == n_stages && mir.n) ? &mir : nullptr;
  };
  auto dst = [&](void) -> float* {  // output buffer of the stage about to run
    ++stage;
    if (stage == n_stages) return out_xyzi;
    float* d = ping;
    ping = pong;
    pong = d;
    return d;
  };
  // index maps (apc_pipeline_run_maps): every selection after the voxel stage also carries, per
  // surviving point, its row in the cloud the voxel stage produced; the last one writes out_row
  fin.dc = dc;
  fin.out = out_counts_dev;
  fin.n_input = n_total;
  fin.has_vox = has_vox; fin.has_stat = has_stat; fin.has_rad = has_rad; fin.has_ground = has_ground;
  uint32_t* const want_row = maps ? maps->out_row_dev : nullptr;
  int sel_left = want_row ? has_stat + has_rad + has_ground : 0;
  const uint32_t* row_in = nullptr;
  uint32_t* row_bufs[2] = {ctx->idx_a, ctx->idx_b};
  int row_flip = 0;
  auto row_out = [&](void) -> uint32_t* {   // destination of the selection stage about to run
    if (!want_row) return nullptr;
    return --sel_left == 0 ? want_row : row_bufs[row_flip++ & 1];
  };
  float* cur = dst();
  uint32_t cur_cnt = DC_FILTERED;
  rc = apc_frontend_nobegin(ctx, clouds, n_clouds, &cfg->filter, cur, maps ? maps->src_idx_dev : nullptr, nullptr,
                            dc + DC_FILTERED, 0, s);
  if (rc) return rc;
  // voxel -> radius with nothing in between: the voxel stage inserts its centroids into the radius
  // grid as it writes them (one launch and one pass over the centroids less)
  const bool grid_in_voxel = has_vox && has_rad && !has_stat && n_total > 0;
  if (has_vox) {
    float* out = dst();
    GridDev grid{};
    if (grid_in_voxel) {
      rc = apc_radius_grid_view(ctx, cfg->radius_search_radius, &grid);
      if (rc) return rc;
    }
    rc = apc_voxel_nobegin(ctx, cur, n_total, dc + cur_cnt, cfg->voxel_size, out, maps ? maps->p2v_dev : nullptr,
                           maps ? maps->voxel_counts_dev : nullptr, dc + DC_VOXELS, 1, grid_in_voxel ? &grid : nullptr, s);
    if (rc) return rc;
    cur = out;
    cur_cnt = DC_VOXELS;
  }
  if (has_stat) {
    float* out = dst();
    // level-0 cell such that the k nearest of a point on a voxelised surface (one point per
    // voxel_size^2: r_k = voxel_size * sqrt(k / pi)) usually lie inside the first 27-cell block; the
    // result does not depend on it (the query climbs levels until the k-th distance is covered).  The factor
    // 1.25 was kept against 1.5 and 2.0 (profiles/r2x_knn_ab.json).
    const float hint = has_vox ? 1.25f * cfg->voxel_size * fmaxf(2.0f, 1.3f * sqrtf((float)cfg->stat_nb_neighbors / 3.14159265f)) : 0.0f;
    rc = apc_statistical_nobegin(ctx, cur, n_total, dc + cur_cnt, cfg->stat_nb_neighbors, cfg->stat_std_ratio, hint,
                                 ctx->mask_a, nullptr, nullptr, s);
    if (rc) return rc;
    uint32_t* rows = row_out();
    rc = apc_select_nobegin(ctx, cur, n_total, dc + cur_cnt, ctx->mask_a, 0, out, rows, dc + DC_STAT, 2, s, row_in, last_mir());
    if (rc) return rc;
    row_in = rows;
    cur = out;
    cur_cnt = DC_STAT;
  }
  if (has_rad) {
    float* out = dst();
    // the select_by_mask of the radius decision also cleans the neighbour grid (one launch)
    uint32_t* rows = row_out();
    rc = apc_radius_select_nobegin(ctx, cur, n_total, dc + cur_cnt, cfg->radius_nb_points, cfg->radius_search_radius,
                                   ctx->mask_a, out, dc + DC_RADIUS, 3, grid_in_voxel ? 1 : 0, s, row_in, rows, last_mir());
    if (rc) return rc;
    row_in = rows;
    cur = out;
    cur_cnt = DC_RADIUS;
  }
  // estimate_normals (pp.py:521-530) on the cloud that enters the ground stage; without a ground
  // stage that cloud IS the output and the normals are written in place
  const float* nrm_in = nullptr;
  if (has_normals && n_total) {
    float* nrm = has_ground ? ctx->nrm_scratch : maps->normals_dev;
    APC_REQUIRE(ctx, nrm, "normals scratch not prepared");
    rc = apc_normals_nobegin(ctx, cur, n_total, dc + cur_cnt, cfg->normals_max_nn, cfg->normals_radius, nrm, nullptr, nullptr, s);
    if (rc) return rc;
    nrm_in = nrm;
  }
  if (has_ground) {
    float* out = dst();
    double* plane = out_plane_dev ? out_plane_dev : ctx->red_b;
    uint32_t* rows = row_out();
    // pp.py:542 select_by_index(inliers, invert=True) is fused into the final RANSAC pass: the
    // non-ground points are written in order straight to `out`
    rc = apc_segment_plane_nobegin(ctx, cur, n_total, dc + cur_cnt, cfg->ground_distance_threshold, cfg->ground_ransac_n,
                                   cfg->ground_num_iterations, cfg->ground_probability, cfg->ground_seed, nullptr, plane,
                                   nullptr, dc + DC_INFO, out, dc + DC_OUT, 4, s, row_in, rows, last_mir(), nrm_in,
                                   nrm_in ? maps->normals_dev : nullptr);
    if (rc) return rc;
    row_in = rows;
    cur = out;
    cur_cnt = DC_OUT;
  }
  if (want_row && !row_in && n_total) {   // no selection stage ran: output row i is row i
    k_iota<<<min(apc_div_up(n_total, 256), (uint32_t)APC_SM_COUNT * 4), 256, 0, s>>>(want_row, n_total, dc + cur_cnt);
    APC_LAUNCH_CHECK(ctx, "k_iota");
  }
  fin.last = cur_cnt;
  apc_klaunch(ctx, k_pipeline_counts, 1, 1, 0, s, fin, ctx->ctrl);
  APC_LAUNCH_CHECK(ctx, "k_pipeline_counts");
  return APC_OK;
}

static int prepare(apc_ctx* ctx, const apc_pipeline_cfg* cfg) {
  int rc = APC_OK;
  if (cfg->radius_enable) rc = apc_neighbors_prepare(ctx, 0);
  if (!rc && cfg->stat_enable) rc = apc_neighbors_prepare(ctx, 1);
  if (!rc && cfg->filter.dedup_mode >= APC_DEDUP_NUMPY) rc = apc_sort_prepare(ctx);
  if (!rc && cfg->normals_enable) {
    rc = apc_normals_prepare(ctx);
    if (!rc && cfg->ground_enable && !ctx->nrm_scratch)
      APC_CUDA(ctx, cudaMalloc((void**)&ctx->nrm_scratch, (size_t)ctx->max_points * 3 * sizeof(float)));
  }
  return rc;
}

extern "C" int apc_pipeline_run(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                double* out_plane_dev, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, cfg, "cfg is NULL");
  int rc = prepare(ctx, cfg);
  if (rc) return rc;
  return run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, (cudaStream_t)stream);
}

extern "C" int apc_pipeline_run_maps(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                     const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                     double* out_plane_dev, const apc_pipeline_maps* maps, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, cfg && maps, "NULL pointer");
  int rc = prepare(ctx, cfg);
  if (rc) return rc;
  return run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, (cudaStream_t)stream, maps);
}

extern "C" int apc_pipeline_run_ex(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                   const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                   double* out_plane_dev, const apc_pipeline_maps* maps, const apc_out_mirror* mirror,
                                   void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, cfg, "cfg is NULL");
  int rc = prepare(ctx, cfg);
  if (rc) return rc;
  return run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, (cudaStream_t)stream, maps, mirror);
}

extern "C" int apc_pipeline_run_mirrored(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                         const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                         double* out_plane_dev, const apc_out_mirror* mirror, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, cfg, "cfg is NULL");
  int rc = prepare(ctx, cfg);
  if (rc) return rc;
  return run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, (cudaStream_t)stream, nullptr,
                      mirror);
}

struct apc_graph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaStream_t capture_stream = nullptr;
};

extern "C" int apc_graph_destroy(apc_graph* g) {
  if (!g) return APC_OK;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  if (g->capture_stream) cudaStreamDestroy(g->capture_stream);
  delete g;
  return APC_OK;
}

extern "C" int apc_graph_capture_pipeline(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                          const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                          double* out_plane_dev, apc_graph** out_graph) {
  return apc_graph_capture_pipeline_mirrored(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, nullptr,
                                             out_graph);
}

extern "C" int apc_graph_capture_pipeline_mirrored(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                                   const apc_pipeline_cfg* cfg, float* out_xyzi,
                                                   uint32_t* out_counts_dev, double* out_plane_dev,
                                                   const apc_out_mirror* mirror, apc_graph** out_graph) {
  return apc_graph_capture_pipeline_ex(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, nullptr, mirror,
                                       out_graph);
}

extern "C" int apc_graph_capture_pipeline_ex(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                             const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                             double* out_plane_dev, const apc_pipeline_maps* maps,
                                             const apc_out_mirror* mirror, apc_graph** out_graph) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, cfg && out_graph, "NULL pointer");
  *out_graph = nullptr;
  APC_CUDA(ctx, cudaSetDevice(ctx->device));
  int rc = prepare(ctx, cfg);
  if (rc) return rc;
  apc_graph* g = new apc_graph();
  cudaError_t e = cudaStreamCreateWithFlags(&g->capture_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { delete g; return apc_set_error(ctx, APC_ERR_CUDA, "cudaStreamCreate", e); }
  // one eager run first: lazily configured attributes (dynamic shared memory limits) are set
  // outside the capture, and argument errors surface before a capture is open
  rc = run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, g->capture_stream, maps, mirror);
  if (!rc && (e = cudaStreamSynchronize(g->capture_stream)) != cudaSuccess)
    rc = apc_set_error(ctx, APC_ERR_CUDA, "pipeline warm-up before capture", e);
  if (rc) { apc_graph_destroy(g); return rc; }
  e = cudaStreamBeginCapture(g->capture_stream, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { apc_graph_destroy(g); return apc_set_error(ctx, APC_ERR_CUDA, "cudaStreamBeginCapture", e); }
  rc = run_pipeline(ctx, clouds, n_clouds, cfg, out_xyzi, out_counts_dev, out_plane_dev, g->capture_stream, maps, mirror);
  e = cudaStreamEndCapture(g->capture_stream, &g->graph);
  if (rc) { apc_graph_destroy(g); return rc; }
  if (e != cudaSuccess) { apc_graph_destroy(g); return apc_set_error(ctx, APC_ERR_CUDA, "cudaStreamEndCapture", e); }
  e = cudaGraphInstantiate(&g->exec, g->graph, 0);
  if (e != cudaSuccess) { apc_graph_destroy(g); return apc_set_error(ctx, APC_ERR_CUDA, "cudaGraphInstantiate", e); }
  *out_graph = g;
  return APC_OK;
}

extern "C" int apc_graph_kernel_count(const apc_graph* g) {
  if (!g || !g->graph) return APC_ERR_BAD_ARG;
  size_t n = 0;
  if (cudaGraphGetNodes(g->graph, nullptr, &n) != cudaSuccess) return APC_ERR_CUDA;
  std::vector<cudaGraphNode_t> nodes(n);
  if (n && cudaGraphGetNodes(g->graph, nodes.data(), &n) != cudaSuccess) return APC_ERR_CUDA;
  int kernels = 0;
  for (size_t i = 0; i < n; ++i) {
    cudaGraphNodeType t;
    if (cudaGraphNodeGetType(nodes[i], &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) ++kernels;
  }
  return kernels;
}

extern "C" int apc_graph_launch(apc_ctx* ctx, apc_graph* g, void* stream) {
  if (!ctx) return APC_ERR_BAD_ARG;
  APC_REQUIRE(ctx, g && g->exec, "graph is NULL");
  APC_CUDA(ctx, cudaGraphLaunch(g->exec, (cudaStream_t)stream));
  return APC_OK;
}
