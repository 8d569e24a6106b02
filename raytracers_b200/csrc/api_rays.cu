// C ABI, part 5: ray queries on a prepared scene - closest hit and path colour of caller-supplied rays
// (include/ray_b200.h "ray queries"; kernel: render_raycast.cu).
#include "api_internal.h"
#include "render_raycast.h"

using namespace rayb200_api;

namespace {

constexpr int64_t kMaxQueryRays = (int64_t)1 << 30;

// Validates, plans the staging like a warp-queue frame with one 32-ray slot set per warp, and enqueues one query on the
// context's stream.  `what` names the entry point in error messages.
int ray_query(futhark_context *ctx, const futhark_opaque_prepared_scene *p, const float *rays, int64_t n, int32_t *index,
              float *t, float *pn, float *colour, bool shade, const char *what) {
  if (n < 0 || n > kMaxQueryRays) { set_error(ctx, "%s: bad ray count %lld (0 <= n <= 2^30)", what, (long long)n); return 1; }
  if (!p || !p->dev.nodes || !p->dev.perm) { set_error(ctx, "%s: invalid prepared scene", what); return 1; }
  if (!ctx->peers.empty()) { set_error(ctx, "%s: not available on a single-process multi-GPU context (RAY_GPUS > 1)", what); return 1; }
  if (n == 0) return 0;
  if (!rays || (shade ? !colour : (!index || !t))) { set_error(ctx, "%s: null output or ray pointer", what); return 1; }
  if (p->max_depth > kStackSize - 1) { set_error(ctx, "%s: BVH depth %d exceeds the traversal stack", what, p->max_depth); return 1; }
  CUDA_TRY(ctx, cudaSetDevice(ctx->cfg.device));

  RenderParams P;
  memset(&P, 0, sizeof P);
  P.nodes = p->dev.nodes; P.nodes_soa = p->dev.nodes_soa; P.geom = p->dev.geom; P.colour = p->dev.colour;
  P.n_inner = (int32_t)(p->n - 1); P.n_leaves = (int32_t)p->n;
  P.max_depth = p->max_depth;
  memcpy(P.root_box, p->root_box, sizeof P.root_box);
  memcpy(P.cam, &p->cam, sizeof P.cam);

  // Shared memory: the warp-queue kernel's K = 1 plan (32 warps, as many as leave 8 KB; the rest stages the BFS prefix of
  // the tree, then the spheres if they fit), with the same stage cap for trees far larger than the caches
  RayQueryLaunch lc;
  lc.sm_count = ctx->sm_count;
  lc.max_dynamic_smem = ctx->max_smem_optin;
  lc.ncap = wq_node_capacity(1, p->max_depth, ctx->cfg.wq_ncap);
  const int64_t per_warp = (int64_t)wq_warp_bytes(1, lc.ncap, false, false);
  int64_t warps = ctx->cfg.wq_warps < 1 ? 32 : std::min<int64_t>(ctx->cfg.wq_warps, kWqMaxWarps);
  while (warps > 1 && warps * per_warp + 8192 > (int64_t)ctx->max_smem_optin) warps--;
  int64_t budget = (int64_t)ctx->max_smem_optin - warps * per_warp - 512;
  if (budget < 256) { set_error(ctx, "%s: the ray-query kernel does not fit shared memory (tree depth %d)", what, p->max_depth); return 1; }
  {
    const bool huge = (int64_t)(p->n - 1) * 64 > ((int64_t)8 << 20);
    const int64_t queues = (int64_t)ctx->max_smem_optin - 512 - budget;
    const int64_t under_196k = std::max<int64_t>(1024, (int64_t)196 * 1024 - 2048 - queues);
    const int64_t cap = ctx->cfg.stage_cap >= 0 ? ctx->cfg.stage_cap : (huge ? under_196k : budget);
    budget = std::min<int64_t>(budget, std::max<int64_t>(cap, 256));
  }
  P.smem_nodes = (int32_t)std::min<int64_t>(P.n_inner, budget / 64);
  const int64_t left = budget - (int64_t)P.smem_nodes * 64;
  P.smem_spheres = (P.smem_nodes == P.n_inner && left >= (int64_t)P.n_leaves * 16) ? P.n_leaves : 0;
  lc.warps = (int)warps;
  const int nring = 1 << (31 - __builtin_clz((unsigned)lc.ncap));
  lc.nlow = ctx->cfg.wq_low < 0 ? 0 : (ctx->cfg.wq_low == 0 ? nring / 2 : std::min(ctx->cfg.wq_low, nring - 96));

  RayQueryParams Q;
  Q.rays = rays; Q.n = (int32_t)n; Q.perm = p->dev.perm;
  Q.index = index; Q.t = t; Q.pn = pn; Q.colour = colour;
  Q.cursor = ctx->lanes[0].work_cursor;   // lane 0 = the context's stream: ordered with that lane's frames
  CUDA_TRY(ctx, cudaMemsetAsync(Q.cursor, 0, sizeof(int32_t), ctx->stream));
  CUDA_TRY(ctx, launch_raycast(P, Q, lc, shade, ctx->stream, &ctx->launches));
  // the query reads the scene's device memory until here: release_scene_block frees / replaces it only after this
  if (!p->last_use[0]) CUDA_TRY(ctx, cudaEventCreateWithFlags(&p->last_use[0], cudaEventDisableTiming));
  CUDA_TRY(ctx, cudaEventRecord(p->last_use[0], ctx->stream));
  p->used[0] = true;
  return 0;
}

// Host-buffer variant: device copies of the rays and the outputs, the query, the copies back, one synchronisation.
int ray_query_host(futhark_context *ctx, const futhark_opaque_prepared_scene *p, const float *rays, int64_t n, int32_t *index,
                   float *t, float *pn, float *colour, bool shade, const char *what) {
  if (n <= 0 || n > kMaxQueryRays || !p || !p->dev.nodes || !p->dev.perm || !ctx->peers.empty() || !rays ||
      (shade ? !colour : (!index || !t)))
    return ray_query(ctx, p, rays, n, index, t, pn, colour, shade, what);  // its validation / n = 0 answer
  CUDA_TRY(ctx, cudaSetDevice(ctx->cfg.device));
  const size_t nn = (size_t)n;
  const size_t bytes = nn * 24 + (shade ? nn * 12 : nn * 8 + (pn ? nn * 24 : 0));
  unsigned char *blk = nullptr;
  CUDA_TRY(ctx, cudaMallocAsync(&blk, bytes, ctx->stream));
  float *d_rays = reinterpret_cast<float *>(blk);
  unsigned char *q = blk + nn * 24;
  float *d_colour = nullptr, *d_t = nullptr, *d_pn = nullptr;
  int32_t *d_index = nullptr;
  if (shade) d_colour = reinterpret_cast<float *>(q);
  else {
    d_t = reinterpret_cast<float *>(q);
    d_index = reinterpret_cast<int32_t *>(q + nn * 4);
    if (pn) d_pn = reinterpret_cast<float *>(q + nn * 8);
  }
  int rc = 0;
  if (cudaMemcpyAsync(d_rays, rays, nn * 24, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) { set_error(ctx, "%s: host-to-device copy failed", what); rc = 1; }
  if (!rc) rc = ray_query(ctx, p, d_rays, n, d_index, d_t, d_pn, d_colour, shade, what);
  if (!rc) {
    cudaError_t e;
    if (shade) e = cudaMemcpyAsync(colour, d_colour, nn * 12, cudaMemcpyDeviceToHost, ctx->stream);
    else {
      e = cudaMemcpyAsync(t, d_t, nn * 4, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaMemcpyAsync(index, d_index, nn * 4, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess && pn) e = cudaMemcpyAsync(pn, d_pn, nn * 24, cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (e != cudaSuccess) { set_error(ctx, "%s: device-to-host copy failed: %s", what, cudaGetErrorString(e)); rc = 1; }
  }
  cudaFreeAsync(blk, ctx->stream);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess && !rc) {
    set_error(ctx, "%s: kernel failed: %s", what, cudaGetErrorString(cudaGetLastError()));
    rc = 1;
  }
  return rc;
}

}  // namespace

extern "C" {

int ray_b200_intersect_into(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p, const float *rays_dev,
                            int64_t n, int32_t *index_dev, float *t_dev, float *pn_dev) {
  if (bad_ctx(ctx)) return 1;
  std::lock_guard<std::mutex> g(ctx->mu);
  return ray_query(ctx, p, rays_dev, n, index_dev, t_dev, pn_dev, nullptr, false, "intersect_into");
}

int ray_b200_trace_into(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p, const float *rays_dev,
                        int64_t n, float *colour_dev) {
  if (bad_ctx(ctx)) return 1;
  std::lock_guard<std::mutex> g(ctx->mu);
  return ray_query(ctx, p, rays_dev, n, nullptr, nullptr, nullptr, colour_dev, true, "trace_into");
}

int ray_b200_intersect_host(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p, const float *rays_host,
                            int64_t n, int32_t *index_host, float *t_host, float *pn_host) {
  if (bad_ctx(ctx)) return 1;
  std::lock_guard<std::mutex> g(ctx->mu);
  return ray_query_host(ctx, p, rays_host, n, index_host, t_host, pn_host, nullptr, false, "intersect_host");
}

int ray_b200_trace_host(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p, const float *rays_host,
                        int64_t n, float *colour_host) {
  if (bad_ctx(ctx)) return 1;
  std::lock_guard<std::mutex> g(ctx->mu);
  return ray_query_host(ctx, p, rays_host, n, nullptr, nullptr, nullptr, colour_host, true, "trace_host");
}

}  // extern "C"
