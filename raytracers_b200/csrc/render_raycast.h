// Ray queries on a prepared scene (include/ray_b200.h "ray queries"): the parameter block of the caller-supplied-ray kernel
// (render_raycast.cu) and its launcher, shared with the C ABI (api_rays.cu).
#pragma once
#include "render_params.h"

namespace rayb200 {

struct RayQueryParams {
  const float *rays;      // [n][6] {origin.xyz, direction.xyz} (device)
  int32_t n;              // rays, <= 2^30
  const int32_t *perm;    // Morton-sorted leaf -> the scene's sphere index (DeviceBvh::perm)
  int32_t *index;         // intersect: [n] sphere index or -1
  float *t;               // intersect: [n] hit.t or +inf
  float *pn;              // intersect, optional: [n][6] hit.p, hit.normal (0 on a miss)
  float *colour;          // trace: [n][3] ray_colour before quantisation
  int32_t *cursor;        // claim cursor (device, zeroed by the launcher)
};

struct RayQueryLaunch {
  int sm_count;
  int warps;              // per CTA (one CTA per SM)
  int ncap;               // node-queue entries per warp
  int nlow;               // node batches take the oldest items while at most this many are queued
  int max_dynamic_smem;
};

// `shade` = false: closest hit (objs_hit bvh r 0 1e9); true: ray_colour objs r 50.  P carries the prepared scene and its
// staging plan (smem_nodes / smem_spheres), as fill_params makes it for a frame.
cudaError_t launch_raycast(const RenderParams &P, const RayQueryParams &Q, const RayQueryLaunch &lc, bool shade,
                           cudaStream_t stream, int64_t *launches);

}  // namespace rayb200
