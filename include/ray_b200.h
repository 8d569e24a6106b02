/*
 * ray_b200.h — extensions next to the Futhark-compatible ABI of ray.h.
 *
 * The reference has no samples-per-pixel, no custom scenes, no float framebuffer and no multi-GPU
 * (ray.fut:150-154, 171-174, 246-247); BASELINE.json's configs need all four.  Because
 * futhark/main.c must stay unmodified, every extension is reachable two ways:
 *   - environment variables read by futhark_context_new (RAY_SPP, RAY_KERNEL, RAY_RANK, RAY_WORLD,
 *     RAY_DEVICE), so the unmodified driver can use them, and
 *   - the explicit C entry points below (plain pointers and sizes; device pointers are raw
 *     CUDA device addresses, e.g. torch.Tensor.data_ptr()).
 *
 * Multi-GPU.  Two ways: (a) one process per GPU (torchrun): ray_b200_context_set_shard + ray_b200_render_shard_into, an
 * NCCL gather by the host, ray_b200_detile — see raytracers_b200/distributed.py; (b) ONE process, several devices:
 * RAY_GPUS=N (or tuning parameter "gpus") makes the context drive devices d..d+N-1; futhark_entry_prepare_scene replicates
 * the scene, futhark_entry_render renders interleaved tiles on every device and pulls the shards to device d with peer
 * copies over NVLink.  This is the mode an unmodified futhark/main.c uses.  In mode (b) the raw-pointer entry points
 * (ray_b200_render_into, ray_b200_render_shard_into) keep addressing device d's shard only.
 *
 * spp semantics (SURVEY.md §8d): sample s of pixel (row j, column i) uses
 *   u = (f32(i) + ox_s) / f32(W),  v = (f32(H - j) + oy_s) / f32(H),
 *   ox_s = frac(f32(s) * 0.7548776662f), oy_s = frac(f32(s) * 0.5698402909f)   [ox_0 = oy_0 = 0]
 * colours are summed in sample order in f32, multiplied by 1/spp, then quantised as ray.fut:158-162.
 * At spp = 1 this is bit-identical to the reference's render.
 */
#ifndef RAY_B200_EXT_H
#define RAY_B200_EXT_H

#include "ray.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Render kernels (tuning param "kernel" / env RAY_KERNEL). */
enum ray_b200_kernel {
  RAY_B200_KERNEL_AUTO = 0,       /* the fastest measured variant (see resolve_kernel in api.cu) */
  RAY_B200_KERNEL_MEGA = 1,       /* one thread per pixel, whole ray_colour loop (parity anchor) */
  RAY_B200_KERNEL_PERSISTENT = 2, /* persistent CTAs, TMA-staged BVH, per-lane dynamic path refill */
  RAY_B200_KERNEL_WAVEFRONT = 3,  /* per-bounce persistent kernel + global ray queues + warp-vote compaction */
  RAY_B200_KERNEL_WARPQUEUE = 4,  /* persistent; lanes bound to (ray,node) items on warp-private smem queues */
  RAY_B200_KERNEL_STREAMQUEUE = 5,/* the same without rounds: per-ray item counters, finished rays refilled continuously */
  RAY_B200_KERNEL_LANEWALK = 6    /* persistent; a lane owns a ray's whole traversal (private smem stack), paths live in
                                     warp-shared slots, finished segments are shaded in dense batches, no rounds */
};

/* ---- context extensions ---------------------------------------------------------------------- */
/* Launch all work of this context on `cuda_stream` (a cudaStream_t / CUstream, e.g.
 * torch.cuda.Stream.cuda_stream).  NULL restores the context's own stream; pass cudaStreamLegacy
 * ((cudaStream_t)0x1) for the legacy default stream (whose raw handle is 0). */
int ray_b200_context_set_stream(struct futhark_context *ctx, void *cuda_stream);
/* Samples per pixel used by futhark_entry_render (default 1 = the reference). */
int ray_b200_context_set_spp(struct futhark_context *ctx, int32_t spp);
int ray_b200_context_set_kernel(struct futhark_context *ctx, int32_t kernel);
/* This process renders tiles t with t % world == rank (8x4-pixel tiles, row-major tile order). */
int ray_b200_context_set_shard(struct futhark_context *ctx, int32_t rank, int32_t world);
int ray_b200_context_device(struct futhark_context *ctx);
/* Device time in ms of the last render (CUDA events on the context's stream; syncs). */
int ray_b200_context_last_render_ms(struct futhark_context *ctx, float *ms);
/* Number of kernel launches issued by this context since creation. */
int64_t ray_b200_context_launch_count(struct futhark_context *ctx);
/* Diagnostic: while enabled, every warp of the warp-queue kernel records when it ran out of work.
 * ray_b200_context_warp_trace returns, for the last traced render, each warp's exit time in microseconds after
 * the first CTA started (exit_us may be NULL to query *count = SMs x warps per CTA).  Syncs the stream. */
int ray_b200_context_trace_warps(struct futhark_context *ctx, int32_t enable);
int ray_b200_context_warp_trace(struct futhark_context *ctx, float *exit_us, int64_t capacity, int64_t *count);

/* ---- scenes ------------------------------------------------------------------------------------ */
/* spheres: n x 7 floats (pos.xyz, colour.xyz, radius) — the `sphere` record of ray.fut:22-24;
 * cam7: look_from.xyz, look_at.xyz, fov — the rest of `scene`, ray.fut:171-174.  n >= 2 (bvh.fut:65). */
int ray_b200_scene_from_arrays(struct futhark_context *ctx, struct futhark_opaque_scene **out0,
                               const float *spheres, int64_t n, const float *cam7);
/* SURVEY.md §8d config 5: splitmix64(seed) stream, 7 draws per sphere, camera (0,0,1100)->(0,0,0). */
int ray_b200_scene_random(struct futhark_context *ctx, struct futhark_opaque_scene **out0, int64_t n,
                          uint64_t seed);
int64_t ray_b200_scene_num_spheres(struct futhark_context *ctx, const struct futhark_opaque_scene *s);
int ray_b200_scene_get_arrays(struct futhark_context *ctx, const struct futhark_opaque_scene *s, float *spheres,
                              float *cam7);

/* ---- prepared scene introspection (tests compare these with the oracle's LBVH) ----------------- */
struct ray_b200_bvh_info {
  int64_t n_leaves, n_inner;
  int32_t max_depth, refit_sweeps, stale_nodes, smem_nodes;
  float root_box[6];
  float camera[12]; /* origin, llc, horizontal, vertical (ray.fut:88-91) */
};
int ray_b200_prepared_info(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                           struct ray_b200_bvh_info *info);
/* Karras-order dump: morton[n], perm[n], left/right/parent[n-1] (leaf i = ~i), boxes[(n-1)*6]. NULLs skipped. */
int ray_b200_prepared_dump(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                           uint32_t *morton, int32_t *perm, int32_t *left, int32_t *right, int32_t *parent,
                           float *boxes);

/* The packed BVH2C arrays as they sit in HBM (tests compare device-built and host-built scenes):
 * nodes / nodes_soa: (n-1) x 16 floats, geom / colour: n x 4 floats.  NULLs skipped.  Synchronous. */
int ray_b200_prepared_packed(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p, float *nodes,
                             float *nodes_soa, float *geom, float *colour);
/* Bytes prepare_scene copies host -> device: the sphere records (LBVH build and packing run on the device);
 * with tuning "host_build" / RAY_HOST_BUILD=1 the host-built arrays instead. */
int64_t ray_b200_prepared_upload_bytes(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p);
/* Bytes of the prepared scene resident in HBM (packed BVH2C + the Karras-order LBVH kept for introspection). */
int64_t ray_b200_prepared_device_bytes(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p);
/* Runs prepare_scene's device work again for an existing handle: H2D of the sphere records from page-locked
 * memory + LBVH build on the device (the H2D leg of bench.py's end-to-end step). */
int ray_b200_prepared_reupload(struct futhark_context *ctx, struct futhark_opaque_prepared_scene *p);

/* ---- render extensions -------------------------------------------------------------------------- */
/* render with explicit spp; optional float framebuffer.  out_pix_dev: device int32[h][w] (REQUIRED);
 * out_rgb_dev: device float[h][w][3] (or NULL).  Asynchronous on the context's stream.
 * With a shard set (world > 1) only this rank's pixels are written.  On a single-process multi-GPU context
 * (RAY_GPUS > 1) this call, ray_b200_render_shard_into and ray_b200_render_batch return an error: only
 * futhark_entry_render / ray_b200_entry_render_spp gather the helper devices' tiles. */
int ray_b200_render_into(struct futhark_context *ctx, int32_t *out_pix_dev, float *out_rgb_dev, int64_t h,
                         int64_t w, int32_t spp, const struct futhark_opaque_prepared_scene *p);
/* Same, host buffers: H2D of nothing (the scene is resident), D2H of the frame, synchronous.
 * This is the call bench.py's e2e leg times. */
int ray_b200_render_host(struct futhark_context *ctx, int32_t *out_pix_host, float *out_rgb_host, int64_t h,
                         int64_t w, int32_t spp, const struct futhark_opaque_prepared_scene *p);
/* Like futhark_entry_render but with explicit spp (library-owned result). */
int ray_b200_entry_render_spp(struct futhark_context *ctx, struct futhark_i32_2d **out0, int64_t h, int64_t w,
                              int32_t spp, const struct futhark_opaque_prepared_scene *p);

/* ---- multi-GPU tile sharding (one process per GPU; the gather itself is NCCL, done by the host) -- */
/* Number of 8x4 tiles rank `rank` of `world` owns for an h x w image, and the padded per-rank count
 * (equal on all ranks, so a plain all_gather / gather works). */
int64_t ray_b200_shard_tiles(int64_t h, int64_t w, int32_t rank, int32_t world);
int64_t ray_b200_shard_tiles_padded(int64_t h, int64_t w, int32_t world);
/* Renders this rank's tiles into a compact tile-major device buffer int32[tiles_padded][32]. */
int ray_b200_render_shard_into(struct futhark_context *ctx, int32_t *out_tiles_dev, int64_t h, int64_t w,
                               int32_t spp, const struct futhark_opaque_prepared_scene *p);
/* Several frames in one call, up to two of them in flight on the device, so that the long-path tail of one frame
 * is covered by the start of the next (the frames are independent: different prepared scenes, sizes or outputs).
 * For the caller the batch is ONE operation on the context's stream: it starts after earlier work on that stream, and
 * later work on that stream starts after every job has finished.  Jobs are launched in array order (put the frame
 * with the longest tail first).  ray_b200_context_last_render_ms then reports the whole batch. */
struct ray_b200_render_job {
  const struct futhark_opaque_prepared_scene *prepared;
  int64_t h, w;
  int32_t spp;          /* 0 = the context's default */
  int32_t shard_layout; /* 0: out_dev = int32[h][w], row-major (ray_b200_render_into);
                           1: out_dev = this rank's compact tiles int32[tiles_padded][32] (ray_b200_render_shard_into) */
  int32_t *out_dev;     /* device (may be a PEER device's memory mapped with ray_b200_ipc_open: row-major layout + a
                           shard set = every rank writes its own pixels straight into rank 0's frame over NVLink) */
  float *out_rgb_dev;   /* device float[h][w][3] or NULL (row-major layout only) */
  /* peer-frame protocol (all optional, NULL = off), see "peer-memory frames" below:
   * before the frame's kernel starts, its stream waits until *wait_flag >= wait_value (back-pressure from the consumer);
   * when the last warp of the frame's kernel has written its pixels, *done_flag is incremented by 1 (system scope). */
  uint32_t *wait_flag;
  uint32_t wait_value;
  uint32_t reserved0;
  uint32_t *done_flag;
};
int ray_b200_render_batch(struct futhark_context *ctx, const struct ray_b200_render_job *jobs, int32_t n);
/* Pipelined submission (off by default).  With it on, ray_b200_render_batch does NOT join its second lane back into the
 * context's stream: consecutive frames alternate between the two lanes ACROSS calls, each lane ordered only after its own
 * previous frame (and after earlier work on the context's stream, e.g. a scene re-upload), so frame k+1 starts on every
 * SM whose CTA of frame k has retired - a frame's last 50-bounce paths no longer idle the GPU at the end of every
 * batch.  The caller orders its reads itself (done_flag / ray_b200_flag_wait, or ray_b200_pipeline_join, or
 * futhark_context_sync, which waits for both lanes).  Prepared scenes may be freed or re-uploaded while frames that use
 * them are in flight: their device memory is reclaimed only after the last such frame (stream-ordered, on a third stream). */
int ray_b200_context_set_pipeline(struct futhark_context *ctx, int32_t on);
/* Makes the context's stream wait for every frame enqueued so far on either lane (no host synchronisation). */
int ray_b200_pipeline_join(struct futhark_context *ctx);
/* sizeof(struct ray_b200_render_job) as the library was compiled: lets a foreign-language binding check its layout. */
int64_t ray_b200_render_job_size(void);
/* gathered_dev: int32[world][tiles_padded][32] (rank-major, as produced by an NCCL gather);
 * writes the row-major image int32[h][w] to out_pix_dev. */
int ray_b200_detile(struct futhark_context *ctx, const int32_t *gathered_dev, int32_t *out_pix_dev, int64_t h,
                    int64_t w, int32_t world);

/* ---- peer-memory frames: the gather fused into the render kernel ----------------------------------------
 * One process per GPU.  Rank 0 allocates a ring of frames with ray_b200_ipc_alloc and hands the 64-byte handle to the
 * other ranks (any transport: torch.distributed object broadcast in raytracers_b200/distributed.py); they map it with
 * ray_b200_ipc_open and pass the mapped address as `out_dev` of a row-major render with their shard set.  The render
 * kernel's pixel stores then ARE the collective: they travel over NVLink into rank 0's frame, no tile buffer, no
 * ncclGather, no de-tiling kernel.  Completion and back-pressure are two 32-bit flags per frame slot in the same
 * allocation (done_flag / wait_flag of ray_b200_render_job); the consumer side enqueues ray_b200_flag_wait on its copy
 * stream, copies the frame out and publishes the slot again with ray_b200_flag_set. */
#define RAY_B200_IPC_HANDLE_BYTES 64
int ray_b200_ipc_alloc(struct futhark_context *ctx, int64_t bytes, void **dev_ptr, unsigned char *handle64);
int ray_b200_ipc_free(struct futhark_context *ctx, void *dev_ptr);
int ray_b200_ipc_open(struct futhark_context *ctx, const unsigned char *handle64, void **dev_ptr);
int ray_b200_ipc_close(struct futhark_context *ctx, void *dev_ptr);
/* Enqueue on `stream` (a cudaStream_t; NULL = the context's stream): spin until *flag >= value (system-scope acquire;
 * gives up after timeout_ms and records an error that the next ray_b200_flag_status call returns). */
int ray_b200_flag_wait(struct futhark_context *ctx, void *stream, uint32_t *flag_dev, uint32_t value, int32_t timeout_ms);
/* Enqueue on `stream`: *flag = value (system-scope release). */
int ray_b200_flag_set(struct futhark_context *ctx, void *stream, uint32_t *flag_dev, uint32_t value);
/* Number of flag waits that timed out since the context was created (0 = healthy). */
int ray_b200_flag_status(struct futhark_context *ctx, int64_t *timeouts);
/* Enqueue on `stream`: device -> host copy (host_dst should be page-locked for the copy to be asynchronous). */
int ray_b200_copy_to_host_async(struct futhark_context *ctx, void *stream, void *host_dst, const void *dev_src, int64_t bytes);

/* ---- ray queries: closest hit and path colour of caller-supplied rays ----------------------------------
 * A ray is 6 floats {origin.xyz, direction.xyz} (the layout of oracle_aabb_hit's ray6); the direction need not be
 * normalised, just as get_ray's is not (ray.fut:109-114).  Output i always belongs to ray i.  0 <= n <= 2^30.
 *
 * intersect = objs_hit bvh r 0.0 1e9 (ray.fut:76-86) exactly as render uses it: boxes are tested against the original
 *   interval, the closest-hit search uses t_min = 0.1 with strict `<`, ties go to the lowest Morton-sorted leaf, and the
 *   winner is re-intersected with (0, t_best + 1); if that re-intersection fails the ray has no hit.  Per ray:
 *     index[i]  int32: the hit sphere's index in the SCENE's order (the order ray_b200_scene_get_arrays returns), -1 = none
 *     t[i]      float: hit.t of the re-intersection, +inf = none
 *     pn[i*6]   float[6] (optional, NULL = not written): hit.p, hit.normal as sphere_hit computes them, 0 = none
 * trace = ray_colour objs r 50 (ray.fut:126-148).  Per ray: colour[i*3] float[3], before quantisation.
 * There are no per-ray t intervals, no depth argument and no any-hit mode: the reference defines none of them.
 *
 * The _into variants take device pointers and are asynchronous on the context's stream; the _host variants take host
 * buffers and return when the results are there.  Bad arguments (n out of range, a NULL ray or required output pointer,
 * an invalid prepared scene) return an error and launch nothing; n = 0 returns 0 and launches nothing.  A shard set with
 * ray_b200_context_set_shard does not apply: every ray is answered.  On a single-process multi-GPU context
 * (RAY_GPUS > 1) these calls return an error.  The prepared scene may be freed right after an asynchronous query: its
 * device memory is released behind the query in stream order. */
int ray_b200_intersect_into(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                            const float *rays_dev, int64_t n, int32_t *index_dev, float *t_dev, float *pn_dev);
int ray_b200_trace_into(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                        const float *rays_dev, int64_t n, float *colour_dev);
int ray_b200_intersect_host(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                            const float *rays_host, int64_t n, int32_t *index_host, float *t_host, float *pn_host);
int ray_b200_trace_host(struct futhark_context *ctx, const struct futhark_opaque_prepared_scene *p,
                        const float *rays_host, int64_t n, float *colour_host);

/* ---- work counters (roofline numerators) ---------------------------------------------------------- */
struct ray_b200_counters { uint64_t segments, node_steps, box_tests, leaf_tests; };
/* Re-renders (1 spp) with counting kernels and returns the work the GPU traversal did. */
int ray_b200_count_work(struct futhark_context *ctx, int64_t h, int64_t w, int32_t spp,
                        const struct futhark_opaque_prepared_scene *p, struct ray_b200_counters *out);

/* ---- host-only entry points (no context, no device needed): the setup path's host logic ------------ */
/* name: "rgbbox" | "irreg" | "random" (n, seed used by "random" only).  spheres may be NULL to query *count. */
int ray_b200_host_scene(const char *name, int64_t n, uint64_t seed, float *spheres, int64_t capacity, float *cam7,
                        int64_t *count);
/* camera look_from look_at (0,1,0) fov (w/h)  (ray.fut:93-107, 243-244) -> origin, llc, horizontal, vertical */
int ray_b200_host_camera(const float *cam7, int64_t h, int64_t w, float *out12);
/* bvh_mk (bvh.fut:30-59) in Karras order; info4 = {refit_sweeps, max_depth, stale_nodes, 0}. 2 = n < 2. */
int ray_b200_host_lbvh(const float *spheres, int64_t n, uint32_t *morton, int32_t *perm, int32_t *left,
                       int32_t *right, int32_t *parent, float *boxes, int32_t *info4);
void ray_b200_host_sample_offsets(int32_t spp, float *table);

const char *ray_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RAY_B200_EXT_H */
