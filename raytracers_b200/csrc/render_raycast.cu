// sm_100a ray-query kernel of the product build: closest hit (objs_hit, ray.fut:76-86) and path colour (ray_colour,
// ray.fut:126-148) of caller-supplied rays on a prepared scene, plus its launcher.  C ABI: api_rays.cu.
//
// The same dense traversal as K3 (render_kernels.cu): one CTA per SM with the top of the tree (and the spheres when they
// fit) TMA-staged in shared memory, every warp keeps 32 rays in flight, and its lanes are bound to (ray, node) box-test and
// (ray, leaf) sphere-test ITEMS on a warp-private node ring and leaf stack, not to rays.  A sphere hit is folded into its
// ray's (t, leaf) pair with fold_hit ("smallest t, lowest Morton-sorted leaf on ties", the reference's strict `<` over
// leaves in ascending order), so the order in which the items run does not matter.  What differs from K3 is where rays
// come from and where they go: a slot takes a ray INDEX from a global cursor (32 per warp-aggregated claim, handed to the
// idle slots in order), reads the ray from the caller's array, and when its query is answered writes the result for that
// index.  There is no camera, no pixel, no sample and no claim-order table.
//
// The drain loop is a copy of K3's item-mode drain (ring + leaf stack, oldest-first below `nlow`), not a shared function:
// in K3 it is a lambda over the kernel's locals whose code shape the 32 instantiations' register allocation was tuned
// with, and hoisting it into render_common.cuh would have to leave every existing kernel's SASS unchanged.  The packet walk
// and the spread / pixel-bound sample machinery are not part of this kernel: caller rays have no known coherence.
#include "render_common.cuh"
#include "render_raycast.h"

namespace rayb200 {

namespace {

// kShade = false: one traversal round per ray, then the owner lane re-intersects the winner (ray.fut:83-85) and writes
// {index, t, p, normal}.  kShade = true: shade_segment after every round, the path bounces until it ends, then the colour
// is written.
template <bool kShade, bool kAllNodes, bool kSpheres>
__global__ void __launch_bounds__(kWqMaxThreads, 1) raycast_kernel(const __grid_constant__ RenderParams P,
                                                                   const __grid_constant__ RayQueryParams Q, const int ncap_arg,
                                                                   const int nlow) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const float4 *s_nodes, *s_geom;
  stage_scene(P, smem_raw, s_nodes, s_geom);
  const StagedScene<kAllNodes, kSpheres> sc{P.nodes, P.geom, s_nodes, s_geom, P.smem_nodes};

  constexpr int R = 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ncap = 1 << (31 - __clz(ncap_arg));
  const unsigned nmask = (unsigned)ncap - 1u;
  auto ring = [&](const int i) { return (int)((unsigned)i & nmask); };
  const unsigned lt_mask = (1u << lane) - 1u;
  const unsigned gt_mask = lane == 31 ? 0u : ~((2u << lane) - 1u);
  // per warp (inside the wq_warp_bytes(1, ncap, false, false) the launcher reserves)
  unsigned char *wbase = smem_raw + ((staging_bytes(P) + 127) & ~(size_t)127) + (size_t)warp * wq_warp_bytes(1, ncap_arg, false, false);
  float4 *ray_o = reinterpret_cast<float4 *>(wbase);   // {o.xyz, a = dot d d}
  float4 *ray_i = ray_o + R;                           // {1/d.xyz, 0}
  float4 *ray_d = ray_i + R;                           // {d.xyz, 0}
  float4 *p_light = ray_d + R;                         // {light.rgb, bits(depth)}   trace only
  uint32_t *best_t = reinterpret_cast<uint32_t *>(p_light + R);  // bits(t) of the closest accepted hit (kItemNoHit = none)
  uint32_t *best_l = best_t + R;                       // ... and its leaf (fold_hit)
  int *p_ray = reinterpret_cast<int *>(best_l + R);    // ray index of the slot, -1 = idle
  uint32_t *lstk = reinterpret_cast<uint32_t *>(p_ray + R);
  uint32_t *nstk = lstk + kWqLeafStack;

  const int n = Q.n;
  p_ray[lane] = -1;
  __syncwarp();
  bool exhausted = false;
  int claim_next = 0, claim_end = 0;  // warp-uniform: claimed ray indices not handed out yet
  int ntop = 0, nhead = 0, ltop = 0;  // warp-uniform: node ring [nhead, ntop), leaf stack height

  // The query of `slot`'s ray is answered (intersect: the fold result j / tb; trace: the path's colour).
  auto finish_intersect = [&](const int slot, const Ray &r, const float a, const int j, const float tb) {
    const int id = p_ray[slot];
    int index = -1;
    float t = __int_as_float(0x7f800000);
    V3 p = v3(0.0f, 0.0f, 0.0f), nrm = v3(0.0f, 0.0f, 0.0f);
    if (j >= 0) {
      // objs_hit, second half (ray.fut:83-85): re-intersect the winner with t_min = 0, t_max = t_best + 1
      const float4 g = sc.sphere(j);
      const float th = sphere_t(g.x, g.y, g.z, g.w, r, a, 0.0f, tb + 1.0f);
      if (th >= 0.0f) {
        index = __ldg(Q.perm + j);
        t = th;
        p = vadd(r.o, vscale(th, r.d));                         // point_at_param, ray.fut:14-15
        nrm = vscale(1.0f / g.w, vsub(p, v3(g.x, g.y, g.z)));   // ray.fut:42-43
      }
    }
    Q.index[id] = index;
    Q.t[id] = t;
    if (Q.pn) {
      float *q = Q.pn + 6 * (size_t)id;
      q[0] = p.x; q[1] = p.y; q[2] = p.z; q[3] = nrm.x; q[4] = nrm.y; q[5] = nrm.z;
    }
    p_ray[slot] = -1;
  };
  auto finish_trace = [&](const int slot, const V3 colour) {
    float *q = Q.colour + 3 * (size_t)p_ray[slot];
    q[0] = colour.x; q[1] = colour.y; q[2] = colour.z;
    p_ray[slot] = -1;
  };

  for (;;) {
    bool go = false;  // this lane's slot traverses this round
    for (int pass = 0; pass < 4; pass++) {
      // ---------------------------------------------------------------- hand ray indices to idle slots
      const bool idle = p_ray[lane] < 0;
      const unsigned im = __ballot_sync(kFullMask, idle);
      if (im && !exhausted) {
        int rank = __popc(im & lt_mask), given = 0;
        const int want = __popc(im);
        while (given < want) {
          if (claim_next == claim_end) {  // claim the next 32 indices for this warp
            int base = 0;
            if (lane == 0) base = atomicAdd(Q.cursor, 32);
            base = __shfl_sync(kFullMask, base, 0);
            if (base >= n) { exhausted = true; break; }
            claim_next = base;
            claim_end = base + 32 < n ? base + 32 : n;
          }
          const int take = min(want - given, claim_end - claim_next);
          if (idle && rank >= given && rank < given + take) {
            const int id = claim_next + (rank - given);
            const float *src = Q.rays + 6 * (size_t)id;
            p_ray[lane] = id;
            ray_o[lane] = make_float4(__ldg(src), __ldg(src + 1), __ldg(src + 2), 0.0f);
            ray_d[lane] = make_float4(__ldg(src + 3), __ldg(src + 4), __ldg(src + 5), 0.0f);
            if (kShade) p_light[lane] = make_float4(1.0f, 1.0f, 1.0f, __int_as_float(0));
          }
          given += take;
          claim_next += take;
        }
      }
      // -------------------------------------------------------------- set up this round's traversals
      // Root box test by the owner lane; a root miss is answered on the spot (no hit / sky), so it never occupies a round.
      if (!go) {
        while (p_ray[lane] >= 0) {
          const float4 ro = ray_o[lane], rd = ray_d[lane];
          Ray r;
          r.o = v3(ro.x, ro.y, ro.z);
          r.d = v3(rd.x, rd.y, rd.z);
          const RayInv q = ray_invariants(r);
          if (box_hit(P.root_box[0], P.root_box[1], P.root_box[2], P.root_box[3], P.root_box[4], P.root_box[5], r, q)) {
            ray_o[lane] = make_float4(ro.x, ro.y, ro.z, q.a);
            ray_i[lane] = make_float4(q.ix, q.iy, q.iz, 0.0f);
            best_t[lane] = kItemNoHit;
            go = true;
            break;
          }
          if (kShade) {
            const float4 pl = p_light[lane];  // miss (ray.fut:141-148)
            V3 light = v3(pl.x, pl.y, pl.z), colour;
            int depth = __float_as_int(pl.w);
            shade_segment(sc, P, r, q.a, -1, 0.0f, light, depth, colour);
            finish_trace(lane, colour);
          } else {
            finish_intersect(lane, r, q.a, -1, 0.0f);
          }
        }
      }
      // another pass only helps if some slot is idle and there are rays left to hand out
      if (exhausted || !__any_sync(kFullMask, p_ray[lane] < 0)) break;
    }
    __syncwarp();
    const unsigned gm = __ballot_sync(kFullMask, go);
    if (gm == 0u) {
      if (exhausted && !__any_sync(kFullMask, p_ray[lane] >= 0)) break;  // no rays left for this warp
      continue;
    }

    // ---------------------------------------------------------------- dense traversal of the round (K3's item mode)
    auto leaf_batch = [&](const int nb) {
      // closest_hit (ray.fut:78-81) for up to 32 (ray, sphere) pairs
      bool hit = false;
      uint32_t tb = 0;
      int slot = 0, li = 0;
      if (lane < nb) {
        const uint32_t it = lstk[ltop - 1 - lane];
        slot = (int)(it >> kSlotShift);
        li = (int)(it & kIndexMask);
        const float4 ro = ray_o[slot], rd = ray_d[slot];
        const float4 g = sc.sphere(li);
        Ray r;
        r.o = v3(ro.x, ro.y, ro.z);
        r.d = v3(rd.x, rd.y, rd.z);
        const float t = sphere_t(g.x, g.y, g.z, g.w, r, ro.w, 0.1f, 1000000000.0f);
        hit = t >= 0.0f;
        tb = __float_as_uint(t);
      }
      ltop -= nb;
      fold_hit(best_t, best_l, slot, hit, tb, (uint32_t)li);
    };
    auto node_batch = [&](const bool bottom, const int nb) {
      // one BVH2C node step (both children's boxes) for up to 32 (ray, node) pairs, from the top of the ring (newest =
      // deepest first) or, `bottom` (warp-uniform), from its bottom (oldest = shallowest first)
      bool pl_node = false, pr_node = false, pl_leaf = false, pr_leaf = false;
      uint32_t tag = 0;
      int lptr = 0, rptr = 0;
      if (lane < nb) {
        const uint32_t it = nstk[ring(bottom ? nhead + lane : ntop + ~lane)];
        tag = it & ~kIndexMask;
        const int slot = (int)(it >> kSlotShift), cur = (int)(it & kIndexMask);
        const float4 ro = ray_o[slot], ri = ray_i[slot];
        float4 q0, q1, q2, q3;
        sc.node(cur, q0, q1, q2, q3);
        Ray r;
        r.o = v3(ro.x, ro.y, ro.z);
        r.d = v3(0.0f, 0.0f, 0.0f);
        RayInv q;
        q.ix = ri.x; q.iy = ri.y; q.iz = ri.z; q.a = ro.w;
        lptr = __float_as_int(q0.w);
        rptr = __float_as_int(q1.w);
        const bool hl = box_hit(q0.x, q0.y, q0.z, q1.x, q1.y, q1.z, r, q);
        const bool hr = box_hit(q2.x, q2.y, q2.z, q3.x, q3.y, q3.z, r, q);
        pl_leaf = lptr < 0;  // a leaf child has no box in the reference (bvh.fut:84): always visited
        pr_leaf = rptr < 0;
        pl_node = hl && !pl_leaf;
        pr_node = hr && !pr_leaf;
      }
      __syncwarp();  // every pop has been read before anything is pushed over it
      if (bottom) nhead += nb; else ntop -= nb;
      const unsigned bl = __ballot_sync(kFullMask, pl_node), br = __ballot_sync(kFullMask, pr_node);
      const int nbase = ntop + __popc(bl & gt_mask) + __popc(br & gt_mask);  // reverse lane order: deepest back on top
      if (pr_node) nstk[ring(nbase)] = tag | (uint32_t)rptr;
      if (pl_node) nstk[ring(nbase + (pr_node ? 1 : 0))] = tag | (uint32_t)lptr;
      ntop += __popc(bl) + __popc(br);
      if (__any_sync(kFullMask, pl_leaf || pr_leaf)) {
        const unsigned cl = __ballot_sync(kFullMask, pl_leaf), cr = __ballot_sync(kFullMask, pr_leaf);
        const int lb = ltop + __popc(cl & lt_mask) + __popc(cr & lt_mask);
        if (pl_leaf) lstk[lb] = tag | (uint32_t)(~lptr);
        if (pr_leaf) lstk[lb + (pl_leaf ? 1 : 0)] = tag | (uint32_t)(~rptr);
        ltop += __popc(cl) + __popc(cr);
      }
    };
    // roots of this round's rays
    if (go) nstk[__popc(gm & lt_mask)] = (uint32_t)lane << kSlotShift;  // (slot, root node 0)
    ntop = __popc(gm);
    nhead = 0;
    // Drain (K3's): full batches, oldest-first while at most nlow node items are queued, newest-first above; once fewer than
    // 96 ring entries are free, one item at a time from the top (a plain DFS adds < 64 before it shrinks).
    {
      __syncwarp();
      const int nroom = ncap - 96;
      for (;;) {
        while ((unsigned)(ntop - nhead - 32) <= (unsigned)(nroom - 32) && ltop < 32) {
          node_batch(ntop - nhead <= nlow, 32);
          __syncwarp();
        }
        const int cnt = ntop - nhead;
        if (ltop >= 32) leaf_batch(32);
        else if (cnt > 0) node_batch(false, cnt > nroom ? 1 : (cnt < 32 ? cnt : 32));
        else if (ltop > 0) leaf_batch(ltop);
        else break;
        __syncwarp();
      }
      ntop = nhead = 0;
    }

    // ---------------------------------------------------------------- owner lanes answer or bounce
    if (go) {
      const float4 ro = ray_o[lane], rd = ray_d[lane];
      const uint32_t bt = best_t[lane];
      Ray r;
      r.o = v3(ro.x, ro.y, ro.z);
      r.d = v3(rd.x, rd.y, rd.z);
      const int j = bt == kItemNoHit ? -1 : (int)best_l[lane];
      const float tb = __uint_as_float(bt);
      if (kShade) {
        const float4 pl = p_light[lane];
        V3 light = v3(pl.x, pl.y, pl.z), colour;
        int depth = __float_as_int(pl.w);
        if (shade_segment(sc, P, r, ro.w, j, tb, light, depth, colour)) {
          ray_o[lane] = make_float4(r.o.x, r.o.y, r.o.z, 0.0f);
          ray_d[lane] = make_float4(r.d.x, r.d.y, r.d.z, 0.0f);
          p_light[lane] = make_float4(light.x, light.y, light.z, __int_as_float(depth));
        } else {
          finish_trace(lane, colour);
        }
      } else {
        finish_intersect(lane, r, ro.w, j, tb);
      }
    }
    __syncwarp();
  }
}

}  // namespace

cudaError_t launch_raycast(const RenderParams &P, const RayQueryParams &Q, const RayQueryLaunch &lc, bool shade,
                           cudaStream_t stream, int64_t *launches) {
  if (Q.n <= 0) return cudaSuccess;
  const bool all_nodes = P.smem_nodes == P.n_inner, sph = P.smem_spheres == P.n_leaves && P.smem_spheres > 0;
  const size_t smem = ((staging_bytes(P) + 127) & ~(size_t)127) + (size_t)lc.warps * wq_warp_bytes(1, lc.ncap, false, false);
  // no more CTAs than 32-ray groups
  long long ctas = lc.sm_count;
  const long long groups = ((long long)Q.n + 32ll * lc.warps - 1) / (32ll * lc.warps);
  if (ctas > groups) ctas = groups;
  cudaError_t e = cudaSuccess;
#define RAYB200_RQ(SH, A, S)                                                                                          \
  do {                                                                                                                \
    e = opt_in_dynamic_smem<raycast_kernel<SH, A, S>>(lc.max_dynamic_smem);                                           \
    if (e == cudaSuccess) raycast_kernel<SH, A, S><<<(unsigned)ctas, 32 * lc.warps, smem, stream>>>(P, Q, lc.ncap, lc.nlow); \
  } while (0)
#define RAYB200_RQ2(SH)                                       \
  do {                                                        \
    if (all_nodes && sph) RAYB200_RQ(SH, true, true);         \
    else if (all_nodes) RAYB200_RQ(SH, true, false);          \
    else if (sph) RAYB200_RQ(SH, false, true);                \
    else RAYB200_RQ(SH, false, false);                        \
  } while (0)
  if (shade) RAYB200_RQ2(true); else RAYB200_RQ2(false);
#undef RAYB200_RQ2
#undef RAYB200_RQ
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e == cudaSuccess) (*launches)++;
  return e;
}

}  // namespace rayb200
