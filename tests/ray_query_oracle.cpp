// TEST INFRASTRUCTURE, NOT PRODUCT CODE: the CPU oracle's answers to the ray queries of include/ray_b200.h.
//
// Compiles oracle/oracle.cpp into the same translation unit (unchanged) and adds two thin, multithreaded loops over its
// objs_hit (ray.fut:76-86) and ray_colour (ray.fut:126-148) for caller-supplied rays.  Loaded by tests/ray_query_oracle.py
// only; built with the oracle's own flags (g++ -O2 -ffp-contract=off -fno-fast-math, no -march).
//
// The sphere index of a hit is the one thing objs_hit does not return: `winning_leaf` restates bvh_fold's closest_hit fold
// (bvh.fut:61-84, ray.fut:78-81) to name the leaf, and oracle_intersect_rays checks that re-intersecting that leaf gives
// bit for bit the hit objs_hit returned (return code 2 otherwise), so the restatement cannot drift from the oracle.
#include "../oracle/oracle.cpp"

namespace {

// bvh_fold with closest_hit (-1, 1e9) (bvh.fut:61-84, ray.fut:77-81): the Morton-sorted leaf objs_hit re-intersects
// (or -1) and its closest-hit t.
int32_t winning_leaf(const Bvh &bvh, const Ray &r, float *t_best) {
  int32_t acc_j = -1;
  float acc_t = 1000000000.0f;
  int32_t cur = 0;
  Ptr prev = inner_ptr(-1);
  while (cur != -1) {
    const Inner &node = bvh.I[cur];
    const bool from_left = ptr_eq(prev, node.left), from_right = ptr_eq(prev, node.right);
    bool rec = false;
    Ptr child = {0, 0};
    if (from_left) { rec = true; child = node.right; }
    else if (!from_right && aabb_hit(node.aabb, r, 0.000f, 1000000000.0f)) { rec = true; child = node.left; }
    if (!rec) { prev = inner_ptr(cur); cur = node.parent; }
    else if (child.tag == 1) { prev = inner_ptr(cur); cur = child.idx; }
    else {
      Hit h;
      if (sphere_hit(bvh.L[child.idx], r, scene_epsilon, acc_t, &h)) { acc_j = child.idx; acc_t = h.t; }
      prev = child;
    }
  }
  *t_best = acc_t;
  return acc_j;
}

inline bool same_bits(float a, float b) { return memcmp(&a, &b, sizeof a) == 0; }

// body(k) for k in [0, n) on `threads` threads (<= 0: all cores), blocks of 256 rays.
template <class F>
void for_rays(int64_t n, int32_t threads, F body) {
  int nthreads = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
  if (nthreads < 1) nthreads = 1;
  const int64_t block = 256, nblocks = (n + block - 1) / block;
  std::atomic<int64_t> next{0};
  auto worker = [&]() {
    for (int64_t b; (b = next.fetch_add(1)) < nblocks;)
      for (int64_t k = b * block; k < std::min(n, (b + 1) * block); k++) body(k);
  };
  if (nthreads == 1) worker();
  else {
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; t++) pool.emplace_back(worker);
    for (auto &t : pool) t.join();
  }
}

}  // namespace

extern "C" {

// rays[n][6] = origin.xyz, direction.xyz.  objs_hit bvh r 0.0 1e9 per ray: index[k] = the hit sphere's index in the
// scene's order (perm of the winning leaf) or -1, t[k] = hit.t or +inf, pn[k][6] (may be NULL) = hit.p, hit.normal or 0.
int oracle_intersect_rays(void *pv, const float *rays, int64_t n, int32_t *index, float *t, float *pn, int32_t threads) {
  Prepared *p = (Prepared *)pv;
  if (!p || n < 0 || (n > 0 && (!rays || !index || !t))) return 1;
  const Bvh &objs = p->objs;
  std::atomic<int> inconsistent{0};
  for_rays(n, threads, [&](int64_t k) {
    const float *q = rays + 6 * k;
    const Ray r = {{q[0], q[1], q[2]}, {q[3], q[4], q[5]}};
    Counters cn;
    Hit h;
    const bool hit = objs_hit(objs, r, 0.000f, 1000000000.0f, &h, &cn);
    // the leaf objs_hit re-intersected: repeating its (0, t_best + 1) re-intersection must give exactly its result
    float tb;
    const int32_t leaf = winning_leaf(objs, r, &tb);
    Hit g;
    const bool again = leaf >= 0 && sphere_hit(objs.L[(size_t)leaf], r, 0.000f, tb + 1.0f, &g);
    if (again != hit || (hit && !same_bits(g.t, h.t))) inconsistent = 1;
    const int32_t idx = hit ? objs.perm[(size_t)leaf] : -1;
    index[k] = idx;
    t[k] = hit ? h.t : INFINITY;
    if (pn) {
      const float v[6] = {h.p.x, h.p.y, h.p.z, h.normal.x, h.normal.y, h.normal.z};
      for (int c = 0; c < 6; c++) pn[6 * k + c] = hit ? v[c] : 0.0f;
    }
  });
  return inconsistent ? 2 : 0;
}

// ray_colour objs r 50 (ray.fut:126-148) per ray: colour[k][3], before quantisation.
int oracle_trace_rays(void *pv, const float *rays, int64_t n, float *colour, int32_t threads) {
  Prepared *p = (Prepared *)pv;
  if (!p || n < 0 || (n > 0 && (!rays || !colour))) return 1;
  for_rays(n, threads, [&](int64_t k) {
    const float *q = rays + 6 * k;
    Counters cn;
    const V3 c = ray_colour(p->objs, Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, 50, &cn);
    colour[3 * k] = c.x; colour[3 * k + 1] = c.y; colour[3 * k + 2] = c.z;
  });
  return 0;
}

}  // extern "C"
