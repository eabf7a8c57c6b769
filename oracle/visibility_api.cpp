// ORACLE — TEST INFRASTRUCTURE ONLY (see ref_math.hpp header).
// The reference's two visibility queries for a batch of rays, over its own acceleration structure (ref_bvh.hpp: SAH tree,
// BFS un-culled candidates) — what the device's ptb_check_hit_index / ptb_occluded are compared against:
//   check_hit_index  Bvh::check_hit_index as it stands (acceleration/mod.rs:226-263);
//   occluded         its blocker scan on its own: a primitive other than `exclude` at 0 < t < tmax (the sky visibility test
//                    of sample_lights, mis.rs:104-115, is this with tmax = +inf), over the same BFS candidates;
//   occluded_brute   the same question over every primitive, no acceleration structure.
// Only geometry matters here: the scene is the primitives alone (one non-emissive material for all of them).
// ctypes binding: oracle/visibility_oracle.py.
#include <atomic>
#include <thread>
#include <vector>

#include "ref_bvh.hpp"

using namespace ref;

struct orv_scene {
  Material mat{};
  std::vector<Prim> prims_original;  // loader order: spheres first, then triangles
  Bvh bvh;
  std::vector<size_t> bvh_index;     // original id -> position in the BVH order
};

template <class F>
static void parallel_for(size_t n, int threads, F f) {
  unsigned nt = threads > 0 ? (unsigned)threads : std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  if (nt == 1 || n < 1024) {
    f((size_t)0, n);
    return;
  }
  std::atomic<size_t> next(0);
  const size_t grain = 4096;
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < nt; ++t)
    pool.emplace_back([&]() {
      for (;;) {
        size_t b = next.fetch_add(grain);
        if (b >= n) break;
        f(b, b + grain < n ? b + grain : n);
      }
    });
  for (auto& th : pool) th.join();
}

static inline Vec3 v3(const ptb_vec3& v) { return Vec3(v.x, v.y, v.z); }

// the blocker scan of Bvh::check_hit_index (acceleration/mod.rs:245-260) with an explicit tmax; exclude in BVH order
static bool occluded_bfs(const Bvh& bvh, const Ray& ray, Float tmax, size_t exclude) {
  thread_local std::vector<std::pair<size_t, size_t>> offset_lens;
  bvh.get_intersection_candidates(ray, offset_lens);
  Hit cur;
  for (const auto& ol : offset_lens)
    for (size_t ci = ol.first; ci < ol.first + ol.second; ++ci) {
      if (ci == exclude) continue;
      if (bvh.primitives[ci].get_int(ray, cur) && cur.t > 0.0f && cur.t < tmax) return true;
    }
  return false;
}

extern "C" {

orv_scene* orv_scene_create(const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt, int split_type) {
  orv_scene* s = new orv_scene();
  s->mat.kind = PTB_MAT_LAMBERTIAN;
  for (size_t i = 0; i < ns; ++i) {
    Prim p{};
    p.is_sphere = 1;
    p.orig_id = (uint32_t)i;
    p.material = &s->mat;
    p.center = v3(spheres[i].center);
    p.radius = spheres[i].radius;
    s->prims_original.push_back(p);
  }
  for (size_t i = 0; i < nt; ++i) {
    Prim p{};
    p.is_sphere = 0;
    p.orig_id = (uint32_t)(ns + i);
    p.material = &s->mat;
    for (int k = 0; k < 3; ++k) { p.p[k] = v3(tris[i].p[k]); p.n[k] = v3(tris[i].n[k]); }
    s->prims_original.push_back(p);
  }
  s->bvh.build(s->prims_original, (SplitType)split_type);
  s->bvh_index.resize(s->bvh.primitives.size());
  for (size_t i = 0; i < s->bvh_index.size(); ++i) s->bvh_index[s->bvh.primitives[i].orig_id] = i;
  return s;
}

void orv_scene_destroy(orv_scene* s) { delete s; }

// index[i]: original primitive id; a target out of range is not visible (the device answers the same way).
// Visible: {t_target, index[i], b1, b2}; otherwise {0, PTB_MISS, 0, 0}.
void orv_check_hit_index(const orv_scene* s, const ptb_ray* rays, const uint32_t* index, size_t n, ptb_hit* out, int threads) {
  parallel_for(n, threads, [&](size_t b, size_t e) {
    for (size_t i = b; i < e; ++i) {
      Ray ray(Vec3(rays[i].ox, rays[i].oy, rays[i].oz), Vec3(rays[i].dx, rays[i].dy, rays[i].dz), 0.0f);
      Hit h;
      const bool vis = index[i] < s->bvh_index.size() && s->bvh.check_hit_index(ray, s->bvh_index[index[i]], h);
      if (vis) out[i] = ptb_hit{h.t, index[i], h.b1, h.b2};
      else out[i] = ptb_hit{0.0f, PTB_MISS, 0.0f, 0.0f};
    }
  });
}

// out[i] = 1 iff a primitive other than rays[i].exclude (original id; PTB_MISS or out of range: none) is hit at
// 0 < t < rays[i].tmax; brute = 0: BFS candidates of the reference's tree, brute != 0: every primitive
void orv_occluded(const orv_scene* s, const ptb_occlusion_ray* rays, size_t n, uint8_t* out, int brute, int threads) {
  parallel_for(n, threads, [&](size_t b, size_t e) {
    for (size_t i = b; i < e; ++i) {
      const ptb_occlusion_ray& r = rays[i];
      Ray ray(Vec3(r.ox, r.oy, r.oz), Vec3(r.dx, r.dy, r.dz), 0.0f);
      bool occ = false;
      if (!brute) {
        const size_t ex = r.exclude < s->bvh_index.size() ? s->bvh_index[r.exclude] : Bvh::MISS;
        occ = occluded_bfs(s->bvh, ray, r.tmax, ex);
      } else {
        Hit h;
        for (const Prim& p : s->prims_original)
          if (p.orig_id != r.exclude && p.get_int(ray, h) && h.t > 0.0f && h.t < r.tmax) { occ = true; break; }
      }
      out[i] = occ ? 1 : 0;
    }
  });
}

}  // extern "C"
