// ORACLE — TEST INFRASTRUCTURE ONLY (see ref_math.hpp header).
// The refit of a kept binary tree (ptb_scene_commit with PTB_BUILD_REFIT), on the CPU: the tree is built once by
// lbvh_ref.hpp (Karras LBVH) or sah_ref.hpp (SAH builder), exactly as liboracle.so builds it, then new primitives of the
// same counts are swapped in and every box is recomputed bottom-up, the topology and the primitive order left as they are.
// The refit is written here on its own, beside Lbvh::build's step 5 rather than through it, so a refit of unchanged
// primitives reproducing the build's nodes bit for bit is a check of two separate statements of the same rule.
// Traversal and counts are Lbvh::closest_hit's. ctypes binding: oracle/refit_oracle.py.
#include <atomic>
#include <thread>
#include <vector>

#include "lbvh_ref.hpp"
#include "sah_ref.hpp"

using namespace ref;

struct orr_tree {
  Material mat{};  // only geometry matters: one non-emissive material for every primitive
  Lbvh lbvh;
};

static inline Vec3 v3(const ptb_vec3& v) { return Vec3(v.x, v.y, v.z); }

static std::vector<Prim> make_prims(const Material* mat, const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt) {
  std::vector<Prim> out;
  out.reserve(ns + nt);
  for (size_t i = 0; i < ns; ++i) {
    Prim p{};
    p.is_sphere = 1;
    p.orig_id = (uint32_t)i;
    p.material = mat;
    p.center = v3(spheres[i].center);
    p.radius = spheres[i].radius;
    out.push_back(p);
  }
  for (size_t i = 0; i < nt; ++i) {
    Prim p{};
    p.is_sphere = 0;
    p.orig_id = (uint32_t)(ns + i);
    p.material = mat;
    for (int k = 0; k < 3; ++k) { p.p[k] = v3(tris[i].p[k]); p.n[k] = v3(tris[i].n[k]); }
    out.push_back(p);
  }
  return out;
}

// box(node) = union of its children's boxes, every node storing both; a leaf's box is Prim::aabb of the primitive in its
// slot. Children before parents: the node array is walked from a post-order stack.
static void refit(Lbvh& l) {
  const size_t m = l.nodes.size();
  if (m == 0) return;
  auto set_box = [](float* mn, float* mx, const Vec3& a, const Vec3& b) {
    mn[0] = a.x; mn[1] = a.y; mn[2] = a.z; mx[0] = b.x; mx[1] = b.y; mx[2] = b.z;
  };
  std::vector<Vec3> nmin(m), nmax(m);
  std::vector<uint32_t> order;  // post-order of the inner nodes
  order.reserve(m);
  std::vector<std::pair<uint32_t, bool>> stack{{0u, false}};
  while (!stack.empty()) {
    const auto [i, expanded] = stack.back();
    stack.pop_back();
    if (expanded) { order.push_back(i); continue; }
    stack.push_back({i, true});
    const ptb_bvh_node& nd = l.nodes[i];
    if (!(nd.left & PTB_LEAF_BIT)) stack.push_back({nd.left, false});
    if (!(nd.right & PTB_LEAF_BIT) && nd.right != nd.left) stack.push_back({nd.right, false});
  }
  auto child = [&](uint32_t ref, Vec3& mn, Vec3& mx) {
    if (ref & PTB_LEAF_BIT) l.prims[l.prim_sorted[ref & ~PTB_LEAF_BIT]].aabb(mn, mx);
    else { mn = nmin[ref]; mx = nmax[ref]; }
  };
  for (uint32_t i : order) {
    ptb_bvh_node& nd = l.nodes[i];
    Vec3 lmn, lmx, rmn, rmx;
    child(nd.left, lmn, lmx);
    child(nd.right, rmn, rmx);
    set_box(nd.lmin, nd.lmax, lmn, lmx);
    set_box(nd.rmin, nd.rmax, rmn, rmx);
    nmin[i] = lmn.min_by_component(rmn);
    nmax[i] = lmx.max_by_component(rmx);
  }
}

template <class F>
static void parallel_for(size_t n, int threads, F f) {
  unsigned nt = threads > 0 ? (unsigned)threads : std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  if (nt == 1 || n < 1024) {
    f(0u, (size_t)0, n);
    return;
  }
  std::atomic<size_t> next(0);
  const size_t grain = 4096;
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < nt; ++t)
    pool.emplace_back([&, t]() {
      for (;;) {
        size_t b = next.fetch_add(grain);
        if (b >= n) break;
        f(t, b, b + grain < n ? b + grain : n);
      }
    });
  for (auto& th : pool) th.join();
}

extern "C" {

// builder 0: Karras LBVH (Lbvh::build); 1: the SAH builder over it (sah_rebuild, nbins / max_depth as the device uses)
orr_tree* orr_create(const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt, int builder, int nbins,
                     uint32_t max_depth) {
  orr_tree* t = new orr_tree();
  t->mat.kind = PTB_MAT_LAMBERTIAN;
  t->lbvh.build(make_prims(&t->mat, spheres, ns, tris, nt));
  if (builder == 1 && ns + nt >= 2) sah_rebuild(t->lbvh, nbins, max_depth);
  return t;
}
void orr_destroy(orr_tree* t) { delete t; }
size_t orr_num_nodes(const orr_tree* t) { return t->lbvh.nodes.size(); }

// new primitives, same counts (returns -1 and changes nothing otherwise), then the refit
int orr_refit(orr_tree* t, const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt) {
  if (ns + nt != t->lbvh.prims.size()) return -1;
  t->lbvh.prims = make_prims(&t->mat, spheres, ns, tris, nt);
  refit(t->lbvh);
  return 0;
}

void orr_export(const orr_tree* t, uint32_t* morton, uint32_t* prim_sorted, ptb_bvh_node* nodes) {
  const Lbvh& l = t->lbvh;
  if (morton) for (size_t i = 0; i < l.morton.size(); ++i) morton[i] = l.morton[i];
  if (prim_sorted) for (size_t i = 0; i < l.prim_sorted.size(); ++i) prim_sorted[i] = l.prim_sorted[i];
  if (nodes) for (size_t i = 0; i < l.nodes.size(); ++i) nodes[i] = l.nodes[i];
}

// Lbvh::closest_hit over the tree as it stands; counts2: nodes fetched, primitives tested (summed over the batch)
void orr_closest_hit(const orr_tree* t, const ptb_ray* rays, size_t n, ptb_hit* out, int threads, uint64_t* counts2) {
  unsigned nt = threads > 0 ? (unsigned)threads : std::thread::hardware_concurrency();
  std::vector<uint64_t> nv(nt ? nt : 1, 0), pt(nt ? nt : 1, 0);
  parallel_for(n, threads, [&](unsigned tid, size_t b, size_t e) {
    for (size_t i = b; i < e; ++i) {
      Ray ray(Vec3(rays[i].ox, rays[i].oy, rays[i].oz), Vec3(rays[i].dx, rays[i].dy, rays[i].dz), 0.0f);
      Hit h;
      uint32_t prim;
      if (t->lbvh.closest_hit(ray, h, prim, &nv[tid], &pt[tid])) out[i] = ptb_hit{h.t, prim, h.b1, h.b2};
      else out[i] = ptb_hit{0.0f, PTB_MISS, 0.0f, 0.0f};
    }
  });
  counts2[0] = counts2[1] = 0;
  for (size_t i = 0; i < nv.size(); ++i) { counts2[0] += nv[i]; counts2[1] += pt[i]; }
}

}  // extern "C"
