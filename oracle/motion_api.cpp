// ORACLE — TEST INFRASTRUCTURE ONLY (see ref_math.hpp header).
// Motion vectors of ptb_render_aov after ptb_motion_mark (include/ptb200.h "motion vectors") restated over the AOV
// oracle's scene (aov_api.cpp: the reference's camera and SAH tree), for every (pixel, sample): the same camera ray and
// first hit, P' from the marked primitives (loader order, ptb_sphere / ptb_triangle records) and both projections in the
// header's order of operations, summed in f32 in increasing sample order. ctypes binding: oracle/motion_oracle.py.
#include <cstring>

#include "aov_api.cpp"

namespace {

// the barycentrics of triangle_int (ref_scene.hpp) for a ray that hits the triangle: the same statements up to b0, b1, b2
void tri_bary(const Ray& ray, const Vec3 p[3], Float& b0, Float& b1, Float& b2) {
  Vec3 p0t = p[0] - ray.origin, p1t = p[1] - ray.origin, p2t = p[2] - ray.origin;
  const Vec3& d = ray.direction;
  const bool swap = (std::fabs(d.x) > std::fabs(d.y) && std::fabs(d.x) > std::fabs(d.z)) || (std::fabs(d.y) > std::fabs(d.z));
  if (swap) {
    Float tmp;
    tmp = p0t.x; p0t.x = p0t.z; p0t.z = tmp;
    tmp = p1t.x; p1t.x = p1t.z; p1t.z = tmp;
    tmp = p2t.x; p2t.x = p2t.z; p2t.z = tmp;
  }
  p0t.x += ray.shear.x * p0t.z; p0t.y += ray.shear.y * p0t.z;
  p1t.x += ray.shear.x * p1t.z; p1t.y += ray.shear.y * p1t.z;
  p2t.x += ray.shear.x * p2t.z; p2t.y += ray.shear.y * p2t.z;
  Float e0 = p1t.x * p2t.y - p1t.y * p2t.x;
  Float e1 = p2t.x * p0t.y - p2t.y * p0t.x;
  Float e2 = p0t.x * p1t.y - p0t.y * p1t.x;
  if (e0 == 0.0f || e1 == 0.0f || e2 == 0.0f) {
    e0 = (Float)((double)p1t.x * (double)p2t.y - (double)p1t.y * (double)p2t.x);
    e1 = (Float)((double)p2t.x * (double)p0t.y - (double)p2t.y * (double)p0t.x);
    e2 = (Float)((double)p0t.x * (double)p1t.y - (double)p0t.y * (double)p1t.x);
  }
  const Float inv_det = 1.0f / (e0 + e1 + e2);
  b0 = e0 * inv_det;
  b1 = e1 * inv_det;
  b2 = e2 * inv_det;
}

// proj(cam, X) of the header: d = X - o, a = ll - o, n = cross(h, vv), s = dot(d, n); λ = s / dot(a, n),
// u = dot(d, cross(vv, a)) / s, v = dot(d, cross(a, h)) / s
void cam_project(const Camera& c, const Vec3& x, Float& u, Float& v, Float& lambda) {
  const Vec3 d = x - c.origin, a = c.lower_left - c.origin, n = c.horizontal.cross(c.vertical);
  const Float s = d.dot(n);
  lambda = s / a.dot(n);
  u = d.dot(c.vertical.cross(a)) / s;
  v = d.dot(a.cross(c.horizontal)) / s;
}

bool same_bits(const float* a, const float* b, int n) { return std::memcmp(a, b, sizeof(float) * n) == 0; }

Vec3 at(const float* f) { return Vec3(f[0], f[1], f[2]); }

}  // namespace

extern "C" {

// Adds the motion of the samples [sample_offset, sample_offset + samples_per_pixel) of the tile's rows into `motion`
// (width * height * 4 floats: Σ Δx, Σ Δy, Σ t', valid samples). The committed frame is the scene `s`; the marked one is
// `prev_spheres` / `prev_tris` (same counts as the scene) and `prev_cam`.
void ora_render_motion(const ora_scene* s, const ptb_render_opts* o, float* motion, const ptb_sphere* prev_spheres,
                       const ptb_triangle* prev_tris, const ptb_camera* prev_cam, int threads) {
  const uint32_t rows = o->row_count ? o->row_count : o->height - o->row_begin;
  const size_t npix = (size_t)o->width * rows;
  size_t ns = 0;
  for (const Prim& p : s->prims_original) ns += p.is_sphere ? 1 : 0;
  Camera pc;
  pc.origin = v3(prev_cam->origin);
  pc.lower_left = v3(prev_cam->lower_left);
  pc.horizontal = v3(prev_cam->horizontal);
  pc.vertical = v3(prev_cam->vertical);
  const Float wm1 = (Float)(o->width - 1), hm1 = (Float)(o->height - 1);
  unsigned nt = threads > 0 ? (unsigned)threads : std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  std::atomic<size_t> next(0);
  auto worker = [&]() {
    g_rng.seed(o->seed);
    for (;;) {
      const size_t k = next.fetch_add(1);
      if (k >= npix) break;
      const uint64_t pixel_i = (uint64_t)o->row_begin * o->width + k;
      const uint64_t x = pixel_i % o->width, y = (pixel_i - x) / o->width;
      float* m = motion + 4 * pixel_i;
      for (uint32_t si = 0; si < o->samples_per_pixel; ++si) {
        g_rng.path((uint32_t)pixel_i, o->sample_offset + si);
        g_rng.select(0, RNG_JITTER);
        const Float u = (g_rng.next_float01() + (Float)x) / (Float)(o->width - 1);
        const Float v = 1.0f - (g_rng.next_float01() + (Float)y) / (Float)(o->height - 1);
        const Ray ray = s->camera.get_ray(u, v);
        Hit hit;
        const Material* mat;
        const size_t idx = s->bvh.check_hit(ray, hit, mat);
        if (idx == Bvh::MISS) continue;
        const Prim& pr = s->bvh.primitives[idx];
        Vec3 q = hit.point;
        if (pr.is_sphere) {
          const ptb_sphere& ps = prev_spheres[pr.orig_id];
          const float cur[4] = {pr.center.x, pr.center.y, pr.center.z, pr.radius};
          if (!same_bits(cur, &ps.center.x, 4)) q = v3(ps.center) + (hit.point - pr.center) * (ps.radius / pr.radius);
        } else {
          const ptb_triangle& pt = prev_tris[pr.orig_id - ns];
          const float cur[9] = {pr.p[0].x, pr.p[0].y, pr.p[0].z, pr.p[1].x, pr.p[1].y, pr.p[1].z, pr.p[2].x, pr.p[2].y, pr.p[2].z};
          if (!same_bits(cur, &pt.p[0].x, 9)) {
            Float b0, b1, b2;
            tri_bary(ray, pr.p, b0, b1, b2);
            q = b0 * at(&pt.p[0].x) + b1 * at(&pt.p[1].x) + b2 * at(&pt.p[2].x);
          }
        }
        Float u0, v0, l0, u1, v1, l1;
        cam_project(s->camera, hit.point, u0, v0, l0);
        cam_project(pc, q, u1, v1, l1);
        if (!(l1 > 0.0f)) continue;
        m[0] += (u1 - u0) * wm1;
        m[1] += -(v1 - v0) * hm1;
        m[2] += (q - pc.origin).mag();
        m[3] += 1.0f;
      }
    }
  };
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < nt; ++t) pool.emplace_back(worker);
  for (auto& th : pool) th.join();
}

}  // extern "C"
