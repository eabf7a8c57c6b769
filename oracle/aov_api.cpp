// ORACLE — TEST INFRASTRUCTURE ONLY (see ref_math.hpp header).
// Denoiser feature buffers (ptb_render_aov) restated over the reference's own scene code, for every (pixel, sample):
//   the camera ray     the jitter and Camera::get_ray of sample_pixel (ref_integrators.hpp:236-242);
//   the first hit      Bvh::check_hit over the reference's SAH tree (a miss answers the zero Hit + the sky's Emit material);
//   albedo             Lambertian: eval_over_scattering_pdf (colour * param); Emit (and the sky): get_emission;
//                      Reflect, Refract, Trowbridge-Reitz: the texture's colour_value(wo, hit.point); each channel clamped
//                      to [0, 1] with fmin(fmax(x, 0), 1) (a NaN becomes 0);
//   normal, depth      hit.normal and hit.t (zero on a miss); coverage 1 on a hit, 0 on a miss;
// summed in f32 in increasing sample order per pixel. ctypes binding: oracle/aov_oracle.py.
#include <atomic>
#include <cmath>
#include <thread>
#include <vector>

#include "ref_integrators.hpp"

namespace ref {
thread_local RngCursor g_rng;
}

using namespace ref;

struct ora_scene {
  std::vector<Texture> textures;
  std::vector<Material> materials;
  std::vector<std::vector<Float>> texture_words;  // owned copies of image pixels / perlin tables
  std::vector<Prim> prims_original;               // loader order: spheres first, then triangles
  Bvh bvh;
  Camera camera;
};

static inline Vec3 v3(const ptb_vec3& v) { return Vec3(v.x, v.y, v.z); }

static inline Float clamp01(Float x) { return std::fmin(std::fmax(x, 0.0f), 1.0f); }

// the albedo of one first hit (mat: the hit's material, or the sky's Emit material on a miss)
static Vec3 albedo(const Material* mat, const Hit& hit, const Vec3& wo) {
  switch (mat->kind) {
    case PTB_MAT_EMIT: return mat->get_emission(hit, wo);
    case PTB_MAT_LAMBERTIAN: return mat->texture->colour_value(wo, hit.point) * mat->param;  // lambertian.rs:48-50
    default: return mat->texture->colour_value(wo, hit.point);
  }
}

extern "C" {

// the scene as liboracle.so's orc_scene_create takes it (same arguments), always with the SAH split
ora_scene* ora_scene_create(const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt, const ptb_material* mats,
                            size_t nm, const ptb_texture* texs, size_t ntex, const ptb_camera* cam, const ptb_sky* sky,
                            const float* const* tex_data, const uint32_t* tex_dims /* width, height, n_words per texture */) {
  ora_scene* s = new ora_scene();
  s->textures.resize(ntex);
  s->texture_words.resize(ntex);
  for (size_t i = 0; i < ntex; ++i) {
    s->textures[i].kind = texs[i].kind;
    s->textures[i].a = v3(texs[i].a);
    s->textures[i].b = v3(texs[i].b);
    if (tex_data && tex_data[i]) {
      s->texture_words[i].assign(tex_data[i], tex_data[i] + tex_dims[3 * i + 2]);
      s->textures[i].data = s->texture_words[i].data();
      s->textures[i].perm = reinterpret_cast<const uint32_t*>(s->texture_words[i].data()) + 256;
      s->textures[i].width = tex_dims[3 * i];
      s->textures[i].height = tex_dims[3 * i + 1];
    }
  }
  s->materials.resize(nm);
  for (size_t i = 0; i < nm; ++i) {
    s->materials[i].kind = mats[i].kind;
    s->materials[i].texture = &s->textures[mats[i].texture];
    s->materials[i].param = mats[i].param;
    s->materials[i].ior = v3(mats[i].ior);
    s->materials[i].metallic = mats[i].metallic;
  }
  for (size_t i = 0; i < ns; ++i) {
    Prim p{};
    p.is_sphere = 1;
    p.orig_id = (uint32_t)i;
    p.material = &s->materials[spheres[i].material];
    p.center = v3(spheres[i].center);
    p.radius = spheres[i].radius;
    s->prims_original.push_back(p);
  }
  for (size_t i = 0; i < nt; ++i) {
    Prim p{};
    p.is_sphere = 0;
    p.orig_id = (uint32_t)(ns + i);
    p.material = &s->materials[tris[i].material];
    for (int k = 0; k < 3; ++k) { p.p[k] = v3(tris[i].p[k]); p.n[k] = v3(tris[i].n[k]); }
    s->prims_original.push_back(p);
  }
  s->camera.origin = v3(cam->origin);
  s->camera.lower_left = v3(cam->lower_left);
  s->camera.horizontal = v3(cam->horizontal);
  s->camera.vertical = v3(cam->vertical);
  s->bvh.sky.init(&s->textures[sky->texture], sky->sampler_res_x, sky->sampler_res_y);
  s->bvh.build(s->prims_original, SPLIT_SAH);
  return s;
}

void ora_scene_destroy(ora_scene* s) { delete s; }

// Adds the samples [sample_offset, sample_offset + samples_per_pixel) of the pixel rows [row_begin, row_begin + rows) into
// `sums` (width * height * 8 floats: albedo.rgb, coverage, normal.xyz, depth per pixel; row-major, top row first).
// `prims` (optional, rows * width * samples_per_pixel words, pixel-major within the tile): the original id of each
// sample's hit, PTB_MISS on a miss.
void ora_render_aov(const ora_scene* s, const ptb_render_opts* o, float* sums, uint32_t* prims, int threads) {
  const uint32_t rows = o->row_count ? o->row_count : o->height - o->row_begin;
  const size_t npix = (size_t)o->width * rows;
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
      float* p = sums + 8 * pixel_i;
      for (uint32_t si = 0; si < o->samples_per_pixel; ++si) {
        // samplers/random_sampler.rs:50-61 as sample_pixel states it
        g_rng.path((uint32_t)pixel_i, o->sample_offset + si);
        g_rng.select(0, RNG_JITTER);
        const Float u = (g_rng.next_float01() + (Float)x) / (Float)(o->width - 1);
        const Float v = 1.0f - (g_rng.next_float01() + (Float)y) / (Float)(o->height - 1);
        const Ray ray = s->camera.get_ray(u, v);
        Hit hit;
        const Material* mat;
        const size_t idx = s->bvh.check_hit(ray, hit, mat);
        const bool is_hit = idx != Bvh::MISS;
        const Vec3 a = albedo(mat, hit, ray.direction);
        p[0] += clamp01(a.x);
        p[1] += clamp01(a.y);
        p[2] += clamp01(a.z);
        p[3] += is_hit ? 1.0f : 0.0f;
        p[4] += hit.normal.x;
        p[5] += hit.normal.y;
        p[6] += hit.normal.z;
        p[7] += hit.t;
        if (prims) prims[k * o->samples_per_pixel + si] = is_hit ? s->bvh.primitives[idx].orig_id : PTB_MISS;
      }
    }
  };
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < nt; ++t) pool.emplace_back(worker);
  for (auto& th : pool) th.join();
}

}  // extern "C"
