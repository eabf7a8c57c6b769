// ptb200 — wavefront path tracer (sm_100a). Replaces RandomSampler::sample_image + the integrators
// (implementations/src/samplers/random_sampler.rs:23-99, integrators/mod.rs:22-78, integrators/mis.rs:6-157) and
// everything they call per bounce (materials/*.rs, sky.rs, textures/mod.rs, primitives light sampling).
//
// Window wavefront (see "window wavefront" below): a call runs in chunks, every camera path of a chunk is resident, path g
// owns slot g, and one iteration traces and shades bounce k of ALL of them:
//   k_win_scan / k_win_prepare / k_win_fill   live counts -> ordered trace queue (slot order, direction-ordered per window)
//   k_trace     K1 + K8      closest hit for every live path (persistent warps pulling 32-ray batches); the first
//                            iteration of a chunk computes its camera rays in the fetch (random_sampler.rs:50-61,
//                            camera.rs:57-63)
//   k_shade     K10 + K12    emission, MIS weights, NEE sample -> shadow queue, BSDF sample -> next ray (written in place),
//                            Russian roulette, path termination -> accumulator
//   k_shadow    K9           any-hit for the NEE queue; unoccluded contributions are added to the path's radiance
//
// The RNG is counter-based (Philox4x32-10 keyed by seed; counter = pixel, absolute sample, depth|purpose, block):
// the image is a pure function of (scene, seed, sample range) — independent of pool size, scheduling and GPU count.
#include "ptb_internal.h"
#include "ptb_traverse.cuh"
#include "ptb_packet.cuh"
#include "ptb_camcand.cuh"

namespace ptb {

struct RenderParams {
  uint32_t width, height, npix;  // npix = width * (rows of this call's image tile)
  uint32_t row_begin;            // first pixel row of the tile (ptb_render_opts::row_begin)
  uint32_t tile_w, tile_h;  // pixel issue order (camera_pixel_sample); tile_h == 1 -> row-major
  uint32_t group;           // samples of one pixel issued back to back (a divisor of the call's spp)
  uint32_t dir_bins;        // order a window's live rays by direction bin (PTB_DIRBINS=0 disables)
  uint32_t sample_offset;
  uint32_t method, max_depth, rr_threshold;
  uint32_t k0, k1;  // Philox key
};

struct Queues {
  uint32_t* live;  // [capacity] this iteration's trace queue: the live slots, ordered by k_win_fill
  float4* shadow;  // 3 x float4 per entry: o.xyz|tmax, d.xyz|exclude slot, contrib.rgb|path slot
  // see "window wavefront" below
  uint32_t* win_count;   // [n_windows] live paths of each kWindow-slot window
  uint32_t* win_prefix;  // [n_windows] exclusive prefix of win_count inside the window's 4096-window segment
  uint32_t* seg_total;   // [n_windows / 4096 + 1] live paths per segment
  uint8_t* bin;          // [capacity] direction bin of the path's next ray, kBinDead once the path has finished
  uint32_t n_windows;
};
constexpr uint32_t kBinDead = 0xFFu;
constexpr unsigned long long kNoCamera = ~0ull;
#ifndef PTB_WINDOW
#define PTB_WINDOW 4096  // slots per window (256 * 1, 2, 4, 8 or 16): the span inside which k_win_fill orders the live rays by direction
#endif
#ifndef PTB_DIR_BITS
#define PTB_DIR_BITS 8   // direction bins per window: 5 = octant x dominant axis, 8 = 16 x 16 octahedral map in Morton order
#endif
constexpr uint32_t kWindow = PTB_WINDOW;
constexpr uint32_t kWinItems = kWindow / 256u;  // slots per k_win_fill thread
static_assert(kWindow % 256u == 0 && kWinItems >= 1 && kWinItems <= 16 && (kWinItems & (kWinItems - 1)) == 0, "window size");
constexpr uint32_t kSegWindows = 4096u;   // windows per scan segment (1024 threads x 4)

constexpr uint32_t kFlagPrevDelta = 1u << 8;  // stored above the 8-bit depth in ray_d.w

// ------------------------------------------------------------------------------------------ textures / sky
// implementations/src/textures/mod.rs (all five kinds; the arithmetic is texture_eval in ptb_common.cuh)
// FULL = false: kernels for scenes that hold only solid / lerp / checkered textures and no Trowbridge-Reitz material
// (the host picks the instantiation at launch), so the common case does not pay registers for the rest.
template <bool FULL>
PTB_DEV v3 texture_colour(const DevTexture* __restrict__ textures, const float* __restrict__ tex_data, uint32_t tex,
                          v3 direction, v3 point) {
  const DevTexture* t = textures + tex;
  const uint32_t kind = __ldg(&t->kind);
  const v3 a = mk(__ldg(&t->a[0]), __ldg(&t->a[1]), __ldg(&t->a[2]));
  if (kind == PTB_TEX_SOLID) return a;
  const v3 b = mk(__ldg(&t->b[0]), __ldg(&t->b[1]), __ldg(&t->b[2]));
  if (!FULL) {
    if (kind == PTB_TEX_LERP) {
      const float tt = direction.z * 0.5f + 0.5f;
      return a * tt + b * (1.0f - tt);
    }
    const float sign = sinf(10.0f * point.x) * sinf(10.0f * point.y) * sinf(10.0f * point.z);
    return sign > 0.0f ? a : b;
  }
  TexWords words{tex_data + __ldg(&t->data_off)};
  return texture_eval(kind, a, b, __ldg(&t->width), __ldg(&t->height), words, direction, point);
}
template <bool FULL>
PTB_DEV v3 texture_colour(const DevScene& sc, uint32_t tex, v3 direction, v3 point) {
  return texture_colour<FULL>(sc.textures, sc.tex_data, tex, direction, point);
}

// statistics/distributions.rs:51-72
PTB_DEV uint32_t dist1d_sample(const float* __restrict__ cdf, uint32_t cdf_len, float num) {
  uint32_t first = 0, len = cdf_len;
  while (len > 0) {
    const uint32_t half = len >> 1;
    const uint32_t middle = first + half;
    if (__ldg(cdf + middle) <= num) {
      first = middle + 1;
      len -= half + 1;
    } else {
      len = half;
    }
  }
  const uint32_t r = first - 1u, hi = cdf_len - 2u;
  return r > hi ? hi : r;
}
// sky.rs:43-60
PTB_DEV float sky_pdf(const DevScene& sc, v3 wi) {
  const float sin_theta = sqrtf(1.0f - wi.z * wi.z);
  if (sin_theta <= 0.0f) return 0.0f;
  const float theta = acosf(wi.z);
  float phi = atan2f(wi.y, wi.x);
  if (phi < 0.0f) phi += 2.0f * kPi;
  const float u = phi / (2.0f * kPi);
  const float v = theta / kPi;
  const uint32_t ui = sat_index((float)sc.sky_rx * u, sc.sky_rx - 1u);
  const uint32_t vi = sat_index((float)sc.sky_ry * v, sc.sky_ry - 1u);
  const float pdf = __ldg(sc.sky_ypdf + vi) * __ldg(sc.sky_xpdf + (size_t)vi * sc.sky_rx + ui);
  return (float)sc.sky_rx * (float)sc.sky_ry * pdf / (sin_theta * kTau * kPi);
}
// sky.rs:64-78 with draws (row, column, u jitter, v jitter)
PTB_DEV v3 sky_sample(const DevScene& sc, float r_row, float r_col, float r_u, float r_v) {
  const uint32_t vi = dist1d_sample(sc.sky_ycdf, sc.sky_ry + 1u, r_row);
  const uint32_t ui = dist1d_sample(sc.sky_xcdf + (size_t)vi * (sc.sky_rx + 1u), sc.sky_rx + 1u, r_col);
  const float u = next_float((float)ui + r_u) / (float)sc.sky_rx;
  const float v = next_float((float)vi + r_v) / (float)sc.sky_ry;
  const float phi = u * 2.0f * kPi;
  const float theta = v * kPi;
  float st, ct, sp, cp;  // sincosf: one range reduction for both; same values as sinf / cosf
  sincosf(theta, &st, &ct);
  sincosf(phi, &sp, &cp);
  return mk(st * cp, st * sp, ct);
}

// ------------------------------------------------------------------------------------------ lights
// sphere.rs:112-154 / triangle.rs:258-277 (MeshTriangle variant, quirk Q8)
PTB_DEV v3 light_sample_dir(const DevScene& sc, uint32_t ref, v3 in_point, float r1, float r2) {
  const float4* g = sc.geom + 3u * (size_t)(ref & kSlotMask);
  const float4 g0 = __ldg(g);
  v3 point;
  if (ref & kSphereBit) {
    const v3 center = from4(g0);
    const float radius = g0.w;
    const float distance_sq = mag_sq(in_point - center);
    if (distance_sq <= radius * radius) {
      const float z = 1.0f - 2.0f * r1;
      const float a = sqrtf(fmaxf(1.0f - z * z, 0.0f));
      const float b = 2.0f * kPi * r2;
      float sb, cb;
      sincosf(b, &sb, &cb);
      point = center + radius * mk(a * cb, a * sb, z);
    } else {
      const float distance = sqrtf(distance_sq);
      const float sin_theta_max_sq = radius * radius / distance_sq;
      const float cos_theta_max = sqrtf(fmaxf(1.0f - sin_theta_max_sq, 0.0f));
      const float cos_theta = (1.0f - r1) + r1 * cos_theta_max;
      const float sin_theta = sqrtf(fmaxf(1.0f - cos_theta * cos_theta, 0.0f));
      const float phi = 2.0f * r2 * kPi;
      const float ds = distance * cos_theta - sqrtf(fmaxf(radius * radius - distance_sq * sin_theta * sin_theta, 0.0f));
      const float cos_alpha = (distance_sq + radius * radius - ds * ds) / (2.0f * distance * radius);
      const float sin_alpha = sqrtf(fmaxf(1.0f - cos_alpha * cos_alpha, 0.0f));
      float sphi, cphi;
      sincosf(phi, &sphi, &cphi);
      const v3 vec = onb_to_world(normalised(in_point - center), mk(sin_alpha * cphi, sin_alpha * sphi, cos_alpha));
      point = center + radius * vec;
    }
  } else {
    const v3 p0 = from4(g0), p1 = from4(__ldg(g + 1)), p2 = from4(__ldg(g + 2));
    const float s = sqrtf(r1);
    const float u0 = 1.0f - s;
    const float u1 = s * sqrtf(r2);
    point = u0 * p0 + u1 * p1 + (1.0f - u0 - u1) * p2;
  }
  return normalised(point - in_point);
}
// sphere.rs:155-170 / triangle.rs:249-257, 278-280
PTB_DEV float light_pdf(const DevScene& sc, uint32_t ref, v3 hit_point, v3 wi, v3 s_point, v3 s_normal) {
  const float4* g = sc.geom + 3u * (size_t)(ref & kSlotMask);
  const float4 g0 = __ldg(g);
  if (ref & kSphereBit) {
    const v3 center = from4(g0);
    const float radius = g0.w;
    const float rsq = radius * radius;
    const float dsq = mag_sq(hit_point - center);
    if (dsq <= rsq) {
      const float area = 4.0f * kPi * radius * radius;
      return mag_sq(s_point - hit_point) / (fabsf(dot(wi, s_normal)) * area);
    }
    const float sin_theta_max_sq = rsq / dsq;
    const float cos_theta_max = sqrtf(fmaxf(1.0f - sin_theta_max_sq, 0.0f));
    return 1.0f / (2.0f * kPi * (1.0f - cos_theta_max));
  }
  const v3 p0 = from4(g0), p1 = from4(__ldg(g + 1)), p2 = from4(__ldg(g + 2));
  const float area = 0.5f * mag(cross(p1 - p0, p2 - p0));
  return mag_sq(s_point - hit_point) / (fabsf(dot(wi, s_normal)) * area);
}

// ------------------------------------------------------------------------------------------ BSDF direction samplers
// The sampling arithmetic of k_shade as functions, so that the chi-squared test hook (k_sample_only below) draws from the
// very code the integrator runs.
// lambertian.rs:30-41, statistics/bxdfs/lambertian.rs:5-18, utility/coord.rs:10-30
PTB_DEV v3 lambertian_sample_dir(v3 normal, float r1, float r2) {
  const float cos_theta = sqrtf(1.0f - r1);
  const float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
  const float phi = 2.0f * kPi * r2;
  float sphi, cphi;
  sincosf(phi, &sphi, &cphi);
  return onb_to_world(normal, mk(cphi * sin_theta, sphi * sin_theta, cos_theta));
}
// random_unit_vector (utility/mod.rs:15-25) is a rejection loop whose result is uniform on the sphere — drawn directly here
// from two uniforms (fixed RNG budget), same distribution
PTB_DEV v3 uniform_sphere_dir(float r1, float r2) {
  const float z = 1.0f - 2.0f * r1;
  const float rr = sqrtf(fmaxf(1.0f - z * z, 0.0f));
  const float phi = 2.0f * kPi * r2;
  float sphi, cphi;
  sincosf(phi, &sphi, &cphi);
  return mk(rr * cphi, rr * sphi, z);
}

// ------------------------------------------------------------------------------------------ bookkeeping kernels
// A slot's counters at the start of a render: work cursors and statistics zeroed, no fused-tail hand-over timed yet
// (k_win_init folds a finished one into tail_ns only when tail_t0 != ~0). k_win_init sets the per-chunk state (mode,
// n_tail, tail_iter, tail_head).
__global__ void k_reset_counters(WaveCounters* wc) {
  wc->n_trace = wc->trace_head = wc->shadow_head = 0;
  wc->shadow_pair = 0;
  wc->rays_camera = wc->rays_bounce = wc->rays_shadow_light = wc->rays_shadow_sky = wc->rays_reference = wc->paths = 0;
  wc->nodes_fetched = wc->prims_tested = wc->rays_counted = 0;
  wc->tail_t0 = ~0ull;
  wc->tail_t1 = wc->tail_ns = 0ull;
}

// ------------------------------------------------------------------------------------------ K1 camera rays
// Global path index g -> pixel (x, y) and absolute sample index.
PTB_DEV void camera_pixel_sample(const RenderParams& rp, unsigned long long g, uint32_t& x, uint32_t& y, uint32_t& sample) {
  // issue order: for each chunk of `group` samples, for each pixel, the chunk's samples — the 32 camera rays of a warp
  // share a pixel (group >= 32) and walk the same nodes down to the last levels. Only the ORDER changes; RNG and
  // accumulator are keyed by (pixel, absolute sample).
  const unsigned long long per_chunk = (unsigned long long)rp.npix * rp.group;
  const uint32_t chunk = (uint32_t)(g / per_chunk);
  const unsigned long long within_chunk = g % per_chunk;
  const uint32_t lin = (uint32_t)(within_chunk / rp.group);
  sample = rp.sample_offset + chunk * rp.group + (uint32_t)(within_chunk % rp.group);
  // A warp's 32 consecutive work items cover a tile_w x tile_h block of pixels (8x4 when the image allows) instead of a
  // 32x1 strip (group == 1 only matters): only the issue ORDER changes.
  if (rp.tile_h > 1u) {
    const uint32_t tile = lin >> 5, within = lin & 31u, tiles_x = rp.width / rp.tile_w;
    x = (tile % tiles_x) * rp.tile_w + within % rp.tile_w;
    y = (tile / tiles_x) * rp.tile_h + within / rp.tile_w;
  } else {
    x = lin % rp.width;
    y = lin / rp.width;
  }
  y += rp.row_begin;  // image tile: pixels keep their full-image coordinates
}
// random_sampler.rs:55-59 (note W-1 / H-1), camera.rs:57-63; the caller's make_ray is Ray::new (ray.rs:13-46)
PTB_DEV v3 camera_direction(const DevScene& sc, const RenderParams& rp, uint32_t x, uint32_t y, uint32_t sample) {
  const uint32_t pixel = y * rp.width + x;
  const uint4 r = philox4x32_10(pixel, sample, (0u << 8) | RNG_JITTER, 0u, rp.k0, rp.k1);
  const float u = (u32_to_unit(r.x) + (float)x) / (float)(rp.width - 1u);
  const float v = 1.0f - (u32_to_unit(r.y) + (float)y) / (float)(rp.height - 1u);
  const v3 dir = sc.cam_lower_left + sc.cam_horizontal * u + sc.cam_vertical * v - sc.cam_origin;
  return dir / mag(dir);
}

// ------------------------------------------------------------------------------------------ K8 closest hit
// CAMERA (first iteration of a chunk): work item i IS slot i and its ray is the camera ray of path first + i, computed
// here — the chunk's camera rays are never written to and read back from memory.
template <bool CAMERA>
struct TraceFetch {
  const PathPool& pool;
  const uint32_t* __restrict__ queue;
  uint32_t slot;
  const DevScene& sc;
  const RenderParams& rp;
  unsigned long long first;
  PTB_DEV void operator()(uint32_t i, Ray& ray, float& /*tmax*/, uint32_t& /*exclude*/) {
    if (CAMERA) {
      slot = i;
      uint32_t x, y, sample;
      camera_pixel_sample(rp, first + i, x, y, sample);
      ray = make_ray(sc.cam_origin, camera_direction(sc, rp, x, y, sample));
      return;
    }
    slot = queue[i];
    float4 o, d;
    ldg256_rw(pool.ray + 4u * (size_t)slot, o, d);
    ray = make_ray(from4(o), from4(d));
  }
};
template <bool CAMERA>
struct TraceRetire {
  const PathPool& pool;
  const TraceFetch<CAMERA>& f;
  // write the hit: the whole 32-byte ray record, so the store is a full sector
  PTB_DEV void operator()(bool fin, const TraceResult& tr, const Ray& ray) {
    if (fin)
      stg256(pool.ray + 4u * (size_t)f.slot, make_float4(ray.o.x, ray.o.y, ray.o.z, tr.t),
             make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(tr.ref)));
  }
};

#ifndef PTB_SHADE_MIN_BLOCKS
#define PTB_SHADE_MIN_BLOCKS 4  // caps k_shade at 64 registers (32 B of spills). The window wavefront streams its records, so
                                // occupancy pays: 2 -> 4 blocks: C3 3664 -> 3746 Mrays/s, rtweekend1 4K MIS 8439 -> 8967
                                // (profiles/r1_sweeps.md)
#endif
template <class TR, bool COUNT, bool CAMERA>
__global__ void __launch_bounds__(256, TR::kTraceMinBlocks)
k_trace(DevScene sc, PathPool pool, Queues q, WaveCounters* wc, RenderParams rp, unsigned long long first) {
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t cnt_nodes = 0, cnt_prims = 0, cnt_rays = 0;
  TraceFetch<CAMERA> fetch{pool, q.live, 0u, sc, rp, first};
  TraceRetire<CAMERA> retire{pool, fetch};
  persistent_trace<TR, false, COUNT>(sc, wc->n_trace, &wc->trace_head, fetch, retire, cnt_nodes, cnt_prims, cnt_rays);
  if (COUNT) {
    for (int off = 16; off > 0; off >>= 1) {
      cnt_nodes += __shfl_xor_sync(0xffffffffu, cnt_nodes, off);
      cnt_prims += __shfl_xor_sync(0xffffffffu, cnt_prims, off);
      cnt_rays += __shfl_xor_sync(0xffffffffu, cnt_rays, off);
    }
    if (lane == 0 && cnt_rays) {
      atomicAdd(&wc->nodes_fetched, (unsigned long long)cnt_nodes);
      atomicAdd(&wc->prims_tested, (unsigned long long)cnt_prims);
      atomicAdd(&wc->rays_counted, (unsigned long long)cnt_rays);
    }
  }
}

// K1 + K8 for the first iteration of a window-mode chunk on the binary tree: packets (ptb_packet.cuh). Work item i is slot i
// and its ray is the camera ray of path first + i, computed here; a warp takes 32 consecutive slots — samples of one pixel
// (or of one 8 x 4 pixel tile when the call has fewer samples) — and walks the tree once for all of them.
// With candidate lists (cl.count set; ptb_camcand.cuh) a warp's 32 samples belong to one pixel, and the warp answers them
// from that pixel's list unless it overflowed — same hits as the packet walk, bit for bit. Counted renders
// (PTB_OPT_COUNT_TRAVERSAL) count a listed ray's primitive tests as prims and no nodes; k_cam_candidates counts the beam
// walk's nodes, once per pixel.
#ifndef PTB_CAMERA_MIN_BLOCKS
// 4 blocks per SM = 64 registers (62 before the candidate-list path), no spills. (Before the octant-specialised slab test the kernel needed 71 registers and
// lost at 4 blocks: 4252 vs 4344 Mrays/s on C3; with it, 3 -> 4 blocks: 4849 -> 4925 at 256 spp, 4475 -> 4570 at 32 spp.)
#define PTB_CAMERA_MIN_BLOCKS 4
#endif
template <bool COUNT>
__global__ void __launch_bounds__(256, PTB_CAMERA_MIN_BLOCKS)
k_trace_camera(DevScene sc, PathPool pool, Queues q, WaveCounters* wc, RenderParams rp, unsigned long long first, CamCandList cl) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t n = wc->n_trace;
  uint32_t cnt_nodes = 0, cnt_prims = 0, cnt_rays = 0;
  for (;;) {
    uint32_t base = 0;
    if (lane == 0u) base = atomicAdd(&wc->trace_head, 32u);
    base = __shfl_sync(0xffffffffu, base, 0);
    if (base >= n) break;
    const uint32_t i = base + lane;
    const bool valid = i < n;
    Ray ray;
    uint32_t lin = 0;
    if (valid) {
      uint32_t x, y, sample;
      camera_pixel_sample(rp, first + i, x, y, sample);
      lin = (y - rp.row_begin) * rp.width + x;
      ray = make_ray(sc.cam_origin, camera_direction(sc, rp, x, y, sample));
      if (COUNT) ++cnt_rays;
    } else {
      ray = make_ray(sc.cam_origin, mk(0.0f, 0.0f, 1.0f));
    }
    float best_t;
    uint32_t best_ref;
    uint32_t cnt = kNone;
    if (cl.count) {  // lane 0 is always valid; a warp whose valid lanes span two pixels keeps the packet walk
      const uint32_t lin0 = __shfl_sync(0xffffffffu, lin, 0);
      if (__all_sync(0xffffffffu, !valid || lin == lin0)) {
        lin = lin0;
        cnt = __ldg(cl.count + lin);
      }
    }
    if (cnt != kNone) cand_trace<COUNT>(sc, cl, lin, cnt, ray, valid, best_t, best_ref, cnt_prims);
    else packet_trace<COUNT>(sc, ray, valid, best_t, best_ref, cnt_nodes, cnt_prims);
    if (valid)
      stg256(pool.ray + 4u * (size_t)i, make_float4(ray.o.x, ray.o.y, ray.o.z, best_ref == kNone ? 0.0f : best_t),
             make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(best_ref == kNone ? kNone : (best_ref & ~PTB_LEAF_BIT))));
  }
  if (COUNT) {
    for (int off = 16; off > 0; off >>= 1) {
      cnt_nodes += __shfl_xor_sync(0xffffffffu, cnt_nodes, off);
      cnt_prims += __shfl_xor_sync(0xffffffffu, cnt_prims, off);
      cnt_rays += __shfl_xor_sync(0xffffffffu, cnt_rays, off);
    }
    if (lane == 0 && cnt_rays) {
      atomicAdd(&wc->nodes_fetched, (unsigned long long)cnt_nodes);
      atomicAdd(&wc->prims_tested, (unsigned long long)cnt_prims);
      atomicAdd(&wc->rays_counted, (unsigned long long)cnt_rays);
    }
  }
}

// ------------------------------------------------------------------------------------------ K10 shade
struct Surface {  // what the integrators read from `hit` + `mat`
  HitRec h;
  uint32_t kind, tex, mat;
  float param;
  bool miss;
};

// ------------------------------------------------------------------------------------------ Trowbridge-Reitz (GGX)
// statistics/bxdfs/trowbridge_reitz.rs:17-24 (d), 62-78 (g2), 80-89 (g1); trowbridge_reitz_vndf.rs:9-15 (vndf),
// 84-113 (sample_vndf, a_x = a_y), 35-52 (sample, pdf); materials/trowbridge_reitz.rs:26-88. Kept out of line: the
// code is only reached for Trowbridge-Reitz surfaces and must not cost the other materials registers.
PTB_DEV float tr_d(float alpha, float cos_theta) {
  if (cos_theta <= 0.0f) return 0.0f;
  const float a_sq = alpha * alpha;
  const float tmp = cos_theta * cos_theta * (a_sq - 1.0f) + 1.0f;
  return a_sq / (kPi * tmp * tmp);
}
PTB_DEV float tr_g1(float alpha, v3 normal, v3 h, v3 v) {
  if (dot(v, h) / dot(v, normal) <= 0.0f) return 0.0f;
  const float c = dot(normal, v);
  const float cos_sq = c * c;
  const float alpha_sq = alpha * alpha;
  const float tmp = alpha_sq + (1.0f - alpha_sq) * cos_sq;
  return 2.0f * c / (sqrtf(tmp) + c);
}
PTB_DEV float tr_g2(float alpha, v3 normal, v3 h, v3 incoming, v3 outgoing) {
  if (dot(incoming, h) / dot(incoming, normal) <= 0.0f || dot(outgoing, h) / dot(outgoing, normal) <= 0.0f) return 0.0f;
  const float alpha_sq = alpha * alpha;
  const float one_minus_alpha_sq = 1.0f - alpha_sq;
  const float cos_i = dot(normal, incoming);
  const float tmp_a = alpha_sq + one_minus_alpha_sq * (cos_i * cos_i);
  const float cos_o = dot(normal, outgoing);
  const float tmp_b = alpha_sq + one_minus_alpha_sq * (cos_o * cos_o);
  return 2.0f * cos_i * cos_o / (cos_o * sqrtf(tmp_a) + cos_i * sqrtf(tmp_b));
}
PTB_DEV void onb_basis(v3 z, v3& x, v3& y) {  // utility/coord.rs:10-22
  if (fabsf(z.x) > fabsf(z.y)) x = mk(-z.z, 0.0f, z.x) / sqrtf(z.x * z.x + z.z * z.z);
  else x = mk(0.0f, z.z, -z.y) / sqrtf(z.y * z.y + z.z * z.z);
  y = cross(x, z);
}
PTB_DEV v3 onb_to_local(v3 x, v3 y, v3 z, v3 v) {  // create_inverse().to_coord(v), coord.rs:23-30
  return v.x * mk(x.x, y.x, z.x) + v.y * mk(x.y, y.y, z.y) + v.z * mk(x.z, y.z, z.z);
}
__device__ __noinline__ float tr_pdf(float alpha, v3 incoming, v3 outgoing, v3 normal) {
  v3 x, y;
  onb_basis(normal, x, y);
  const v3 in = onb_to_local(x, y, normal, incoming), out = onb_to_local(x, y, normal, outgoing);
  v3 h = normalised(out + in);
  if (h.z < 0.0f) h = -h;
  // vndf (h.z >= 0 here)
  const float vndf = tr_g1(alpha, mk(0.0f, 0.0f, 1.0f), h, in) * fmaxf(dot(in, h), 0.0f) * tr_d(alpha, h.z) / in.z;
  return vndf / (4.0f * dot(in, h));
}
__device__ __noinline__ v3 tr_sample(float a, v3 incoming, v3 normal, float u1, float u2) {
  v3 x, y;
  onb_basis(normal, x, y);
  const v3 in = onb_to_local(x, y, normal, incoming);
  const v3 vh = normalised(mk(a * in.x, a * in.y, in.z));
  const float len_sq = vh.x * vh.x + vh.y * vh.y;
  const v3 b2 = len_sq > 0.0f ? mk(-vh.y, vh.x, 0.0f) / sqrtf(len_sq) : mk(1.0f, 0.0f, 0.0f);
  const v3 b3 = cross(vh, b2);
  const float r = sqrtf(u1);
  const float phi = kTau * u2;
  float sphi, cphi;
  sincosf(phi, &sphi, &cphi);
  const float tx = r * cphi;
  float ty = r * sphi;
  const float sh = 0.5f * (1.0f + vh.z);
  ty = (1.0f - sh) * sqrtf(1.0f - tx * tx) + sh * ty;
  const v3 hh = tx * b2 + ty * b3 + sqrtf(fmaxf(1.0f - tx * tx - ty * ty, 0.0f)) * vh;
  const v3 hl = normalised(mk(a * hh.x, a * hh.y, fmaxf(hh.z, 0.0f)));
  const v3 h = hl.x * x + hl.y * y + hl.z * normal;
  return reflected(incoming, h);
}
// eval (which == 0) or eval_over_scattering_pdf (which == 1); wo is the integrator's wo (ray direction, INTO the surface).
// Everything is passed by value: a reference to the kernel's DevScene / Surface would force them into local memory.
struct TrArgs {
  const DevMaterial* m;
  const DevTexture* textures;
  const float* tex_data;
  uint32_t tex;
  float alpha;
  v3 normal, point;
};
__device__ __noinline__ v3 tr_eval_impl(TrArgs s, v3 wo_in, v3 wi, int which) {
  const v3 wo = -wo_in;
  const v3 h = normalised(wi + wo);
  if (dot(wi, s.normal) < 0.0f || dot(h, wo) < 0.0f) return mk(0.0f, 0.0f, 0.0f);
  const DevMaterial* m = s.m;
  const v3 ior = mk(__ldg(&m->ior[0]), __ldg(&m->ior[1]), __ldg(&m->ior[2]));
  const float metallic = __ldg(&m->metallic);
  v3 f0 = vabs((mk(1.0f, 1.0f, 1.0f) - ior) / (mk(1.0f, 1.0f, 1.0f) + ior));
  f0 = f0 * f0;
  f0 = (1.0f - metallic) * f0 + metallic * texture_colour<true>(s.textures, s.tex_data, s.tex, wi, s.point);
  const v3 f = f0 + (mk(1.0f, 1.0f, 1.0f) - f0) * powf(1.0f - dot(wo, h), 5.0f);  // refract.rs:59-61
  const float g = tr_g2(s.alpha, s.normal, h, wo, wi);
  if (which == 0) {
    const float d = tr_d(s.alpha, dot(s.normal, h));
    return f * g * d / (4.0f * fabsf(dot(wo, s.normal)) * dot(wi, s.normal));
  }
  return f * g / tr_g1(s.alpha, s.normal, h, wo);
}
PTB_DEV v3 tr_eval(const DevScene& sc, const Surface& s, v3 wo_in, v3 wi, int which) {
  TrArgs a{sc.materials + s.mat, sc.textures, sc.tex_data, s.tex, s.param, s.h.normal, s.h.point};
  return tr_eval_impl(a, wo_in, wi, which);
}

// rt_core/src/material.rs:20-26 + materials/lambertian.rs:42-47 / reflect.rs:37-39 / refract.rs:51-53
template <bool FULL>
PTB_DEV float mat_scattering_pdf(const Surface& s, v3 wo, v3 wi) {
  if (s.kind == PTB_MAT_LAMBERTIAN) return fmaxf(dot(wi, s.h.normal), 0.0f) / kPi;
  if (FULL && s.kind == PTB_MAT_TROWBRIDGE_REITZ) {  // trowbridge_reitz.rs:51-59
    const float a = tr_pdf(s.param, -wo, wi, s.h.normal);
    return a == 0.0f ? __int_as_float(0x7f800000) : a;
  }
  return 0.0f;  // Reflect / Refract keep the trait default (quirk Q4)
}
template <bool FULL>
PTB_DEV v3 mat_eval(const DevScene& sc, const Surface& s, v3 wo, v3 wi) {
  if (FULL && s.kind == PTB_MAT_TROWBRIDGE_REITZ) return tr_eval(sc, s, wo, wi, 0);
  const v3 col = texture_colour<FULL>(sc, s.tex, wo, s.h.point);
  if (s.kind == PTB_MAT_LAMBERTIAN) return col * s.param * fmaxf(dot(s.h.normal, wi), 0.0f) / kPi;
  return col;
}

// Adds the radiance of the paths that finished in this warp iteration to the accumulator. Called by all 32 lanes.
// The samples of a pixel are issued back to back, so the finishing lanes of a warp usually share ONE pixel: their sum
// is formed with shuffles and added with three atomics instead of 3 x 32 same-address ones.
PTB_DEV void finish_paths(float* __restrict__ accum, bool contributes, uint32_t pixel, v3 L) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t m = __ballot_sync(0xffffffffu, contributes);
  if (!m) return;
  const uint32_t peers = __match_any_sync(0xffffffffu, contributes ? pixel : 0xffffffffu);
  if (__all_sync(0xffffffffu, !contributes || peers == m)) {
    if (!contributes) L = mk(0.0f, 0.0f, 0.0f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      L.x += __shfl_xor_sync(0xffffffffu, L.x, o);
      L.y += __shfl_xor_sync(0xffffffffu, L.y, o);
      L.z += __shfl_xor_sync(0xffffffffu, L.z, o);
    }
    if (lane == (uint32_t)__ffs(m) - 1u) {
      atomicAdd(accum + 3u * (size_t)pixel + 0, L.x);
      atomicAdd(accum + 3u * (size_t)pixel + 1, L.y);
      atomicAdd(accum + 3u * (size_t)pixel + 2, L.z);
    }
  } else if (contributes) {
    atomicAdd(accum + 3u * (size_t)pixel + 0, L.x);
    atomicAdd(accum + 3u * (size_t)pixel + 1, L.y);
    atomicAdd(accum + 3u * (size_t)pixel + 2, L.z);
  }
}

// Direction bin of a unit vector. Window-mode k_shade leaves it per slot and k_win_fill orders the live rays of a window
// by it, so the 32 consecutive rays a k_trace warp fetches start in the same few pixels AND point the same way.
//   5 bits: octant (signs) x dominant axis;
//   8 bits: 16 x 16 cells of the octahedral map (|x|+|y|+|z| = 1 unfolded onto the square), cell index in Morton
//           order so that neighbouring bins are neighbouring directions; bin 255 is reserved for finished paths.
PTB_DEV uint32_t direction_bin(v3 d) {
#if PTB_DIR_BITS == 5
  const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
  const uint32_t major = ax >= ay ? (ax >= az ? 0u : 2u) : (ay >= az ? 1u : 2u);
  return ((d.x < 0.0f ? 4u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 1u : 0u)) * 4u + major;
#else
  const float inv = 1.0f / (fabsf(d.x) + fabsf(d.y) + fabsf(d.z));
  float u = d.x * inv, v = d.y * inv;
  if (d.z < 0.0f) {
    const float fu = (1.0f - fabsf(v)) * (u < 0.0f ? -1.0f : 1.0f), fv = (1.0f - fabsf(u)) * (v < 0.0f ? -1.0f : 1.0f);
    u = fu;
    v = fv;
  }
  const uint32_t iu = (uint32_t)fminf(fmaxf((u * 0.5f + 0.5f) * 16.0f, 0.0f), 15.0f);
  const uint32_t iv = (uint32_t)fminf(fmaxf((v * 0.5f + 0.5f) * 16.0f, 0.0f), 15.0f);
  uint32_t m = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b) m |= (((iu >> b) & 1u) << (2 * b + 1)) | (((iv >> b) & 1u) << (2 * b));
  return m < 255u ? m : 254u;
#endif
}

// One path, one bounce: everything the integrators do between two check_hit calls (emission, MIS weights, NEE sample, BSDF
// sample, Russian roulette, termination). Reads the path's records (ray + hit, colour) from the pool and writes the
// continuing path's records back; what the caller has to route (direction bin, accumulator, shadow ray) comes back in `o`.
// Shared by the wavefront kernel k_shade and the fused tail kernel k_tail.
struct ShadeOut {
  bool alive = false;       // path continues: its next ray is in the slot's ray record
  bool finished = false;    // path ended: the slot is marked dead
  bool shadow = false;      // an NEE ray was produced
  bool contributes = false; // finished with a radiance that passes the NaN test (integrators/mod.rs:74-76, mis.rs:88-90)
  uint32_t shadow_is_sky = 0, fin_pixel = 0;
  uint32_t bin = 0;         // direction bin of the continuing ray
  float4 sh_o, sh_d, sh_c;  // NEE ray: o.xyz|tmax, d.xyz|exclude slot, contribution.rgb|path slot
  v3 fin_L;
};
// Next-event estimation of one departing path (integrators/mis.rs:36-43, 95-157): one light or the sky, sampled, its
// shadow ray and weighted contribution left in `o`. Out of line (PTB_NEE_NOINLINE): its sampling code — sky tables, cone
// sampling, the light's own hit record, two Philox blocks — then holds registers only while it runs.
#ifndef PTB_NEE_NOINLINE
#define PTB_NEE_NOINLINE 0
#endif
#if PTB_NEE_NOINLINE
#define PTB_NEE_ATTR __device__ __noinline__
#else
#define PTB_NEE_ATTR PTB_DEV
#endif
template <bool FULL>
PTB_NEE_ATTR void nee_sample(const DevScene& sc, const RenderParams& rp, const Surface& s, v3 wo, v3 T, uint32_t pixel, uint32_t sample,
                             uint32_t depth, uint32_t slot, ShadeOut& o) {
  bool& shadow = o.shadow;
  uint32_t& shadow_is_sky = o.shadow_is_sky;
  float4 &sh_o = o.sh_o, &sh_d = o.sh_d, &sh_c = o.sh_c;
    const uint32_t n_l = sc.n_lights;
    const bool sky_s = (sc.sky_rx | sc.sky_ry) != 0u;
    if (n_l != 0u || sky_s) {
      const uint4 r = philox4x32_10(pixel, sample, (depth << 8) | RNG_NEE, 0u, rp.k0, rp.k1);
      bool do_sky;
      float mult;
      uint32_t li = 0;
      if (n_l == 0u) { do_sky = true; mult = 1.0f; }
      else if (!sky_s) { do_sky = false; mult = 1.0f / (float)n_l; li = rng_below(r.x, n_l); }
      else { mult = 1.0f / (float)(n_l + 1u); li = rng_below(r.x, n_l + 1u); do_sky = li == n_l; }
      const v3 so = s.h.point + 0.0001f * s.h.normal;  // mis.rs:106,124
      v3 l_wi, le;
      float l_pdf = 0.0f, tmax = __int_as_float(0x7f800000);
      uint32_t exclude = kNone;
      bool usable = false;
      if (do_sky) {
        const uint4 r2 = philox4x32_10(pixel, sample, (depth << 8) | RNG_NEE, 1u, rp.k0, rp.k1);
        l_wi = sky_sample(sc, u32_to_unit(r.y), u32_to_unit(r.z), u32_to_unit(r.w), u32_to_unit(r2.x));
        const v3 point = offset_ray(s.h.point, s.h.normal, s.h.error, true);
        le = 1.0f * texture_colour<FULL>(sc, sc.sky_tex, l_wi, point);
        l_pdf = sky_pdf(sc, l_wi) * mult;
        usable = true;
        shadow_is_sky = 1u;
      } else {
        const uint32_t lref = __ldg(sc.lights + li);
        l_wi = light_sample_dir(sc, lref, s.h.point, u32_to_unit(r.y), u32_to_unit(r.z));
        const Ray sray = make_ray_from_raw(so, l_wi);
        HitRec si;
        if (prim_hit(sc, sray, lref, si) && si.t > 0.0f) {  // acceleration/mod.rs:231-243
          const float pdf = light_pdf(sc, lref, s.h.point, l_wi, si.point, si.normal);
          if (pdf > 0.0f) {
            const uint32_t lmi = __ldg(sc.slot_mat + (lref & kSlotMask)) & 0x00FFFFFFu;
            const DevMaterial* lm = sc.materials + lmi;
            const v3 lpoint = offset_ray(si.point, si.normal, si.error, true);
            le = __ldg(&lm->param) * texture_colour<FULL>(sc, __ldg(&lm->tex), l_wi, lpoint);
            l_pdf = pdf * mult;
            tmax = si.t;
            exclude = lref & kSlotMask;
            usable = true;
          }
        }
      }
      if (usable) {
        const float mp = mat_scattering_pdf<FULL>(s, wo, l_wi);
        const float w = power_heuristic(l_pdf, mp);
        const v3 contrib = T * mat_eval<FULL>(sc, s, wo, l_wi) * w * le / l_pdf;  // mis.rs:42
        const v3 sd = l_wi / mag(l_wi);  // Ray::new normalises (ray.rs:14)
        sh_o = make_float4(so.x, so.y, so.z, tmax);
        sh_d = make_float4(sd.x, sd.y, sd.z, __uint_as_float(exclude));
        sh_c = make_float4(contrib.x, contrib.y, contrib.z, __uint_as_float(slot));
        shadow = true;
      }
    }
}

template <int METHOD, bool FULL>
PTB_DEV void shade_path(const DevScene& sc, const PathPool& pool, const RenderParams& rp, uint32_t slot, bool depth0,
                        unsigned long long camera_first, ShadeOut& o) {
  bool &alive = o.alive, &finished = o.finished, &shadow = o.shadow, &contributes = o.contributes;
  uint32_t &shadow_is_sky = o.shadow_is_sky, &fin_pixel = o.fin_pixel;
  float4 &sh_o = o.sh_o, &sh_d = o.sh_d, &sh_c = o.sh_c;
  v3& fin_L = o.fin_L;
  float4 ro, rd, th, ra;
  ldg256_rw(pool.ray + 4u * (size_t)slot, ro, rd);
  if (depth0) {
    uint32_t x, y, smp;
    camera_pixel_sample(rp, camera_first + slot, x, y, smp);
    th = make_float4(1.0f, 1.0f, 1.0f, __uint_as_float(y * rp.width + x));
    ra = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(smp << 9));
  } else {
    ldg256_rw(pool.col + 4u * (size_t)slot, th, ra);
  }
  const uint2 ht = make_uint2(__float_as_uint(ro.w), __float_as_uint(rd.w));
  const uint32_t pixel = __float_as_uint(th.w);
  const uint32_t df = __float_as_uint(ra.w);
  const uint32_t sample = df >> 9;
  uint32_t depth = df & 0xFFu;
  const bool prev_delta = (df & kFlagPrevDelta) != 0u;
  const Ray ray = make_ray(from4(ro), from4(rd));
  const v3 wo = ray.d;
  v3 T = from4(th), L = from4(ra);

  Surface s;
  s.miss = ht.y == kNone;
  if (s.miss) {  // sky.rs:79-91: zero Hit + Emit(sky texture, 1.0)
    s.h.t = 0.0f;
    s.h.point = s.h.error = s.h.normal = mk(0.0f, 0.0f, 0.0f);
    s.h.out = false;
    s.kind = PTB_MAT_EMIT;
    s.tex = sc.sky_tex;
    s.mat = 0u;
    s.param = 1.0f;
  } else {
    prim_hit(sc, ray, ht.y, s.h);  // same arithmetic as the traversal: reproduces t, adds point/normal/error/out
    const uint32_t mi = __ldg(sc.slot_mat + (ht.y & kSlotMask)) & 0x00FFFFFFu;
    const DevMaterial* m = sc.materials + mi;
    s.mat = mi;
    s.kind = __ldg(&m->kind);
    s.tex = __ldg(&m->tex);
    s.param = __ldg(&m->param);
  }
  const bool is_emit = s.kind == PTB_MAT_EMIT;
  bool depart = false;
  bool nan_check = true;

  if (METHOD == PTB_METHOD_NAIVE) {
    // integrators/mod.rs:29-72
    if (is_emit) {
      const v3 point = offset_ray(s.h.point, s.h.normal, s.h.error, true);        // emissive.rs:23-26
      const v3 emission = s.param * texture_colour<FULL>(sc, s.tex, wo, point);
      L = L + T * emission;  // depth 0: throughput is exactly (1,1,1)
      finished = true;
    } else {
      depart = true;
    }
  } else {
    // integrators/mis.rs:17-31 (first hit) and :52-80 (after each bounce)
    if (depth == 0u) {
      if (is_emit) {
        const v3 point = offset_ray(s.h.point, s.h.normal, s.h.error, true);
        L = L + s.param * texture_colour<FULL>(sc, s.tex, wo, point);
        finished = true;
        nan_check = false;  // mis.rs:29-31 returns before the NaN test
      } else {
        depth = 1u;
        depart = true;
      }
    } else {
      if (is_emit) {
        // mis.rs:55: emission of the NEW material evaluated with the PREVIOUS hit record (quirk Q6); the
        // previous hit's offset point is this ray's origin (lambertian.rs:37, reflect.rs:29)
        const v3 le = s.param * texture_colour<FULL>(sc, s.tex, wo, ray.o);
        if (!is_zero(le)) {
          const bool sky_samplable = (sc.sky_rx | sc.sky_ry) != 0u;
          const bool use_mis = s.miss ? sky_samplable : !prev_delta;  // mis.rs:57-60 (an emissive prim is in `lights`)
          if (use_mis) {
            const float divisor = (float)(sky_samplable ? sc.n_lights + 1u : sc.n_lights);  // acceleration/mod.rs:299-318
            const float4 pv = pool.prev[slot];  // previous hit point | m_pdf of the BSDF sample that got us here
            const float l_pdf = s.miss ? sky_pdf(sc, wo) / divisor
                                       : light_pdf(sc, ht.y, from4(pv), wo, s.h.point, s.h.normal) / divisor;
            const float w = power_heuristic(pv.w, l_pdf);
            L = L + T * le * w;
          } else {
            L = L + T * le;
          }
        }
        finished = true;  // mis.rs:69-71
      } else {
        bool survive = true;
        if (depth > rp.rr_threshold) {  // mis.rs:73-80
          const float p = cmax3(T.x, T.y, T.z);
          const uint4 r = philox4x32_10(pixel, sample, (depth << 8) | RNG_RR, 0u, rp.k0, rp.k1);
          if (u32_to_unit(r.x) > p) survive = false;
          else T = T / p;
        }
        depth += 1u;
        if (survive && depth < rp.max_depth) depart = true;
        else finished = true;
      }
    }
  }

  if (depart) {
    float m_pdf = 0.0f;
    // ---- next-event estimation (MIS only): integrators/mis.rs:36-43, 95-157
    if (METHOD == PTB_METHOD_MIS) nee_sample<FULL>(sc, rp, s, wo, T, pixel, sample, depth, slot, o);
    // ---- BSDF sample -> next ray
    const uint4 r = philox4x32_10(pixel, sample, (depth << 8) | RNG_SCATTER, 0u, rp.k0, rp.k1);
    v3 new_o, new_dir;
    bool delta = false;
    if (s.kind == PTB_MAT_LAMBERTIAN) {
      new_dir = lambertian_sample_dir(s.h.normal, u32_to_unit(r.x), u32_to_unit(r.y));
      new_o = offset_ray(s.h.point, s.h.normal, s.h.error, true);
    } else if (FULL && s.kind == PTB_MAT_TROWBRIDGE_REITZ) {
      // trowbridge_reitz.rs:38-50: VNDF sample about the normal, draws (r, phi) = (sqrt(u1), tau * u2)
      new_dir = tr_sample(s.param, -wo, s.h.normal, u32_to_unit(r.x), u32_to_unit(r.y));
      new_o = offset_ray(s.h.point, s.h.normal, s.h.error, true);
    } else if (s.kind == PTB_MAT_REFLECT) {
      // reflect.rs:26-36
      const v3 unit = uniform_sphere_dir(u32_to_unit(r.x), u32_to_unit(r.y));
      new_dir = reflected(-wo, s.h.normal) + s.param * unit;
      new_o = offset_ray(s.h.point, s.h.normal, s.h.error, true);
      delta = true;
    } else {  // PTB_MAT_REFRACT — refract.rs:27-50
      float eta_fraction = 1.0f / s.param;
      if (!s.h.out) eta_fraction = s.param;
      const float cos_theta = fminf(dot(-wo, s.h.normal), 1.0f);
      const float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
      const bool cannot_refract = eta_fraction * sin_theta > 1.0f;
      float f0 = (1.0f - eta_fraction) / (1.0f + eta_fraction);
      f0 = f0 * f0 * 1.0f;
      const float fres = f0 + (1.0f - f0) * powf(1.0f - cos_theta, 5.0f);  // refract.rs:59-61
      if (cannot_refract || fres > u32_to_unit(r.x)) {
        new_dir = reflected(-wo, s.h.normal);  // Reflect{fuzz: 0}: the unit vector is multiplied by 0
        new_o = offset_ray(s.h.point, s.h.normal, s.h.error, true);
      } else {
        const v3 perp = eta_fraction * (wo + cos_theta * s.h.normal);
        const v3 para = -1.0f * sqrtf(fabsf(1.0f - mag_sq(perp))) * s.h.normal;
        new_dir = perp + para;
        new_o = offset_ray(s.h.point, s.h.normal, s.h.error, false);
      }
      delta = true;
    }
    const v3 nd = new_dir / mag(new_dir);  // Ray::new
    const bool is_tr = FULL && s.kind == PTB_MAT_TROWBRIDGE_REITZ;
    const v3 col = is_tr ? tr_eval(sc, s, wo, nd, 1) : texture_colour<FULL>(sc, s.tex, wo, s.h.point);
    if (METHOD == PTB_METHOD_NAIVE) {
      // integrators/mod.rs:57-70
      if (s.kind == PTB_MAT_LAMBERTIAN) T = T * (col * s.param);
      else T = T * col;  // Trowbridge-Reitz: col is already eval_over_scattering_pdf
      bool survive = true;
      if (depth > rp.rr_threshold) {
        const float p = cmax3(T.x, T.y, T.z);
        const uint4 r3 = philox4x32_10(pixel, sample, (depth << 8) | RNG_RR, 0u, rp.k0, rp.k1);
        if (u32_to_unit(r3.x) > p) survive = false;
        else T = T / p;
      }
      depth += 1u;
      if (survive && depth < rp.max_depth) alive = true;
      else finished = true;
    } else {
      // mis.rs:54-56: m_pdf and throughput use the previous hit only, so they are folded in at departure
      if (s.kind == PTB_MAT_LAMBERTIAN) {
        m_pdf = fmaxf(dot(nd, s.h.normal), 0.0f) / kPi;
        T = T * (col * s.param);
      } else if (is_tr) {
        m_pdf = mat_scattering_pdf<FULL>(s, wo, nd);
        T = T * col;
      } else {
        m_pdf = 0.0f;
        T = T * (col / 0.0f);  // eval / scattering_pdf with the default pdf 0 (quirk Q4)
      }
      pool.prev[slot] = make_float4(s.h.point.x, s.h.point.y, s.h.point.z, m_pdf);
      alive = true;
    }
    if (alive) {
      stg256(pool.ray + 4u * (size_t)slot, make_float4(new_o.x, new_o.y, new_o.z, 0.0f),
             make_float4(nd.x, nd.y, nd.z, __uint_as_float(kNone)));
      stg256(pool.col + 4u * (size_t)slot, make_float4(T.x, T.y, T.z, th.w),
             make_float4(L.x, L.y, L.z, __uint_as_float((sample << 9) | (delta ? kFlagPrevDelta : 0u) | depth)));
      o.bin = rp.dir_bins ? direction_bin(nd) : 0u;
    }
  }
  if (finished) {
    contributes = !(nan_check && (contains_nan(L) || !any_finite(L)));
    fin_pixel = pixel;
    fin_L = L;
  }
}

// Ordered live-slot queue in, per-slot direction bin and per-window live count out.
// MIS shades at one block more per SM than naive (48 registers): rtweekend1 4K 9133 -> 9179 Mrays/s, C3 (naive) would lose 2 %
template <int METHOD, bool FULL>
__global__ void __launch_bounds__(256, PTB_SHADE_MIN_BLOCKS + (METHOD == PTB_METHOD_MIS ? 1 : 0))
k_shade(DevScene sc, PathPool pool, Queues q, WaveCounters* wc, RenderParams rp, float* __restrict__ accum,
        unsigned long long camera_first, uint32_t sort_kinds) {
  // first iteration of a chunk (camera_first != kNoCamera): work item i is slot i, every slot is live and its colour
  // record is the camera path's initial state, derived from the path index instead of read from memory
  const bool depth0 = camera_first != kNoCamera;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t n_total = wc->n_trace;
  // grid-stride over the ordered live-slot queue; whole blocks iterate together (ballots below)
  for (uint32_t base = blockIdx.x * blockDim.x; base < n_total; base += gridDim.x * blockDim.x) {
  const uint32_t i = base + threadIdx.x;
  bool active = i < n_total;

  uint32_t slot = 0;
  ShadeOut so;
  so.fin_L = mk(0.0f, 0.0f, 0.0f);

  if (active) slot = depth0 ? i : q.live[i];
  if (sort_kinds) {
    // The window wavefront orders a window's rays by direction, so the hits a block shades arrive with their materials mixed. A
    // scene with more than two material kinds (sort_kinds, decided at commit) has its block's work items counting-sorted
    // by the kind of the surface hit (0 = sky, 1 + PTB_MAT_*) before they are shaded: warps then run one material's code
    // instead of all of them one after the other. Costs one extra 16-byte read per path (the hit reference) and two
    // block barriers; scenes with one or two kinds (C1 - C5) skip it.
    __shared__ uint32_t s_slot[256];
    __shared__ uint32_t s_cnt[(kNumKinds + 1) * 8];  // [kind][warp], kind kNumKinds = no work item
    const uint32_t warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    uint32_t kind = (uint32_t)kNumKinds;
    if (active) {
      const uint32_t ref = __float_as_uint(pool.ray[4u * (size_t)slot + 1u].w);
      kind = ref == kNone ? 0u : 1u + (__ldg(sc.slot_mat + (ref & kSlotMask)) >> 24);
    }
    uint32_t rank = 0;
#pragma unroll
    for (uint32_t k = 0; k <= (uint32_t)kNumKinds; ++k) {
      const uint32_t m = __ballot_sync(0xffffffffu, kind == k);
      if (kind == k) rank = (uint32_t)__popc(m & ((1u << lane) - 1u));
      if (lane == 0u) s_cnt[k * 8u + warp] = (uint32_t)__popc(m);
    }
    __syncthreads();
    uint32_t pos = rank;
    for (uint32_t e = 0; e < kind * 8u + warp; ++e)
      if ((e & 7u) < n_warps) pos += s_cnt[e];
    s_slot[pos] = slot;
    __syncthreads();
    uint32_t n_here = 0;
    for (uint32_t e = 0; e < (uint32_t)kNumKinds * 8u; ++e)
      if ((e & 7u) < n_warps) n_here += s_cnt[e];
    active = threadIdx.x < n_here;
    slot = s_slot[threadIdx.x];
    __syncthreads();  // the tables are reused by the block's next batch
  }
  if (active) shade_path<METHOD, FULL>(sc, pool, rp, slot, depth0, camera_first, so);
  finish_paths(accum, so.contributes, so.fin_pixel, so.fin_L);

  // Paths stay in their slot. A finished path is marked dead and leaves its window's live count (lanes of a warp nearly
  // always share the window: one atomic per warp); NEE rays go to the shadow queue.
  if (so.alive) q.bin[slot] = (uint8_t)so.bin;
  if (so.finished) q.bin[slot] = (uint8_t)kBinDead;
  const uint32_t window = slot / kWindow;
  const uint32_t peers = __match_any_sync(0xffffffffu, so.finished ? window : 0xffffffffu);
  if (so.finished && lane == (uint32_t)__ffs(peers) - 1u) atomicSub(&q.win_count[window], (uint32_t)__popc(peers));
  if (METHOD == PTB_METHOD_MIS) {
    const uint32_t m_sh = __ballot_sync(0xffffffffu, so.shadow), m_sky = __ballot_sync(0xffffffffu, so.shadow && so.shadow_is_sky);
    unsigned long long p2 = 0ull;
    if (lane == 0u && m_sh)
      p2 = atomicAdd(&wc->shadow_pair, ((unsigned long long)__popc(m_sky) << 32) | (unsigned long long)__popc(m_sh));
    p2 = __shfl_sync(0xffffffffu, p2, 0);
    if (so.shadow) {
      float4* e = q.shadow + 3u * (size_t)((uint32_t)p2 + __popc(m_sh & ((1u << lane) - 1u)));
      e[0] = so.sh_o;
      e[1] = so.sh_d;
      e[2] = so.sh_c;
    }
  }
  }  // grid-stride
}

// ------------------------------------------------------------------------------------------ window wavefront
// Every camera path of a chunk is resident, so the wavefront needs no free list and no compaction of scattered slots:
// path g of the chunk lives in slot g for its whole life (pixel-major, the samples of a pixel adjacent), and each
// iteration's trace queue is rebuilt IN SLOT ORDER from per-slot state: k_shade leaves a direction bin (or "dead") per
// slot and keeps a live count per 4096-slot window; a prefix sum over the window counts places every window's live slots
// in the queue, ordered by direction bin inside the window. Consequences, all measured (profiles/r1_sweeps.md): the rays a
// k_trace warp fetches share a pixel (origin) and roughly a direction at every depth, path records are gathered from one
// 256 KB window at a time instead of from the whole pool, and iteration k holds exactly the rays of bounce k.
//   k_win_init       window counts of a fresh chunk (its camera rays are computed by the first k_trace itself)
//   k_win_scan       per 4096-window segment: exclusive prefix of the counts + segment total
//   k_win_prepare    1 warp: statistics of the finished iteration, total of live paths, cursor resets
//   k_win_fill       ordered live-slot queue (one block per window: counting sort of its live slots by direction bin)
__global__ void __launch_bounds__(256) k_win_init(Queues q, WaveCounters* wc, uint32_t n_paths) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w == 0u) {
    wc->mode = 0u; wc->n_tail = 0u; wc->tail_iter = 0xFFFFFFFFu; wc->n_trace = 0u; wc->tail_head = 0u;
    if (wc->tail_t0 != ~0ull && wc->tail_t1 > wc->tail_t0) wc->tail_ns += wc->tail_t1 - wc->tail_t0;  // the slot's previous hand-over
    wc->tail_t0 = ~0ull;
    wc->tail_t1 = 0ull;
  }
  if (w < q.n_windows) {
    const unsigned long long first = (unsigned long long)w * kWindow;
    q.win_count[w] = first >= n_paths ? 0u : (n_paths - first < kWindow ? (uint32_t)(n_paths - first) : kWindow);
  }
}

__global__ void __launch_bounds__(1024) k_win_scan(Queues q) {
  __shared__ uint32_t warp_sum[32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t w0 = blockIdx.x * kSegWindows + threadIdx.x * 4u;
  uint32_t c[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) c[k] = w0 + k < q.n_windows ? q.win_count[w0 + k] : 0u;
  const uint32_t mine = c[0] + c[1] + c[2] + c[3];
  uint32_t inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += t;
  }
  if (lane == 31u) warp_sum[warp] = inc;
  __syncthreads();
  if (warp == 0u) {
    const uint32_t v = warp_sum[lane];
    uint32_t winc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= (uint32_t)o) winc += t;
    }
    warp_sum[lane] = winc - v;
    if (lane == 31u) q.seg_total[blockIdx.x] = winc;
  }
  __syncthreads();
  uint32_t run = warp_sum[warp] + inc - mine;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (w0 + k < q.n_windows) q.win_prefix[w0 + k] = run;
    run += c[k];
  }
}

// `prev` = what the finished iteration traced: 0 nothing (first of a chunk), 1 camera rays, 2 bounce rays.
// Also the chunk's state machine (WaveCounters::mode): from iteration 2 on, a chunk with at most `tail_paths` live paths is
// handed to k_tail (mode 1 for this iteration, 3 afterwards); with no live path left it is finished (2). The wavefront
// kernels of an iteration in any state but 0 find n_trace == 0, so the host may enqueue iterations without waiting.
__global__ void k_win_prepare(WaveCounters* wc, Queues q, uint32_t n_segments, uint32_t method, uint32_t prev, uint32_t depth,
                              uint32_t tail_paths) {
#ifdef PTB_DRAIN_STATS
  if (threadIdx.x == 0u && g_drain[0] != ~0ull && g_drain[2] != ~0ull) {  // fold the previous persistent launch
    if (g_drain[1] > g_drain[0]) g_drain[3] += g_drain[1] - g_drain[0];
    if (g_drain[1] > g_drain[2]) g_drain[4] += g_drain[1] - g_drain[2];
    if (g_drain[1] > g_drain[2] + 200000ull) g_drain[5] += 1ull;  // launches longer than 0.2 ms
    g_drain[0] = ~0ull; g_drain[1] = 0ull; g_drain[2] = ~0ull;
  }
#endif
  const uint32_t lane = threadIdx.x;
  uint32_t total = 0;
  for (uint32_t s = lane; s < n_segments; s += 32u) total += q.seg_total[s];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
  if (lane != 0u) return;
  uint32_t mode = wc->mode;
  if (prev && mode == 0u) {
    const uint32_t traced = wc->n_trace, survivors = total;
    const unsigned long long sp = wc->shadow_pair;
    wc->rays_shadow_sky += sp >> 32;
    wc->rays_shadow_light += (uint32_t)sp - (uint32_t)(sp >> 32);
    if (prev == 1u) wc->rays_camera += traced;
    else wc->rays_bounce += traced;
    wc->rays_reference += method == PTB_METHOD_NAIVE ? traced : survivors;  // Q7: naive 1/check_hit, MIS 1/bounce iteration
    wc->paths += traced - survivors;
  }
  if (mode == 0u) {
    if (total == 0u) mode = 2u;
    else if (depth >= 2u && total <= tail_paths) { mode = 1u; wc->n_tail = total; wc->tail_iter = depth; }
  } else if (mode == 1u) {
    mode = 3u;  // n_tail / tail_iter stay: the k_tail launch of the hand-over iteration may not have started yet
  }
  wc->mode = mode;
  wc->n_trace = mode == 0u ? total : 0u;
  wc->shadow_pair = 0;
  wc->trace_head = wc->shadow_head = 0;
}

constexpr uint32_t kFillGroup = 8u;  // windows whose live counts a k_win_fill block fetches (and skips) together
__global__ void __launch_bounds__(256) k_win_fill(Queues q, WaveCounters* wc) {
  __shared__ uint32_t s_cnt[kFillGroup];
  __shared__ uint32_t s_hist[2][256];  // per direction bin: count, then running output offset (double-buffered)
  __shared__ uint32_t s_warp[8];
  __shared__ uint32_t s_seg_base;
  const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const uint32_t n_groups = (q.n_windows + kFillGroup - 1u) / kFillGroup;
  if (wc->mode > 1u) return;  // chunk finished or handed over earlier: the live list must stay as the tail reads it
  uint32_t seg_cached = 0xffffffffu, buf = 0;
  s_hist[0][tid] = 0u;
  for (uint32_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
    const uint32_t wmine = g * kFillGroup + tid;
    const uint32_t cmine = tid < kFillGroup && wmine < q.n_windows ? q.win_count[wmine] : 0u;
    __syncthreads();  // the previous group's readers of s_cnt are done; s_hist[buf] is zero and visible
    if (tid < kFillGroup) s_cnt[tid] = cmine;
    if (!__syncthreads_or(cmine != 0u)) continue;
    for (uint32_t j = 0; j < kFillGroup; ++j) {
      const uint32_t cnt = s_cnt[j];
      if (cnt == 0u) continue;  // uniform
      const uint32_t w = g * kFillGroup + j;
      const uint32_t seg = w / kSegWindows;
      if (seg != seg_cached) {  // uniform, rare: base of the segment = live paths of all earlier segments
        uint32_t b = 0;
        for (uint32_t sgi = tid; sgi < seg; sgi += 256u) b += q.seg_total[sgi];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
        __syncthreads();
        if (lane == 0u) s_warp[warp] = b;
        __syncthreads();
        if (tid == 0u) {
          uint32_t t = 0;
          for (int k = 0; k < 8; ++k) t += s_warp[k];
          s_seg_base = t;
        }
        __syncthreads();
        seg_cached = seg;
      }
      const uint32_t out = s_seg_base + q.win_prefix[w];
      const uint32_t first_slot = w * kWindow;
      uint32_t* hist = s_hist[buf];
      // this thread's kWinItems consecutive slots: their bins, and (from the returning atomic) their place inside the bin
      uint32_t bins[kWinItems], offs[kWinItems];
      {
        const uint8_t* src = q.bin + first_slot + tid * kWinItems;
        if (kWinItems == 16) {
          const uint4 raw = *reinterpret_cast<const uint4*>(src);
          const uint32_t r4[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
          for (uint32_t k = 0; k < kWinItems; ++k) bins[k] = (r4[(k >> 2) & 3u] >> (8u * (k & 3u))) & 0xFFu;
        } else {
#pragma unroll
          for (uint32_t k = 0; k < kWinItems; ++k) bins[k] = src[k];
        }
      }
#pragma unroll
      for (uint32_t k = 0; k < kWinItems; ++k) offs[k] = bins[k] != kBinDead ? atomicAdd(&hist[bins[k]], 1u) : 0u;
      __syncthreads();
      {  // exclusive scan over the 256 bins; the other buffer is cleared for the next window meanwhile
        const uint32_t c = hist[tid];
        uint32_t inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= (uint32_t)o) inc += t;
        }
        if (lane == 31u) s_warp[warp] = inc;
        s_hist[buf ^ 1u][tid] = 0u;
        __syncthreads();
        uint32_t before = 0;
#pragma unroll
        for (uint32_t k = 0; k < 8u; ++k) before += k < warp ? s_warp[k] : 0u;
        hist[tid] = out + before + inc - c;
      }
      __syncthreads();
#pragma unroll
      for (uint32_t k = 0; k < kWinItems; ++k)
        if (bins[k] != kBinDead) q.live[hist[bins[k]] + offs[k]] = first_slot + tid * kWinItems + k;
      buf ^= 1u;
    }
  }
}

// ------------------------------------------------------------------------------------------ K9 shadow rays
struct ShadowFetch {
  const Queues& q;
  float4 contrib;  // rgb | path slot
  PTB_DEV void operator()(uint32_t i, Ray& ray, float& tmax, uint32_t& exclude) {
    const float4* e = q.shadow + 3u * (size_t)i;
    const float4 o = e[0], d = e[1];
    contrib = e[2];
    ray = make_ray(from4(o), from4(d));
    tmax = o.w;
    exclude = __float_as_uint(d.w);
  }
};
struct ShadowRetire {
  const PathPool& pool;
  const ShadowFetch& f;
  PTB_DEV void operator()(bool fin, const TraceResult& tr, const Ray&) {
    if (fin && tr.ref == kNone) {  // unoccluded
      const uint32_t slot = __float_as_uint(f.contrib.w);
      float4 ra = pool.col[4u * (size_t)slot + 1u];
      ra.x += f.contrib.x; ra.y += f.contrib.y; ra.z += f.contrib.z;  // output += throughput*eval*mis*le/l_pdf (mis.rs:42)
      pool.col[4u * (size_t)slot + 1u] = ra;
    }
  }
};
// same-run A/B (profiles/r1_sweeps.md): k_closest_hit_api at 6 blocks / SM (40 registers) C5 4116 -> 4816 Mrays/s; k_shadow
// prefers its unconstrained 63 registers (rtweekend1 4K: 10 ms vs 13 - 14 ms of shadow per 3 steps)
#ifndef PTB_SHADOW_MIN_BLOCKS
#define PTB_SHADOW_MIN_BLOCKS 1
#endif
template <class TR>
__global__ void __launch_bounds__(256, PTB_SHADOW_MIN_BLOCKS) k_shadow(DevScene sc, PathPool pool, Queues q, WaveCounters* wc) {
  uint32_t a = 0, b = 0, r = 0;
  ShadowFetch fetch{q, make_float4(0.f, 0.f, 0.f, 0.f)};
  ShadowRetire retire{pool, fetch};
  persistent_trace<TR, true, false>(sc, (uint32_t)wc->shadow_pair, &wc->shadow_head, fetch, retire, a, b, r);
}

// ------------------------------------------------------------------------------------------ fused tail
// The last few thousand paths of a chunk (glass paths bouncing up to max_depth times) used to cost ~45 wavefront iterations
// of five dependent, nearly empty launches each: 5 - 8 ms per chunk whatever its size. k_tail finishes them in ONE launch:
// a lane owns a path and alternates closest hit -> shade (-> NEE any-hit) until the path ends — the paths are independent,
// so nothing synchronises; the launch is latency bound (one traversal after the other per lane) and runs on a side stream
// underneath the next chunk's wide iterations. Same functions, same records, same RNG counters as the wavefront: the image
// does not depend on where the hand-over happens (tests: PTB_TAIL_PATHS=0 disables it).
PTB_DEV unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// One bounce of the path in `slot` whose closest hit `tr` has just been found: the hit goes into the ray record, where
// shade_path reads it; then the shading step of k_shade. Returns the shading outcome; the NEE visibility test (MIS) is the
// caller's (a lane walk or a cooperative walk).
template <int METHOD, bool FULL>
PTB_DEV void tail_shade(const DevScene& sc, const PathPool& pool, const RenderParams& rp, uint32_t slot, const Ray& ray,
                        const TraceResult& tr, ShadeOut& so) {
  stg256(pool.ray + 4u * (size_t)slot, make_float4(ray.o.x, ray.o.y, ray.o.z, tr.t),
         make_float4(ray.d.x, ray.d.y, ray.d.z, __uint_as_float(tr.ref)));
  so.fin_L = mk(0.0f, 0.0f, 0.0f);
  shade_path<METHOD, FULL>(sc, pool, rp, slot, false, kNoCamera, so);
}
PTB_DEV void tail_add_nee(const PathPool& pool, uint32_t slot, const ShadeOut& so) {  // unoccluded NEE joins the path's radiance
  float4 ra = pool.col[4u * (size_t)slot + 1u];
  ra.x += so.sh_c.x; ra.y += so.sh_c.y; ra.z += so.sh_c.z;
  pool.col[4u * (size_t)slot + 1u] = ra;
}
PTB_DEV void tail_finish(float* __restrict__ accum, const Queues& q, uint32_t slot, const ShadeOut& so) {
  if (so.contributes) {
    atomicAdd(accum + 3u * (size_t)so.fin_pixel + 0, so.fin_L.x);
    atomicAdd(accum + 3u * (size_t)so.fin_pixel + 1, so.fin_L.y);
    atomicAdd(accum + 3u * (size_t)so.fin_pixel + 2, so.fin_L.z);
  }
  q.bin[slot] = (uint8_t)kBinDead;
}

// Binary tree: the warp advances its (up to 32) paths one bounce at a time, in lock step, and traverses their rays
// TOGETHER (ptb_coop.cuh: the rays of up to kCoopRays paths share one frontier, all 32 lanes work on it); shading stays with
// the lane that owns the path, and a lane whose path has ended takes the next one from the queue. A lane that walks its ray
// alone pays one dependent memory round trip per node (~150 for a ray inside the glass sphere of C3: 60 us per bounce, and
// the launch used to last as long as its longest path — 3.5 ms exposed at the end of a C3 render at 5 of 32 lanes); the
// cooperative walk pays about the depth of the tree, and as the warp's paths die its lanes move over to the survivors.
// Every step of the loop is warp-convergent on purpose: a lane that leaves a divergent loop early waits at the compiler's
// reconvergence point until the others arrive, so "a lane pulls the next path when its own has ended" did not do what it
// says (measured: hand-over tests that relied on idle lanes making progress never fired).
// Wide tree, and scenes of a handful of primitives (a two-level tree: nothing to share, the rounds' bookkeeping would be
// most of the work — rtweekend1 measured 3 % slower cooperatively): the lane walk (one lane per path, trace_lane).
constexpr uint32_t kCoopMinPrims = 4096u;
#ifndef PTB_TAIL_WARPS
#define PTB_TAIL_WARPS 4  // warps per k_tail block (each owns one cooperative frontier in shared memory)
#endif
constexpr int kTailThreads = 32 * PTB_TAIL_WARPS;
template <class TR, int METHOD, bool FULL>
__global__ void __launch_bounds__(kTailThreads)
k_tail(DevScene sc, PathPool pool, Queues q, WaveCounters* wc, RenderParams rp, float* __restrict__ accum, uint32_t depth) {
  if (wc->tail_iter != depth) return;  // launched after every iteration >= 2; only the hand-over iteration's launch has work
  const uint32_t n = wc->n_tail;   // live paths, listed in q.live by k_win_fill
  if (threadIdx.x == 0u) atomicMin(&wc->tail_t0, global_timer_ns());
#ifdef PTB_TAIL_STATS
  if (threadIdx.x == 0u) atomicMin(&g_tail_stats[9], global_timer_ns());
#endif
  constexpr bool COOP = TR::kCoop;
  __shared__ CoopWarp s_coop[COOP ? PTB_TAIL_WARPS : 1];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  unsigned long long c_bounce = 0, c_sky = 0, c_light = 0, c_ref = 0, c_paths = 0;
  // Ticket t -> path: cycle walking over x -> (x * odd) mod 2^k, a bijection of [0, n) that sends the 32 consecutive
  // tickets of a warp to paths ~0.618 * 2^k apart (Fibonacci hashing): neighbouring paths — the same glass pixels, the long
  // ones — land in different warps.
  const uint32_t mask = n <= 1u ? 0u : (1u << (32 - __clz(n - 1u))) - 1u;
  if (COOP && sc.n_prims >= kCoopMinPrims) {
    CoopWarp& cw = s_coop[warp];
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t slot = kNone;
    bool exhausted = false;
    for (;;) {
      if (slot == kNone && !exhausted) {
        const uint32_t t = atomicAdd(&wc->tail_head, 1u);
        if (t < n) {
          uint32_t i = t;
          do { i = (i * 0x9E3779B1u) & mask; } while (i >= n);
          slot = q.live[i];
        } else {
          exhausted = true;
        }
      }
      const uint32_t live = __ballot_sync(0xffffffffu, slot != kNone);
      if (!live) break;
      const bool active = slot != kNone;
      // ---- closest hit (k_trace), kCoopRays rays at a time
      Ray ray;
      TraceResult tr;
      tr.t = 0.0f;
      tr.ref = kNone;
      if (active) {
        float4 o4, d4;
        ldg256_rw(pool.ray + 4u * (size_t)slot, o4, d4);
        ray = make_ray(from4(o4), from4(d4));
      }
      for (uint32_t todo = live; todo;) {
        const bool mine = ((todo >> lane) & 1u) && (uint32_t)__popc(todo & lt) < kCoopRays;
        const uint32_t bm = __ballot_sync(0xffffffffu, mine);
        const uint32_t r = (uint32_t)__popc(bm & lt);
        if (mine) coop_set_ray(sc, cw, r, ray, __int_as_float(0x7f800000), kNone);
        __syncwarp();
        coop_trace<false>(sc, cw, (uint32_t)__popc(bm));
        if (mine) {
          tr.ref = cw.ref[r];
          tr.t = tr.ref == kNone ? 0.0f : __uint_as_float((uint32_t)(cw.best[r] >> 32));
        }
        __syncwarp();  // answers read before the next batch overwrites them
        todo &= ~bm;
      }
      // ---- shade (k_shade)
      ShadeOut so;
      if (active) {
        ++c_bounce;
        tail_shade<METHOD, FULL>(sc, pool, rp, slot, ray, tr, so);
        if (METHOD == PTB_METHOD_NAIVE) ++c_ref;            // Q7: naive counts every check_hit ...
        else if (so.alive) ++c_ref;                         // ... MIS every bounce iteration that continues
      }
      // ---- NEE visibility (k_shadow): unoccluded contributions join the path's radiance
      if (METHOD == PTB_METHOD_MIS) {
        const bool sh = active && so.shadow;
        if (sh) { if (so.shadow_is_sky) ++c_sky; else ++c_light; }
        for (uint32_t todo = __ballot_sync(0xffffffffu, sh); todo;) {
          const bool mine = ((todo >> lane) & 1u) && (uint32_t)__popc(todo & lt) < kCoopRays;
          const uint32_t bm = __ballot_sync(0xffffffffu, mine);
          const uint32_t r = (uint32_t)__popc(bm & lt);
          if (mine) coop_set_ray(sc, cw, r, make_ray(from4(so.sh_o), from4(so.sh_d)), so.sh_o.w, __float_as_uint(so.sh_d.w));
          __syncwarp();
          coop_trace<true>(sc, cw, (uint32_t)__popc(bm));
          if (mine && cw.ref[r] == kNone) tail_add_nee(pool, slot, so);
          __syncwarp();
          todo &= ~bm;
        }
      }
      if (active && so.finished) {
        ++c_paths;
        tail_finish(accum, q, slot, so);
        slot = kNone;
      }
    }
  } else {
    typename TR::Scratch scratch;
    for (;;) {
      const uint32_t i = atomicAdd(&wc->tail_head, 1u);
      if (i >= n) break;
      const uint32_t s = q.live[i];
      for (;;) {
        float4 o4, d4;
        ldg256_rw(pool.ray + 4u * (size_t)s, o4, d4);
        const Ray ray = make_ray(from4(o4), from4(d4));
        const TraceResult tr = trace_lane<TR, false>(sc, ray, __int_as_float(0x7f800000), kNone, scratch);
        ++c_bounce;
        ShadeOut so;
        tail_shade<METHOD, FULL>(sc, pool, rp, s, ray, tr, so);
        if (METHOD == PTB_METHOD_NAIVE) ++c_ref;
        else if (so.alive) ++c_ref;
        if (METHOD == PTB_METHOD_MIS && so.shadow) {
          if (so.shadow_is_sky) ++c_sky; else ++c_light;
          const Ray sray = make_ray(from4(so.sh_o), from4(so.sh_d));
          const TraceResult ss = trace_lane<TR, true>(sc, sray, so.sh_o.w, __float_as_uint(so.sh_d.w), scratch);
          if (ss.ref == kNone) tail_add_nee(pool, s, so);
        }
        if (so.finished) {
          ++c_paths;
          tail_finish(accum, q, s, so);
          break;
        }
      }
    }
  }
  // statistics: one set of atomics per warp
  __syncwarp();
#ifdef PTB_TAIL_STATS
  PTB_TS(4, c_bounce);
  if (threadIdx.x == 0u && blockIdx.x == 0u) { PTB_TS(0, 1); PTB_TS(1, n); }
  if (lane == 0u) atomicMax(&g_tail_stats[10], global_timer_ns());
#endif
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    c_bounce += __shfl_xor_sync(0xffffffffu, c_bounce, o);
    c_sky += __shfl_xor_sync(0xffffffffu, c_sky, o);
    c_light += __shfl_xor_sync(0xffffffffu, c_light, o);
    c_ref += __shfl_xor_sync(0xffffffffu, c_ref, o);
    c_paths += __shfl_xor_sync(0xffffffffu, c_paths, o);
  }
  if (threadIdx.x == 0u) atomicMax(&wc->tail_t1, global_timer_ns());
  if ((threadIdx.x & 31u) == 0u && c_bounce) {
    atomicAdd(&wc->rays_bounce, c_bounce);
    if (c_sky) atomicAdd(&wc->rays_shadow_sky, c_sky);
    if (c_light) atomicAdd(&wc->rays_shadow_light, c_light);
    atomicAdd(&wc->rays_reference, c_ref);
    atomicAdd(&wc->paths, c_paths);
  }
}

// ------------------------------------------------------------------------------------------ closest-hit API kernel
// check_hit for a batch of caller rays (acceleration/mod.rs:265-298): 2 x float4 in, 16 B out.
// The caller's rays arrive in no order. A warp that holds a few rays which walk deep while the others miss the scene at
// the root runs at 8 of 32 lanes (ncu, 100 M random rays vs 10 M triangles), so the batch is ordered first: key = does the
// ray reach the scene's box at all, then the 6-bit-per-axis Morton code of the point where it enters the box and its
// direction octant (21 bits, three radix passes). Rays are traced in key order through an index array; hits are written
// to the caller's positions.
__global__ void __launch_bounds__(256)
k_ray_sort_keys(DevScene sc, const float4* __restrict__ rays, uint32_t n, uint32_t* __restrict__ keys, uint32_t* __restrict__ idx) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // scene box = union of the root's two child boxes
  const BvhNode root = sc.nodes[0];
  const v3 bmin = mk(fminf(root.n0.x, root.n1.z), fminf(root.n0.y, root.n1.w), fminf(root.n0.z, root.n2.x));
  const v3 bmax = mk(fmaxf(root.n0.w, root.n2.y), fmaxf(root.n1.x, root.n2.z), fmaxf(root.n1.y, root.n2.w));
  const float4 o4 = __ldg(rays + 2u * (size_t)i), d4 = __ldg(rays + 2u * (size_t)i + 1u);
  const v3 o = from4(o4), d = from4(d4);
  // plain slab test (ordering only: a wrong key costs coherence, never correctness)
  const v3 inv = mk(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
  const v3 t0 = (bmin - o) * inv, t1 = (bmax - o) * inv;
  const float tn = fmaxf(fmaxf(fminf(t0.x, t1.x), fminf(t0.y, t1.y)), fmaxf(fminf(t0.z, t1.z), 0.0f));
  const float tf = fminf(fminf(fmaxf(t0.x, t1.x), fmaxf(t0.y, t1.y)), fmaxf(t0.z, t1.z));
  uint32_t key = 0x1FFFFFu;  // misses the scene box: all such rays together, after the others
  if (tn <= tf) {
    const v3 p = o + tn * d;
    const v3 ext = bmax - bmin;
    auto q = [](float x, float lo, float e) {
      const float f = e > 0.0f ? (x - lo) / e * 64.0f : 0.0f;
      return (uint32_t)fminf(fmaxf(f, 0.0f), 63.0f);
    };
    uint32_t m = 0;
    const uint32_t qx = q(p.x, bmin.x, ext.x), qy = q(p.y, bmin.y, ext.y), qz = q(p.z, bmin.z, ext.z);
#pragma unroll
    for (int b = 0; b < 6; ++b) m |= (((qx >> b) & 1u) << (3 * b + 2)) | (((qy >> b) & 1u) << (3 * b + 1)) | (((qz >> b) & 1u) << (3 * b));
    key = (m << 3) | (d.x < 0.0f ? 4u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 1u : 0u);
    if (key >= 0x1FFFFFu) key = 0x1FFFFEu;
  }
  keys[i] = key;
  idx[i] = i;
}

struct ApiFetch {
  const float4* __restrict__ rays;
  const uint32_t* __restrict__ order;  // nullptr: trace in the caller's order
  uint32_t idx;
  Ray ray;
  PTB_DEV void operator()(uint32_t i, Ray& r, float& /*tmax*/, uint32_t& /*exclude*/) {
    idx = order ? order[i] : i;
    const float4 o = __ldg(rays + 2u * (size_t)idx), d = __ldg(rays + 2u * (size_t)idx + 1u);
    r = make_ray_from_raw(from4(o), from4(d));
    ray = r;
  }
};
struct ApiRetire {
  const DevScene& sc;
  uint4* __restrict__ hits;
  const ApiFetch& f;
  PTB_DEV void operator()(bool fin, const TraceResult& tr, const Ray&) {
    if (!fin) return;
    uint4 out = make_uint4(__float_as_uint(0.0f), PTB_MISS, 0u, 0u);
    if (tr.ref != kNone) {
      HitRec h;
      prim_hit(sc, f.ray, tr.ref, h);
      out = make_uint4(__float_as_uint(tr.t), __ldg(sc.slot_prim + (tr.ref & kSlotMask)), __float_as_uint(h.b1),
                       __float_as_uint(h.b2));
    }
    hits[f.idx] = out;
  }
};
template <class TR, bool COUNT>
__global__ void __launch_bounds__(256, TR::kApiMinBlocks)
k_closest_hit_api(DevScene sc, const float4* __restrict__ rays, const uint32_t* __restrict__ order, uint32_t n,
                  uint4* __restrict__ hits, uint32_t* head, unsigned long long* counts) {
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t cnt_nodes = 0, cnt_prims = 0, cnt_rays = 0;
  ApiFetch fetch{rays, order, 0u, Ray()};
  ApiRetire retire{sc, hits, fetch};
  persistent_trace<TR, false, COUNT>(sc, n, head, fetch, retire, cnt_nodes, cnt_prims, cnt_rays);
  if (COUNT) {
    for (int off = 16; off > 0; off >>= 1) {
      cnt_nodes += __shfl_xor_sync(0xffffffffu, cnt_nodes, off);
      cnt_prims += __shfl_xor_sync(0xffffffffu, cnt_prims, off);
    }
    if (lane == 0) {
      atomicAdd(counts + 0, (unsigned long long)cnt_nodes);
      atomicAdd(counts + 1, (unsigned long long)cnt_prims);
    }
  }
}

// ------------------------------------------------------------------------------------------ denoiser feature buffers
// ptb_render_aov: the first hit of the camera ray of every (pixel, sample) that ptb_render traces, reduced to what a
// denoiser reads. One launch per sample; work item i is the i-th pixel of the tile in the render's issue order
// (camera_pixel_sample with group 1, so rp.sample_offset is the launch's sample), and its ray is the render's camera
// ray: camera_direction + make_ray. Each pixel occurs once per launch, so its sums are updated with a plain
// read-add-write and are formed in sample order: deterministic, and independent of how a call is split.
// Sums per pixel, two 16-byte records: [albedo.rgb | coverage], [normal.xyz | depth].
struct AovFetch {
  const DevScene& sc;
  const RenderParams& rp;
  uint32_t pixel;
  PTB_DEV void operator()(uint32_t i, Ray& r, float& /*tmax*/, uint32_t& /*exclude*/) {
    uint32_t x, y, sample;
    camera_pixel_sample(rp, i, x, y, sample);
    pixel = y * rp.width + x;
    r = make_ray(sc.cam_origin, camera_direction(sc, rp, x, y, sample));
  }
};
struct AovRetire {
  const DevScene& sc;
  float4* __restrict__ sums;
  const AovFetch& f;
  PTB_DEV void operator()(bool fin, const TraceResult& tr, const Ray& ray) {
    if (!fin) return;
    const bool hit = tr.ref != kNone;
    HitRec h;
    uint32_t kind = PTB_MAT_EMIT, tex = sc.sky_tex;
    float param = 1.0f;
    if (hit) {
      prim_hit(sc, ray, tr.ref, h);
      const DevMaterial* m = sc.materials + (__ldg(sc.slot_mat + (tr.ref & kSlotMask)) & 0x00FFFFFFu);
      kind = __ldg(&m->kind);
      tex = __ldg(&m->tex);
      param = __ldg(&m->param);
    } else {  // sky.rs:79-91: zero Hit + Emit(sky texture, 1.0), as k_shade treats a miss
      h.t = 0.0f;
      h.point = h.error = h.normal = mk(0.0f, 0.0f, 0.0f);
    }
    v3 a;
    if (kind == PTB_MAT_EMIT) {  // the emission the depth-0 integrator adds (emissive.rs:23-26)
      a = param * texture_colour<true>(sc, tex, ray.d, offset_ray(h.point, h.normal, h.error, true));
    } else {
      a = texture_colour<true>(sc, tex, ray.d, h.point);
      if (kind == PTB_MAT_LAMBERTIAN) a = a * param;  // the colour factor of mat_eval
    }
    // denoisers expect albedo in [0, 1]; fminf / fmaxf also turn a NaN into 0
    a = mk(fminf(fmaxf(a.x, 0.0f), 1.0f), fminf(fmaxf(a.y, 0.0f), 1.0f), fminf(fmaxf(a.z, 0.0f), 1.0f));
    float4* p = sums + 2u * (size_t)f.pixel;
    float4 s0 = p[0], s1 = p[1];
    s0.x += a.x; s0.y += a.y; s0.z += a.z; s0.w += hit ? 1.0f : 0.0f;
    s1.x += h.normal.x; s1.y += h.normal.y; s1.z += h.normal.z; s1.w += h.t;
    p[0] = s0;
    p[1] = s1;
  }
};
template <class TR>
__global__ void __launch_bounds__(256, TR::kApiMinBlocks)
k_aov(DevScene sc, RenderParams rp, float4* __restrict__ sums, uint32_t* head) {
  uint32_t a = 0, b = 0, r = 0;
  AovFetch fetch{sc, rp, 0u};
  AovRetire retire{sc, sums, fetch};
  persistent_trace<TR, false, false>(sc, rp.npix, head, fetch, retire, a, b, r);
}

// ------------------------------------------------------------------------------------------ visibility API kernel
// Batch any-hit through the walk k_shadow runs (persistent_trace<TR, ANYHIT = true>), fed from caller records.
//   CHI  : check_hit_index (acceleration/mod.rs:226-263): ptb_ray + target id in, ptb_hit out. The target's own hit is
//          computed first, as k_shade does for a light sample; the walk then looks for a blocker at 0 < t < t_target with
//          the target excluded. A missed target keeps its lane with tmax = 0, which nothing can block, and answers a miss.
//   !CHI : occlusion: ptb_occlusion_ray in (origin | tmax, direction | excluded original id), one byte out.
// Ids arrive in the original order and are mapped to slots through prim_slot (k_gather's map, kept with the scene).
template <bool CHI>
struct VisFetch {
  const DevScene& sc;
  const float4* __restrict__ rays;
  const uint32_t* __restrict__ index;      // CHI: target id per record
  const uint32_t* __restrict__ order;      // nullptr: trace in the caller's order
  const uint32_t* __restrict__ prim_slot;  // original id -> slot
  uint32_t n_spheres;
  uint32_t idx;
  uint4 hit;  // CHI: the target's record, written when nothing blocks it
  PTB_DEV void operator()(uint32_t i, Ray& r, float& tmax, uint32_t& exclude) {
    idx = order ? order[i] : i;
    const float4 o = __ldg(rays + 2u * (size_t)idx), d = __ldg(rays + 2u * (size_t)idx + 1u);
    r = make_ray_from_raw(from4(o), from4(d));
    if (CHI) {
      const uint32_t p = __ldg(index + idx);
      hit = make_uint4(__float_as_uint(0.0f), PTB_MISS, 0u, 0u);
      tmax = 0.0f;
      exclude = kNone;
      if (p < sc.n_prims) {
        const uint32_t slot = __ldg(prim_slot + p);
        HitRec h;
        if (prim_hit(sc, r, (p < n_spheres ? kSphereBit : 0u) | slot, h) && h.t > 0.0f) {  // acceleration/mod.rs:231-243
          hit = make_uint4(__float_as_uint(h.t), p, __float_as_uint(h.b1), __float_as_uint(h.b2));
          tmax = h.t;
          exclude = slot;
        }
      }
    } else {
      const uint32_t x = __float_as_uint(d.w);
      tmax = o.w;
      exclude = x < sc.n_prims ? __ldg(prim_slot + x) : kNone;
    }
  }
};
template <bool CHI>
struct VisRetire {
  void* __restrict__ out;
  const VisFetch<CHI>& f;
  PTB_DEV void operator()(bool fin, const TraceResult& tr, const Ray&) {
    if (!fin) return;
    if (CHI) static_cast<uint4*>(out)[f.idx] = tr.ref == kNone ? f.hit : make_uint4(__float_as_uint(0.0f), PTB_MISS, 0u, 0u);
    else static_cast<uint8_t*>(out)[f.idx] = tr.ref != kNone ? 1u : 0u;
  }
};
template <class TR, bool CHI>
__global__ void __launch_bounds__(256, TR::kApiMinBlocks)
k_visibility_api(DevScene sc, const float4* __restrict__ rays, const uint32_t* __restrict__ index,
                 const uint32_t* __restrict__ order, const uint32_t* __restrict__ prim_slot, uint32_t n_spheres, uint32_t n,
                 void* __restrict__ out, uint32_t* head) {
  uint32_t a = 0, b = 0, r = 0;
  VisFetch<CHI> fetch{sc, rays, index, order, prim_slot, n_spheres, 0u, make_uint4(0u, 0u, 0u, 0u)};
  VisRetire<CHI> retire{out, fetch};
  persistent_trace<TR, true, false>(sc, n, head, fetch, retire, a, b, r);
}

// ------------------------------------------------------------------------------------------ sampler test hook
// ptb_sample_only / ptb_sampler_pdf (include/ptb200.h): the reference's best-pinned tests are chi-squared tests of its
// samplers against their pdfs (statistics/spherical_sampling.rs:64-226, bxdfs/lambertian.rs:30-48,
// bxdfs/trowbridge_reitz_vndf.rs:156-218, distributions.rs:186-300). These two kernels expose the DEVICE samplers — the
// functions k_shade calls — to the same harness: sample k draws its uniforms from Philox counter (k, 0, RNG_TEST, block).
constexpr uint32_t RNG_TEST = 7;
// light sampling as k_shade runs it (integrators/mis.rs:117-133, acceleration/mod.rs:231-243): pdf of direction `wi` from
// the shading point (point, normal) towards light `lref`, 0 when the light is not hit
PTB_DEV float light_dir_pdf(const DevScene& sc, uint32_t lref, v3 point, v3 normal, v3 wi) {
  const v3 so = point + 0.0001f * normal;
  const Ray sray = make_ray_from_raw(so, wi);
  HitRec si;
  if (prim_hit(sc, sray, lref, si) && si.t > 0.0f) return light_pdf(sc, lref, point, wi, si.point, si.normal);
  return 0.0f;
}
__global__ void k_sample_only(DevScene sc, ptb_sampler_query q, uint32_t n, float* __restrict__ dirs, float* __restrict__ pdf) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t k0 = (uint32_t)q.seed, k1 = (uint32_t)(q.seed >> 32);
  const uint4 r = philox4x32_10(k, 0u, RNG_TEST, 0u, k0, k1);
  const v3 normal = mk(q.normal.x, q.normal.y, q.normal.z), aux = mk(q.aux.x, q.aux.y, q.aux.z);
  v3 d = mk(0.0f, 0.0f, 0.0f);
  float p = 0.0f;
  switch (q.kind) {
    case PTB_SAMPLER_LAMBERTIAN:
      d = lambertian_sample_dir(normal, u32_to_unit(r.x), u32_to_unit(r.y));
      p = fmaxf(dot(d, normal), 0.0f) / kPi;
      break;
    case PTB_SAMPLER_TR_VNDF:
      d = tr_sample(q.alpha, aux, normal, u32_to_unit(r.x), u32_to_unit(r.y));
      p = tr_pdf(q.alpha, aux, d, normal);
      break;
    case PTB_SAMPLER_SKY: {
      const uint4 r2 = philox4x32_10(k, 0u, RNG_TEST, 1u, k0, k1);
      d = sky_sample(sc, u32_to_unit(r.y), u32_to_unit(r.z), u32_to_unit(r.w), u32_to_unit(r2.x));  // draws as in k_shade
      p = sky_pdf(sc, d);
      break;
    }
    case PTB_SAMPLER_LIGHT: {
      const uint32_t lref = __ldg(sc.lights + q.light_index);
      d = light_sample_dir(sc, lref, aux, u32_to_unit(r.y), u32_to_unit(r.z));
      p = light_dir_pdf(sc, lref, aux, normal, d);
      break;
    }
    default:
      d = uniform_sphere_dir(u32_to_unit(r.x), u32_to_unit(r.y));
      p = 1.0f / (4.0f * kPi);
  }
  dirs[3u * (size_t)k + 0] = d.x; dirs[3u * (size_t)k + 1] = d.y; dirs[3u * (size_t)k + 2] = d.z;
  if (pdf) pdf[k] = p;
}
__global__ void k_sampler_pdf(DevScene sc, ptb_sampler_query q, uint32_t n, const float* __restrict__ dirs, float* __restrict__ pdf) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const v3 normal = mk(q.normal.x, q.normal.y, q.normal.z), aux = mk(q.aux.x, q.aux.y, q.aux.z);
  const v3 d = mk(dirs[3u * (size_t)k], dirs[3u * (size_t)k + 1], dirs[3u * (size_t)k + 2]);
  float p;
  switch (q.kind) {
    case PTB_SAMPLER_LAMBERTIAN: p = fmaxf(dot(d, normal), 0.0f) / kPi; break;
    case PTB_SAMPLER_TR_VNDF: p = tr_pdf(q.alpha, aux, d, normal); break;
    case PTB_SAMPLER_SKY: p = sky_pdf(sc, d); break;
    case PTB_SAMPLER_LIGHT: p = light_dir_pdf(sc, __ldg(sc.lights + q.light_index), aux, normal, d); break;
    default: p = 1.0f / (4.0f * kPi);
  }
  pdf[k] = p;
}
int32_t sampler_hook(Ctx* c, const ptb_sampler_query& q, size_t n, const float* dirs_in, float* dirs_out, float* pdf_out) {
  if (q.kind > PTB_SAMPLER_UNIFORM_SPHERE) return set_error(c, PTB_ERR_INVALID, "unknown sampler kind %u", q.kind);
  if ((q.kind == PTB_SAMPLER_SKY || q.kind == PTB_SAMPLER_LIGHT) && !c->committed)
    return set_error(c, PTB_ERR_INVALID, "sky / light samplers need a committed scene");
  if (q.kind == PTB_SAMPLER_SKY && (c->dev.sky_rx | c->dev.sky_ry) == 0u) return set_error(c, PTB_ERR_INVALID, "the scene's sky is not samplable");
  if (q.kind == PTB_SAMPLER_LIGHT && q.light_index >= c->dev.n_lights) return set_error(c, PTB_ERR_INVALID, "light index out of range");
  if (n == 0) return PTB_OK;
  if (n > 0x7FFFFFFFull) return set_error(c, PTB_ERR_INVALID, "too many samples");
  PTB_CUDA_TRY(c, c->d_rays.reserve(n * 12));
  PTB_CUDA_TRY(c, c->d_hits.reserve(n * 4));
  float* d_dirs = c->d_rays.as<float>();
  float* d_pdf = c->d_hits.as<float>();
  const uint32_t n32 = (uint32_t)n, grid = (n32 + 255u) / 256u;
  if (dirs_in) {
    PTB_CUDA_TRY(c, cudaMemcpyAsync(d_dirs, dirs_in, n * 12, cudaMemcpyHostToDevice, c->stream));
    k_sampler_pdf<<<grid, 256, 0, c->stream>>>(c->dev, q, n32, d_dirs, d_pdf);
  } else {
    k_sample_only<<<grid, 256, 0, c->stream>>>(c->dev, q, n32, d_dirs, d_pdf);
    PTB_CUDA_TRY(c, cudaMemcpyAsync(dirs_out, d_dirs, n * 12, cudaMemcpyDeviceToHost, c->stream));
  }
  c->stats.kernel_launches += 1;
  if (pdf_out) PTB_CUDA_TRY(c, cudaMemcpyAsync(pdf_out, d_pdf, n * 4, cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  PTB_CUDA_TRY(c, cudaGetLastError());
  return PTB_OK;
}

// ---- kernel tables: every persistent traversal kernel exists once per tree (BinTrav / CwTrav)
template <class TR>
static const void* trace_kernel_of(bool count, bool camera) {
  if (camera) return count ? (const void*)k_trace<TR, true, true> : (const void*)k_trace<TR, false, true>;
  return count ? (const void*)k_trace<TR, true, false> : (const void*)k_trace<TR, false, false>;
}
static const void* trace_kernel(const Ctx* c, bool count, bool camera) {
  return c->wide ? trace_kernel_of<CwTrav>(count, camera) : trace_kernel_of<BinTrav>(count, camera);
}
static const void* shadow_kernel(const Ctx* c) { return c->wide ? (const void*)k_shadow<CwTrav> : (const void*)k_shadow<BinTrav>; }
static const void* api_kernel(const Ctx* c, bool count) {
  if (c->wide) return count ? (const void*)k_closest_hit_api<CwTrav, true> : (const void*)k_closest_hit_api<CwTrav, false>;
  return count ? (const void*)k_closest_hit_api<BinTrav, true> : (const void*)k_closest_hit_api<BinTrav, false>;
}
static const void* aov_kernel(const Ctx* c) { return c->wide ? (const void*)k_aov<CwTrav> : (const void*)k_aov<BinTrav>; }
static const void* visibility_kernel(const Ctx* c, bool chi) {
  if (c->wide) return chi ? (const void*)k_visibility_api<CwTrav, true> : (const void*)k_visibility_api<CwTrav, false>;
  return chi ? (const void*)k_visibility_api<BinTrav, true> : (const void*)k_visibility_api<BinTrav, false>;
}
template <class TR>
static const void* tail_kernel_of(bool mis, bool full) {
  if (mis) return full ? (const void*)k_tail<TR, PTB_METHOD_MIS, true> : (const void*)k_tail<TR, PTB_METHOD_MIS, false>;
  return full ? (const void*)k_tail<TR, PTB_METHOD_NAIVE, true> : (const void*)k_tail<TR, PTB_METHOD_NAIVE, false>;
}
static cudaError_t launch_trace(const void* fn, int grid, cudaStream_t st, const DevScene& sc, const PathPool& pool, const Queues& q,
                                WaveCounters* wc, const RenderParams& rp, unsigned long long first) {
  void* args[] = {(void*)&sc, (void*)&pool, (void*)&q, (void*)&wc, (void*)&rp, (void*)&first};
  return cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, st);
}
static cudaError_t launch_trace_camera(const void* fn, int grid, cudaStream_t st, const DevScene& sc, const PathPool& pool,
                                       const Queues& q, WaveCounters* wc, const RenderParams& rp, unsigned long long first,
                                       const CamCandList& cl) {
  void* args[] = {(void*)&sc, (void*)&pool, (void*)&q, (void*)&wc, (void*)&rp, (void*)&first, (void*)&cl};
  return cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, st);
}
static cudaError_t launch_shadow(const void* fn, int grid, cudaStream_t st, const DevScene& sc, const PathPool& pool, const Queues& q,
                                 WaveCounters* wc) {
  void* args[] = {(void*)&sc, (void*)&pool, (void*)&q, (void*)&wc};
  return cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, st);
}

// ------------------------------------------------------------------------------------------ host side
static int persistent_grid(Ctx* c, const void* kernel, int threads) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  return c->sm_count * per_sm;
}

// Work cursor and counters of one batch-API launch (in the scratch after the wavefront counters: [0] work cursor,
// [8..24) node / primitive counters), zeroed on the stream, and the order the batch is traced in: batches of >= 65 536
// rays are ordered by k_ray_sort_keys (which reads only the .xyz of the two float4 of a record, so ptb_ray and
// ptb_occlusion_ray sort alike); PTB_HIT_SORT=0 traces in the caller's order (*order = nullptr).
static int32_t prepare_batch(Ctx* c, const float4* r4, size_t n, uint32_t** head, unsigned long long** counts,
                             const uint32_t** order) {
  if (n > 0xFFFFFFF0ull) return set_error(c, PTB_ERR_INVALID, "too many rays in one batch");
  PTB_CUDA_TRY(c, c->d_counters.reserve(sizeof(WaveCounters) + 64));
  char* scratch = c->d_counters.as<char>() + sizeof(WaveCounters);
  *head = reinterpret_cast<uint32_t*>(scratch);
  *counts = reinterpret_cast<unsigned long long*>(scratch + 8);
  PTB_CUDA_TRY(c, cudaMemsetAsync(scratch, 0, 24, c->stream));
  *order = nullptr;
  bool sort = n >= (1u << 16) && c->n_prims > 0;
  if (const char* e = getenv("PTB_HIT_SORT")) sort = sort && atoi(e) != 0;
  if (sort) {
    const uint32_t n32 = (uint32_t)n;
    PTB_CUDA_TRY(c, c->d_hit_sort.reserve(((size_t)n32 * 4 + radix_sort_hist_words(n32)) * 4));
    uint32_t* w = c->d_hit_sort.as<uint32_t>();
    uint32_t *ka = w, *va = w + n, *kb = w + 2 * n, *vb = w + 3 * n, *hist = w + 4 * n;
    k_ray_sort_keys<<<(n32 + 255u) / 256u, 256, 0, c->stream>>>(c->dev, r4, n32, ka, va);
    c->stats.kernel_launches += 1;
    radix_sort_pairs(c, ka, va, kb, vb, n32, 3, hist);
    *order = va;
  }
  return PTB_OK;
}

int32_t launch_closest_hit(Ctx* c, const void* d_rays, size_t n, void* d_hits) {
  if (n == 0) return PTB_OK;
  const float4* r4 = reinterpret_cast<const float4*>(d_rays);
  uint4* h4 = reinterpret_cast<uint4*>(d_hits);
  uint32_t* head;
  unsigned long long* counts;
  const uint32_t* order;
  const int32_t rc = prepare_batch(c, r4, n, &head, &counts, &order);
  if (rc != PTB_OK) return rc;
  {
    const void* fn = api_kernel(c, c->opt_count_traversal);
    const int grid = persistent_grid(c, fn, 256);
    uint32_t n32 = (uint32_t)n;
    void* args[] = {(void*)&c->dev, (void*)&r4, (void*)&order, (void*)&n32, (void*)&h4, (void*)&head, (void*)&counts};
    PTB_CUDA_TRY(c, cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, c->stream));
  }
  if (c->opt_count_traversal) {
    unsigned long long hc[2] = {0, 0};
    PTB_CUDA_TRY(c, cudaMemcpyAsync(hc, counts, 16, cudaMemcpyDeviceToHost, c->stream));
    PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->stats.nodes_fetched += hc[0];
    c->stats.prims_tested += hc[1];
    c->stats.rays_counted += n;
  }
  c->stats.kernel_launches += 1;
  c->stats.trace_launches += 1;
  PTB_CUDA_TRY(c, cudaGetLastError());
  return PTB_OK;
}

int32_t launch_visibility(Ctx* c, const void* d_rays, const void* d_index, size_t n, void* d_out) {
  if (n == 0) return PTB_OK;
  const float4* r4 = reinterpret_cast<const float4*>(d_rays);
  const uint32_t* index = static_cast<const uint32_t*>(d_index);
  uint32_t* head;
  unsigned long long* counts;
  const uint32_t* order;
  const int32_t rc = prepare_batch(c, r4, n, &head, &counts, &order);
  if (rc != PTB_OK) return rc;
  const void* fn = visibility_kernel(c, index != nullptr);
  const int grid = persistent_grid(c, fn, 256);
  const uint32_t* prim_slot = c->d_prim_slot.as<uint32_t>();
  uint32_t ns = (uint32_t)c->n_spheres, n32 = (uint32_t)n;
  void* args[] = {(void*)&c->dev, (void*)&r4, (void*)&index, (void*)&order, (void*)&prim_slot, (void*)&ns, (void*)&n32,
                  (void*)&d_out, (void*)&head};
  PTB_CUDA_TRY(c, cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, c->stream));
  c->stats.kernel_launches += 1;
  c->stats.trace_launches += 1;
  PTB_CUDA_TRY(c, cudaGetLastError());
  return PTB_OK;
}

// Pixel issue order: 32 consecutive pixel indices cover an 8 x 4 tile when the image allows (else 16 x 2, else a row), so
// the 16 pixels of a 4096-slot window are an 8 x 2 block instead of a 16 x 1 strip: the origins of a window's rays lie
// closer together. C3: 3793 -> 3834 Mrays/s. PTB_TILES=0 keeps rows.
static void pick_tiles(RenderParams& rp, uint32_t width, uint32_t rows) {
  rp.tile_w = 32u; rp.tile_h = 1u;
  bool tiles = true;
  if (const char* e = getenv("PTB_TILES")) tiles = atoi(e) != 0;
  if (tiles)
    for (uint32_t th = 4u; th > 1u; th >>= 1)
      if (rows % th == 0u && width % (32u / th) == 0u) { rp.tile_h = th; rp.tile_w = 32u / th; break; }
}

// ptb_render_aov after validation: one k_aov launch per sample of the call, each over the tile's pixels in the render's
// tile order. Every launch has its own work cursor, all zeroed by one memset.
int32_t launch_aov(Ctx* c, const ptb_render_opts& o) {
  const uint32_t rows = o.row_count ? o.row_count : o.height - o.row_begin;
  const uint32_t spp = o.samples_per_pixel;
  if (spp == 0) return PTB_OK;
  RenderParams rp{};
  rp.width = o.width; rp.height = o.height; rp.npix = o.width * rows;
  rp.row_begin = o.row_begin;
  pick_tiles(rp, o.width, rows);
  rp.group = 1u;
  rp.k0 = (uint32_t)o.seed; rp.k1 = (uint32_t)(o.seed >> 32);
  PTB_CUDA_TRY(c, c->d_aov_heads.reserve((size_t)spp * 4));
  PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_aov_heads.p, 0, (size_t)spp * 4, c->stream));
  const void* fn = aov_kernel(c);
  const int grid = persistent_grid(c, fn, 256);
  float4* sums = c->d_aov.as<float4>();
  for (uint32_t s = 0; s < spp; ++s) {
    rp.sample_offset = o.sample_offset + s;
    uint32_t* head = c->d_aov_heads.as<uint32_t>() + s;
    void* args[] = {(void*)&c->dev, (void*)&rp, (void*)&sums, (void*)&head};
    PTB_CUDA_TRY(c, cudaLaunchKernel(fn, dim3((unsigned)grid), dim3(256), args, 0, c->stream));
    c->stats.kernel_launches += 1;
    c->stats.trace_launches += 1;
  }
  PTB_CUDA_TRY(c, cudaGetLastError());
  return PTB_OK;
}

// bytes of device state per path in flight
static unsigned long long bytes_per_path(bool mis) {
  // 64-byte path block + the live-slot queue + one bin byte + MIS: previous-hit record, 48-byte shadow entry
  return 64ull + 4ull + 1ull + (mis ? 16ull + 48ull : 0ull);
}

void free_render_state(Ctx* c) {
  for (DevBuf* b : {&c->d_pool_mem, &c->d_prev, &c->d_queues, &c->d_shadow, &c->d_windows, &c->d_pool_mem2, &c->d_prev2,
                    &c->d_queues2, &c->d_shadow2, &c->d_windows2})
    b->release();
  c->pool = PathPool();
}

// Paths in flight. Round 1 kept EVERY camera path of a call resident (36 GB for 1080p x 256 spp) to amortise the ~45
// nearly empty iterations at the end of a wavefront; the fused tail kernel on a side stream removes that cost instead, so
// the path state is bounded: two chunk slots of together PTB_POOL_BYTES (default 8 GiB), never more than half of the
// device memory that was free at the context's first large render. A call is cut into equal chunks of at most one slot;
// all tails but the last chunk's are hidden under the next chunk.
// PTB_POOL_PATHS sets the slot size directly (tests).
struct PoolPlan {
  uint32_t slot_paths;  // capacity of one slot (multiple of kWindow)
  uint32_t n_chunks;
  uint32_t chunk_paths; // paths per chunk (the last one may be shorter)
};
static PoolPlan plan_pool(Ctx* c, unsigned long long total, bool mis) {
  unsigned long long budget = 8ull << 30;
  if (const char* e = getenv("PTB_POOL_BYTES")) { unsigned long long v = strtoull(e, nullptr, 10); if (v >= (64ull << 20)) budget = v; }
  const unsigned long long per_path = bytes_per_path(mis);
  unsigned long long cap = 0;
  if (const char* e = getenv("PTB_POOL_PATHS")) {
    unsigned long long v = strtoull(e, nullptr, 10);
    if (v >= 1024 && v <= (1ull << 29)) cap = v;
  }
  if (!cap) {
    if (total * per_path > (1ull << 30)) {
      // asked once per context (cudaMemGetInfo costs milliseconds once tens of GB are allocated)
      if (c->pool_budget_bytes == 0) {
        size_t free_b = 0, total_b = 0;
        c->pool_budget_bytes = cudaMemGetInfo(&free_b, &total_b) == cudaSuccess ? free_b / 2 + 1 : ~(size_t)0;
      }
      if (budget > c->pool_budget_bytes) budget = c->pool_budget_bytes;
    }
    // a call that fits the whole budget runs as ONE chunk in one slot (its only tail is exposed either way, and every
    // extra chunk adds the drain of five more persistent launches: measured, profiles/r2_sweeps.md); a larger one
    // alternates between two slots of half the budget each
    cap = budget / per_path;
    if (total > cap) cap = budget / 2ull / per_path;
    if (cap > (1ull << 29)) cap = 1ull << 29;
    if (cap < (1ull << 20)) cap = 1ull << 20;
  }
  const unsigned long long gran = kWindow;
  cap = cap / gran * gran;
  if (cap < gran) cap = gran;
  unsigned long long n_chunks = (total + cap - 1ull) / cap;
  unsigned long long chunk = (total + n_chunks - 1ull) / n_chunks;
  chunk = (chunk + gran - 1ull) / gran * gran;
  if (chunk > cap) chunk = cap;
  PoolPlan p;
  p.chunk_paths = (uint32_t)chunk;
  p.n_chunks = (uint32_t)((total + chunk - 1ull) / chunk);
  p.slot_paths = (uint32_t)(chunk < 1024ull ? ((1024ull + gran - 1ull) / gran * gran) : chunk);
  return p;
}

struct RenderSetup {
  RenderParams rp;
  Queues q;            // slot 0
  Queues q2;           // slot 1 (calls of more than one chunk)
  PathPool pool2;
  WaveCounters* wc;
  WaveCounters* wc2;
  float* accum;
  uint32_t chunk_paths, n_chunks;
  bool mis, full, count, prof;
  bool sort_kinds = false;  // k_shade sorts each block's hits by material kind
};

static int32_t render_window_mode(Ctx* c, const ptb_render_opts& o, const RenderSetup& rs, ptb_progress_fn progress, void* user);

// carve one slot's queue / window arrays out of its buffers
static void bind_slot(Queues& q, PathPool& pool, uint32_t P, DevBuf& pool_mem, DevBuf& prev, DevBuf& queues, DevBuf& shadow,
                      DevBuf& win) {
  pool.capacity = P;
  pool.ray = pool_mem.as<float4>();
  pool.col = pool.ray + 2;
  pool.prev = prev.as<float4>();
  q.live = queues.as<uint32_t>();
  q.shadow = shadow.as<float4>();
  q.n_windows = P / kWindow;  // P is a multiple of kWindow
  const size_t n_seg = (q.n_windows + kSegWindows - 1) / kSegWindows;
  const size_t words = ((size_t)q.n_windows * 2 + n_seg + 3) & ~(size_t)3;  // keeps the byte array 16-byte aligned
  uint32_t* w = win.as<uint32_t>();
  q.win_count = w;
  q.win_prefix = w + q.n_windows;
  q.seg_total = w + 2 * (size_t)q.n_windows;
  q.bin = reinterpret_cast<uint8_t*>(w + words);  // k_win_fill reads a window's 256 bytes as 32 x uint2
}

int32_t render_wavefront(Ctx* c, const ptb_render_opts& o, ptb_progress_fn progress, void* user) {
  const uint32_t rows = o.row_count ? o.row_count : o.height - o.row_begin;  // validated by ptb_render
  const uint32_t npix = o.width * rows;
  const unsigned long long total = (unsigned long long)npix * o.samples_per_pixel;
  if (total == 0) return PTB_OK;
  RenderSetup rs;
  rs.mis = o.method == PTB_METHOD_MIS;
  PoolPlan plan = plan_pool(c, total, rs.mis);
  // ---- device state (grow-only across calls; the MIS-only arrays are allocated by the first MIS call)
  // one 64-byte block per path: ray record then colour record (a DRAM access atom; two scattered 32-byte sectors per
  // path cost ~1 TB/s of effective write bandwidth). If the device cannot provide the slots (another
  // process holds the memory), they are halved and the call runs in more chunks.
  uint32_t P = plan.slot_paths;
  for (;;) {
    const bool two = plan.n_chunks > 1;
    const size_t n_seg = ((size_t)P / kWindow + kSegWindows - 1) / kSegWindows;
    const size_t win_bytes = (((size_t)P / kWindow * 2 + n_seg + 3) & ~(size_t)3) * 4 + (size_t)P;
    cudaError_t e = cudaSuccess;
    DevBuf* sets[2][5] = {{&c->d_pool_mem, &c->d_queues, &c->d_prev, &c->d_shadow, &c->d_windows},
                          {&c->d_pool_mem2, &c->d_queues2, &c->d_prev2, &c->d_shadow2, &c->d_windows2}};
    for (int sl = 0; sl < (two ? 2 : 1) && e == cudaSuccess; ++sl) {
      e = sets[sl][0]->reserve((size_t)P * 64);
      if (e == cudaSuccess) e = sets[sl][1]->reserve((size_t)P * 4);
      if (e == cudaSuccess && rs.mis) e = sets[sl][2]->reserve((size_t)P * 16);
      if (e == cudaSuccess && rs.mis) e = sets[sl][3]->reserve((size_t)P * 48);
      if (e == cudaSuccess) e = sets[sl][4]->reserve(win_bytes);
    }
    if (e == cudaSuccess) break;
    if (e != cudaErrorMemoryAllocation || P <= (1u << 20)) return check_cuda(c, e, "path pool allocation");
    cudaGetLastError();  // clear the sticky allocation error
    free_render_state(c);
    P = (P / 2 + kWindow - 1) / kWindow * kWindow;
    plan.slot_paths = plan.chunk_paths = P;
    plan.n_chunks = (uint32_t)((total + P - 1ull) / P);
  }
  rs.chunk_paths = plan.chunk_paths;
  rs.n_chunks = plan.n_chunks;
  PTB_CUDA_TRY(c, c->d_counters.reserve(sizeof(WaveCounters) + 64));
  PTB_CUDA_TRY(c, c->d_counters2.reserve(sizeof(WaveCounters) + 64));
  bind_slot(rs.q, c->pool, P, c->d_pool_mem, c->d_prev, c->d_queues, c->d_shadow, c->d_windows);
  rs.q2 = rs.q;
  rs.pool2 = c->pool;
  if (plan.n_chunks > 1) bind_slot(rs.q2, rs.pool2, P, c->d_pool_mem2, c->d_prev2, c->d_queues2, c->d_shadow2, c->d_windows2);
  rs.wc = c->d_counters.as<WaveCounters>();
  rs.wc2 = c->d_counters2.as<WaveCounters>();
  if (!c->h_counters) PTB_CUDA_TRY(c, cudaMallocHost(&c->h_counters, 10 * sizeof(WaveCounters)));

  RenderParams& rp = rs.rp;
  rp.width = o.width; rp.height = o.height; rp.npix = npix;
  rp.row_begin = o.row_begin;
  pick_tiles(rp, o.width, rows);
  // samples of one pixel issued back to back: the largest divisor of spp <= 1024 (PTB_SAMPLE_GROUP). Measured on C3 at
  // 256 spp: group 1 -> 2760 Mrays/s, 32 -> 3066, 256 -> 3197 (camera rays of a warp walk the same nodes).
  rp.group = 1u;
  {
    uint32_t want = 1024u;
    if (const char* e = getenv("PTB_SAMPLE_GROUP")) { int v = atoi(e); if (v >= 1 && v <= 1024) want = (uint32_t)v; }
    for (uint32_t g = want < o.samples_per_pixel ? want : o.samples_per_pixel; g > 1u; --g)
      if (o.samples_per_pixel % g == 0u) { rp.group = g; break; }
  }
  rp.dir_bins = 1u;
  if (const char* e = getenv("PTB_DIRBINS")) rp.dir_bins = atoi(e) != 0;
  rp.sample_offset = o.sample_offset;
  rp.method = o.method;
  rp.max_depth = o.max_depth ? o.max_depth : 50u;
  if (rp.max_depth > 255u) return set_error(c, PTB_ERR_INVALID, "max_depth must be <= 255");
  if ((uint64_t)o.sample_offset + o.samples_per_pixel > kMaxSampleIndex)
    return set_error(c, PTB_ERR_INVALID, "sample_offset + samples_per_pixel must be <= %u", kMaxSampleIndex);
  rp.rr_threshold = o.rr_threshold == PTB_RR_DEFAULT ? 3u : o.rr_threshold;
  rp.k0 = (uint32_t)o.seed; rp.k1 = (uint32_t)(o.seed >> 32);

  rs.accum = c->accum_target ? c->accum_target : c->d_accum.as<float>();
  rs.full = c->scene_needs_full_shade;
  // k_shade sorts a block's hits by material kind (PTB_SHADE_SORT=0|1 overrides). Measured on the five-sphere showcase scene
  // (three kinds, 1080p x 64 spp, profiles/r2_sweeps.md §11): MIS 4370 -> 4494 Mrays/s (k_shade 107 -> 101 ms), naive 9376 ->
  // 8538 (its shading is too short to pay for the sort): on for MIS.
  rs.sort_kinds = c->scene_material_kinds > 2 && rs.mis;
  if (const char* e = getenv("PTB_SHADE_SORT")) rs.sort_kinds = atoi(e) != 0;
  rs.count = c->opt_count_traversal;
  rs.prof = c->opt_time_kernels;
  if (rs.prof) {
    for (cudaEvent_t& e : c->ev_prof)
      if (!e) PTB_CUDA_TRY(c, cudaEventCreate(&e));
  }
  return render_window_mode(c, o, rs, progress, user);
}

// ev_prof[(slot * 4 + (iter & 3)) * 8 + 2 * k + {0,1}] brackets kernel class k (0 window bookkeeping, 1 trace, 2 shade,
// 3 shadow)
static void prof_collect(Ctx* c, int half, bool mis) {  // half = ring position (+ 4 for the second slot's ring)
  double* prof_ms[4] = {&c->stats.ms_generate, &c->stats.ms_trace, &c->stats.ms_shade, &c->stats.ms_shadow};
  static const bool timeline = getenv("PTB_TIMELINE") != nullptr;  // tuning aid: where each iteration sits inside the render
  for (int k = 0; k < (mis ? 4 : 3); ++k) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_prof[half * 8 + 2 * k], c->ev_prof[half * 8 + 2 * k + 1]) == cudaSuccess)
      *prof_ms[k] += ms;
    if (timeline) {
      float t0 = 0.f;
      cudaEventElapsedTime(&t0, c->ev_a, c->ev_prof[half * 8 + 2 * k]);
      fprintf(stderr, "timeline ring %d class %d start %.3f ms dur %.3f ms\n", half, k, t0, ms);
    }
  }
}
static void dump_lane_stats() {
#ifdef PTB_DRAIN_STATS
  {
    unsigned long long d[6];
    cudaMemcpyFromSymbol(d, g_drain, sizeof(d));
    if (d[5])
      fprintf(stderr, "drain_stats launches %llu: %.3f ms of %.3f ms ran after the queue was empty (%.1f us per launch)\n", d[5],
              1e-6 * (double)d[3], 1e-6 * (double)d[4], 1e-3 * (double)d[3] / (double)d[5]);
    unsigned long long z[6] = {~0ull, 0ull, ~0ull, 0ull, 0ull, 0ull};
    cudaMemcpyToSymbol(g_drain, z, sizeof(z));
  }
#endif
#ifdef PTB_TAIL_STATS  // tuning builds: what the fused tail's two phases did (per ptb_render call)
  {
    unsigned long long ts[16];
    cudaMemcpyFromSymbol(ts, g_tail_stats, sizeof(ts));
    fprintf(stderr, "tail_stats launches %llu paths %llu bounces %llu | cooperative traces %llu, rounds %llu (%.1f per trace, %.2f us each), "
            "entries %llu (%.1f per round), culled at pop %llu | all warps done after %.3f ms\n", ts[0], ts[1], ts[4], ts[5], ts[6],
            (double)ts[6] / (ts[5] ? ts[5] : 1), 1e-3 * (double)ts[13] / (ts[6] ? ts[6] : 1), ts[7], (double)ts[7] / (ts[6] ? ts[6] : 1), ts[12],
            1e-6 * (double)(ts[10] - ts[9]));
    unsigned long long z[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, ~0ull, 0, 0, 0, 0, 0, 0};
    cudaMemcpyToSymbol(g_tail_stats, z, sizeof(z));
  }
#endif
#ifdef PTB_LANE_STATS  // tuning builds (scripts/lane_stats.sh): where the lanes of persistent_trace spent their iterations
  unsigned long long ls[8];
  cudaMemcpyFromSymbol(ls, g_lane_stats, sizeof(ls));
  fprintf(stderr, "lane_stats iters %llu work_lanes/iter %.2f node_phases %llu (%.2f ready lanes) prim_phases %llu (%.2f ready lanes) "
          "services %llu node_steps %llu\n", ls[0], (double)ls[1] / (ls[0] ? ls[0] : 1), ls[2], (double)ls[3] / (ls[2] ? ls[2] : 1), ls[4],
          (double)ls[5] / (ls[4] ? ls[4] : 1), ls[6], ls[7]);
  unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaMemcpyToSymbol(g_lane_stats, z, sizeof(z));
#endif
}
static void fold_counters(Ctx* c, const WaveCounters& h, uint64_t iterations) {
  dump_lane_stats();
  c->stats.nodes_fetched += h.nodes_fetched;
  c->stats.prims_tested += h.prims_tested;
  c->stats.rays_counted += h.rays_counted;
  c->stats.rays_camera += h.rays_camera;
  c->stats.rays_bounce += h.rays_bounce;
  c->stats.rays_shadow_light += h.rays_shadow_light;
  c->stats.rays_shadow_sky += h.rays_shadow_sky;
  c->stats.rays_reference += h.rays_reference;
  c->stats.paths += h.paths;
  c->stats.wavefront_iterations += iterations;
}
struct SlotRefs {  // the device state one chunk runs in
  const PathPool& pool;
  const Queues& q;
  WaveCounters* wc;
};
static void launch_shade(const RenderSetup& rs, Ctx* c, const SlotRefs& sl, uint32_t grid, int threads, cudaStream_t st,
                         unsigned long long camera_first) {
  const uint32_t sort = rs.sort_kinds ? 1u : 0u;
  if (rs.mis) {
    if (rs.full) k_shade<PTB_METHOD_MIS, true><<<grid, threads, 0, st>>>(c->dev, sl.pool, sl.q, sl.wc, rs.rp, rs.accum, camera_first, sort);
    else k_shade<PTB_METHOD_MIS, false><<<grid, threads, 0, st>>>(c->dev, sl.pool, sl.q, sl.wc, rs.rp, rs.accum, camera_first, sort);
  } else {
    if (rs.full) k_shade<PTB_METHOD_NAIVE, true><<<grid, threads, 0, st>>>(c->dev, sl.pool, sl.q, sl.wc, rs.rp, rs.accum, camera_first, sort);
    else k_shade<PTB_METHOD_NAIVE, false><<<grid, threads, 0, st>>>(c->dev, sl.pool, sl.q, sl.wc, rs.rp, rs.accum, camera_first, sort);
  }
}
static const void* tail_fn(const RenderSetup& rs, Ctx* c) {
  return c->wide ? tail_kernel_of<CwTrav>(rs.mis, rs.full) : tail_kernel_of<BinTrav>(rs.mis, rs.full);
}
static void launch_tail(const RenderSetup& rs, Ctx* c, const SlotRefs& sl, uint32_t grid, cudaStream_t st, uint32_t depth) {
  const void* fn = tail_fn(rs, c);
  WaveCounters* wc = sl.wc;
  float* accum = rs.accum;
  void* args[] = {(void*)&c->dev, (void*)&sl.pool, (void*)&sl.q, (void*)&wc, (void*)&rs.rp, (void*)&accum, (void*)&depth};
  cudaLaunchKernel(fn, dim3(grid), dim3(kTailThreads), args, 0, st);
}
static const void* shade_fn(const RenderSetup& rs) {
  return rs.mis ? (rs.full ? (const void*)k_shade<PTB_METHOD_MIS, true> : (const void*)k_shade<PTB_METHOD_MIS, false>)
                : (rs.full ? (const void*)k_shade<PTB_METHOD_NAIVE, true> : (const void*)k_shade<PTB_METHOD_NAIVE, false>);
}

// ---- window mode: chunk by chunk, every path of a chunk resident, one bounce of all of them per iteration.
// Chunk k runs its wide iterations on the main stream in slot k & 1; once fewer than `tail_paths` of its paths are alive
// they are handed to ONE k_tail launch on the side stream, and chunk k+1 starts in the other slot right away.
static int32_t render_window_mode(Ctx* c, const ptb_render_opts& o, const RenderSetup& rs, ptb_progress_fn progress, void* user) {
  cudaStream_t st = c->stream;
  const uint32_t npix = rs.rp.npix, P = rs.chunk_paths;
  const unsigned long long total = (unsigned long long)npix * o.samples_per_pixel;
  const bool mis = rs.mis, prof = rs.prof, count = rs.count;
  const int T = 256;
  const SlotRefs slots[2] = {{c->pool, rs.q, rs.wc}, {rs.pool2, rs.q2, rs.wc2}};
  const uint32_t n_windows = rs.q.n_windows;
  const uint32_t n_seg = (n_windows + kSegWindows - 1) / kSegWindows;
  auto capped = [&](const void* k, uint32_t items_per_block, uint32_t items) {
    const uint32_t g = (uint32_t)persistent_grid(c, k, T), need = (items + items_per_block - 1) / items_per_block;
    return g < need ? g : (need ? need : 1u);
  };
  const uint32_t grid_fill = capped((const void*)k_win_fill, kFillGroup, n_windows);
  // k_shade is register-heavy (84 naive / 116 MIS): 128-thread blocks let more of them share an SM's register file
  // (window mode, C3: 256 threads 3438 Mrays/s, 128 -> 3500, 64 -> 3499)
  int TS = 128;
  if (const char* e = getenv("PTB_SHADE_THREADS")) { int v = atoi(e); if (v == 64 || v == 128 || v == 256) TS = v; }
  uint32_t grid_shade = (uint32_t)persistent_grid(c, shade_fn(rs), TS);
  if (grid_shade > (P + TS - 1) / TS) grid_shade = (P + TS - 1) / TS;
  const void* fn_trace = trace_kernel(c, count, false);
  // camera rays of the binary tree walk it in packets (PTB_CAMERA_PACKET=0: the persistent kernel, as the wide tree does)
  // — when a warp's 32 work items are samples of ONE pixel (group a multiple of 32). C3 on B200: 256 spp 4256 -> 4344 Mrays/s;
  // with 4 samples per pixel a warp spans eight pixels and the packet loses (7.32 vs 6.75 ms per 4-spp step).
  bool cam_packet = !c->wide && rs.rp.group % 32u == 0u;
  if (const char* e = getenv("PTB_CAMERA_PACKET")) cam_packet = !c->wide && atoi(e) != 0;
  const void* fn_trace_cam = cam_packet ? (count ? (const void*)k_trace_camera<true> : (const void*)k_trace_camera<false>)
                                        : trace_kernel(c, count, true);
  // Camera samples answered from per-pixel candidate lists (ptb_camcand.cuh): one beam walk per pixel and call, then each
  // sample tests only what its pixel can see. Taken where the packets run, on scenes whose geometry is not L1 resident
  // anyway (>= 4096 primitives, as for the chunk streams below); PTB_CAMERA_CAND=0|1 overrides, PTB_CAMERA_CAND_K=1..16
  // shortens the lists (tests: forces the overflow fallback).
  const bool cand_ok = cam_packet && rs.rp.group % 32u == 0u;
  bool cam_cand = cand_ok && c->n_prims >= 4096;
  if (const char* e = getenv("PTB_CAMERA_CAND")) cam_cand = cand_ok && atoi(e) != 0;
  CamCandList cand{nullptr, nullptr, kCamCandMaxK};
  if (const char* e = getenv("PTB_CAMERA_CAND_K")) { int v = atoi(e); if (v >= 1 && v <= (int)kCamCandMaxK) cand.k = (uint32_t)v; }
  if (cam_cand) {
    PTB_CUDA_TRY(c, c->d_camcand.reserve((size_t)npix * cand.k * sizeof(uint4)));
    PTB_CUDA_TRY(c, c->d_camcand_count.reserve((size_t)npix * sizeof(uint32_t)));
    cand.entries = c->d_camcand.as<uint4>();
    cand.count = c->d_camcand_count.as<uint32_t>();
  }
  const void* fn_shadow = shadow_kernel(c);
  const int grid_trace = persistent_grid(c, fn_trace, T);
  const int grid_trace_cam = persistent_grid(c, fn_trace_cam, T);
  const int grid_shadow = persistent_grid(c, fn_shadow, T);
  int cam_fetch = c->dev.trace_fetch_threshold < 4 ? c->dev.trace_fetch_threshold : 4;
  if (const char* e = getenv("PTB_TRACE_FETCH_CAMERA")) { int v = atoi(e); if (v >= 1 && v <= 32) cam_fetch = v; }
  // hand-over point: live paths of a chunk at or below which the fused tail takes it (0: never; the traversal statistics
  // build counts in k_trace only, so it keeps the wavefront to the end)
  uint32_t tail_paths = 65536u;
  if (const char* e = getenv("PTB_TAIL_PATHS")) { long v = atol(e); if (v >= 0 && v <= (1l << 24)) tail_paths = (uint32_t)v; }
  if (count) tail_paths = 0u;
  if (tail_paths) {
    if (!c->s_tail) {
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = greatest priority: the tail's few blocks go first when slots free up
      PTB_CUDA_TRY(c, cudaStreamCreateWithPriority(&c->s_tail, cudaStreamNonBlocking, hi));
    }
    for (int k = 0; k < 2; ++k) {
      if (!c->ev_head_done[k]) PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_head_done[k], cudaEventDisableTiming));
      if (!c->ev_tail_done[k]) PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_tail_done[k], cudaEventDisableTiming));
    }
  }
  for (cudaEvent_t& e : c->ev_ring)
    if (!e) PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  if (!c->ev_fork) PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  if (!c->ev_join) PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  const bool two = rs.n_chunks > 1;
  // How many chunks run their wide iterations at the same time. Two (each on its own stream) fill each other's kernel
  // drains, but their rays compete for L1 / L2: measured on B200 (profiles/r2_sweeps.md) it loses 4 - 13 % on the 1 M-triangle
  // mesh and gains 5 % on the two-sphere / 14-primitive scenes, whose geometry lives in L1 whatever happens. One chunk at a
  // time still alternates between the two slots, so its fused tail overlaps the next chunk's iterations.
  int chunk_streams = c->n_prims < 4096 ? 2 : 1;
  if (const char* e = getenv("PTB_CHUNK_STREAMS")) { int v = atoi(e); if (v == 1 || v == 2) chunk_streams = v; }
  if (!two) chunk_streams = 1;
  if (chunk_streams == 2 && !c->s_work2) PTB_CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_work2, cudaStreamNonBlocking));
  uint32_t grid_tail = (uint32_t)c->sm_count * (4u / PTB_TAIL_WARPS);  // four warps per SM beside the next chunk (PTB_TAIL_BLOCKS)
  if (const char* e = getenv("PTB_TAIL_BLOCKS")) { int v = atoi(e); if (v >= 1 && v <= 65535) grid_tail = (uint32_t)v; }
  const uint32_t tail_blocks_max = (tail_paths + (uint32_t)kTailThreads - 1u) / (uint32_t)kTailThreads;  // one lane per path
  if (grid_tail > tail_blocks_max) grid_tail = tail_blocks_max;
  // The call's last tail has the machine to itself: one lane per path, but never more blocks than are resident at once
  // (45 KB of shared memory each) — a block that starts only when another has finished would keep the work queue from
  // running empty, which is what lets a warp go cooperative.
  uint32_t grid_tail_last = tail_blocks_max;
  if (tail_paths) {
#ifdef PTB_TAIL_CARVEOUT
    cudaFuncSetAttribute(tail_fn(rs, c), cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
#endif
    const uint32_t resident = (uint32_t)persistent_grid(c, tail_fn(rs, c), kTailThreads);
    if (grid_tail_last > resident) grid_tail_last = resident;
    if (grid_tail > resident) grid_tail = resident;
  }
  // Two chunks are in flight at any time, one per slot, each on its own stream: the block scheduler fills the drain of
  // one chunk's persistent kernel (its last long rays) and its small late iterations with the other chunk's blocks. The
  // FIRST chunk is half as long as the others, so the two streams stay half a chunk out of phase — while one is in its
  // narrow iterations the other is in its wide ones.
  // The host never waits for the iteration it has just enqueued: the chunk's state machine runs on the device
  // (k_win_prepare) and every kernel of an iteration that has nothing to do returns at once. The host stays at most
  // kAhead iterations in front of each chunk and reads the mirror of iteration d - kAhead to learn that the chunk is over.
  constexpr uint64_t kAhead = 3;
  struct ChunkRun {
    bool active = false;
    unsigned long long first = 0;
    uint32_t n_paths = 0;
    uint64_t depth = 0;    // iterations enqueued
    uint64_t drained = 0;  // iterations whose mirror has been read
    bool over = false;
    bool tail_pending = false;  // a k_tail launch of this slot may still be running
    uint64_t rays_ref_seen = 0;
    bool last = false;          // the call's last chunk: its tail runs alone and may take the whole machine
  };
  ChunkRun run[2];
  cudaStream_t wst[2] = {st, chunk_streams == 2 ? c->s_work2 : st};

  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_a, st));
  k_reset_counters<<<1, 1, 0, st>>>(rs.wc);
  k_reset_counters<<<1, 1, 0, st>>>(rs.wc2);
  c->stats.kernel_launches += 2;
  if (cam_cand) {
    const DevScene& d = c->dev;
    k_cam_candidates<<<(npix + 127) / 128, 128, 0, st>>>(d, rs.rp.width, rs.rp.height, rs.rp.row_begin, npix,
                                                        cam_cand_camera(d.cam_origin, d.cam_lower_left, d.cam_horizontal, d.cam_vertical),
                                                        cand.k, c->d_camcand.as<uint4>(), c->d_camcand_count.as<uint32_t>(),
                                                        count ? &rs.wc->nodes_fetched : nullptr);
    c->stats.kernel_launches += 1;
  }
  if (chunk_streams == 2) {  // the second stream starts after whatever the caller queued before this render
    PTB_CUDA_TRY(c, cudaEventRecord(c->ev_fork, st));
    PTB_CUDA_TRY(c, cudaStreamWaitEvent(wst[1], c->ev_fork, 0));
  }
  int32_t rc = PTB_OK;
  uint64_t iterations = 0;
  unsigned long long next_first = 0, paths_done = 0;
  uint32_t chunks_started = 0;

  auto prof_rec = [&](int sl, uint64_t it, int k, int which) {
    if (prof) cudaEventRecord(c->ev_prof[(sl * 4 + (int)(it & 3u)) * 8 + 2 * k + which], wst[sl]);
  };
  // start the next chunk in slot sl
  auto start_chunk = [&](int sl) -> int32_t {
    ChunkRun& R = run[sl];
    const SlotRefs& S = slots[sl];
    // chunk 0 is half a chunk long (see above); the others P, the last one what is left
    unsigned long long len = P;
    if (chunk_streams == 2 && chunks_started == 0 && total > (unsigned long long)P) len = (P / 2 + kWindow - 1) / kWindow * kWindow;
    if (len > total - next_first) len = total - next_first;
    R = ChunkRun();
    R.active = true;
    R.first = next_first;
    R.n_paths = (uint32_t)len;
    next_first += len;
    R.last = next_first >= total;
    ++chunks_started;
    cudaStream_t s = wst[sl];
    if (tail_paths)  // the slot's previous chunk has left it (a no-op while the event has never been recorded)
      PTB_CUDA_TRY(c, cudaStreamWaitEvent(s, c->ev_tail_done[sl], 0));
    PTB_CUDA_TRY(c, cudaMemsetAsync(S.q.win_count, 0, (size_t)S.q.n_windows * 4, s));
    if (R.n_paths % kWindow)  // slots of the last window that hold no path
      PTB_CUDA_TRY(c, cudaMemsetAsync(S.q.bin + R.n_paths, (int)kBinDead, kWindow - R.n_paths % kWindow, s));
    prof_rec(sl, 0, 0, 0);
    k_win_init<<<(S.q.n_windows + T - 1) / T, T, 0, s>>>(S.q, S.wc, R.n_paths);
    c->stats.kernel_launches += 1;
    return PTB_OK;
  };
  // enqueue iteration R.depth of the chunk in slot sl
  auto enqueue_iteration = [&](int sl) -> int32_t {
    ChunkRun& R = run[sl];
    const SlotRefs& S = slots[sl];
    const Queues& q = S.q;
    WaveCounters* wc = S.wc;
    cudaStream_t s = wst[sl];
    const uint64_t depth = R.depth;
    if (depth) prof_rec(sl, depth, 0, 0);
    k_win_scan<<<n_seg, 1024, 0, s>>>(q);
    k_win_prepare<<<1, 32, 0, s>>>(wc, q, n_seg, o.method, depth == 0 ? 0u : (depth == 1 ? 1u : 2u), (uint32_t)depth, tail_paths);
    if (depth) k_win_fill<<<grid_fill, T, 0, s>>>(q, wc);  // depth 0: work item i is slot i, no queue
    prof_rec(sl, depth, 0, 1);
    if (tail_paths && depth >= 2) {
      // k_tail runs in the iteration whose k_win_prepare hands the chunk over (and returns at once in all the others):
      // everything left of the chunk is then ONE launch on the side stream
      PTB_CUDA_TRY(c, cudaEventRecord(c->ev_head_done[sl], s));
      PTB_CUDA_TRY(c, cudaStreamWaitEvent(c->s_tail, c->ev_head_done[sl], 0));
      // (the last chunk's tail has nothing beside it: one lane per path instead of one block per SM)
      launch_tail(rs, c, S, R.last ? grid_tail_last : grid_tail, c->s_tail, (uint32_t)depth);
      PTB_CUDA_TRY(c, cudaEventRecord(c->ev_tail_done[sl], c->s_tail));
      R.tail_pending = true;
      c->stats.kernel_launches += 1;
    }
    prof_rec(sl, depth, 1, 0);
    if (depth == 0) {
      // camera rays of a warp finish together: refilling later (fewer, fuller service passes) suits them
      // (C3, camera rays only: threshold 8 -> 8105 Mrays/s, 4 -> 8311; bounce rays prefer 8, profiles/r1_sweeps.md)
      DevScene cam = c->dev;
      cam.trace_fetch_threshold = cam_fetch;
      if (cam_packet) PTB_CUDA_TRY(c, launch_trace_camera(fn_trace_cam, grid_trace_cam, s, cam, S.pool, q, wc, rs.rp, R.first, cand));
      else PTB_CUDA_TRY(c, launch_trace(fn_trace_cam, grid_trace_cam, s, cam, S.pool, q, wc, rs.rp, R.first));
    } else {
      PTB_CUDA_TRY(c, launch_trace(fn_trace, grid_trace, s, c->dev, S.pool, q, wc, rs.rp, 0ull));
    }
    prof_rec(sl, depth, 1, 1);
    prof_rec(sl, depth, 2, 0);
    launch_shade(rs, c, S, grid_shade, TS, s, depth == 0 ? R.first : kNoCamera);
    prof_rec(sl, depth, 2, 1);
    c->stats.kernel_launches += depth ? 5 : 4;
    c->stats.trace_launches += 1;
    if (mis) {
      prof_rec(sl, depth, 3, 0);
      PTB_CUDA_TRY(c, launch_shadow(fn_shadow, grid_shadow, s, c->dev, S.pool, q, wc));
      prof_rec(sl, depth, 3, 1);
      c->stats.kernel_launches += 1;
    }
    // pinned mirror + event of this iteration, a ring of four per slot
    const int r = sl * 4 + (int)(depth & 3u);
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->h_counters + r, wc, sizeof(WaveCounters), cudaMemcpyDeviceToHost, s));
    PTB_CUDA_TRY(c, cudaEventRecord(c->ev_ring[r], s));
    ++R.depth;
    ++iterations;
    if (R.depth > 4096) return set_error(c, PTB_ERR_INVALID, "wavefront did not terminate");
    return PTB_OK;
  };
  // reads the mirror of the oldest undrained iteration (its event must be complete)
  auto drain_one = [&](int sl) {
    ChunkRun& R = run[sl];
    const int r = sl * 4 + (int)(R.drained & 3u);
    if (prof) prof_collect(c, r, mis);
    if (c->h_counters[r].mode != 0u) R.over = true;
    R.rays_ref_seen = c->h_counters[r].rays_reference;
    ++R.drained;
  };

  while (rc == PTB_OK) {
    while (next_first < total && (int)run[0].active + (int)run[1].active < chunk_streams) {
      const int sl = two ? (int)(chunks_started & 1u) : 0;  // slots alternate: chunk k's tail may still be running in slot k & 1
      if (run[sl].active) break;
      const int32_t e = start_chunk(sl);
      if (e != PTB_OK) return e;
    }
    if (!run[0].active && !run[1].active) break;
    bool progress_made = false;
    for (int sl = 0; sl < 2 && rc == PTB_OK; ++sl) {
      ChunkRun& R = run[sl];
      if (!R.active) continue;
      if (R.depth - R.drained >= kAhead) {
        const int r = sl * 4 + (int)(R.drained & 3u);
        if (cudaEventQuery(c->ev_ring[r]) != cudaSuccess) continue;  // still running: look at the other chunk
        drain_one(sl);
        progress_made = true;
      } else if (!R.over) {
        const int32_t e = enqueue_iteration(sl);
        if (e != PTB_OK) return e;
        progress_made = true;
        continue;
      }
      if (R.over) {
        // the iterations still in flight are empty (or the hand-over itself); the timing build collects their events
        if (prof)
          while (R.drained < R.depth) {
            PTB_CUDA_TRY(c, cudaEventSynchronize(c->ev_ring[sl * 4 + (int)(R.drained & 3u)]));
            drain_one(sl);
          }
        R.active = false;
        paths_done += R.n_paths;
        progress_made = true;
        if (progress && paths_done < total && progress(user, paths_done / npix, R.rays_ref_seen)) rc = PTB_ERR_ABORTED;
      }
    }
    if (!progress_made) {
      // both chunks are kAhead iterations ahead of the device: wait for the older of the two oldest iterations
      int sl = run[0].active ? 0 : 1;
      if (run[0].active && run[1].active && run[1].depth - run[1].drained >= kAhead && run[0].depth - run[0].drained < kAhead) sl = 1;
      PTB_CUDA_TRY(c, cudaEventSynchronize(c->ev_ring[sl * 4 + (int)(run[sl].drained & 3u)]));
    }
  }
  // join: everything the second stream and the tail stream still hold comes back to the caller's stream
  if (chunk_streams == 2) {
    PTB_CUDA_TRY(c, cudaEventRecord(c->ev_join, wst[1]));
    PTB_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_join, 0));
  }
  if (tail_paths)
    for (int sl = 0; sl < 2; ++sl) PTB_CUDA_TRY(c, cudaStreamWaitEvent(st, c->ev_tail_done[sl], 0));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->h_counters + 8, rs.wc, sizeof(WaveCounters), cudaMemcpyDeviceToHost, st));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->h_counters + 9, rs.wc2, sizeof(WaveCounters), cudaMemcpyDeviceToHost, st));
  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_b, st));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(st));
  PTB_CUDA_TRY(c, cudaGetLastError());
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev_a, c->ev_b);
  const uint64_t ref_before = c->stats.rays_reference;
  fold_counters(c, c->h_counters[8], iterations);
  fold_counters(c, c->h_counters[9], 0);
  for (int k = 8; k < 10; ++k) {
    const WaveCounters& h = c->h_counters[k];
    c->stats.ms_tail += 1e-6 * (double)(h.tail_ns + (h.tail_t0 != ~0ull && h.tail_t1 > h.tail_t0 ? h.tail_t1 - h.tail_t0 : 0ull));
  }
  c->stats.render_ms = ms;
  if (rc == PTB_OK) {
    c->accum_samples += o.samples_per_pixel;
    if (progress) progress(user, o.samples_per_pixel, c->stats.rays_reference - ref_before);
  }
  return rc;
}

}  // namespace ptb
