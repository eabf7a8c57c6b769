// CPU statement of the per-pixel camera candidate lists (csrc/ptb_camcand.cuh) on the device SAH tree's CPU definition
// (oracle/sah_ref.hpp), and the check that answers every camera ray from its pixel's list gives the ordered walk's hit
// bit for bit. Test and evidence infrastructure (tests/test_camcand_oracle.py, scripts/camcand_probe.py); not on the
// product path. Built like the oracle: strict IEEE, no contraction.
#include <atomic>
#include <cmath>
#include <cstdint>
#include <thread>
#include <vector>

#include "../oracle/sah_ref.hpp"
#include "../oracle/ref_integrators.hpp"
#include "../raytracing-rust_b200/csrc/ptb_camcand_frustum.h"

namespace ref {
thread_local RngCursor g_rng;
}
using namespace ref;

namespace {

// ---- the frustum of one pixel (restates ptb_camcand.cuh: cam_candidates_pixel / cc_box; the f64 camera and the margins
// are the device's own, ptb_camcand_frustum.h) ------------------------------------------------------------------------
using ptb::CamCandCamera;
using ptb::kCcEps;
using ptb::kCcUvMargin;
using ptb::kCcBoxGrow;
using ptb::kCcKeySlack;
struct CcPixel {
  double n[4][3];  // outward unit normals of the four side planes (through the apex)
};

void cross3(const double a[3], const double b[3], double r[3]) { ptb::cc_cross(a, b, r); }
double dot3(const double a[3], const double b[3]) { return ptb::cc_dot(a, b); }
void unit3(double a[3]) {
  const double m = std::sqrt(dot3(a, a));
  for (int k = 0; k < 3; ++k) a[k] /= m;
}

CamCandCamera cc_camera(const Camera& cam) {
  const Vec3* src[4] = {&cam.origin, &cam.lower_left, &cam.horizontal, &cam.vertical};
  float v[4][3];
  for (int i = 0; i < 4; ++i) { v[i][0] = src[i]->x; v[i][1] = src[i]->y; v[i][2] = src[i]->z; }
  return ptb::cam_cand_camera(v[0], v[1], v[2], v[3]);
}
CcPixel cc_pixel(const CamCandCamera& c, uint32_t x, uint32_t y, uint32_t W, uint32_t H) {
  const double u0 = (double)x / (double)(W - 1) - kCcUvMargin, u1 = (double)(x + 1) / (double)(W - 1) + kCcUvMargin;
  const double v0 = 1.0 - (double)(y + 1) / (double)(H - 1) - kCcUvMargin, v1 = 1.0 - (double)y / (double)(H - 1) + kCcUvMargin;
  const double us[4] = {u0, u1, u1, u0}, vs[4] = {v0, v0, v1, v1};
  double d[4][3], dc[3] = {0, 0, 0};
  for (int i = 0; i < 4; ++i)
    for (int k = 0; k < 3; ++k) {
      d[i][k] = c.ll[k] - c.o[k] + c.h[k] * us[i] + c.vv[k] * vs[i];
      dc[k] += d[i][k];
    }
  CcPixel p;
  for (int i = 0; i < 4; ++i) {
    cross3(d[i], d[(i + 1) & 3], p.n[i]);
    if (dot3(p.n[i], dc) > 0.0) for (int k = 0; k < 3; ++k) p.n[i][k] = -p.n[i][k];
    unit3(p.n[i]);
  }
  return p;
}
// may a camera ray of the pixel reach the box? On acceptance `key` is a lower bound on the box_entry cull key of every
// such ray (float, rounded down). grow = false: the box as given, without the 2^-16 growth (the directed frustum check).
// rejected (may be null): 1 = outside a side plane, 2 = behind the apex.
bool cc_box(const CamCandCamera& c, const CcPixel& p, const double* bmn, const double* bmx, float& key, bool grow = true,
            int* rejected = nullptr) {
  double mx_abs = 0.0;
  for (int k = 0; k < 3; ++k) mx_abs = std::fmax(mx_abs, std::fmax(std::fabs(c.o[k]), std::fmax(std::fabs(bmn[k]), std::fabs(bmx[k]))));
  const double g = grow ? kCcBoxGrow * mx_abs : 0.0;
  double lo[3], hi[3], far2 = 0.0, near2 = 0.0;
  for (int k = 0; k < 3; ++k) {
    lo[k] = bmn[k] - g - c.o[k];
    hi[k] = bmx[k] + g - c.o[k];
    far2 += std::fmax(lo[k] * lo[k], hi[k] * hi[k]);
    const double nd = std::fmax(std::fmax(lo[k], 0.0), -hi[k]);
    near2 += nd * nd;
  }
  const double rmax = std::sqrt(far2);
  for (int i = 0; i < 4; ++i) {
    const double* n = p.n[i];
    const double pmin = n[0] * (n[0] > 0.0 ? lo[0] : hi[0]) + n[1] * (n[1] > 0.0 ? lo[1] : hi[1]) + n[2] * (n[2] > 0.0 ? lo[2] : hi[2]);
    if (pmin > c.sin_a * rmax) {
      if (rejected) *rejected = 1;
      return false;
    }
  }
  const double fmax_ = c.f[0] * (c.f[0] > 0.0 ? hi[0] : lo[0]) + c.f[1] * (c.f[1] > 0.0 ? hi[1] : lo[1]) + c.f[2] * (c.f[2] > 0.0 ? hi[2] : lo[2]);
  if (fmax_ < 0.0) {
    if (rejected) *rejected = 2;
    return false;
  }
  const double kd = std::sqrt(near2) * (1.0 - kCcEps) - kCcKeySlack * rmax;
  float kf = (float)kd;
  if ((double)kf > kd) kf = std::nextafter(kf, -INF_F);
  key = kf;
  return true;
}
bool cc_box(const CamCandCamera& c, const CcPixel& p, const float* bmn, const float* bmx, float& key) {
  const double dmn[3] = {bmn[0], bmn[1], bmn[2]}, dmx[3] = {bmx[0], bmx[1], bmx[2]};
  return cc_box(c, p, dmn, dmx, key);
}

struct Entry {
  float key;
  uint32_t ref;   // PTB_LEAF_BIT | slot
  uint32_t node;  // parent node | side << 31
};

template <class F>
void parallel_for(size_t n, int threads, F f) {
  unsigned nt = threads > 0 ? (unsigned)threads : std::thread::hardware_concurrency();
  if (nt == 0) nt = 1;
  std::atomic<size_t> next(0);
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < nt; ++t)
    pool.emplace_back([&]() {
      for (;;) {
        const size_t b = next.fetch_add(256);
        if (b >= n) break;
        f(b, b + 256 < n ? b + 256 : n);
      }
    });
  for (auto& th : pool) th.join();
}

}  // namespace

struct ccr_scene {
  std::vector<Prim> prims;
  Lbvh l;
  Camera cam;
};

extern "C" {

ccr_scene* ccr_create(const ptb_sphere* spheres, size_t ns, const ptb_triangle* tris, size_t nt, const ptb_camera* cam) {
  ccr_scene* s = new ccr_scene();
  for (size_t i = 0; i < ns; ++i) {
    Prim p{};
    p.is_sphere = 1;
    p.orig_id = (uint32_t)i;
    p.center = Vec3(spheres[i].center.x, spheres[i].center.y, spheres[i].center.z);
    p.radius = spheres[i].radius;
    s->prims.push_back(p);
  }
  for (size_t i = 0; i < nt; ++i) {
    Prim p{};
    p.orig_id = (uint32_t)(ns + i);
    for (int k = 0; k < 3; ++k) {
      p.p[k] = Vec3(tris[i].p[k].x, tris[i].p[k].y, tris[i].p[k].z);
      p.n[k] = Vec3(tris[i].n[k].x, tris[i].n[k].y, tris[i].n[k].z);
    }
    s->prims.push_back(p);
  }
  s->l.build(s->prims);
  sah_rebuild(s->l, 8);
  auto v = [](const ptb_vec3& a) { return Vec3(a.x, a.y, a.z); };
  s->cam.origin = v(cam->origin);
  s->cam.lower_left = v(cam->lower_left);
  s->cam.horizontal = v(cam->horizontal);
  s->cam.vertical = v(cam->vertical);
  return s;
}
void ccr_destroy(ccr_scene* s) { delete s; }

// Candidate lists of the pixels of rows [row_begin, row_begin + rows) of a W x H image: every leaf whose ancestors'
// boxes and own box pass cc_box, nearest key first. count[i] = the full number of candidates (the list holds the first
// min(count, K) of them, sorted; count > K: overflowed); visits[i] = nodes expanded by the beam walk.
void ccr_lists(const ccr_scene* s, uint32_t W, uint32_t H, uint32_t row_begin, uint32_t rows, uint32_t K, uint32_t* count,
               float* keys, uint32_t* refs, uint32_t* nodes, uint32_t* visits, int threads) {
  const CamCandCamera c = cc_camera(s->cam);
  const std::vector<ptb_bvh_node>& nd = s->l.nodes;
  parallel_for((size_t)W * rows, threads, [&](size_t b, size_t e) {
    std::vector<Entry> list;
    for (size_t i = b; i < e; ++i) {
      const uint32_t x = (uint32_t)(i % W), y = row_begin + (uint32_t)(i / W);
      const CcPixel p = cc_pixel(c, x, y, W, H);
      list.clear();
      uint32_t stack[128];
      int sp = 0;
      uint32_t nv = 0;
      if (!nd.empty()) stack[sp++] = 0;
      while (sp > 0) {
        const uint32_t n = stack[--sp];
        ++nv;
        const ptb_bvh_node& q = nd[n];
        for (int side = 0; side < 2; ++side) {
          float key;
          if (!cc_box(c, p, side ? q.rmin : q.lmin, side ? q.rmax : q.lmax, key)) continue;
          const uint32_t ch = side ? q.right : q.left;
          if (ch & PTB_LEAF_BIT) list.push_back(Entry{key, ch, n | ((uint32_t)side << 31)});
          else stack[sp++] = ch;
        }
      }
      std::stable_sort(list.begin(), list.end(), [](const Entry& a, const Entry& b) { return a.key < b.key; });
      count[i] = (uint32_t)list.size();
      visits[i] = nv;
      for (uint32_t k = 0; k < K; ++k) {
        const bool have = k < list.size();
        keys[i * K + k] = have ? list[k].key : INF_F;
        refs[i * K + k] = have ? list[k].ref : 0xFFFFFFFFu;
        nodes[i * K + k] = have ? list[k].node : 0u;
      }
    }
  });
}

// Every camera ray of samples [sample_offset, sample_offset + spp) of the pixels ccr_lists described, built with the
// device's camera arithmetic (wavefront.cu camera_direction + make_ray), answered twice: by the ordered walk
// (Lbvh::closest_hit) and, for pixels that did not overflow, from the pixel's list as k_trace_camera does (entries in key
// order, stop at the first key above the best t, the walk's box test on the leaf box, ties to the lower primitive id).
// out[0] rays, [1] rays answered from a list, [2] of those whose hit differs (t bits or primitive), [3] list entries
// tested (box + primitive), [4] primitive tests of the list path, [5] walk nodes, [6] walk primitive tests over the list
// rays, [7] list entries whose primitive is hit (t > 0) although the walk's box test rejects its leaf box, [8] list
// entries (all of the list, not only those a ray reached) whose key exceeds the cull key box_entry computes for the ray on
// their leaf box while its geometric test passes, and is positive (the key must bound the cull key from below wherever
// that decides anything: a best t is positive, so a key at or below 0, a box around the apex, never stops a list). hist (3 x kHistBins, may be null): per
// list ray, the entries tested, the primitive tests of the list path and the ordered walk's nodes (last bin: that many or
// more).
static const int kHistBins = 256;
void ccr_check(const ccr_scene* s, uint32_t W, uint32_t H, uint32_t row_begin, uint32_t rows, uint32_t K, const uint32_t* count,
               const float* keys, const uint32_t* refs, const uint32_t* nodes, uint32_t spp, uint32_t sample_offset, uint64_t seed,
               int threads, uint64_t out[9], uint64_t* hist) {
  std::vector<std::atomic<uint64_t>> hacc(3 * kHistBins);
  for (auto& a : hacc) a = 0;
  std::atomic<uint64_t> acc[9];
  for (auto& a : acc) a = 0;
  const Lbvh& l = s->l;
  const uint32_t key2[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  parallel_for((size_t)W * rows, threads, [&](size_t b, size_t e) {
    uint64_t loc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<uint64_t> hl(3 * kHistBins, 0);
    auto bin = [](uint64_t v) { return v < (uint64_t)kHistBins - 1 ? (size_t)v : (size_t)kHistBins - 1; };
    for (size_t i = b; i < e; ++i) {
      const uint32_t x = (uint32_t)(i % W), y = row_begin + (uint32_t)(i / W);
      const uint32_t pixel = y * W + x;
      const bool listed = count[i] <= K;
      for (uint32_t smp = sample_offset; smp < sample_offset + spp; ++smp) {
        uint32_t ctr[4] = {pixel, smp, (0u << 8) | RNG_JITTER, 0u}, r[4];
        Philox::block(ctr, key2, r);
        const Float u = (u32_to_unit(r[0]) + (Float)x) / (Float)(W - 1u);
        const Float v = 1.0f - (u32_to_unit(r[1]) + (Float)y) / (Float)(H - 1u);
        const Ray ray = s->cam.get_ray(u, v);
        Hit hw;
        uint32_t pw;
        uint64_t wn = 0, wp = 0;
        l.closest_hit(ray, hw, pw, &wn, &wp);
        ++loc[0];
        if (!listed) continue;
        ++loc[1];
        loc[5] += wn;
        loc[6] += wp;
        const Lbvh::SlabRay slab = Lbvh::make_slab_ray(ray);
        for (uint32_t k = 0; k < count[i]; ++k) {
          const size_t j = i * K + k;
          const ptb_bvh_node& q = l.nodes[nodes[j] & 0x7FFFFFFFu];
          const bool side = (nodes[j] >> 31) != 0;
          Float tk;
          if (Lbvh::box_hit(side ? q.rmin : q.lmin, side ? q.rmax : q.lmax, slab, INF_F, tk) && keys[j] > tk && keys[j] > 0.0f) ++loc[8];
        }
        const uint64_t e0 = loc[3], p0 = loc[4];
        Float best_t = INF_F;
        uint32_t best = PTB_MISS;
        Hit h;
        for (uint32_t k = 0; k < count[i]; ++k) {
          const size_t j = i * K + k;
          if (keys[j] > best_t) break;
          const uint32_t slot = refs[j] & ~PTB_LEAF_BIT;
          const ptb_bvh_node& q = l.nodes[nodes[j] & 0x7FFFFFFFu];
          const bool side = (nodes[j] >> 31) != 0;
          Float tk;
          const bool pass = Lbvh::box_hit(side ? q.rmin : q.lmin, side ? q.rmax : q.lmax, slab, best_t, tk);
          ++loc[3];
          const uint32_t pid = l.prim_sorted[slot];
          if (!pass) {
            if (l.prims[pid].get_int(ray, h) && h.t > 0.0f && h.t <= best_t) ++loc[7];
            continue;
          }
          ++loc[4];
          if (l.prims[pid].get_int(ray, h) && h.t > 0.0f) {
            if (h.t < best_t || (h.t == best_t && pid < best)) { best_t = h.t; best = pid; }
          }
        }
        hl[bin(loc[3] - e0)]++;
        hl[kHistBins + bin(loc[4] - p0)]++;
        hl[2 * kHistBins + bin(wn)]++;
        const bool same = best == pw && (pw == PTB_MISS || f2u(best_t) == f2u(hw.t));
        if (!same) ++loc[2];
      }
    }
    for (int k = 0; k < 9; ++k) acc[k] += loc[k];
    for (size_t k = 0; k < hl.size(); ++k) hacc[k] += hl[k];
  });
  for (int k = 0; k < 9; ++k) out[k] = acc[k];
  if (hist) for (size_t k = 0; k < hacc.size(); ++k) hist[k] = hacc[k];
}

// Directed check of the frustum predicate alone (argument (b) of ptb_camcand.cuh: sin_a and the uv margin cover the
// rounding of the computed camera directions; the box growth is switched off). For every pixel of rows [row_begin,
// row_begin + rows): the four corner rays of its jitter square (jitter 0 and 1 - 2^-24 on each axis, the extremes of
// u32_to_unit), built with the device's camera arithmetic (camera_direction + make_ray), and on each of them the
// zero-extent boxes at dist[j] times the ray's distance from the apex to the image plane, placed in f64 on the computed
// ray. Every such box must pass the pixel's side planes and lie ahead of the apex. out[0] boxes tested, [1] rejected by a
// side plane, [2] rejected as behind the apex. worst[0]: the largest (signed distance outside a side plane) / (sin_a *
// distance from the apex) over the boxes, which stays below 1 while the check passes.
void ccr_frustum_corners(const ccr_scene* s, uint32_t W, uint32_t H, uint32_t row_begin, uint32_t rows, const double* dist,
                         uint32_t ndist, int threads, uint64_t out[3], double* worst) {
  const CamCandCamera c = cc_camera(s->cam);
  std::atomic<uint64_t> acc[3];
  for (auto& a : acc) a = 0;
  std::vector<double> worst_part((size_t)W * rows, -INFINITY);
  const Float j1 = u32_to_unit(0xFFFFFFFFu);  // 1 - 2^-24
  parallel_for((size_t)W * rows, threads, [&](size_t b, size_t e) {
    uint64_t loc[3] = {0, 0, 0};
    for (size_t i = b; i < e; ++i) {
      const uint32_t x = (uint32_t)(i % W), y = row_begin + (uint32_t)(i / W);
      const CcPixel p = cc_pixel(c, x, y, W, H);
      double wmax = -INFINITY;
      for (int corner = 0; corner < 4; ++corner) {
        const Float ju = (corner & 1) ? j1 : 0.0f, jv = (corner & 2) ? j1 : 0.0f;
        const Float u = (ju + (Float)x) / (Float)(W - 1u);
        const Float v = 1.0f - (jv + (Float)y) / (Float)(H - 1u);
        const Ray ray = s->cam.get_ray(u, v);
        const double d[3] = {ray.direction.x, ray.direction.y, ray.direction.z};
        const double llo[3] = {c.ll[0] - c.o[0], c.ll[1] - c.o[1], c.ll[2] - c.o[2]};
        const double to_plane = dot3(llo, c.f) / dot3(d, c.f);  // along the ray, to the image plane
        for (uint32_t j = 0; j < ndist; ++j) {
          double pt[3], rel[3];
          for (int k = 0; k < 3; ++k) {
            pt[k] = c.o[k] + dist[j] * to_plane * d[k];
            rel[k] = pt[k] - c.o[k];
          }
          float key;
          int why = 0;
          ++loc[0];
          if (!cc_box(c, p, pt, pt, key, false, &why)) ++loc[why];
          const double r = std::sqrt(dot3(rel, rel));
          for (int q = 0; q < 4; ++q) wmax = std::fmax(wmax, dot3(p.n[q], rel) / (c.sin_a * r));
        }
      }
      worst_part[i] = wmax;
    }
    for (int k = 0; k < 3; ++k) acc[k] += loc[k];
  });
  for (int k = 0; k < 3; ++k) out[k] = acc[k];
  double w = -INFINITY;
  for (double v : worst_part) w = std::fmax(w, v);
  *worst = w;
}

}  // extern "C"
