// Per-pixel camera candidate lists (device): one beam walk per pixel and render call, reused by every sample of the pixel.
//
// Why. Every camera ray starts at the pinhole (the device camera has no aperture: ptb_camera holds the four vectors of
// camera.rs:57-63 and nothing else) and passes through its pixel's jitter square. The primitives a pixel's rays can hit
// are a property of the pixel, not of the sample; the packet walk (ptb_packet.cuh) nevertheless walks the top of the
// tree again for every 32 samples. k_cam_candidates walks the tree ONCE per pixel with the pixel's frustum and stores the
// leaves it reaches, nearest first; k_trace_camera then answers each sample from that list.
//
// Frustum. The cone from cam_origin through u in [x/(W-1), (x+1)/(W-1)], v in [1-(y+1)/(H-1), 1-y/(H-1)] (random_sampler.rs
// with the reference's W-1 / H-1), the square widened by 2^-20 on each side. A box is rejected only when it lies entirely
// outside one of the four side planes (p-vertex test) or entirely behind the apex. All of it in f64: once per pixel.
// Error budget (eps = 2^-23). (a) u = fl(fl(jitter + x) / (W-1)) lies in [x/(W-1)(1-eps), (x+1)/(W-1)(1+eps)] (rounding is
// monotone and x, x+1 are exact), |u| <= 2: the 2^-20 widening covers it; v likewise. (b) camera_direction's sum
// ll + h u + vv v - o takes four roundings per component, each at most eps/2 of a partial sum bounded by
// S_k = |ll_k| + 2|h_k| + 2|vv_k| + |o_k|: the computed vector is D(u, v) + delta with |delta| <= 2 eps |S| (taken as 4);
// |D| >= dmin, the distance of the image plane from the apex; the normalisation rounds each component by eps/2 and
// scales all of them alike. So the computed direction lies within angle a of the exact cone, sin a <= 4 eps |S| / dmin +
// eps; the test uses twice that (`sin_a`) and accepts a box unless its nearest point lies more than sin_a * (its farthest
// distance from the apex) outside a side plane. (c) box_entry accepts a box up to its widened slabs: near planes moved by
// 2 eps |o_i| along axis i, far side stretched by 1 + 4 gamma(3), one rounding of the fma: a few eps of the box's distance.
// Every box is grown by 2^-16 * max(|o|, |box|) per side, which covers (c) many times over. The CPU statement of all
// this (scripts/camcand_ref.cpp) checks the lists against the ordered walk over millions of jittered camera rays, and
// checks (b) alone on the corner rays of every pixel's jitter square with the growth switched off. The f64 camera and
// the margins live in ptb_camcand_frustum.h, which that statement includes. sin_a alone also covers (a): it is twice
// (b)'s bound, and the spare half, 4 eps |S| / dmin >= 4 eps (|h| + |vv|) / dmin, exceeds the angle of at most
// 2 eps (|h| + |vv|) / dmin by which (a) turns a direction. So the uv margin is redundant (the corner check passes
// without it).
//
// List. Up to K entries per pixel, sorted by key: (key, leaf reference, parent node | side << 31). The key is the
// distance from the apex to the grown box, times (1 - eps), less 2^-16 of its farthest distance, rounded down to f32: a
// lower bound, for every ray of the pixel, on box_entry's cull key tmin - kCullSlack * max(|tmin|, |hmin|) of the leaf box
// (tmin * |d| >= that distance, |d| = 1 within 2 eps, and kCullSlack = 32 eps < 2^-16) wherever that key is positive. A
// box around the apex has a key below 0 and a cull key that may be lower still; neither stops anything, since every best
// t is positive. More than K candidates: the pixel
// is marked overflowed (count = kNone) and its samples take the packet walk.
//
// Why the answer is the walk's, bit for bit (the argument k_trace_camera's list path rests on):
// 1. The ordered walk returns the minimum (t, then the lower primitive id) over the primitives whose ancestor boxes pass
//    box_entry. Its culling never removes a closer hit: a box is culled only when its key tkey exceeds the best t so far,
//    and the key of a box holding a hit at t is at most t (kCullSlack, ptb_intersect.cuh). The geometric part of
//    box_entry is monotone under box inclusion (every plane distance is one correctly rounded fma, monotone in the plane),
//    and each child box lies inside its parent's, so a leaf whose own box passes has ancestors that pass: the walk's
//    answer is the minimum over the primitives whose LEAF box passes box_entry.
// 2. The list holds every primitive whose leaf box any ray of the pixel can pass box_entry on (the frustum above is a
//    superset of the computed rays, grown beyond box_entry's widening). Each lane applies box_entry to the entry's leaf
//    box itself (a prim_t hit outside the box the walk accepts is then rejected as the walk rejects it), and stops at
//    the first entry whose key exceeds its best t, which is at most that entry's tkey for this ray, so the walk would cull
//    it too. So the lane computes the same minimum over the same set, with the same tie rule.
#pragma once
#include <cmath>
#include "ptb_camcand_frustum.h"
#include "ptb_intersect.cuh"

namespace ptb {

#ifndef PTB_CAMCAND_K
#define PTB_CAMCAND_K 16  // entries per pixel (scripts/camcand_probe.py: overflow fraction on C3 at 1080p)
#endif
constexpr uint32_t kCamCandMaxK = PTB_CAMCAND_K;
// The frustum starts every ray at the pinhole: a camera with an aperture (a lens radius in ptb_camera) would break the lists.
static_assert(sizeof(ptb_camera) == 4 * sizeof(ptb_vec3), "camera candidate lists assume a pinhole camera (no aperture)");

struct CamCandList {  // what k_trace_camera reads; count == nullptr: the list path is off
  const uint4* entries;   // [npix * k] (key bits, leaf reference, parent node | side << 31, 0), nearest key first
  const uint32_t* count;  // [npix] entries of the pixel, kNone: overflowed
  uint32_t k;
};

// host: cam_cand_camera (ptb_camcand_frustum.h) of the device scene's camera
inline CamCandCamera cam_cand_camera(v3 o, v3 ll, v3 h, v3 vv) {
  const float fo[3] = {o.x, o.y, o.z}, fll[3] = {ll.x, ll.y, ll.z}, fh[3] = {h.x, h.y, h.z}, fvv[3] = {vv.x, vv.y, vv.z};
  return cam_cand_camera(fo, fll, fh, fvv);
}

#ifdef __CUDACC__
// May a camera ray of the pixel (side planes n[4]) reach the box? On acceptance `key` bounds box_entry's cull key from below.
__device__ __forceinline__ bool cc_box(const CamCandCamera& c, const double n[4][3], const float* b, float& key) {
  double mx_abs = 0.0;
  for (int k = 0; k < 3; ++k) mx_abs = fmax(mx_abs, fmax(fabs(c.o[k]), fmax(fabs((double)b[k]), fabs((double)b[3 + k]))));
  const double g = kCcBoxGrow * mx_abs;
  double lo[3], hi[3], far2 = 0.0, near2 = 0.0;
  for (int k = 0; k < 3; ++k) {
    lo[k] = (double)b[k] - g - c.o[k];
    hi[k] = (double)b[3 + k] + g - c.o[k];
    far2 += fmax(lo[k] * lo[k], hi[k] * hi[k]);
    const double nd = fmax(fmax(lo[k], 0.0), -hi[k]);
    near2 += nd * nd;
  }
  const double rmax = sqrt(far2);
  for (int i = 0; i < 4; ++i) {
    const double pmin = n[i][0] * (n[i][0] > 0.0 ? lo[0] : hi[0]) + n[i][1] * (n[i][1] > 0.0 ? lo[1] : hi[1]) +
                        n[i][2] * (n[i][2] > 0.0 ? lo[2] : hi[2]);
    if (pmin > c.sin_a * rmax) return false;
  }
  const double fmx = c.f[0] * (c.f[0] > 0.0 ? hi[0] : lo[0]) + c.f[1] * (c.f[1] > 0.0 ? hi[1] : lo[1]) + c.f[2] * (c.f[2] > 0.0 ? hi[2] : lo[2]);
  if (fmx < 0.0) return false;
  key = __double2float_rd(__dmul_rn(sqrt(near2), 1.0 - kCcEps) - kCcKeySlack * rmax);
  return true;
}

// One pixel's list; returns the nodes the beam walk visited.
PTB_DEV uint32_t cam_candidates_pixel(const DevScene& sc, uint32_t width, uint32_t height, uint32_t row_begin, uint32_t lin,
                                     const CamCandCamera& c, uint32_t k, uint4* entries, uint32_t* count) {
  const uint32_t x = lin % width, y = row_begin + lin / width;
  const double u0 = (double)x / (double)(width - 1u) - kCcUvMargin, u1 = (double)(x + 1u) / (double)(width - 1u) + kCcUvMargin;
  const double v0 = 1.0 - (double)(y + 1u) / (double)(height - 1u) - kCcUvMargin, v1 = 1.0 - (double)y / (double)(height - 1u) + kCcUvMargin;
  double n[4][3];
  {
    const double us[4] = {u0, u1, u1, u0}, vs[4] = {v0, v0, v1, v1};
    double d[4][3], dc[3] = {0.0, 0.0, 0.0};
    for (int i = 0; i < 4; ++i)
      for (int a = 0; a < 3; ++a) {
        d[i][a] = c.ll[a] - c.o[a] + c.h[a] * us[i] + c.vv[a] * vs[i];
        dc[a] += d[i][a];
      }
    for (int i = 0; i < 4; ++i) {
      cc_cross(d[i], d[(i + 1) & 3], n[i]);
      const double s = (cc_dot(n[i], dc) > 0.0 ? -1.0 : 1.0) / sqrt(cc_dot(n[i], n[i]));
      for (int a = 0; a < 3; ++a) n[i][a] *= s;
    }
  }
  float keys[kCamCandMaxK];
  uint32_t refs[kCamCandMaxK], parents[kCamCandMaxK];
  uint32_t m = 0;
  bool over = false;
  uint32_t stack[64];
  int sp = 0;
  uint32_t visits = 0;
  if (sc.n_prims) stack[sp++] = 0u;
  while (sp > 0 && !over) {
    const uint32_t nd = stack[--sp];
    ++visits;
    const float* box = reinterpret_cast<const float*>(sc.nodes + nd);
    const uint32_t ch[2] = {__ldg(&sc.nodes[nd].n3.x), __ldg(&sc.nodes[nd].n3.y)};
    for (int side = 0; side < 2; ++side) {
      float key;
      if (!cc_box(c, n, box + 6 * side, key)) continue;
      if (!(ch[side] & PTB_LEAF_BIT)) {
        if (sp < 64) stack[sp++] = ch[side];
        else over = true;  // deeper than the builders go: leave the pixel to the packet walk
        continue;
      }
      if (m == k) { over = true; break; }
      uint32_t j = m++;  // insertion, nearest key first (ties: walk order)
      while (j > 0 && keys[j - 1] > key) {
        keys[j] = keys[j - 1]; refs[j] = refs[j - 1]; parents[j] = parents[j - 1];
        --j;
      }
      keys[j] = key; refs[j] = ch[side]; parents[j] = nd | ((uint32_t)side << 31);
    }
  }
  count[lin] = over ? kNone : m;
  if (over) return visits;
  uint4* out = entries + (size_t)lin * k;
  for (uint32_t j = 0; j < m; ++j) out[j] = make_uint4(__float_as_uint(keys[j]), refs[j], parents[j], 0u);
  return visits;
}

// One thread per pixel of the call's image tile (lin = (y - row_begin) * width + x): the pixel's candidate list.
// nodes_counted (traversal statistics only, else null): receives the beam walk's node visits, once per pixel.
__global__ void __launch_bounds__(128) k_cam_candidates(DevScene sc, uint32_t width, uint32_t height, uint32_t row_begin,
                                                        uint32_t npix, CamCandCamera c, uint32_t k, uint4* entries, uint32_t* count,
                                                        unsigned long long* nodes_counted) {
  const uint32_t lin = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t visits = 0;
  if (lin < npix) visits = cam_candidates_pixel(sc, width, height, row_begin, lin, c, k, entries, count);
  if (nodes_counted) {
    for (int off = 16; off > 0; off >>= 1) visits += __shfl_xor_sync(0xffffffffu, visits, off);
    if ((threadIdx.x & 31u) == 0u && visits) atomicAdd(nodes_counted, (unsigned long long)visits);
  }
}

// The camera ray of each valid lane answered from its pixel's list (all 32 lanes call this together; the list is the same
// for all of them and each entry is one broadcast load). Same result as packet_trace (see the argument above).
// n_prims counts the lane's primitive tests (COUNT).
template <bool COUNT>
PTB_DEV void cand_trace(const DevScene& sc, const CamCandList& cl, uint32_t lin, uint32_t cnt, const Ray& ray, bool valid,
                        float& best_t, uint32_t& best_ref, uint32_t& n_prims) {
  best_t = __int_as_float(0x7f800000);
  best_ref = kNone;
  const SlabRay sr = make_slab_ray(ray);
  const uint4* e = cl.entries + (size_t)lin * cl.k;
  for (uint32_t j = 0; j < cnt; ++j) {
    const uint4 en = __ldg(e + j);
    const float key = __uint_as_float(en.x);
    const bool want = valid && key <= best_t;
    if (!__any_sync(0xffffffffu, want)) break;  // keys ascend: no later entry is wanted either
    if (!want) continue;
    const float* b = reinterpret_cast<const float*>(sc.nodes + (en.z & 0x7FFFFFFFu)) + ((en.z >> 31) ? 6 : 0);
    float tk;
    if (!box_entry(__ldg(b), __ldg(b + 1), __ldg(b + 2), __ldg(b + 3), __ldg(b + 4), __ldg(b + 5), sr, best_t, tk)) continue;
    const float t = prim_t(sc, ray, en.y);
    if (COUNT) ++n_prims;
    if (t > 0.0f) {
      if (t < best_t) {
        best_t = t;
        best_ref = en.y;
      } else if (t == best_t) {
        const uint32_t a = __ldg(sc.slot_prim + (en.y & kSlotMask));
        const uint32_t bb = __ldg(sc.slot_prim + (best_ref & kSlotMask));
        if (a < bb) best_ref = en.y;
      }
    }
  }
}
#endif

}  // namespace ptb
