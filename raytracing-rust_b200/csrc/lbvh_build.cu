// ptb200 — device LBVH build (sm_100a). Replaces Bvh::new / build_bvh
// (implementations/src/acceleration/mod.rs:58-160; split.rs) with a fully parallel construction:
//   K2  primitive AABB + centroid + scene centroid bounds   (PrimitiveInfo::new, acceleration/mod.rs:29-41;
//                                                            get_aabb sphere.rs:175-181, triangle.rs:285-307)
//   K3  30-bit Morton codes
//   K4  stable LSD radix sort, 4 passes x 8 bits, (key = Morton, value = primitive id)
//   K5  Karras-2012 hierarchy, duplicate keys tie-broken by index
//   K6  bottom-up AABB refit with atomic arrival flags (AABB::merge, aabb.rs:59-67); every 64-byte node stores
//       both children's boxes
//   then primitives are gathered into Morton (slot) order as 3 x float4 records.
// The result is bit-exact against oracle/lbvh_ref.hpp (tests/test_gpu_lbvh.py): min/max and the Morton arithmetic are
// order-independent and IEEE-exact, the sort is stable, the hierarchy is a pure function of the sorted keys.
#include <cstdarg>
#include <cstring>

#include "ptb_internal.h"

namespace ptb {

// ------------------------------------------------------------------------------------------ helpers
__device__ __forceinline__ uint32_t float_flip(float f) {  // order-preserving float -> uint
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float float_unflip(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}
__device__ __forceinline__ uint32_t expand_bits10(uint32_t v) {
  v = (v * 0x00010001u) & 0xFF0000FFu;
  v = (v * 0x00000101u) & 0x0F00F00Fu;
  v = (v * 0x00000011u) & 0xC30C30C3u;
  v = (v * 0x00000005u) & 0x49249249u;
  return v;
}
__device__ __forceinline__ uint32_t quantise10(float c, float cmin, float ext) {
  float n = ext > 0.0f ? (c - cmin) / ext : 0.0f;
  float s = fminf(fmaxf(n * 1024.0f, 0.0f), 1023.0f);
  return (uint32_t)s;
}

// ------------------------------------------------------------------------------------------ K2
// bounds[0..2] = flipped min of centroids, bounds[3..5] = flipped max; bounds[6..8] / [9..11] = the same of the boxes
// themselves (the root box of the SAH builder)
__global__ void k_prim_bounds(const ptb_sphere* __restrict__ spheres, uint32_t n_spheres,
                              const ptb_triangle* __restrict__ tris, uint32_t n_tris, float4* __restrict__ bmin,
                              float4* __restrict__ bmax, uint32_t* __restrict__ bounds) {
  const uint32_t n = n_spheres + n_tris;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const float inf = __int_as_float(0x7f800000);
  v3 cmin = mk(inf, inf, inf), cmax = mk(-inf, -inf, -inf);
  uint32_t bx[6] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u};
  if (i < n) {
    v3 mn, mx;
    if (i < n_spheres) {
      const ptb_sphere s = spheres[i];
      const v3 c = mk(s.center.x, s.center.y, s.center.z);
      mn = c - s.radius * mk(1.0f, 1.0f, 1.0f);
      mx = c + s.radius * mk(1.0f, 1.0f, 1.0f);
    } else {
      const ptb_triangle* t = tris + (i - n_spheres);
      const v3 p0 = mk(t->p[0].x, t->p[0].y, t->p[0].z), p1 = mk(t->p[1].x, t->p[1].y, t->p[1].z),
               p2 = mk(t->p[2].x, t->p[2].y, t->p[2].z);
      mn = vmin(p0, vmin(p1, p2));
      mx = vmax(p0, vmax(p1, p2));
    }
    bmin[i] = make_float4(mn.x, mn.y, mn.z, 0.0f);
    bmax[i] = make_float4(mx.x, mx.y, mx.z, 0.0f);
    const v3 c = 0.5f * (mn + mx);
    cmin = c;
    cmax = c;
    bx[0] = float_flip(mn.x); bx[1] = float_flip(mn.y); bx[2] = float_flip(mn.z);
    bx[3] = float_flip(mx.x); bx[4] = float_flip(mx.y); bx[5] = float_flip(mx.z);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) bx[k] = __reduce_min_sync(0xffffffffu, bx[k]);
#pragma unroll
  for (int k = 3; k < 6; ++k) bx[k] = __reduce_max_sync(0xffffffffu, bx[k]);
  // warp reduce then one atomic per warp per component
  for (int off = 16; off > 0; off >>= 1) {
    cmin.x = fminf(cmin.x, __shfl_xor_sync(0xffffffffu, cmin.x, off));
    cmin.y = fminf(cmin.y, __shfl_xor_sync(0xffffffffu, cmin.y, off));
    cmin.z = fminf(cmin.z, __shfl_xor_sync(0xffffffffu, cmin.z, off));
    cmax.x = fmaxf(cmax.x, __shfl_xor_sync(0xffffffffu, cmax.x, off));
    cmax.y = fmaxf(cmax.y, __shfl_xor_sync(0xffffffffu, cmax.y, off));
    cmax.z = fmaxf(cmax.z, __shfl_xor_sync(0xffffffffu, cmax.z, off));
  }
  // block reduce (12 words x warps), then ONE atomic per word per block: at 10 M primitives the per-warp atomics on twelve
  // addresses were a quarter of the kernel. Warps without a primitive contribute the identities (+inf / -inf).
  __shared__ uint32_t red[12][32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, n_warps = (blockDim.x + 31u) >> 5;
  if (lane == 0u) {
    red[0][warp] = float_flip(cmin.x); red[1][warp] = float_flip(cmin.y); red[2][warp] = float_flip(cmin.z);
    red[3][warp] = float_flip(cmax.x); red[4][warp] = float_flip(cmax.y); red[5][warp] = float_flip(cmax.z);
#pragma unroll
    for (int k = 0; k < 6; ++k) red[6 + k][warp] = bx[k];
  }
  __syncthreads();
  if (threadIdx.x < 12u) {
    const bool is_min = threadIdx.x < 3u || (threadIdx.x >= 6u && threadIdx.x < 9u);
    uint32_t v = red[threadIdx.x][0];
    for (uint32_t w = 1; w < n_warps; ++w) v = is_min ? min(v, red[threadIdx.x][w]) : max(v, red[threadIdx.x][w]);
    if (is_min) atomicMin(bounds + threadIdx.x, v);
    else atomicMax(bounds + threadIdx.x, v);
  }
}

// ------------------------------------------------------------------------------------------ K3
__global__ void k_morton(const float4* __restrict__ bmin, const float4* __restrict__ bmax, uint32_t n,
                         const uint32_t* __restrict__ bounds, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const v3 cmin = mk(float_unflip(bounds[0]), float_unflip(bounds[1]), float_unflip(bounds[2]));
  const v3 cmax = mk(float_unflip(bounds[3]), float_unflip(bounds[4]), float_unflip(bounds[5]));
  const v3 ext = cmax - cmin;
  const v3 c = 0.5f * (from4(bmin[i]) + from4(bmax[i]));
  const float e = fmaxf(ext.x, fmaxf(ext.y, ext.z));  // cubic grid (see oracle/lbvh_ref.hpp)
  const uint32_t qx = quantise10(c.x, cmin.x, e), qy = quantise10(c.y, cmin.y, e), qz = quantise10(c.z, cmin.z, e);
  keys[i] = (expand_bits10(qx) << 2) | (expand_bits10(qy) << 1) | expand_bits10(qz);
  vals[i] = i;
}

// ------------------------------------------------------------------------------------------ K4: radix sort
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_ITEMS = 16;                       // keys per thread
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;     // 4096 keys per block
constexpr int RS_WARP_TILE = 32 * RS_ITEMS;        // contiguous keys per warp (keeps the sort stable)

// Per-warp digit counts of this block's tile. Warp w owns tile elements [w*512, (w+1)*512), walked 32 at a time in
// order; lanes holding the same digit are grouped with match.any so only the group leader touches shared memory.
template <bool SCATTER>
__global__ void __launch_bounds__(RS_THREADS)
k_radix_pass(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, uint32_t* __restrict__ keys_out,
             uint32_t* __restrict__ vals_out, uint32_t n, int shift, uint32_t* __restrict__ hist, uint32_t n_tiles,
             const uint32_t* __restrict__ row_base) {
  __shared__ uint32_t cnt[RS_WARPS][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tile = blockIdx.x;
  for (int d = threadIdx.x; d < RS_WARPS * 256; d += RS_THREADS) (&cnt[0][0])[d] = 0;
  __syncthreads();

  uint32_t key[RS_ITEMS];
  const uint32_t base = tile * RS_TILE + warp * RS_WARP_TILE + lane;
#pragma unroll
  for (int c = 0; c < RS_ITEMS; ++c) {
    const uint32_t idx = base + c * 32;
    key[c] = idx < n ? keys_in[idx] : 0xFFFFFFFFu;
  }
#pragma unroll
  for (int c = 0; c < RS_ITEMS; ++c) {
    const uint32_t idx = base + c * 32;
    const bool valid = idx < n;
    const uint32_t digit = (key[c] >> shift) & 255u;
    const uint32_t peers = __match_any_sync(0xffffffffu, valid ? digit : (256u + lane));
    if (valid && (__ffs(peers) - 1) == lane) cnt[warp][digit] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  if (!SCATTER) {
    const int d = threadIdx.x;  // RS_THREADS == 256 digits
    uint32_t total = 0;
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) total += cnt[w][d];
    hist[(size_t)d * n_tiles + tile] = total;
    return;
  }
  {  // turn counts into running output offsets: global digit offset + counts of the earlier warps of this tile
    const int d = threadIdx.x;
    uint32_t run = hist[(size_t)d * n_tiles + tile] + row_base[d];
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      const uint32_t c = cnt[w][d];
      cnt[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int c = 0; c < RS_ITEMS; ++c) {
    const uint32_t idx = base + c * 32;
    const bool valid = idx < n;
    const uint32_t digit = (key[c] >> shift) & 255u;
    const uint32_t peers = __match_any_sync(0xffffffffu, valid ? digit : (256u + lane));
    if (valid) {
      const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
      const uint32_t dst = cnt[warp][digit] + rank;
      keys_out[dst] = key[c];
      vals_out[dst] = vals_in[idx];
    }
    __syncwarp();
    if (valid && (__ffs(peers) - 1) == lane) cnt[warp][digit] += __popc(peers);
    __syncwarp();
  }
}

// Exclusive scan of hist in digit-major order (256 rows x n_tiles), in two launches: one block per digit row scans its
// row in place and leaves the row total in row_base[digit]; a single block then turns the 256 totals into row bases,
// which k_radix_pass<true> adds. (The first version scanned all rows in ONE block: 0.6 ms per pass at 4096 tiles.)
__global__ void __launch_bounds__(256) k_radix_scan(uint32_t* __restrict__ hist, uint32_t n_tiles, uint32_t* __restrict__ row_base) {
  __shared__ uint32_t warp_sum[8];
  __shared__ uint32_t carry_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t* r = hist + (size_t)blockIdx.x * n_tiles;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (uint32_t b = 0; b < n_tiles; b += 256) {
    const uint32_t i = b + threadIdx.x;
    const uint32_t v = i < n_tiles ? r[i] : 0;
    uint32_t inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
      if (lane >= off) inc += t;
    }
    if (lane == 31) warp_sum[warp] = inc;
    __syncthreads();
    uint32_t before = carry_s;
#pragma unroll
    for (int w = 0; w < 8; ++w) before += w < warp ? warp_sum[w] : 0u;
    if (i < n_tiles) r[i] = before + inc - v;
    __syncthreads();
    if (threadIdx.x == 255) carry_s = before + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) row_base[blockIdx.x] = carry_s;
}
__global__ void __launch_bounds__(256) k_radix_bases(uint32_t* __restrict__ row_base) {
  __shared__ uint32_t warp_sum[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t v = row_base[threadIdx.x];
  uint32_t inc = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= off) inc += t;
  }
  if (lane == 31) warp_sum[warp] = inc;
  __syncthreads();
  uint32_t before = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) before += w < warp ? warp_sum[w] : 0u;
  row_base[threadIdx.x] = before + inc - v;
}

// Stable LSD radix sort of (key, value) pairs, `passes` x 8 bits from bit 0; ping-pongs between (ka, va) and (kb, vb)
// and returns with the result in (ka, va) (the pointers are swapped). `hist` holds 256 * ceil(n / 4096) words.
// Also used by the closest-hit batch API to order its rays (wavefront.cu).
void radix_sort_pairs(Ctx* c, uint32_t*& ka, uint32_t*& va, uint32_t*& kb, uint32_t*& vb, uint32_t n, int passes, uint32_t* hist) {
  const uint32_t n_tiles = (n + RS_TILE - 1) / RS_TILE;
  for (int pass = 0; pass < passes; ++pass) {
    const int shift = pass * 8;
    uint32_t* row_base = hist + (size_t)256 * n_tiles;
    k_radix_pass<false><<<n_tiles, RS_THREADS, 0, c->stream>>>(ka, va, kb, vb, n, shift, hist, n_tiles, row_base);
    k_radix_scan<<<256, 256, 0, c->stream>>>(hist, n_tiles, row_base);
    k_radix_bases<<<1, 256, 0, c->stream>>>(row_base);
    k_radix_pass<true><<<n_tiles, RS_THREADS, 0, c->stream>>>(ka, va, kb, vb, n, shift, hist, n_tiles, row_base);
    c->stats.kernel_launches += 4;
    uint32_t* t;
    t = ka; ka = kb; kb = t;
    t = va; va = vb; vb = t;
  }
}
size_t radix_sort_hist_words(uint32_t n) { return (size_t)256 * ((n + RS_TILE - 1) / RS_TILE) + 256; }

// ------------------------------------------------------------------------------------------ K5
__device__ __forceinline__ int lbvh_delta(const uint32_t* __restrict__ keys, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  const uint32_t a = keys[i], b = keys[j];
  if (a == b) return 32 + __clz((uint32_t)i ^ (uint32_t)j);
  return __clz(a ^ b);
}
__global__ void k_hierarchy(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ prim_sorted, uint32_t n_prims,
                            uint32_t n_spheres, BvhNode* __restrict__ nodes, uint32_t* __restrict__ leaf_parent,
                            uint2* __restrict__ range) {
  const int n = (int)n_prims;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  const int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) < 0 ? -1 : 1;
  const int dmin = lbvh_delta(keys, n, i, i - d);
  int lmax = 2;
  while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
  int l = 0;
  for (int t = lmax / 2; t >= 1; t /= 2)
    if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
  const int j = i + l * d;
  const int dnode = lbvh_delta(keys, n, i, j);
  int s = 0;
  for (int t = (l + 1) / 2;; t = (t + 1) / 2) {
    if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    if (t == 1) break;
  }
  const int gam = i + s * d + (d < 0 ? -1 : 0);
  const int lo = min(i, j), hi = max(i, j);
  if (range) range[i] = make_uint2((uint32_t)lo, (uint32_t)hi);  // Morton positions the node covers (wide collapse)
  uint32_t left, right;
  if (lo == gam) {
    left = PTB_LEAF_BIT | (prim_sorted[gam] < n_spheres ? kSphereBit : 0u) | (uint32_t)gam;
    leaf_parent[gam] = (uint32_t)i;
  } else {
    left = (uint32_t)gam;
    nodes[gam].n3.z = (uint32_t)i;
  }
  if (hi == gam + 1) {
    right = PTB_LEAF_BIT | (prim_sorted[gam + 1] < n_spheres ? kSphereBit : 0u) | (uint32_t)(gam + 1);
    leaf_parent[gam + 1] = (uint32_t)i;
  } else {
    right = (uint32_t)(gam + 1);
    nodes[gam + 1].n3.z = (uint32_t)i;
  }
  nodes[i].n3.x = left;
  nodes[i].n3.y = right;
  nodes[i].n3.w = 0u;
  if (i == 0) nodes[0].n3.z = kNone;
}

// ------------------------------------------------------------------------------------------ K6
__device__ __forceinline__ void child_box(uint32_t ref, const uint32_t* __restrict__ prim_sorted,
                                          const float4* __restrict__ bmin, const float4* __restrict__ bmax,
                                          const float4* nbmin, const float4* nbmax, v3& mn, v3& mx) {
  if (ref & PTB_LEAF_BIT) {
    const uint32_t p = prim_sorted[ref & kSlotMask];
    mn = from4(bmin[p]);
    mx = from4(bmax[p]);
  } else {
    mn = from4(__ldcg(nbmin + ref));  // written by another SM: read through L2
    mx = from4(__ldcg(nbmax + ref));
  }
}
__global__ void k_refit(uint32_t n_prims, const uint32_t* __restrict__ prim_sorted, const uint32_t* __restrict__ leaf_parent,
                        const float4* __restrict__ bmin, const float4* __restrict__ bmax, BvhNode* nodes, float4* nbmin,
                        float4* nbmax, uint32_t* flags) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_prims) return;
  uint32_t cur = leaf_parent[s];
  while (cur != kNone) {
    __threadfence();
    if (atomicAdd(flags + cur, 1u) == 0u) return;  // first arrival: the sibling subtree is not finished yet
    __threadfence();
    const uint4 links = nodes[cur].n3;  // written by k_hierarchy (previous launch)
    v3 lmn, lmx, rmn, rmx;
    child_box(links.x, prim_sorted, bmin, bmax, nbmin, nbmax, lmn, lmx);
    child_box(links.y, prim_sorted, bmin, bmax, nbmin, nbmax, rmn, rmx);
    nodes[cur].n0 = make_float4(lmn.x, lmn.y, lmn.z, lmx.x);
    nodes[cur].n1 = make_float4(lmx.y, lmx.z, rmn.x, rmn.y);
    nodes[cur].n2 = make_float4(rmn.z, rmx.x, rmx.y, rmx.z);
    const v3 mn = vmin(lmn, rmn), mx = vmax(lmx, rmx);
    __stcg(nbmin + cur, make_float4(mn.x, mn.y, mn.z, 0.0f));
    __stcg(nbmax + cur, make_float4(mx.x, mx.y, mx.z, 0.0f));
    cur = links.z;
  }
}

// single primitive: one node, both child slots reference leaf 0 (see oracle/lbvh_ref.hpp)
__global__ void k_single_node(const uint32_t* __restrict__ prim_sorted, uint32_t n_spheres, const float4* __restrict__ bmin,
                              const float4* __restrict__ bmax, BvhNode* nodes) {
  const uint32_t p = prim_sorted[0];
  const v3 mn = from4(bmin[p]), mx = from4(bmax[p]);
  const uint32_t ref = PTB_LEAF_BIT | (p < n_spheres ? kSphereBit : 0u);
  nodes[0].n0 = make_float4(mn.x, mn.y, mn.z, mx.x);
  nodes[0].n1 = make_float4(mx.y, mx.z, mn.x, mn.y);
  nodes[0].n2 = make_float4(mn.z, mx.x, mx.y, mx.z);
  nodes[0].n3 = make_uint4(ref, ref, kNone, 0u);
}

// ------------------------------------------------------------------------------------------ 16-bit traversal nodes
// The traversal kernels read 32-byte nodes (ptb_intersect.cuh: 16-bit boxes); CPU definition: oracle/lbvh_ref.hpp
// quantise(). Grid: the scene box = union of the root's two child boxes; per axis q_step = (float)(extent / 65535), moved
// up until q_min + 65535 * q_step reaches the far side (f64), 0 for a flat axis. A box is snapped OUTWARDS in f64:
// q_lo = floor((lo - q_min) / q_step) stepped down while q_min + q_lo * q_step > lo, q_hi the mirror image.
__global__ void k_qframe(const BvhNode* __restrict__ nodes, float* __restrict__ frame) {
  const BvhNode r = nodes[0];
  const float mn[3] = {fminf(r.n0.x, r.n1.z), fminf(r.n0.y, r.n1.w), fminf(r.n0.z, r.n2.x)};
  const float mx[3] = {fmaxf(r.n0.w, r.n2.y), fmaxf(r.n1.x, r.n2.z), fmaxf(r.n1.y, r.n2.w)};
  for (int k = 0; k < 3; ++k) {
    const double ext = (double)mx[k] - (double)mn[k];
    float step = (float)(ext / 65535.0);
    if (ext > 0.0)
      while ((double)mn[k] + 65535.0 * (double)step < (double)mx[k]) step = __uint_as_float(__float_as_uint(step) + 1u);
    else
      step = 0.0f;
    frame[k] = mn[k];
    frame[3 + k] = step;
  }
}
PTB_DEV uint32_t q_floor(float v, float mn, float step) {
  if (!(step > 0.0f)) return 0u;
  double q = floor(((double)v - (double)mn) / (double)step);
  q = q < 0.0 ? 0.0 : (q > 65535.0 ? 65535.0 : q);
  while (q > 0.0 && (double)mn + q * (double)step > (double)v) q -= 1.0;
  return (uint32_t)q;
}
PTB_DEV uint32_t q_ceil(float v, float mn, float step) {
  if (!(step > 0.0f)) return 0u;
  double q = ceil(((double)v - (double)mn) / (double)step);
  q = q < 0.0 ? 0.0 : (q > 65535.0 ? 65535.0 : q);
  while (q < 65535.0 && (double)mn + q * (double)step < (double)v) q += 1.0;
  return (uint32_t)q;
}
__global__ void __launch_bounds__(256)
k_quantise_nodes(const BvhNode* __restrict__ nodes, uint32_t n_nodes, const float* __restrict__ frame, uint4* __restrict__ qnodes) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_nodes) return;
  const BvhNode nd = nodes[i];
  const float mn[3] = {frame[0], frame[1], frame[2]}, st[3] = {frame[3], frame[4], frame[5]};
  const float llo[3] = {nd.n0.x, nd.n0.y, nd.n0.z}, lhi[3] = {nd.n0.w, nd.n1.x, nd.n1.y};
  const float rlo[3] = {nd.n1.z, nd.n1.w, nd.n2.x}, rhi[3] = {nd.n2.y, nd.n2.z, nd.n2.w};
  uint32_t l[3], r[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    l[k] = q_floor(llo[k], mn[k], st[k]) | (q_ceil(lhi[k], mn[k], st[k]) << 16);
    r[k] = q_floor(rlo[k], mn[k], st[k]) | (q_ceil(rhi[k], mn[k], st[k]) << 16);
  }
  qnodes[2u * (size_t)i] = make_uint4(l[0], l[1], l[2], r[0]);
  qnodes[2u * (size_t)i + 1u] = make_uint4(r[1], r[2], nd.n3.x, nd.n3.y);
}

// ------------------------------------------------------------------------------------------ gather into slot order
__global__ void k_gather(const ptb_sphere* __restrict__ spheres, uint32_t n_spheres, const ptb_triangle* __restrict__ tris,
                         uint32_t n_prims, const uint32_t* __restrict__ prim_sorted, const DevMaterial* __restrict__ mats,
                         uint32_t n_mats, float4* __restrict__ geom, float4* __restrict__ normals, uint32_t* __restrict__ slot_mat,
                         uint32_t* __restrict__ prim_slot) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_prims) return;
  const uint32_t p = prim_sorted[slot];
  prim_slot[p] = slot;
  uint32_t mat;
  float4 g0, g1, g2, m0, m1, m2;
  if (p < n_spheres) {
    const ptb_sphere s = spheres[p];
    g0 = make_float4(s.center.x, s.center.y, s.center.z, s.radius);
    g1 = g2 = m0 = m1 = m2 = make_float4(0.f, 0.f, 0.f, 0.f);
    mat = s.material;
  } else {
    const ptb_triangle* t = tris + (p - n_spheres);
    g0 = make_float4(t->p[0].x, t->p[0].y, t->p[0].z, 0.f);
    g1 = make_float4(t->p[1].x, t->p[1].y, t->p[1].z, 0.f);
    g2 = make_float4(t->p[2].x, t->p[2].y, t->p[2].z, 0.f);
    m0 = make_float4(t->n[0].x, t->n[0].y, t->n[0].z, 0.f);
    m1 = make_float4(t->n[1].x, t->n[1].y, t->n[1].z, 0.f);
    m2 = make_float4(t->n[2].x, t->n[2].y, t->n[2].z, 0.f);
    mat = t->material;
  }
  geom[3 * (size_t)slot + 0] = g0;
  geom[3 * (size_t)slot + 1] = g1;
  geom[3 * (size_t)slot + 2] = g2;
  normals[3 * (size_t)slot + 0] = m0;
  normals[3 * (size_t)slot + 1] = m1;
  normals[3 * (size_t)slot + 2] = m2;
  // an out-of-range index is reported by k_collect_lights (commit then fails with PTB_ERR_INVALID); it must not be
  // dereferenced here, the primitives never passed through the host
  const uint32_t kind = mat < n_mats ? mats[mat].kind : 0u;
  slot_mat[slot] = (kind << 24) | (mat & 0x00FFFFFFu);
}
__global__ void k_light_slots(const uint32_t* __restrict__ light_prims, uint32_t n_lights, uint32_t n_spheres,
                              const uint32_t* __restrict__ prim_slot, uint32_t* __restrict__ lights) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_lights) return;
  const uint32_t p = light_prims[i];
  lights[i] = (p < n_spheres ? kSphereBit : 0u) | prim_slot[p];
}

// ------------------------------------------------------------------------------------------ refit of a kept tree
// PTB_BUILD_REFIT: one thread per slot of the binary tree of the last full commit. It reads its primitive once, writes the
// slot's records as k_gather does, computes the box with k_prim_bounds' arithmetic (bit-identical), stores it in slot order
// and climbs leaf_parent with k_refit's arrival flags. A leaf child's box comes from the slot-ordered array, so an arrival
// costs no dependent prim_sorted -> bmin[p] load, and nothing goes through original order or the global bounds atomics.
__global__ void k_refit_slots(const ptb_sphere* __restrict__ spheres, uint32_t n_spheres, const ptb_triangle* __restrict__ tris,
                              uint32_t n_prims, const uint32_t* __restrict__ slot_prim, const uint32_t* __restrict__ leaf_parent,
                              const DevMaterial* __restrict__ mats, uint32_t n_mats, float4* __restrict__ geom,
                              float4* __restrict__ normals, uint32_t* __restrict__ slot_mat, float4* sbmin, float4* sbmax,
                              BvhNode* nodes, float4* nbmin, float4* nbmax, uint32_t* flags) {
  const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_prims) return;
  const uint32_t p = slot_prim[slot];
  uint32_t mat;
  float4 g0, g1, g2, m0, m1, m2;
  v3 mn, mx;
  if (p < n_spheres) {
    const ptb_sphere s = spheres[p];
    const v3 c = mk(s.center.x, s.center.y, s.center.z);
    mn = c - s.radius * mk(1.0f, 1.0f, 1.0f);
    mx = c + s.radius * mk(1.0f, 1.0f, 1.0f);
    g0 = make_float4(s.center.x, s.center.y, s.center.z, s.radius);
    g1 = g2 = m0 = m1 = m2 = make_float4(0.f, 0.f, 0.f, 0.f);
    mat = s.material;
  } else {
    const ptb_triangle* t = tris + (p - n_spheres);
    const v3 p0 = mk(t->p[0].x, t->p[0].y, t->p[0].z), p1 = mk(t->p[1].x, t->p[1].y, t->p[1].z),
             p2 = mk(t->p[2].x, t->p[2].y, t->p[2].z);
    mn = vmin(p0, vmin(p1, p2));
    mx = vmax(p0, vmax(p1, p2));
    g0 = make_float4(p0.x, p0.y, p0.z, 0.f);
    g1 = make_float4(p1.x, p1.y, p1.z, 0.f);
    g2 = make_float4(p2.x, p2.y, p2.z, 0.f);
    m0 = make_float4(t->n[0].x, t->n[0].y, t->n[0].z, 0.f);
    m1 = make_float4(t->n[1].x, t->n[1].y, t->n[1].z, 0.f);
    m2 = make_float4(t->n[2].x, t->n[2].y, t->n[2].z, 0.f);
    mat = t->material;
  }
  geom[3 * (size_t)slot + 0] = g0;
  geom[3 * (size_t)slot + 1] = g1;
  geom[3 * (size_t)slot + 2] = g2;
  normals[3 * (size_t)slot + 0] = m0;
  normals[3 * (size_t)slot + 1] = m1;
  normals[3 * (size_t)slot + 2] = m2;
  const uint32_t kind = mat < n_mats ? mats[mat].kind : 0u;  // out of range: reported by k_collect_lights, as in k_gather
  slot_mat[slot] = (kind << 24) | (mat & 0x00FFFFFFu);
  __stcg(sbmin + slot, make_float4(mn.x, mn.y, mn.z, 0.0f));
  __stcg(sbmax + slot, make_float4(mx.x, mx.y, mx.z, 0.0f));
  if (n_prims < 2) return;  // the single node is k_single_node's
  uint32_t cur = leaf_parent[slot];
  while (cur != kNone) {
    __threadfence();
    if (atomicAdd(flags + cur, 1u) == 0u) return;  // first arrival: the sibling subtree is not finished yet
    __threadfence();
    const uint4 links = nodes[cur].n3;
    v3 lmn, lmx, rmn, rmx;
    const float4 *lo = (links.x & PTB_LEAF_BIT) ? sbmin + (links.x & kSlotMask) : nbmin + links.x,
                 *hi = (links.x & PTB_LEAF_BIT) ? sbmax + (links.x & kSlotMask) : nbmax + links.x;
    lmn = from4(__ldcg(lo));  // written by another thread of this launch: read through L2
    lmx = from4(__ldcg(hi));
    lo = (links.y & PTB_LEAF_BIT) ? sbmin + (links.y & kSlotMask) : nbmin + links.y;
    hi = (links.y & PTB_LEAF_BIT) ? sbmax + (links.y & kSlotMask) : nbmax + links.y;
    rmn = from4(__ldcg(lo));
    rmx = from4(__ldcg(hi));
    nodes[cur].n0 = make_float4(lmn.x, lmn.y, lmn.z, lmx.x);
    nodes[cur].n1 = make_float4(lmx.y, lmx.z, rmn.x, rmn.y);
    nodes[cur].n2 = make_float4(rmn.z, rmx.x, rmx.y, rmx.z);
    const v3 bmn = vmin(lmn, rmn), bmx = vmax(lmx, rmx);
    __stcg(nbmin + cur, make_float4(bmn.x, bmn.y, bmn.z, 0.0f));
    __stcg(nbmax + cur, make_float4(bmx.x, bmx.y, bmx.z, 0.0f));
    cur = links.z;
  }
}

// ------------------------------------------------------------------------------------------ SAH cost of the binary tree
// (0.125 * sum over inner nodes of SA(node) + sum over leaves of SA(leaf box)) / SA(root), SA = 2 (xy + yz + zx) of the f32
// box in f64 (the reference's cost model, split.rs:161-163,176). A node's own box is the union of its two child boxes, a
// leaf's box is the child box its parent stores. Fixed summation order: block partials, then one block in index order.
PTB_DEV double box_area(float lx, float ly, float lz, float hx, float hy, float hz) {
  const double dx = (double)hx - (double)lx, dy = (double)hy - (double)ly, dz = (double)hz - (double)lz;
  return 2.0 * (dx * dy + dy * dz + dz * dx);
}
constexpr int kCostThreads = 256;
__device__ __forceinline__ double block_sum_fixed(double v, double* sh) {
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int s = kCostThreads / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  return sh[0];
}
__global__ void __launch_bounds__(kCostThreads)
k_sah_cost_partial(const BvhNode* __restrict__ nodes, uint32_t n_nodes, uint32_t n_prims, double* __restrict__ partial) {
  __shared__ double sh[kCostThreads];
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  double v = 0.0;
  if (i < n_nodes) {
    const BvhNode nd = nodes[i];
    v = 0.125 * box_area(fminf(nd.n0.x, nd.n1.z), fminf(nd.n0.y, nd.n1.w), fminf(nd.n0.z, nd.n2.x), fmaxf(nd.n0.w, nd.n2.y),
                         fmaxf(nd.n1.x, nd.n2.z), fmaxf(nd.n1.y, nd.n2.w));
    if (nd.n3.x & PTB_LEAF_BIT) v += box_area(nd.n0.x, nd.n0.y, nd.n0.z, nd.n0.w, nd.n1.x, nd.n1.y);
    if ((nd.n3.y & PTB_LEAF_BIT) && n_prims > 1)  // one primitive: both child slots name the same leaf
      v += box_area(nd.n1.z, nd.n1.w, nd.n2.x, nd.n2.y, nd.n2.z, nd.n2.w);
  }
  const double s = block_sum_fixed(v, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}
__global__ void __launch_bounds__(kCostThreads)
k_sah_cost_final(const double* __restrict__ partial, uint32_t n_partial, const BvhNode* __restrict__ nodes, double* __restrict__ out) {
  __shared__ double sh[kCostThreads];
  const uint32_t per = (n_partial + kCostThreads - 1) / kCostThreads;
  const uint32_t b = threadIdx.x * per, e = min(b + per, n_partial);
  double v = 0.0;
  for (uint32_t k = b; k < e; ++k) v += partial[k];
  const double s = block_sum_fixed(v, sh);
  if (threadIdx.x == 0) {
    const BvhNode r = nodes[0];
    const double root = box_area(fminf(r.n0.x, r.n1.z), fminf(r.n0.y, r.n1.w), fminf(r.n0.z, r.n2.x), fmaxf(r.n0.w, r.n2.y),
                                 fmaxf(r.n1.x, r.n2.z), fmaxf(r.n1.y, r.n2.w));
    *out = root > 0.0 ? s / root : 0.0;
  }
}
int32_t tree_sah_cost(Ctx* c, double* cost) {
  *cost = 0.0;
  if (c->n_prims == 0) return PTB_OK;
  const uint32_t n_nodes = (uint32_t)c->n_nodes, nb = (n_nodes + kCostThreads - 1) / kCostThreads;
  DevBuf& tmp = c->scratch[2];  // build temporary (the bounds words), free between commits
  PTB_CUDA_TRY(c, tmp.reserve(((size_t)nb + 1) * sizeof(double)));
  double* d = tmp.as<double>();
  k_sah_cost_partial<<<nb, kCostThreads, 0, c->stream>>>(c->d_nodes.as<BvhNode>(), n_nodes, (uint32_t)c->n_prims, d + 1);
  k_sah_cost_final<<<1, kCostThreads, 0, c->stream>>>(d + 1, nb, c->d_nodes.as<BvhNode>(), d);
  c->stats.kernel_launches += 2;
  PTB_CUDA_TRY(c, cudaMemcpyAsync(cost, d, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

// ------------------------------------------------------------------------------------------ host: sky table
// Sky::new (implementations/src/sky.rs:20-37) = generate_values (textures/mod.rs:32-50) + Distribution2D::new
// (statistics/distributions.rs:11-44, 82-99), in the reference's f32 operation order.
static void host_texture_colour(const Ctx* c, uint32_t tex, const float d[3], const float p[3], float out[3]) {
  const ptb_texture& t = c->textures[tex];
  auto it = c->texture_data.find(tex);
  TexWords words{it == c->texture_data.end() ? nullptr : it->second.data.data()};
  const uint32_t w = it == c->texture_data.end() ? 0u : it->second.width, h = it == c->texture_data.end() ? 0u : it->second.height;
  const v3 col = texture_eval(t.kind, mk(t.a.x, t.a.y, t.a.z), mk(t.b.x, t.b.y, t.b.z), w, h, words, mk(d[0], d[1], d[2]),
                              mk(p[0], p[1], p[2]));
  out[0] = col.x; out[1] = col.y; out[2] = col.z;
}
static void dist1d(const float* values, size_t n, std::vector<float>& pdf, std::vector<float>& cdf) {
  cdf.assign(1, 0.0f);
  for (size_t i = 1; i <= n; ++i) cdf.push_back(cdf[i - 1] + values[i - 1]);
  const float c = cdf[n];
  for (auto& v : cdf)
    if (c != 0.0f) v /= c;
  pdf.clear();
  float last = 0.0f;
  for (size_t i = 1; i <= n; ++i) {
    pdf.push_back(cdf[i] - last);
    last = cdf[i];
  }
}
static int32_t build_sky(Ctx* c) {
  const uint32_t rx = c->sky.sampler_res_x, ry = c->sky.sampler_res_y;
  c->dev.sky_tex = c->sky.texture;
  c->dev.sky_rx = rx;
  c->dev.sky_ry = ry;
  c->dev.sky_ycdf = c->dev.sky_ypdf = c->dev.sky_xcdf = c->dev.sky_xpdf = nullptr;
  if ((rx | ry) == 0) return PTB_OK;
  if (rx == 0 || ry == 0) return set_error(c, PTB_ERR_INVALID, "sky sampler_res must be (0,0) or both non-zero");
  std::vector<float> values;
  values.reserve((size_t)rx * ry);
  const float step_x = 1.0f / (float)rx, step_y = 1.0f / (float)ry;
  for (uint32_t y = 0; y < ry; ++y)
    for (uint32_t x = 0; x < rx; ++x) {
      float u = ((float)x + 0.5f) * step_x, v = ((float)y + 0.5f) * step_y;
      float phi = u * 2.0f * kPi, theta = v * kPi;
      float sin_theta = sinf(theta);
      float dir[3] = {cosf(phi) * sin_theta, sinf(phi) * sin_theta, cosf(theta)};
      float zero[3] = {0, 0, 0}, col[3];
      host_texture_colour(c, c->sky.texture, dir, zero, col);
      values.push_back((0.2126f * col[0] + 0.7152f * col[1] + 0.0722f * col[2]) * sin_theta);
    }
  std::vector<float> ycdf, ypdf, xcdf, xpdf, yvals, p, q;
  for (uint32_t y = 0; y < ry; ++y) {
    dist1d(&values[(size_t)y * rx], rx, p, q);
    xpdf.insert(xpdf.end(), p.begin(), p.end());
    xcdf.insert(xcdf.end(), q.begin(), q.end());
    float row_sum = 0.0f;
    for (uint32_t x = 0; x < rx; ++x) row_sum += values[(size_t)y * rx + x];
    yvals.push_back(row_sum);
  }
  dist1d(yvals.data(), ry, ypdf, ycdf);
  PTB_CUDA_TRY(c, c->d_sky_ycdf.reserve(ycdf.size() * 4));
  PTB_CUDA_TRY(c, c->d_sky_ypdf.reserve(ypdf.size() * 4));
  PTB_CUDA_TRY(c, c->d_sky_xcdf.reserve(xcdf.size() * 4));
  PTB_CUDA_TRY(c, c->d_sky_xpdf.reserve(xpdf.size() * 4));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_sky_ycdf.p, ycdf.data(), ycdf.size() * 4, cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_sky_ypdf.p, ypdf.data(), ypdf.size() * 4, cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_sky_xcdf.p, xcdf.data(), xcdf.size() * 4, cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_sky_xpdf.p, xpdf.data(), xpdf.size() * 4, cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // the host vectors die at scope exit
  c->dev.sky_ycdf = c->d_sky_ycdf.as<float>();
  c->dev.sky_ypdf = c->d_sky_ypdf.as<float>();
  c->dev.sky_xcdf = c->d_sky_xcdf.as<float>();
  c->dev.sky_xpdf = c->d_sky_xpdf.as<float>();
  return PTB_OK;
}

// ------------------------------------------------------------------------------------------ indexed mesh expansion
// ptb_scene_set_mesh: mesh triangle i becomes ptb_triangle record i of d_raw_tris, before anything else of the commit reads
// that array. The words are copied, never computed on, so the records are bit-identical to a host-side gather. An index out
// of range is not dereferenced: its corner becomes (0, 0, 0) and the commit fails through the word the material check uses
// (out[1] |= 2 for a vertex index, 4 for a normal index; out[2] / out[3] = max of ~triangle, i.e. the first such triangle).
constexpr uint32_t kExpandThreads = 256;
constexpr uint32_t kMeshWords = sizeof(ptb_mesh_triangle) / 4, kTriWords = sizeof(ptb_triangle) / 4;  // 7, 19
static_assert(sizeof(ptb_mesh_triangle) == 28 && sizeof(ptb_triangle) == 76, "record layouts");

__device__ __forceinline__ void expand_record(const uint32_t* idx, uint32_t* rec, uint32_t tri, const uint32_t* __restrict__ vtx,
                                              uint32_t nv, const uint32_t* __restrict__ nrm, uint32_t nn, uint32_t* out) {
  bool bad_v = false, bad_n = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint32_t a = idx[k], b = idx[3 + k];
    uint32_t p[3] = {0u, 0u, 0u}, q[3] = {0u, 0u, 0u};
    if (a < nv) { p[0] = vtx[3 * (size_t)a]; p[1] = vtx[3 * (size_t)a + 1]; p[2] = vtx[3 * (size_t)a + 2]; }
    else bad_v = true;
    if (b < nn) { q[0] = nrm[3 * (size_t)b]; q[1] = nrm[3 * (size_t)b + 1]; q[2] = nrm[3 * (size_t)b + 2]; }
    else bad_n = true;
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      rec[3 * k + w] = p[w];
      rec[9 + 3 * k + w] = q[w];
    }
  }
  rec[18] = idx[6];
  if (bad_v) { atomicOr(out + 1, 2u); atomicMax(out + 2, ~tri); }
  if (bad_n) { atomicOr(out + 1, 4u); atomicMax(out + 3, ~tri); }
}
__global__ void __launch_bounds__(kExpandThreads)
k_expand_mesh(const uint32_t* __restrict__ vtx, uint32_t nv, const uint32_t* __restrict__ nrm, uint32_t nn,
              const uint32_t* __restrict__ mesh_tris, uint32_t n_tris, uint32_t* __restrict__ tris, uint32_t* out) {
  // A block reads its index records and writes its output records with 16-byte accesses through shared memory: 3.3x
  // faster on B200 than 4-byte per-thread accesses to the 28- and 76-byte records (profiles/mesh_b200.md). A block's
  // records start at 16-byte boundaries (256 x 28 and 256 x 76 bytes per block from cudaMalloc'd bases).
  __shared__ __align__(16) uint32_t s_idx[kExpandThreads * kMeshWords];
  __shared__ __align__(16) uint32_t s_rec[kExpandThreads * kTriWords];
  const uint32_t first = blockIdx.x * kExpandThreads, count = min(kExpandThreads, n_tris - first);
  const uint32_t in_words = count * kMeshWords, out_words = count * kTriWords;
  const uint32_t* src = mesh_tris + (size_t)first * kMeshWords;
  for (uint32_t q = threadIdx.x; q < in_words / 4; q += kExpandThreads)
    reinterpret_cast<uint4*>(s_idx)[q] = __ldg(reinterpret_cast<const uint4*>(src) + q);
  for (uint32_t w = (in_words & ~3u) + threadIdx.x; w < in_words; w += kExpandThreads) s_idx[w] = src[w];
  __syncthreads();
  if (threadIdx.x < count)  // odd word strides (7, 19): no bank conflicts
    expand_record(s_idx + threadIdx.x * kMeshWords, s_rec + threadIdx.x * kTriWords, first + threadIdx.x, vtx, nv, nrm, nn, out);
  __syncthreads();
  uint32_t* dst = tris + (size_t)first * kTriWords;
  for (uint32_t q = threadIdx.x; q < out_words / 4; q += kExpandThreads)
    reinterpret_cast<uint4*>(dst)[q] = reinterpret_cast<const uint4*>(s_rec)[q];
  for (uint32_t w = (out_words & ~3u) + threadIdx.x; w < out_words; w += kExpandThreads) dst[w] = s_rec[w];
}
// ptb_scene_set_mesh_instances: output triangle t belongs to the last instance whose first triangle id (the exclusive prefix
// sum `inst_first`) is <= t; empty instances share their successor's prefix and are never chosen. The record is gathered
// as k_expand_mesh gathers it, with the same index checks naming the mesh triangle, then transformed in shared memory in
// the header's statement order (__fmul_rn / __fadd_rn: never contracted into an FMA).
constexpr uint32_t kInstWords = sizeof(ptb_mesh_instance) / 4, kXformWords = sizeof(ptb_instance_xform) / 4;  // 3, 21
static_assert(sizeof(ptb_mesh_instance) == 12 && sizeof(ptb_instance_xform) == 84, "record layouts");

__device__ __forceinline__ float xf_point(const float* r, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[0], x), __fmul_rn(r[1], y)), __fmul_rn(r[2], z)), r[3]);
}
__device__ __forceinline__ float xf_normal(const float* r, float x, float y, float z) {
  return __fadd_rn(__fadd_rn(__fmul_rn(r[0], x), __fmul_rn(r[1], y)), __fmul_rn(r[2], z));
}
__global__ void __launch_bounds__(kExpandThreads)
k_expand_instances(const uint32_t* __restrict__ vtx, uint32_t nv, const uint32_t* __restrict__ nrm, uint32_t nn,
                   const uint32_t* __restrict__ mesh_tris, const uint32_t* __restrict__ inst, const uint32_t* __restrict__ inst_first,
                   const float* __restrict__ xforms, uint32_t n_inst, uint32_t n_tris, uint32_t* __restrict__ tris, uint32_t* out) {
  // the output side is k_expand_mesh's: records staged in shared memory, stored with 16-byte accesses
  __shared__ __align__(16) uint32_t s_rec[kExpandThreads * kTriWords];
  const uint32_t first = blockIdx.x * kExpandThreads, count = min(kExpandThreads, n_tris - first);
  if (threadIdx.x < count) {
    const uint32_t t = first + threadIdx.x;
    uint32_t lo = 0, hi = n_inst;  // the first instance whose prefix is > t, minus one
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (__ldg(inst_first + mid) <= t) lo = mid;
      else hi = mid;
    }
    const uint32_t mt = __ldg(inst + kInstWords * lo) + (t - __ldg(inst_first + lo)), material = __ldg(inst + kInstWords * lo + 2);
    uint32_t idx[kMeshWords];
#pragma unroll
    for (uint32_t w = 0; w < kMeshWords; ++w) idx[w] = __ldg(mesh_tris + (size_t)mt * kMeshWords + w);
    uint32_t* rec = s_rec + threadIdx.x * kTriWords;
    expand_record(idx, rec, mt, vtx, nv, nrm, nn, out);
    const float* m = xforms + (size_t)lo * kXformWords;
    float mr[12], nr[9];
#pragma unroll
    for (int w = 0; w < 12; ++w) mr[w] = __ldg(m + w);
#pragma unroll
    for (int w = 0; w < 9; ++w) nr[w] = __ldg(m + 12 + w);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float* p = reinterpret_cast<float*>(rec + 3 * k);
      float* q = reinterpret_cast<float*>(rec + 9 + 3 * k);
      const float x = p[0], y = p[1], z = p[2], a = q[0], b = q[1], d = q[2];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        p[r] = xf_point(mr + 4 * r, x, y, z);
        q[r] = xf_normal(nr + 3 * r, a, b, d);
      }
    }
    if (material != PTB_MISS) rec[18] = material;
  }
  __syncthreads();
  const uint32_t out_words = count * kTriWords;
  uint32_t* dst = tris + (size_t)first * kTriWords;
  for (uint32_t q = threadIdx.x; q < out_words / 4; q += kExpandThreads)
    reinterpret_cast<uint4*>(dst)[q] = reinterpret_cast<const uint4*>(s_rec)[q];
  for (uint32_t w = (out_words & ~3u) + threadIdx.x; w < out_words; w += kExpandThreads) dst[w] = s_rec[w];
}
// Enqueued after the memset of the light-list words and before k_collect_lights, in both commit paths.
static void expand_mesh(Ctx* c, uint32_t* out) {
  if (!c->mesh || !c->mesh_dirty || c->n_tris == 0) return;
  const uint32_t nt = (uint32_t)c->n_tris;
  if (c->instanced) {
    k_expand_instances<<<(nt + kExpandThreads - 1) / kExpandThreads, kExpandThreads, 0, c->stream>>>(
        c->d_mesh_vertices.as<uint32_t>(), (uint32_t)c->n_mesh_vertices, c->d_mesh_normals.as<uint32_t>(), (uint32_t)c->n_mesh_normals,
        c->d_mesh_tris.as<uint32_t>(), c->d_inst.as<uint32_t>(), c->d_inst_first.as<uint32_t>(), c->d_inst_xforms.as<float>(),
        (uint32_t)c->n_instances, nt, c->d_raw_tris.as<uint32_t>(), out);
    c->stats.kernel_launches += 1;
    return;
  }
  k_expand_mesh<<<(nt + kExpandThreads - 1) / kExpandThreads, kExpandThreads, 0, c->stream>>>(
      c->d_mesh_vertices.as<uint32_t>(), (uint32_t)c->n_mesh_vertices, c->d_mesh_normals.as<uint32_t>(), (uint32_t)c->n_mesh_normals,
      c->d_mesh_tris.as<uint32_t>(), nt, c->d_raw_tris.as<uint32_t>(), out);
  c->stats.kernel_launches += 1;
}

// ------------------------------------------------------------------------------------------ host: build
// Material-index validation + light list, on the device: the host never walks the primitive arrays.
// out[0] = number of lights, out[1] = 1 if some material index is out of range; list = light primitive ids (unordered).
__global__ void k_collect_lights(const ptb_sphere* __restrict__ spheres, uint32_t n_spheres, const ptb_triangle* __restrict__ tris,
                                 uint32_t n_prims, const DevMaterial* __restrict__ mats, uint32_t n_mats, uint32_t* out,
                                 uint32_t* __restrict__ list) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_prims) return;
  const uint32_t mat = i < n_spheres ? spheres[i].material : tris[i - n_spheres].material;
  if (mat >= n_mats) { atomicOr(out + 1, 1u); return; }
  if (mats[mat].kind == PTB_MAT_EMIT) list[atomicAdd(out, 1u)] = i;  // material.is_light() (acceleration/mod.rs:84-88)
}

#ifndef PTB_DEFAULT_WIDE
#define PTB_DEFAULT_WIDE 0  // tree behind PTB_BUILD_DEFAULT (see the comment at its use); decided by measurement, DESIGN.md
#endif
#ifndef PTB_DEFAULT_SAH
// builder of the binary tree behind PTB_BUILD_DEFAULT: 0 Karras LBVH, 1 SAH (sah_build.cu). Measured on B200: C3 4335 -> 4850
// Mrays/s (256 spp per step), 4010 -> 4467 (32 spp), C5 4625 -> 4918, for a commit of 4.3 instead of 0.55 ms at 1 M
// triangles and 38.8 instead of 4.2 ms at 10 M (profiles/r2_sweeps.md section 12); the reference's own default is its SAH split
#define PTB_DEFAULT_SAH 1
#endif
// What every commit redoes, full or refit: validation of the small tables, materials / textures / camera to the device, the
// sky table.
static int32_t commit_tables(Ctx* c) {
  const size_t n = c->n_spheres + c->n_tris;
  if (n >= (size_t)kSlotMask) return set_error(c, PTB_ERR_INVALID, "too many primitives (%zu)", n);
  if (!c->have_camera) return set_error(c, PTB_ERR_INVALID, "scene has no camera");
  if (c->materials.empty() || c->textures.empty()) return set_error(c, PTB_ERR_INVALID, "scene has no materials/textures");
  for (const auto& m : c->materials)
    if (m.texture >= c->textures.size()) return set_error(c, PTB_ERR_INVALID, "material texture index out of range");
  if (!c->have_sky) {  // loader default: __DEFAULT_TEX, 100x100 (loader/src/misc.rs:22-25) needs an explicit sky here
    return set_error(c, PTB_ERR_INVALID, "scene has no sky (ptb_scene_set_sky)");
  }
  if (c->sky.texture >= c->textures.size()) return set_error(c, PTB_ERR_INVALID, "sky texture index out of range");
  for (size_t i = 0; i < c->textures.size(); ++i)
    if ((c->textures[i].kind == PTB_TEX_IMAGE || c->textures[i].kind == PTB_TEX_PERLIN) && !c->texture_data.count((uint32_t)i))
      return set_error(c, PTB_ERR_MISSING, "texture %zu needs ptb_scene_set_texture_data before commit", i);

  cudaStream_t st = c->stream;
  c->committed = false;
  c->scene_needs_full_shade = false;
  for (const auto& t : c->textures) c->scene_needs_full_shade |= t.kind == PTB_TEX_IMAGE || t.kind == PTB_TEX_PERLIN;
  for (const auto& m : c->materials) c->scene_needs_full_shade |= m.kind == PTB_MAT_TROWBRIDGE_REITZ;
  {
    uint32_t kinds = 0;
    for (const auto& m : c->materials) kinds |= 1u << (m.kind & 31u);
    c->scene_material_kinds = (uint32_t)__builtin_popcount(kinds);
  }

  // materials / textures / camera
  std::vector<DevMaterial> dm(c->materials.size());
  for (size_t i = 0; i < dm.size(); ++i) {
    const ptb_material& m = c->materials[i];
    dm[i].kind = m.kind; dm[i].tex = m.texture; dm[i].param = m.param; dm[i].metallic = m.metallic;
    dm[i].ior[0] = m.ior.x; dm[i].ior[1] = m.ior.y; dm[i].ior[2] = m.ior.z; dm[i]._pad = 0;
  }
  std::vector<DevTexture> dt(c->textures.size());
  std::vector<float> tex_words;
  for (size_t i = 0; i < dt.size(); ++i) {
    const ptb_texture& t = c->textures[i];
    dt[i] = DevTexture{};
    dt[i].kind = t.kind;
    dt[i].a[0] = t.a.x; dt[i].a[1] = t.a.y; dt[i].a[2] = t.a.z;
    dt[i].b[0] = t.b.x; dt[i].b[1] = t.b.y; dt[i].b[2] = t.b.z;
    auto it = c->texture_data.find((uint32_t)i);
    if (it != c->texture_data.end()) {
      if (tex_words.size() + it->second.data.size() > 0xFFFFFFF0ull) return set_error(c, PTB_ERR_INVALID, "texture data exceeds 16 GiB");
      dt[i].data_off = (uint32_t)tex_words.size();
      dt[i].width = it->second.width;
      dt[i].height = it->second.height;
      tex_words.insert(tex_words.end(), it->second.data.begin(), it->second.data.end());
    }
  }
  PTB_CUDA_TRY(c, c->d_tex_data.reserve(tex_words.size() * sizeof(float)));
  if (!tex_words.empty())
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_tex_data.p, tex_words.data(), tex_words.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  c->dev.tex_data = c->d_tex_data.as<float>();
  PTB_CUDA_TRY(c, c->d_materials.reserve(dm.size() * sizeof(DevMaterial)));
  PTB_CUDA_TRY(c, c->d_textures.reserve(dt.size() * sizeof(DevTexture)));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_materials.p, dm.data(), dm.size() * sizeof(DevMaterial), cudaMemcpyHostToDevice, st));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_textures.p, dt.data(), dt.size() * sizeof(DevTexture), cudaMemcpyHostToDevice, st));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(st));
  c->dev.materials = c->d_materials.as<DevMaterial>();
  c->dev.textures = c->d_textures.as<DevTexture>();
  c->dev.cam_origin = mk(c->camera.origin.x, c->camera.origin.y, c->camera.origin.z);
  c->dev.cam_lower_left = mk(c->camera.lower_left.x, c->camera.lower_left.y, c->camera.lower_left.z);
  c->dev.cam_horizontal = mk(c->camera.horizontal.x, c->camera.horizontal.y, c->camera.horizontal.z);
  c->dev.cam_vertical = mk(c->camera.vertical.x, c->camera.vertical.y, c->camera.vertical.z);
  return build_sky(c);
}

// Light list, after k_collect_lights: count + validation flags back to the host (16 bytes, with whatever else the stream
// has queued for the host), ids sorted into original order with the radix passes, then mapped to slots.
static int32_t light_list(Ctx* c, uint32_t ns32, uint32_t* n_lights) {
  cudaStream_t st = c->stream;
  DevBuf &keys_b = c->scratch[4], &vals_b = c->scratch[6], &hist = c->scratch[7], &d_light_prims = c->scratch[12],
         &d_light_tmp = c->scratch[13], &d_light_out = c->scratch[14];
  uint32_t h_light_out[4] = {0u, 0u, 0u, 0u};
  PTB_CUDA_TRY(c, cudaMemcpyAsync(h_light_out, d_light_out.p, 16, cudaMemcpyDeviceToHost, st));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(st));
  if (h_light_out[1] & 2u)
    return set_error(c, PTB_ERR_INVALID, "mesh triangle %u: vertex index out of range (the mesh has %zu vertices)", ~h_light_out[2],
                     c->n_mesh_vertices);
  if (h_light_out[1] & 4u)
    return set_error(c, PTB_ERR_INVALID, "mesh triangle %u: normal index out of range (the mesh has %zu normals)", ~h_light_out[3],
                     c->n_mesh_normals);
  if (h_light_out[1]) return set_error(c, PTB_ERR_INVALID, "primitive material index out of range");
  const uint32_t nl = h_light_out[0];
  if (nl) {
    PTB_CUDA_TRY(c, c->d_lights.reserve((size_t)nl * 4));
    uint32_t *la = d_light_prims.as<uint32_t>(), *lb = d_light_tmp.as<uint32_t>();
    if (nl > 1) {
      // nl <= n: the histogram scratch is large enough
      // values ride along unused: keys double as values (keys_b / vals_b are free again)
      uint32_t *lva = keys_b.as<uint32_t>(), *lvb = vals_b.as<uint32_t>();
      radix_sort_pairs(c, la, lva, lb, lvb, nl, 4, hist.as<uint32_t>());
    }
    k_light_slots<<<(nl + 255) / 256, 256, 0, st>>>(la, nl, ns32, c->d_prim_slot.as<uint32_t>(), c->d_lights.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  *n_lights = nl;
  return PTB_OK;
}

// PTB_BUILD_REFIT: keeps the binary tree of the last full commit (links, leaf_parent, slot order, Morton codes) and refits
// its boxes to the primitives as they are now; materials, textures, camera, sky and the light list are redone as in a
// full commit.
static int32_t refit_scene(Ctx* c, uint32_t build_flags) {
  if (build_flags != PTB_BUILD_REFIT)
    return set_error(c, PTB_ERR_INVALID, "PTB_BUILD_REFIT cannot be combined with another build flag (flags 0x%x)", build_flags);
  if (!c->refittable)
    return set_error(c, PTB_ERR_INVALID, "PTB_BUILD_REFIT needs a tree to keep: the last full commit of this context failed or there was none");
  if (c->wide)
    return set_error(c, PTB_ERR_UNSUPPORTED, "PTB_BUILD_REFIT: the compressed 8-wide tree cannot be refitted; commit with a binary builder");
  if (c->n_spheres != c->topo_spheres || c->n_tris != c->topo_tris)
    return set_error(c, PTB_ERR_INVALID, "PTB_BUILD_REFIT keeps the tree of %zu spheres and %zu triangles, the scene now has %zu and %zu",
                     c->topo_spheres, c->topo_tris, c->n_spheres, c->n_tris);
  int32_t rc = commit_tables(c);
  if (rc != PTB_OK) return rc;
  const size_t n = c->n_prims;
  if (n == 0) {
    c->committed = true;
    c->stats.build_ms = 0.0;
    return PTB_OK;
  }
  cudaStream_t st = c->stream;
  // the full commit of the same counts reserved every one of these (grow-only): no allocation happens here
  DevBuf &sbmin = c->scratch[0], &sbmax = c->scratch[1], &nbmin = c->scratch[9], &nbmax = c->scratch[10], &flags = c->scratch[11],
         &d_light_prims = c->scratch[12], &d_light_out = c->scratch[14], &d_qframe = c->scratch[15];
  PTB_CUDA_TRY(c, sbmin.reserve(n * 16));
  PTB_CUDA_TRY(c, sbmax.reserve(n * 16));
  const uint32_t n32 = (uint32_t)n, ns32 = (uint32_t)c->n_spheres;
  const int T = 256;
  const uint32_t gn = (n32 + T - 1) / T;
  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_a, st));
  PTB_CUDA_TRY(c, cudaMemsetAsync(d_light_out.p, 0, 16, st));
  expand_mesh(c, d_light_out.as<uint32_t>());
  k_collect_lights<<<gn, T, 0, st>>>(c->d_raw_spheres.as<ptb_sphere>(), ns32, c->d_raw_tris.as<ptb_triangle>(), n32,
                                     c->d_materials.as<DevMaterial>(), (uint32_t)c->materials.size(), d_light_out.as<uint32_t>(),
                                     d_light_prims.as<uint32_t>());
  if (n > 1) PTB_CUDA_TRY(c, cudaMemsetAsync(flags.p, 0, c->n_nodes * 4, st));
  k_refit_slots<<<gn, T, 0, st>>>(c->d_raw_spheres.as<ptb_sphere>(), ns32, c->d_raw_tris.as<ptb_triangle>(), n32,
                                  c->d_slot_prim.as<uint32_t>(), c->d_leaf_parent.as<uint32_t>(), c->d_materials.as<DevMaterial>(),
                                  (uint32_t)c->materials.size(), c->d_geom.as<float4>(), c->d_normals.as<float4>(),
                                  c->d_slot_mat.as<uint32_t>(), sbmin.as<float4>(), sbmax.as<float4>(), c->d_nodes.as<BvhNode>(),
                                  nbmin.as<float4>(), nbmax.as<float4>(), flags.as<uint32_t>());
  c->stats.kernel_launches += 2;
  if (n == 1) {  // slot 0 holds primitive 0: the slot-ordered box is also the original-order one k_single_node reads
    k_single_node<<<1, 1, 0, st>>>(c->d_slot_prim.as<uint32_t>(), ns32, sbmin.as<float4>(), sbmax.as<float4>(), c->d_nodes.as<BvhNode>());
    c->stats.kernel_launches += 1;
  }
  float h_qframe[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (PTB_QNODES) {  // the grid follows the root box
    k_qframe<<<1, 1, 0, st>>>(c->d_nodes.as<BvhNode>(), d_qframe.as<float>());
    k_quantise_nodes<<<((uint32_t)c->n_nodes + T - 1) / T, T, 0, st>>>(c->d_nodes.as<BvhNode>(), (uint32_t)c->n_nodes, d_qframe.as<float>(),
                                                                     c->d_qnodes.as<uint4>());
    PTB_CUDA_TRY(c, cudaMemcpyAsync(h_qframe, d_qframe.p, sizeof h_qframe, cudaMemcpyDeviceToHost, st));
    c->stats.kernel_launches += 2;
  }
  uint32_t nl = 0;
  rc = light_list(c, ns32, &nl);
  if (rc != PTB_OK) return rc;
  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_b, st));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(st));
  PTB_CUDA_TRY(c, cudaGetLastError());
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev_a, c->ev_b);
  c->stats.build_ms = ms;
  if (PTB_QNODES)
    for (int k = 0; k < 3; ++k) { c->dev.q_min[k] = h_qframe[k]; c->dev.q_step[k] = h_qframe[3 + k]; }
  c->dev.lights = c->d_lights.as<uint32_t>();
  c->dev.n_lights = nl;
  c->committed = true;
  c->mesh_dirty = false;
  return PTB_OK;
}

int32_t build_scene(Ctx* c, uint32_t build_flags) {
  if (build_flags & PTB_BUILD_REFIT) return refit_scene(c, build_flags);
  c->refittable = false;  // from here on the kept topology is being replaced
  {
    int32_t rc = commit_tables(c);
    if (rc != PTB_OK) return rc;
  }
  const size_t ns = c->n_spheres, nt = c->n_tris;
  const size_t n = ns + nt;
  cudaStream_t st = c->stream;

  c->n_prims = n;
  c->n_nodes = n == 0 ? 0 : (n == 1 ? 1 : n - 1);
  c->dev.n_prims = (uint32_t)n;
  c->dev.n_lights = 0;
  c->dev.geom = nullptr; c->dev.normals = nullptr; c->dev.slot_prim = nullptr; c->dev.slot_mat = nullptr;
  c->dev.nodes = nullptr; c->dev.qnodes = nullptr; c->dev.lights = nullptr; c->dev.cw_nodes = nullptr;
  c->wide = false;
  if (n == 0) {
    c->committed = true;
    c->refittable = true;
    c->topo_spheres = ns;
    c->topo_tris = nt;
    c->stats.build_ms = 0.0;
    return PTB_OK;
  }

  // Primitives were uploaded by ptb_scene_set_* (c->d_raw_spheres / d_raw_tris). Build temporaries live in the context
  // and only ever grow: a re-commit of a same-sized scene performs no cudaMalloc / cudaFree at all.
  DevBuf &raw_spheres = c->d_raw_spheres, &raw_tris = c->d_raw_tris;
  DevBuf &bmin = c->scratch[0], &bmax = c->scratch[1], &bounds = c->scratch[2], &keys_a = c->scratch[3], &keys_b = c->scratch[4],
         &vals_a = c->scratch[5], &vals_b = c->scratch[6], &hist = c->scratch[7], &leaf_parent = c->d_leaf_parent,
         &nbmin = c->scratch[9], &nbmax = c->scratch[10], &flags = c->scratch[11], &prim_slot = c->d_prim_slot,
         &d_light_prims = c->scratch[12], &d_light_tmp = c->scratch[13], &d_light_out = c->scratch[14], &d_qframe = c->scratch[15];
  const uint32_t n32 = (uint32_t)n, ns32 = (uint32_t)ns, nt32 = (uint32_t)nt;
  PTB_CUDA_TRY(c, bmin.reserve(n * 16));
  PTB_CUDA_TRY(c, bmax.reserve(n * 16));
  PTB_CUDA_TRY(c, bounds.reserve(12 * 4));
  PTB_CUDA_TRY(c, keys_a.reserve(n * 4));
  PTB_CUDA_TRY(c, keys_b.reserve(n * 4));
  PTB_CUDA_TRY(c, vals_a.reserve(n * 4));
  PTB_CUDA_TRY(c, vals_b.reserve(n * 4));
  PTB_CUDA_TRY(c, hist.reserve(radix_sort_hist_words(n32) * 4));
  PTB_CUDA_TRY(c, leaf_parent.reserve(n * 4));
  PTB_CUDA_TRY(c, nbmin.reserve(c->n_nodes * 16));
  PTB_CUDA_TRY(c, nbmax.reserve(c->n_nodes * 16));
  PTB_CUDA_TRY(c, flags.reserve(c->n_nodes * 4));
  PTB_CUDA_TRY(c, prim_slot.reserve(n * 4));
  PTB_CUDA_TRY(c, d_light_prims.reserve(n * 4));
  PTB_CUDA_TRY(c, d_light_tmp.reserve(n * 4));
  PTB_CUDA_TRY(c, d_light_out.reserve(16));
  PTB_CUDA_TRY(c, c->d_nodes.reserve(c->n_nodes * sizeof(BvhNode)));
  if (PTB_QNODES) PTB_CUDA_TRY(c, c->d_qnodes.reserve(c->n_nodes * 32));
  PTB_CUDA_TRY(c, d_qframe.reserve(6 * 4));
  PTB_CUDA_TRY(c, c->d_geom.reserve(n * 48));
  PTB_CUDA_TRY(c, c->d_normals.reserve(n * 48));
  PTB_CUDA_TRY(c, c->d_slot_mat.reserve(n * 4));
  PTB_CUDA_TRY(c, c->d_morton.reserve(n * 4));
  PTB_CUDA_TRY(c, c->d_slot_prim.reserve(n * 4));

  // Which tree the traversal kernels walk: the binary LBVH or its collapse into the compressed 8-wide tree
  // (cwbvh_build.cu). build_flags picks; PTB_BUILD_DEFAULT follows PTB_BVH=binary|wide, else the measured default.
  bool wide = PTB_DEFAULT_WIDE != 0;
  if (const char* e = getenv("PTB_BVH")) wide = strcmp(e, "wide") == 0 ? true : (strcmp(e, "binary") == 0 ? false : wide);
  // ... and which builder makes the binary tree: the Karras hierarchy over the Morton order, or the SAH builder
  // (sah_build.cu) started from that order. The wide tree is always collapsed from the Karras hierarchy.
  bool sah = PTB_DEFAULT_SAH != 0;
  if (const char* e = getenv("PTB_BVH")) {
    if (strcmp(e, "sah") == 0) { sah = true; wide = false; }
    else if (strcmp(e, "binary") == 0 || strcmp(e, "lbvh") == 0 || strcmp(e, "wide") == 0) sah = false;
  }
  if (build_flags & PTB_BUILD_BINARY) { wide = false; sah = false; }
  if (build_flags & PTB_BUILD_WIDE) { wide = true; sah = false; }
  if (build_flags & PTB_BUILD_SAH) { wide = false; sah = true; }
  if (wide || n < 2 || n > (1u << 24)) sah = false;
  c->cw_max_leaf = 3u;
  if (const char* e = getenv("PTB_WIDE_LEAF")) { int v = atoi(e); if (v >= 1 && v <= 3) c->cw_max_leaf = (uint32_t)v; }
  DevBuf &range = c->cw_scratch[8], &final_prim = c->cw_scratch[9];
  if (wide) {
    PTB_CUDA_TRY(c, range.reserve(c->n_nodes * 8));
    PTB_CUDA_TRY(c, final_prim.reserve(n * 4));
    PTB_CUDA_TRY(c, c->d_prim_sorted.reserve(n * 4));
  }
  if (sah) {
    const int32_t rcs = reserve_sah(c, n32);
    if (rcs != PTB_OK) return rcs;
  }
  const int T = 256;
  const uint32_t gn = (n32 + T - 1) / T;
  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_a, st));
  // lights + material-index validation (device), then the light ids are put in ORIGINAL primitive order (deterministic)
  PTB_CUDA_TRY(c, cudaMemsetAsync(d_light_out.p, 0, 16, st));
  expand_mesh(c, d_light_out.as<uint32_t>());
  k_collect_lights<<<gn, T, 0, st>>>(raw_spheres.as<ptb_sphere>(), ns32, raw_tris.as<ptb_triangle>(), n32,
                                     c->d_materials.as<DevMaterial>(), (uint32_t)c->materials.size(), d_light_out.as<uint32_t>(),
                                     d_light_prims.as<uint32_t>());
  c->stats.kernel_launches += 1;
  {
    const uint32_t init[12] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u};
    PTB_CUDA_TRY(c, cudaMemcpyAsync(bounds.p, init, sizeof init, cudaMemcpyHostToDevice, st));
  }
  k_prim_bounds<<<gn, T, 0, st>>>(raw_spheres.as<ptb_sphere>(), ns32, raw_tris.as<ptb_triangle>(), nt32, bmin.as<float4>(),
                                  bmax.as<float4>(), bounds.as<uint32_t>());
  k_morton<<<gn, T, 0, st>>>(bmin.as<float4>(), bmax.as<float4>(), n32, bounds.as<uint32_t>(), keys_a.as<uint32_t>(),
                             vals_a.as<uint32_t>());
  c->stats.kernel_launches += 2;
  uint32_t *ka = keys_a.as<uint32_t>(), *kb = keys_b.as<uint32_t>(), *va = vals_a.as<uint32_t>(), *vb = vals_b.as<uint32_t>();
  radix_sort_pairs(c, ka, va, kb, vb, n32, 4, hist.as<uint32_t>());
  // after 4 passes the sorted data is back in (keys_a, vals_a) == (ka, va)
  if (n == 1) {
    k_single_node<<<1, 1, 0, st>>>(va, ns32, bmin.as<float4>(), bmax.as<float4>(), c->d_nodes.as<BvhNode>());
    c->stats.kernel_launches += 1;
  } else {
    PTB_CUDA_TRY(c, cudaMemsetAsync(flags.p, 0, c->n_nodes * 4, st));
    if (sah) {
      SahBuildInputs si{bmin.as<float4>(), bmax.as<float4>(), bounds.as<uint32_t>() + 6, va, vb, c->d_nodes.as<BvhNode>(), leaf_parent.as<uint32_t>(), n32, ns32};
      const uint32_t* order = nullptr;
      const int32_t rcs = build_sah(c, si, &order);
      if (rcs != PTB_OK) return rcs;
      va = const_cast<uint32_t*>(order);  // the tree's own primitive order from here on
    } else {
      k_hierarchy<<<(n32 - 1 + T - 1) / T, T, 0, st>>>(ka, va, n32, ns32, c->d_nodes.as<BvhNode>(), leaf_parent.as<uint32_t>(),
                                                       wide ? range.as<uint2>() : nullptr);
      c->stats.kernel_launches += 1;
    }
    k_refit<<<gn, T, 0, st>>>(n32, va, leaf_parent.as<uint32_t>(), bmin.as<float4>(), bmax.as<float4>(),
                              c->d_nodes.as<BvhNode>(), nbmin.as<float4>(), nbmax.as<float4>(), flags.as<uint32_t>());
    c->stats.kernel_launches += 1;
  }
  // the 32-byte nodes the traversal kernels read, and their grid (6 floats, read back with the light count below)
  float h_qframe[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (!wide && PTB_QNODES) {
    k_qframe<<<1, 1, 0, st>>>(c->d_nodes.as<BvhNode>(), d_qframe.as<float>());
    k_quantise_nodes<<<((uint32_t)c->n_nodes + T - 1) / T, T, 0, st>>>(c->d_nodes.as<BvhNode>(), (uint32_t)c->n_nodes, d_qframe.as<float>(),
                                                                     c->d_qnodes.as<uint4>());
    PTB_CUDA_TRY(c, cudaMemcpyAsync(h_qframe, d_qframe.p, sizeof h_qframe, cudaMemcpyDeviceToHost, st));
    c->stats.kernel_launches += 2;
  }
  // slot order of the geometry: Morton order for the binary tree, the wide tree's own primitive order otherwise
  const uint32_t* slot_order = va;
  if (wide) {
    CwBuildInputs bi{c->d_nodes.as<BvhNode>(), range.as<uint2>(), nbmin.as<float4>(), nbmax.as<float4>(), bmin.as<float4>(),
                     bmax.as<float4>(), va, n32};
    const int32_t rcw = build_wide(c, bi, final_prim.as<uint32_t>());
    if (rcw != PTB_OK) return rcw;
    slot_order = final_prim.as<uint32_t>();
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_prim_sorted.p, va, n * 4, cudaMemcpyDeviceToDevice, st));
  }
  k_gather<<<gn, T, 0, st>>>(raw_spheres.as<ptb_sphere>(), ns32, raw_tris.as<ptb_triangle>(), n32, slot_order,
                             c->d_materials.as<DevMaterial>(), (uint32_t)c->materials.size(), c->d_geom.as<float4>(),
                             c->d_normals.as<float4>(),
                             c->d_slot_mat.as<uint32_t>(), prim_slot.as<uint32_t>());
  c->stats.kernel_launches += 1;
  // keep the sorted keys / ids for ptb_bvh_export and the traversal's tie-break
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_morton.p, ka, n * 4, cudaMemcpyDeviceToDevice, st));
  PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_slot_prim.p, slot_order, n * 4, cudaMemcpyDeviceToDevice, st));
  uint32_t nl = 0;
  {
    const int32_t rcl = light_list(c, ns32, &nl);
    if (rcl != PTB_OK) return rcl;
  }
  PTB_CUDA_TRY(c, cudaEventRecord(c->ev_b, st));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(st));
  PTB_CUDA_TRY(c, cudaGetLastError());
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev_a, c->ev_b);
  c->stats.build_ms = ms;

  c->dev.geom = c->d_geom.as<float4>();
  c->dev.normals = c->d_normals.as<float4>();
  c->dev.slot_prim = c->d_slot_prim.as<uint32_t>();
  c->dev.slot_mat = c->d_slot_mat.as<uint32_t>();
  c->dev.nodes = c->d_nodes.as<BvhNode>();
  c->dev.qnodes = (wide || !PTB_QNODES) ? nullptr : c->d_qnodes.as<uint4>();
  for (int k = 0; k < 3; ++k) { c->dev.q_min[k] = h_qframe[k]; c->dev.q_step[k] = h_qframe[3 + k]; }
  c->dev.cw_nodes = wide ? c->d_cw_nodes.as<CwNode>() : nullptr;
  c->wide = wide;
  c->sah = sah;
  if (!wide) c->n_cw_nodes = 0;
  c->dev.lights = c->d_lights.as<uint32_t>();
  c->dev.n_lights = nl;
  c->committed = true;
  c->mesh_dirty = false;
  c->refittable = true;
  c->topo_spheres = ns;
  c->topo_tris = nt;
  return PTB_OK;
}

}  // namespace ptb
