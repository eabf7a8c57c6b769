// ptb200 internal host-side declarations shared by the .cu translation units (not part of the ABI).
#pragma once
#include <cuda_runtime.h>

#include <cstdio>
#include <map>
#include <string>
#include <vector>

#include "ptb_common.cuh"

namespace ptb {

// RAII device allocation
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  cudaError_t alloc(size_t n) {
    release();
    if (n == 0) n = 16;
    cudaError_t e = cudaMalloc(&p, n);
    if (e == cudaSuccess) bytes = n;
    else p = nullptr;
    return e;
  }
  // grow-only
  cudaError_t reserve(size_t n) { return n <= bytes ? cudaSuccess : alloc(n); }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// Wavefront state for one render call (device pointers). See wavefront.cu.
struct PathPool {
  uint32_t capacity = 0;
  // Records are 32-byte sectors written whole by one thread (a 16-byte store to a scattered slot costs a
  // read-modify-write at the DRAM side; two adjacent 16-byte stores do not).
  // one 64-byte block per path (4 x float4); col == ray + 2
  float4* ray = nullptr;   // [4*slot]   origin.xyz | hit t        [4*slot+1] normalised direction.xyz | hit leaf ref (bits)
  float4* col = nullptr;   // [4*slot]   throughput.rgb | pixel    [4*slot+1] radiance so far .rgb | sample<<9 | flags<<8 | depth
  float4* prev = nullptr;  // MIS only: previous (un-offset) hit point.xyz | m_pdf of the last BSDF sample
};
constexpr uint32_t kMaxSampleIndex = 1u << 23;  // sample index shares a word with depth (8 bits) and one flag

constexpr int kNumKinds = 6;  // material kinds of k_shade's block sort: 0 = miss (sky), 1 + PTB_MAT_* otherwise

struct WaveCounters {  // one per chunk slot, in device memory; mirrored to pinned host memory once per iteration
  uint32_t n_trace;         // rays to trace this iteration
  uint32_t trace_head, shadow_head;  // persistent-kernel work cursors
  // decided ON THE DEVICE by k_win_prepare so that the host never has to wait for an iteration before it enqueues the
  // next: 0 wavefront iterations running, 1 this iteration hands the chunk's last n_tail paths to k_tail, 2 chunk
  // finished, 3 handed over earlier — in every state but 0 the wavefront kernels find n_trace == 0 and return
  uint32_t mode;
  uint32_t n_tail, tail_iter;  // set ONCE per chunk: live paths handed over, and the iteration whose k_tail launch takes them
  uint32_t tail_head, _pad2;   // k_tail's work cursor (its lanes pull paths one by one)
  // k_shade's shadow-queue cursor, packed so that one warp needs ONE returning atomic: sky NEE rays << 32 | entries.
  // k_win_prepare unpacks it between iterations.
  unsigned long long shadow_pair;
  // statistics (ptb_stats)
  unsigned long long rays_camera, rays_bounce, rays_shadow_light, rays_shadow_sky, rays_reference, paths;
  unsigned long long nodes_fetched, prims_tested, rays_counted;  // PTB_OPT_COUNT_TRAVERSAL
  // k_tail times itself (%globaltimer: first block in, last block out) — it runs on a side stream, detached from the
  // host's view of the iterations; tail_ns sums the finished hand-overs of this slot
  unsigned long long tail_t0, tail_t1, tail_ns;
};

struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string last_error;
  int sm_count = 148;

  // scene as handed over by ptb_scene_set_*: primitives go straight to the device (no host copy), the small tables
  // are kept on the host until commit
  DevBuf d_raw_spheres, d_raw_tris;
  size_t n_spheres = 0, n_tris = 0;
  // indexed mesh (ptb_scene_set_mesh): when `mesh` is set, d_raw_tris is the mesh's expansion (k_expand_mesh), redone at
  // the next commit whenever `mesh_dirty`; n_tris is the number of mesh triangles, n_mesh_tris too unless `instanced`
  DevBuf d_mesh_vertices, d_mesh_normals, d_mesh_tris;
  size_t n_mesh_vertices = 0, n_mesh_normals = 0, n_mesh_tris = 0;
  bool mesh = false, mesh_dirty = false;
  // mesh instances (ptb_scene_set_mesh_instances): when `instanced` is set (on a mesh scene), d_raw_tris is the expansion
  // of every instance (k_expand_instances) and n_tris the sum of their n_triangles; d_inst_first is the exclusive prefix
  // sum of n_triangles (the first triangle id of each instance)
  DevBuf d_inst, d_inst_first, d_inst_xforms;
  size_t n_instances = 0;
  bool instanced = false;
  DevBuf scratch[16];  // LBVH build temporaries, grow-only (lbvh_build.cu)
  std::vector<ptb_material> materials;
  std::vector<ptb_texture> textures;
  struct TexData { uint32_t width = 0, height = 0; std::vector<float> data; };
  std::map<uint32_t, TexData> texture_data;  // ptb_scene_set_texture_data
  ptb_camera camera{};
  ptb_sky sky{};
  bool have_camera = false, have_sky = false;
  bool committed = false;
  uint32_t scene_material_kinds = 0;    // distinct PTB_MAT_* kinds among the scene's materials (k_shade's block-level sort)
  bool scene_needs_full_shade = false;  // any Trowbridge-Reitz material or image / perlin texture (k_shade<.., FULL>)

  // device scene
  DevScene dev{};
  DevBuf d_prim_slot;  // original primitive id -> slot (k_gather; valid until the next commit: lights, visibility API)
  DevBuf d_leaf_parent;  // slot -> parent node of the binary tree (k_hierarchy / SAH build; the refit climbs from it)
  // The binary tree of the last full commit can be refitted (PTB_BUILD_REFIT): set when a full commit succeeds, cleared
  // when one starts. Its topology (d_nodes links, d_leaf_parent, d_slot_prim) belongs to these primitive counts.
  bool refittable = false;
  size_t topo_spheres = 0, topo_tris = 0;
  DevBuf d_geom, d_normals, d_slot_prim, d_slot_mat, d_nodes, d_qnodes, d_cw_nodes, d_prim_sorted, d_morton, d_materials, d_textures, d_tex_data, d_lights;
  DevBuf d_sky_ycdf, d_sky_ypdf, d_sky_xcdf, d_sky_xpdf;
  uint64_t n_prims = 0, n_nodes = 0, n_cw_nodes = 0;
  bool wide = false;          // the committed scene is traversed through the compressed 8-wide tree (d_cw_nodes)
  uint32_t cw_max_leaf = 3;   // primitives per leaf group of the wide tree (1..3)
  DevBuf cw_scratch[10];      // wide-tree build temporaries, grow-only (cwbvh_build.cu; [8] LBVH ranges, [9] final order)
  bool sah = false;           // the committed scene's binary tree was built by the SAH builder (sah_build.cu)
  uint32_t sah_levels = 0;    // levels of large tasks the last SAH build took
  DevBuf sah_scratch[12];     // SAH build temporaries, grow-only
  uint32_t* h_sah = nullptr;  // pinned: the per-level counters of the SAH build

  // render state
  DevBuf d_accum;
  float* accum_target = nullptr;  // ptb_render_passes: render into the single-pass buffer instead of d_accum
  DevBuf d_pass;
  float* h_pass[2] = {nullptr, nullptr};  // pinned
  size_t h_pass_floats = 0;
  uint32_t accum_w = 0, accum_h = 0;
  uint64_t accum_samples = 0;
  // denoiser feature buffers (ptb_render_aov): 8 float sums per pixel, [albedo.rgb | coverage] [normal.xyz | depth],
  // and the work cursors of one call's k_aov launches (one per sample)
  DevBuf d_aov, d_aov_heads;
  uint32_t aov_w = 0, aov_h = 0;
  uint64_t aov_samples = 0;
  // denoiser scratch (denoise.cu), dn_w x dn_h pixels: ping-pong [e.rgb | var] and the guide records [n.xyz | z],
  // coverage α and the depth gradient [∂x z, ∂y z]
  DevBuf d_dn_e[2], d_dn_nz, d_dn_alpha, d_dn_grad;
  uint32_t dn_w = 0, dn_h = 0;
  // camera candidate lists of the window wavefront (ptb_camcand.cuh), grow-only: entries [npix * k] and counts [npix]
  DevBuf d_camcand, d_camcand_count;
  DevBuf d_pool_mem, d_prev, d_queues, d_shadow, d_counters, d_windows;
  // second chunk slot of the window wavefront: chunk k+1's wide iterations run on the main stream while chunk k's fused
  // tail (k_tail) finishes on `s_tail` in the other slot
  DevBuf d_pool_mem2, d_prev2, d_queues2, d_shadow2, d_counters2, d_windows2;
  cudaStream_t s_tail = nullptr;
  cudaStream_t s_work2 = nullptr;  // the odd chunks' wide iterations run here, concurrently with the even chunks' on `stream`
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_head_done[2] = {}, ev_tail_done[2] = {};
  cudaEvent_t ev_ring[8] = {};  // per-slot ring of 4: iteration completion (the host runs at most 3 iterations ahead)
  PathPool pool;
  size_t pool_budget_bytes = 0;  // half of the device memory that was free at the first large render (0 = not asked yet)
  WaveCounters* h_counters = nullptr;  // pinned: [0..7] per-iteration mirrors (a ring of 4 per slot), [8..9] end-of-render copy of each slot
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  cudaEvent_t ev_prof[64] = {};  // PTB_OPT_TIME_KERNELS: 2 slots x 4 iterations (ring) x 4 kernel classes x (start, stop)
  bool opt_time_kernels = false, opt_count_traversal = false;

  // closest-hit staging: two buffer pairs + copy streams so that the upload of batch k+1, the traversal of batch k and the
  // read-back of batch k-1 overlap (ptb_closest_hit with host buffers)
  DevBuf d_rays, d_hits, d_rays2, d_hits2;
  DevBuf d_index, d_index2;  // the second input of ptb_check_hit_index (target ids), staged with the rays
  DevBuf d_hit_sort;  // ray ordering scratch of the closest-hit API: 4 x n words (keys / indices, ping-pong) + histogram
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[2] = {}, ev_kernel[2] = {}, ev_out[2] = {};

  ptb_stats stats{};
};

int32_t set_error(Ctx* c, int32_t code, const char* fmt, ...);
int32_t check_cuda(Ctx* c, cudaError_t e, const char* what);

// lbvh_build.cu — uploads the host scene and builds the device LBVH (K2..K6)
int32_t build_scene(Ctx* c, uint32_t flags);
// SAH cost of the committed binary tree (ptb_bvh_sah_cost)
int32_t tree_sah_cost(Ctx* c, double* cost);
// cwbvh_build.cu — collapses the LBVH into the compressed 8-wide tree; leaves the final primitive order in
// `final_prim` (final slot -> original primitive id, n words, device)
struct CwBuildInputs {
  const BvhNode* nodes;          // LBVH (n - 1 nodes)
  const uint2* range;            // Morton range [lo, hi] of every LBVH node
  const float4 *nbmin, *nbmax;   // box of every LBVH node
  const float4 *bmin, *bmax;     // box of every primitive (original order)
  const uint32_t* prim_sorted;   // Morton position -> original primitive id
  uint32_t n_prims;
};
int32_t build_wide(Ctx* c, const CwBuildInputs& in, uint32_t* final_prim);
// in-place exclusive prefix sum of n <= 2^24 words (block_sum: 4096 words of scratch; *total_out receives the sum)
int32_t exclusive_scan(Ctx* c, uint32_t* data, uint32_t n, uint32_t* block_sum, uint32_t* total_out);
void scan_block_sums(Ctx* c, uint32_t* block_sum, uint32_t n_blocks, uint32_t* total_out);
// sah_build.cu — top-down SAH hierarchy in the LBVH's node format (links in nodes[].n3 + leaf_parent; k_refit fills the boxes)
struct SahBuildInputs {
  const float4 *bmin, *bmax;      // box of every primitive (original order)
  const uint32_t* box6;           // union of those boxes: min xyz, max xyz as order-preserving uints (k_prim_bounds)
  uint32_t *order_a, *order_b;    // order_a: Morton position -> original primitive id (the starting order); order_b: scratch
  BvhNode* nodes;                 // n - 1 nodes
  uint32_t* leaf_parent;          // n words
  uint32_t n_prims, n_spheres;
};
int32_t build_sah(Ctx* c, const SahBuildInputs& in, const uint32_t** order_out);
int32_t reserve_sah(Ctx* c, uint32_t n_prims);
void radix_sort_pairs(Ctx* c, uint32_t*& ka, uint32_t*& va, uint32_t*& kb, uint32_t*& vb, uint32_t n, int passes, uint32_t* hist);
size_t radix_sort_hist_words(uint32_t n);
// wavefront.cu
int32_t render_wavefront(Ctx* c, const ptb_render_opts& o, ptb_progress_fn progress, void* user);
int32_t launch_closest_hit(Ctx* c, const void* d_rays, size_t n, void* d_hits);
// ptb_render_aov's launches, opts validated; adds into d_aov
int32_t launch_aov(Ctx* c, const ptb_render_opts& o);
// check_hit_index (d_index != nullptr: ptb_ray in, ptb_hit out) or occlusion (ptb_occlusion_ray in, one byte out)
int32_t launch_visibility(Ctx* c, const void* d_rays, const void* d_index, size_t n, void* d_out);
void free_render_state(Ctx* c);
int32_t sampler_hook(Ctx* c, const ptb_sampler_query& q, size_t n, const float* dirs_in, float* dirs_out, float* pdf_out);

}  // namespace ptb

struct ptb_ctx {
  ptb::Ctx c;
};

#define PTB_CUDA_TRY(ctx, expr)                                   \
  do {                                                            \
    cudaError_t _e = (expr);                                      \
    if (_e != cudaSuccess) return ptb::check_cuda(ctx, _e, #expr); \
  } while (0)
