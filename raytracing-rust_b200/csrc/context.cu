// ptb200 — C ABI (include/ptb200.h): context lifecycle, scene upload, closest-hit batches, render, accumulator.
// No CPU fallback: every compute entry point needs a CUDA device and fails with PTB_ERR_CUDA otherwise.
#include <cstdarg>
#include <cstring>
#include <new>

#include "ptb_internal.h"

namespace ptb {

static thread_local std::string g_create_error;

int32_t set_error(Ctx* c, int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->last_error = buf;
  else g_create_error = buf;
  return code;
}
int32_t check_cuda(Ctx* c, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return PTB_OK;
  const int32_t code = e == cudaErrorMemoryAllocation ? PTB_ERR_OOM : PTB_ERR_CUDA;
  return set_error(c, code, "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
}

__global__ void k_scale_copy(const float* __restrict__ in, float* __restrict__ out, size_t n, float scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] * scale;
}

}  // namespace ptb

using namespace ptb;

#define CTX_OR_FAIL(ctx)                 \
  if (!(ctx)) return PTB_ERR_INVALID;    \
  Ctx* c = &(ctx)->c;                    \
  if (cudaSetDevice(c->device) != cudaSuccess) return set_error(c, PTB_ERR_CUDA, "cudaSetDevice(%d) failed", c->device)

extern "C" {

uint32_t ptb_abi_version(void) { return PTB_ABI_VERSION; }

int32_t ptb_device_count(int32_t* count) {
  if (!count) return PTB_ERR_INVALID;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    *count = 0;
    return set_error(nullptr, PTB_ERR_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  *count = n;
  return PTB_OK;
}

int32_t ptb_create(int32_t device, ptb_ctx** out) {
  if (!out) return PTB_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_error(nullptr, PTB_ERR_CUDA, "no CUDA device available (%s); ptb200 has no CPU fallback",
                     e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= n) return set_error(nullptr, PTB_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  ptb_ctx* ctx = new (std::nothrow) ptb_ctx();
  if (!ctx) return PTB_ERR_OOM;
  Ctx* c = &ctx->c;
  c->device = device;
  auto fail = [&](cudaError_t err, const char* what) {
    int32_t rc = set_error(nullptr, PTB_ERR_CUDA, "%s: %s", what, cudaGetErrorString(err));
    delete ctx;
    return rc;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(e, "cudaSetDevice");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(e, "cudaGetDeviceProperties");
  if (prop.major < 10) {
    int32_t rc = set_error(nullptr, PTB_ERR_CUDA, "device %d is sm_%d%d; ptb200 is built for sm_100a only", device, prop.major,
                           prop.minor);
    delete ctx;
    return rc;
  }
  c->sm_count = prop.multiProcessorCount;
  c->dev.trace_burst = 8;  // window mode, C3: 2 -> 3285, 4 -> 3425, 8 -> 3472 Mrays/s (profiles/r1_sweeps.md)
  c->dev.trace_fetch_threshold = 8;
  c->dev.trace_prim_bias = 0;
  if (const char* e = getenv("PTB_TRACE_PRIM_BIAS")) { int v = atoi(e); if (v >= 0 && v <= 32) c->dev.trace_prim_bias = v; }
  if (const char* e = getenv("PTB_TRACE_BURST")) { int v = atoi(e); if (v >= 1 && v <= 64) c->dev.trace_burst = v; }
  if (const char* e = getenv("PTB_TRACE_FETCH")) { int v = atoi(e); if (v >= 1 && v <= 32) c->dev.trace_fetch_threshold = v; }
  if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
  c->own_stream = true;
  if ((e = cudaEventCreate(&c->ev_a)) != cudaSuccess) return fail(e, "cudaEventCreate");
  if ((e = cudaEventCreate(&c->ev_b)) != cudaSuccess) return fail(e, "cudaEventCreate");
  *out = ctx;
  return PTB_OK;
}

int32_t ptb_destroy(ptb_ctx* ctx) {
  if (!ctx) return PTB_OK;
  Ctx* c = &ctx->c;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->h_counters) cudaFreeHost(c->h_counters);
  if (c->h_sah) cudaFreeHost(c->h_sah);
  for (float* h : c->h_pass)
    if (h) cudaFreeHost(h);
  if (c->ev_a) cudaEventDestroy(c->ev_a);
  if (c->ev_b) cudaEventDestroy(c->ev_b);
  for (int b = 0; b < 2; ++b) {
    if (c->ev_in[b]) cudaEventDestroy(c->ev_in[b]);
    if (c->ev_kernel[b]) cudaEventDestroy(c->ev_kernel[b]);
    if (c->ev_out[b]) cudaEventDestroy(c->ev_out[b]);
  }
  for (cudaEvent_t e : c->ev_head_done) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_tail_done) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : c->ev_ring) if (e) cudaEventDestroy(e);
  if (c->s_tail) { cudaStreamSynchronize(c->s_tail); cudaStreamDestroy(c->s_tail); }
  if (c->s_work2) { cudaStreamSynchronize(c->s_work2); cudaStreamDestroy(c->s_work2); }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  for (cudaEvent_t e : c->ev_prof)
    if (e) cudaEventDestroy(e);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete ctx;  // DevBuf destructors release device memory
  return PTB_OK;
}

const char* ptb_last_error(const ptb_ctx* ctx) { return ctx ? ctx->c.last_error.c_str() : g_create_error.c_str(); }

int32_t ptb_set_stream(ptb_ctx* ctx, void* cuda_stream) {
  CTX_OR_FAIL(ctx);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  c->own_stream = false;
  return PTB_OK;
}

int32_t ptb_set_option(ptb_ctx* ctx, uint32_t option, uint32_t value) {
  CTX_OR_FAIL(ctx);
  if (option == PTB_OPT_TIME_KERNELS) c->opt_time_kernels = value != 0;
  else if (option == PTB_OPT_COUNT_TRAVERSAL) c->opt_count_traversal = value != 0;
  else return set_error(c, PTB_ERR_INVALID, "unknown option %u", option);
  return PTB_OK;
}

int32_t ptb_synchronize(ptb_ctx* ctx) {
  CTX_OR_FAIL(ctx);
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

// ---------------------------------------------------------------- scene
int32_t ptb_scene_set_spheres(ptb_ctx* ctx, const ptb_sphere* p, size_t n) {
  CTX_OR_FAIL(ctx);
  if (n && !p) return set_error(c, PTB_ERR_INVALID, "null spheres");
  // "the library copies on upload": straight into device memory (pinned caller buffers DMA at PCIe rate), no host
  // staging copy; the stream is drained before returning so the caller may reuse its buffer immediately.
  c->committed = false;
  c->n_spheres = 0;
  PTB_CUDA_TRY(c, c->d_raw_spheres.reserve(n * sizeof(ptb_sphere)));
  if (n) PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_raw_spheres.p, p, n * sizeof(ptb_sphere), cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  c->n_spheres = n;
  return PTB_OK;
}
// the instance list goes with ptb_scene_set_mesh and ptb_scene_set_triangles (the caller has drained the stream)
static void drop_instances(Ctx* c) {
  c->instanced = false;
  c->n_instances = 0;
  c->d_inst.release();
  c->d_inst_first.release();
  c->d_inst_xforms.release();
}
int32_t ptb_scene_set_triangles(ptb_ctx* ctx, const ptb_triangle* p, size_t n) {
  CTX_OR_FAIL(ctx);
  if (n && !p) return set_error(c, PTB_ERR_INVALID, "null triangles");
  c->committed = false;
  c->n_tris = 0;
  if (c->mesh) {  // flat mode: the mesh and its instances are dropped
    PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // a device update may still read into its buffers
    c->mesh = c->mesh_dirty = false;
    c->n_mesh_vertices = c->n_mesh_normals = c->n_mesh_tris = 0;
    c->d_mesh_vertices.release();
    c->d_mesh_normals.release();
    c->d_mesh_tris.release();
    drop_instances(c);
  }
  PTB_CUDA_TRY(c, c->d_raw_tris.reserve(n * sizeof(ptb_triangle)));
  if (n) PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_raw_tris.p, p, n * sizeof(ptb_triangle), cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  c->n_tris = n;
  return PTB_OK;
}
int32_t ptb_scene_set_mesh(ptb_ctx* ctx, const ptb_vec3* v, size_t nv, const ptb_vec3* nrm, size_t nn, const ptb_mesh_triangle* t,
                           size_t nt) {
  CTX_OR_FAIL(ctx);
  if ((nv && !v) || (nn && !nrm) || (nt && !t)) return set_error(c, PTB_ERR_INVALID, "null mesh array");
  if (nv > 0xFFFFFFFFull || nn > 0xFFFFFFFFull)
    return set_error(c, PTB_ERR_INVALID, "a mesh holds at most 2^32 - 1 vertices and normals (%zu vertices, %zu normals)", nv, nn);
  c->committed = false;
  c->n_tris = 0;
  c->mesh = false;
  c->n_mesh_vertices = c->n_mesh_normals = c->n_mesh_tris = 0;
  if (c->instanced) {
    PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // a device transform update may still write into its buffer
    drop_instances(c);
  }
  PTB_CUDA_TRY(c, c->d_mesh_vertices.reserve(nv * sizeof(ptb_vec3)));
  PTB_CUDA_TRY(c, c->d_mesh_normals.reserve(nn * sizeof(ptb_vec3)));
  PTB_CUDA_TRY(c, c->d_mesh_tris.reserve(nt * sizeof(ptb_mesh_triangle)));
  PTB_CUDA_TRY(c, c->d_raw_tris.reserve(nt * sizeof(ptb_triangle)));  // the expansion's output
  if (nv) PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_mesh_vertices.p, v, nv * sizeof(ptb_vec3), cudaMemcpyHostToDevice, c->stream));
  if (nn) PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_mesh_normals.p, nrm, nn * sizeof(ptb_vec3), cudaMemcpyHostToDevice, c->stream));
  if (nt) PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_mesh_tris.p, t, nt * sizeof(ptb_mesh_triangle), cudaMemcpyHostToDevice, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  c->n_mesh_vertices = nv;
  c->n_mesh_normals = nn;
  c->n_mesh_tris = c->n_tris = nt;
  c->mesh = c->mesh_dirty = true;
  return PTB_OK;
}
int32_t ptb_scene_set_mesh_instances(ptb_ctx* ctx, const ptb_mesh_instance* inst, const ptb_instance_xform* xf, size_t n) {
  CTX_OR_FAIL(ctx);
  if (!c->mesh)
    return set_error(c, PTB_ERR_INVALID, "mesh instances: the scene's triangles are flat, not an indexed mesh (ptb_scene_set_mesh)");
  if (n && (!inst || !xf)) return set_error(c, PTB_ERR_INVALID, "null mesh instances or transforms (%zu instances)", n);
  if (n > 0xFFFFFFFFull) return set_error(c, PTB_ERR_INVALID, "at most 2^32 - 1 mesh instances (%zu)", n);
  // every instance is checked before anything is allocated; the prefix sums are what k_expand_instances searches
  std::vector<uint32_t> first(n);
  uint64_t total = 0;
  for (size_t i = 0; i < n; ++i) {
    if ((uint64_t)inst[i].first_triangle + inst[i].n_triangles > c->n_mesh_tris)
      return set_error(c, PTB_ERR_INVALID, "mesh instance %zu: triangles [%u, %u + %u) outside the %zu the mesh holds", i,
                       inst[i].first_triangle, inst[i].first_triangle, inst[i].n_triangles, c->n_mesh_tris);
    first[i] = (uint32_t)total;
    total += inst[i].n_triangles;
    if (total > 0xFFFFFFFFull)
      return set_error(c, PTB_ERR_INVALID, "mesh instance %zu: the instances place more than 2^32 - 1 triangles", i);
  }
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // a device transform update may still write into the old list
  c->committed = false;
  c->n_tris = 0;
  c->instanced = false;
  c->n_instances = 0;
  PTB_CUDA_TRY(c, c->d_inst.reserve(n * sizeof(ptb_mesh_instance)));
  PTB_CUDA_TRY(c, c->d_inst_first.reserve(n * sizeof(uint32_t)));
  PTB_CUDA_TRY(c, c->d_inst_xforms.reserve(n * sizeof(ptb_instance_xform)));
  PTB_CUDA_TRY(c, c->d_raw_tris.reserve(total * sizeof(ptb_triangle)));  // the expansion's output
  if (n) {
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_inst.p, inst, n * sizeof(ptb_mesh_instance), cudaMemcpyHostToDevice, c->stream));
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_inst_first.p, first.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_inst_xforms.p, xf, n * sizeof(ptb_instance_xform), cudaMemcpyHostToDevice, c->stream));
  }
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  c->n_instances = n;
  c->n_tris = total;
  c->instanced = c->mesh_dirty = true;
  return PTB_OK;
}
// ptb_scene_update_*: primitives [first, first + n) of `raw` (count `have`, records of `rec` bytes) in place
static int32_t update_prims(Ctx* c, DevBuf& raw, size_t have, size_t rec, size_t first, const void* p, size_t n,
                            cudaMemcpyKind kind, const char* what) {
  if (first > have || n > have - first)
    return set_error(c, PTB_ERR_INVALID, "%s update [%zu, %zu + %zu) outside the %zu the scene holds", what, first, first, n, have);
  if (n == 0) return PTB_OK;
  if (!p) return set_error(c, PTB_ERR_INVALID, "null %s", what);
  c->committed = false;
  PTB_CUDA_TRY(c, cudaMemcpyAsync(static_cast<char*>(raw.p) + first * rec, p, n * rec, kind, c->stream));
  if (kind == cudaMemcpyHostToDevice) PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));  // the caller may reuse its buffer
  return PTB_OK;
}
int32_t ptb_scene_update_spheres(ptb_ctx* ctx, size_t first, const ptb_sphere* p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_prims(c, c->d_raw_spheres, c->n_spheres, sizeof(ptb_sphere), first, p, n, cudaMemcpyHostToDevice, "spheres");
}
// the triangles of a mesh scene are the mesh's expansion: the next commit would overwrite a flat update
#define FLAT_TRIANGLES_OR_FAIL(c)                                                                                        \
  if ((c)->mesh)                                                                                                         \
    return set_error(c, PTB_ERR_INVALID,                                                                                 \
                     "the scene's triangles are an indexed mesh: update it with ptb_scene_update_mesh_* (or go back to " \
                     "flat triangles with ptb_scene_set_triangles)")
int32_t ptb_scene_update_triangles(ptb_ctx* ctx, size_t first, const ptb_triangle* p, size_t n) {
  CTX_OR_FAIL(ctx);
  FLAT_TRIANGLES_OR_FAIL(c);
  return update_prims(c, c->d_raw_tris, c->n_tris, sizeof(ptb_triangle), first, p, n, cudaMemcpyHostToDevice, "triangles");
}
int32_t ptb_scene_update_spheres_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_prims(c, c->d_raw_spheres, c->n_spheres, sizeof(ptb_sphere), first, d_p, n, cudaMemcpyDeviceToDevice, "spheres");
}
int32_t ptb_scene_update_triangles_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  FLAT_TRIANGLES_OR_FAIL(c);
  return update_prims(c, c->d_raw_tris, c->n_tris, sizeof(ptb_triangle), first, d_p, n, cudaMemcpyDeviceToDevice, "triangles");
}
// ptb_scene_update_mesh_*: update_prims on one of the mesh arrays, which the next commit expands again
static int32_t update_mesh(Ctx* c, DevBuf& raw, size_t have, size_t rec, size_t first, const void* p, size_t n,
                           cudaMemcpyKind kind, const char* what) {
  if (!c->mesh)
    return set_error(c, PTB_ERR_INVALID, "%s update: the scene's triangles are flat, not an indexed mesh (ptb_scene_set_mesh)", what);
  const int32_t rc = update_prims(c, raw, have, rec, first, p, n, kind, what);
  if (rc == PTB_OK && n) c->mesh_dirty = true;
  return rc;
}
int32_t ptb_scene_update_mesh_vertices(ptb_ctx* ctx, size_t first, const ptb_vec3* p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_vertices, c->n_mesh_vertices, sizeof(ptb_vec3), first, p, n, cudaMemcpyHostToDevice, "mesh vertices");
}
int32_t ptb_scene_update_mesh_normals(ptb_ctx* ctx, size_t first, const ptb_vec3* p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_normals, c->n_mesh_normals, sizeof(ptb_vec3), first, p, n, cudaMemcpyHostToDevice, "mesh normals");
}
int32_t ptb_scene_update_mesh_triangles(ptb_ctx* ctx, size_t first, const ptb_mesh_triangle* p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_tris, c->n_mesh_tris, sizeof(ptb_mesh_triangle), first, p, n, cudaMemcpyHostToDevice, "mesh triangles");
}
int32_t ptb_scene_update_mesh_vertices_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_vertices, c->n_mesh_vertices, sizeof(ptb_vec3), first, d_p, n, cudaMemcpyDeviceToDevice, "mesh vertices");
}
int32_t ptb_scene_update_mesh_normals_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_normals, c->n_mesh_normals, sizeof(ptb_vec3), first, d_p, n, cudaMemcpyDeviceToDevice, "mesh normals");
}
int32_t ptb_scene_update_mesh_triangles_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_mesh(c, c->d_mesh_tris, c->n_mesh_tris, sizeof(ptb_mesh_triangle), first, d_p, n, cudaMemcpyDeviceToDevice, "mesh triangles");
}
// ptb_scene_update_instance_xforms*: update_prims on the transform list, which the next commit expands again
static int32_t update_xforms(Ctx* c, size_t first, const void* p, size_t n, cudaMemcpyKind kind) {
  if (!c->instanced)
    return set_error(c, PTB_ERR_INVALID, "instance transform update: the scene has no instance list (ptb_scene_set_mesh_instances)");
  const int32_t rc = update_prims(c, c->d_inst_xforms, c->n_instances, sizeof(ptb_instance_xform), first, p, n, kind, "instance transforms");
  if (rc == PTB_OK && n) c->mesh_dirty = true;
  return rc;
}
int32_t ptb_scene_update_instance_xforms(ptb_ctx* ctx, size_t first, const ptb_instance_xform* p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_xforms(c, first, p, n, cudaMemcpyHostToDevice);
}
int32_t ptb_scene_update_instance_xforms_device(ptb_ctx* ctx, size_t first, const void* d_p, size_t n) {
  CTX_OR_FAIL(ctx);
  return update_xforms(c, first, d_p, n, cudaMemcpyDeviceToDevice);
}
int32_t ptb_scene_set_materials(ptb_ctx* ctx, const ptb_material* p, size_t n) {
  CTX_OR_FAIL(ctx);
  if (n && !p) return set_error(c, PTB_ERR_INVALID, "null materials");
  for (size_t i = 0; i < n; ++i)
    if (p[i].kind > PTB_MAT_REFRACT) return set_error(c, PTB_ERR_INVALID, "material %zu: unknown kind %u", i, p[i].kind);
  c->materials.assign(p, p + n);
  c->committed = false;
  return PTB_OK;
}
int32_t ptb_scene_set_textures(ptb_ctx* ctx, const ptb_texture* p, size_t n) {
  CTX_OR_FAIL(ctx);
  if (n && !p) return set_error(c, PTB_ERR_INVALID, "null textures");
  for (size_t i = 0; i < n; ++i)
    if (p[i].kind > PTB_TEX_PERLIN) return set_error(c, PTB_ERR_INVALID, "texture %zu: unknown kind %u", i, p[i].kind);
  c->textures.assign(p, p + n);
  c->texture_data.clear();
  c->committed = false;
  return PTB_OK;
}
int32_t ptb_scene_set_texture_data(ptb_ctx* ctx, uint32_t texture, uint32_t width, uint32_t height, const float* data,
                                   size_t n_floats) {
  CTX_OR_FAIL(ctx);
  if (texture >= c->textures.size()) return set_error(c, PTB_ERR_INVALID, "texture index %u out of range", texture);
  if (!data) return set_error(c, PTB_ERR_INVALID, "null texture data");
  const uint32_t kind = c->textures[texture].kind;
  if (kind == PTB_TEX_IMAGE) {
    if (width == 0 || height == 0 || n_floats != (size_t)width * height * 3)  // textures/mod.rs:229 asserts non-zero
      return set_error(c, PTB_ERR_INVALID, "image texture %u: need 3*width*height floats and non-zero dimensions", texture);
  } else if (kind == PTB_TEX_PERLIN) {
    if (n_floats != PTB_PERLIN_TABLE_WORDS) return set_error(c, PTB_ERR_INVALID, "perlin texture %u: need %u words", texture, PTB_PERLIN_TABLE_WORDS);
    const uint32_t* perm = reinterpret_cast<const uint32_t*>(data) + 256;
    for (uint32_t i = 0; i < 768; ++i)
      if (perm[i] > 255u) return set_error(c, PTB_ERR_INVALID, "perlin texture %u: permutation entry out of range", texture);
  } else {
    return set_error(c, PTB_ERR_INVALID, "texture %u takes no bulk data", texture);
  }
  Ctx::TexData& td = c->texture_data[texture];
  td.width = width;
  td.height = height;
  td.data.assign(data, data + n_floats);
  c->committed = false;
  return PTB_OK;
}
int32_t ptb_scene_set_camera(ptb_ctx* ctx, const ptb_camera* cam) {
  CTX_OR_FAIL(ctx);
  if (!cam) return set_error(c, PTB_ERR_INVALID, "null camera");
  c->camera = *cam;
  c->have_camera = true;
  c->committed = false;
  return PTB_OK;
}
int32_t ptb_scene_set_sky(ptb_ctx* ctx, const ptb_sky* sky) {
  CTX_OR_FAIL(ctx);
  if (!sky) return set_error(c, PTB_ERR_INVALID, "null sky");
  c->sky = *sky;
  c->have_sky = true;
  c->committed = false;
  return PTB_OK;
}

int32_t ptb_scene_upload(ptb_ctx* ctx, const ptb_host_scene* s) {
  if (!ctx || !s) return PTB_ERR_INVALID;
  const ptb_sphere* sp; const ptb_triangle* tr; const ptb_material* ma; const ptb_texture* te;
  size_t ns = ptb_host_scene_spheres(s, &sp), nt = ptb_host_scene_triangles(s, &tr);
  size_t nm = ptb_host_scene_materials(s, &ma), nx = ptb_host_scene_textures(s, &te);
  ptb_camera cam; ptb_sky sky;
  ptb_host_scene_camera(s, &cam);
  ptb_host_scene_sky(s, &sky);
  int32_t rc;
  if ((rc = ptb_scene_set_textures(ctx, te, nx)) != PTB_OK) return rc;
  for (size_t i = 0; i < nx; ++i) {
    uint32_t w = 0, h = 0;
    const float* data = nullptr;
    const size_t n = ptb_host_scene_texture_data(s, (uint32_t)i, &w, &h, &data);
    if (n && (rc = ptb_scene_set_texture_data(ctx, (uint32_t)i, w, h, data, n)) != PTB_OK) return rc;
  }
  if ((rc = ptb_scene_set_materials(ctx, ma, nm)) != PTB_OK) return rc;
  if ((rc = ptb_scene_set_spheres(ctx, sp, ns)) != PTB_OK) return rc;
  if ((rc = ptb_scene_set_triangles(ctx, tr, nt)) != PTB_OK) return rc;
  if ((rc = ptb_scene_set_camera(ctx, &cam)) != PTB_OK) return rc;
  return ptb_scene_set_sky(ctx, &sky);
}

int32_t ptb_scene_commit(ptb_ctx* ctx, uint32_t build_flags) {
  CTX_OR_FAIL(ctx);
  return build_scene(c, build_flags);
}

int32_t ptb_bvh_info(ptb_ctx* ctx, uint64_t* n_prims, uint64_t* n_nodes) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n_prims) *n_prims = c->n_prims;
  if (n_nodes) *n_nodes = c->n_nodes;
  return PTB_OK;
}

int32_t ptb_bvh_builder(ptb_ctx* ctx, uint32_t* builder, uint32_t* sah_levels) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (builder) *builder = c->wide ? PTB_BUILD_WIDE : (c->sah ? PTB_BUILD_SAH : PTB_BUILD_BINARY);
  if (sah_levels) *sah_levels = c->sah ? c->sah_levels : 0u;
  return PTB_OK;
}

int32_t ptb_bvh_sah_cost(ptb_ctx* ctx, double* cost) {
  CTX_OR_FAIL(ctx);
  if (!cost) return set_error(c, PTB_ERR_INVALID, "null cost");
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (c->wide) return set_error(c, PTB_ERR_UNSUPPORTED, "the SAH cost is defined for the binary tree; the committed scene uses the 8-wide tree");
  return tree_sah_cost(c, cost);
}

int32_t ptb_bvh_export(ptb_ctx* ctx, uint32_t* morton_sorted, uint32_t* prim_sorted, ptb_bvh_node* nodes) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (c->n_prims == 0) return PTB_OK;
  if (morton_sorted)
    PTB_CUDA_TRY(c, cudaMemcpyAsync(morton_sorted, c->d_morton.p, c->n_prims * 4, cudaMemcpyDeviceToHost, c->stream));
  if (prim_sorted)  // Morton order (the wide tree keeps its own primitive order in d_slot_prim)
    PTB_CUDA_TRY(c, cudaMemcpyAsync(prim_sorted, c->wide ? c->d_prim_sorted.p : c->d_slot_prim.p, c->n_prims * 4, cudaMemcpyDeviceToHost, c->stream));
  if (nodes)
    PTB_CUDA_TRY(c, cudaMemcpyAsync(nodes, c->d_nodes.p, c->n_nodes * sizeof(ptb_bvh_node), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  if (nodes)  // the sphere flag of leaf references is device-internal
    for (uint64_t i = 0; i < c->n_nodes; ++i) {
      if (nodes[i].left & PTB_LEAF_BIT) nodes[i].left &= ~kSphereBit;
      if (nodes[i].right & PTB_LEAF_BIT) nodes[i].right &= ~kSphereBit;
    }
  return PTB_OK;
}

int32_t ptb_bvh_export_quantised(ptb_ctx* ctx, float frame[6], void* nodes32) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (!PTB_QNODES) return set_error(c, PTB_ERR_UNSUPPORTED, "this build walks the 64-byte nodes (compile with -DPTB_QNODES=1)");
  if (frame)
    for (int k = 0; k < 3; ++k) { frame[k] = c->dev.q_min[k]; frame[3 + k] = c->dev.q_step[k]; }
  if (c->n_prims == 0 || c->wide || !nodes32) return PTB_OK;
  PTB_CUDA_TRY(c, cudaMemcpyAsync(nodes32, c->d_qnodes.p, c->n_nodes * 32, cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  uint32_t* w = static_cast<uint32_t*>(nodes32);  // the sphere flag of leaf references is device-internal
  for (uint64_t i = 0; i < c->n_nodes; ++i)
    for (int k = 6; k < 8; ++k)
      if (w[8 * i + k] & PTB_LEAF_BIT) w[8 * i + k] &= ~kSphereBit;
  return PTB_OK;
}

int32_t ptb_bvh_wide_info(ptb_ctx* ctx, uint64_t* n_nodes, uint32_t* max_leaf) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n_nodes) *n_nodes = c->wide ? c->n_cw_nodes : 0;
  if (max_leaf) *max_leaf = c->cw_max_leaf;
  return PTB_OK;
}
int32_t ptb_bvh_wide_export(ptb_ctx* ctx, void* nodes96, uint32_t* slot_prim) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (!c->wide) return set_error(c, PTB_ERR_INVALID, "the committed scene uses the binary tree");
  if (c->n_prims == 0) return PTB_OK;
  if (nodes96) PTB_CUDA_TRY(c, cudaMemcpyAsync(nodes96, c->d_cw_nodes.p, c->n_cw_nodes * sizeof(CwNode), cudaMemcpyDeviceToHost, c->stream));
  if (slot_prim) PTB_CUDA_TRY(c, cudaMemcpyAsync(slot_prim, c->d_slot_prim.p, c->n_prims * 4, cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

// ---------------------------------------------------------------- batch queries (closest hit, visibility)
// A query over host buffers: in_bytes per record of `in` (plus in2_bytes of `in2`, when given) up, out_bytes per record of
// `out` back. Batches of 4 Mi records through two staging pairs: upload k+1 | traverse k | read back k-1. With pinned
// host buffers the three overlap and the call runs at PCIe speed; pageable buffers still work (the copies then serialise
// inside the driver).
typedef int32_t (*BatchLaunch)(Ctx* c, const void* d_in, const void* d_in2, size_t n, void* d_out);
static int32_t staged_batches(Ctx* c, size_t n, const void* in, size_t in_bytes, const void* in2, size_t in2_bytes, void* out,
                              size_t out_bytes, BatchLaunch launch) {
  size_t chunk = (size_t)1 << 22;
  if (const char* e = getenv("PTB_HIT_BATCH")) { size_t v = strtoull(e, nullptr, 10); if (v >= 1024) chunk = v; }
  const size_t cap = n < chunk ? n : chunk;
  DevBuf* dr[2] = {&c->d_rays, &c->d_rays2};
  DevBuf* dx[2] = {&c->d_index, &c->d_index2};
  DevBuf* dh[2] = {&c->d_hits, &c->d_hits2};
  const int nbuf = n > chunk ? 2 : 1;
  for (int b = 0; b < nbuf; ++b) {
    PTB_CUDA_TRY(c, dr[b]->reserve(cap * in_bytes));
    if (in2) PTB_CUDA_TRY(c, dx[b]->reserve(cap * in2_bytes));
    PTB_CUDA_TRY(c, dh[b]->reserve(cap * out_bytes));
  }
  if (!c->s_in) {
    PTB_CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
    PTB_CUDA_TRY(c, cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_in[b], cudaEventDisableTiming));
      PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_kernel[b], cudaEventDisableTiming));
      PTB_CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_out[b], cudaEventDisableTiming));
    }
  }
  // On any failure the copies of earlier batches may still be in flight against the caller's buffers: drain all three
  // streams before returning, the caller is free to release its buffers as soon as the call is back.
  auto drain = [&](int32_t rc) {
    cudaStreamSynchronize(c->s_out);
    cudaStreamSynchronize(c->s_in);
    cudaStreamSynchronize(c->stream);
    return rc;
  };
#define PTB_TRY_DRAIN(expr)                                                  \
  do {                                                                       \
    cudaError_t _e = (expr);                                                 \
    if (_e != cudaSuccess) return drain(ptb::check_cuda(c, _e, #expr));      \
  } while (0)
  const char* src = static_cast<const char*>(in);
  const char* src2 = static_cast<const char*>(in2);
  char* dst = static_cast<char*>(out);
  // the staging buffers may still be in use by earlier work on the main stream
  PTB_TRY_DRAIN(cudaEventRecord(c->ev_kernel[0], c->stream));
  PTB_TRY_DRAIN(cudaStreamWaitEvent(c->s_in, c->ev_kernel[0], 0));
  size_t k = 0;
  for (size_t off = 0; off < n; off += chunk, ++k) {
    const size_t m = n - off < chunk ? n - off : chunk;
    const int b = (int)(k & 1u);
    if (k >= 2) PTB_TRY_DRAIN(cudaStreamWaitEvent(c->s_in, c->ev_kernel[b], 0));  // batch k-2 no longer reads d_rays[b]
    PTB_TRY_DRAIN(cudaMemcpyAsync(dr[b]->p, src + off * in_bytes, m * in_bytes, cudaMemcpyHostToDevice, c->s_in));
    if (in2) PTB_TRY_DRAIN(cudaMemcpyAsync(dx[b]->p, src2 + off * in2_bytes, m * in2_bytes, cudaMemcpyHostToDevice, c->s_in));
    PTB_TRY_DRAIN(cudaEventRecord(c->ev_in[b], c->s_in));
    PTB_TRY_DRAIN(cudaStreamWaitEvent(c->stream, c->ev_in[b], 0));
    if (k >= 2) PTB_TRY_DRAIN(cudaStreamWaitEvent(c->stream, c->ev_out[b], 0));     // batch k-2's results left d_hits[b]
    int32_t rc = launch(c, dr[b]->p, in2 ? dx[b]->p : nullptr, m, dh[b]->p);
    if (rc != PTB_OK) return drain(rc);
    PTB_TRY_DRAIN(cudaEventRecord(c->ev_kernel[b], c->stream));
    PTB_TRY_DRAIN(cudaStreamWaitEvent(c->s_out, c->ev_kernel[b], 0));
    PTB_TRY_DRAIN(cudaMemcpyAsync(dst + off * out_bytes, dh[b]->p, m * out_bytes, cudaMemcpyDeviceToHost, c->s_out));
    PTB_TRY_DRAIN(cudaEventRecord(c->ev_out[b], c->s_out));
  }
  PTB_TRY_DRAIN(cudaStreamSynchronize(c->s_out));
  PTB_TRY_DRAIN(cudaStreamSynchronize(c->stream));
#undef PTB_TRY_DRAIN
  return PTB_OK;
}
static int32_t closest_hit_batch(Ctx* c, const void* d_rays, const void*, size_t n, void* d_hits) {
  return launch_closest_hit(c, d_rays, n, d_hits);
}
static int32_t visibility_batch(Ctx* c, const void* d_rays, const void* d_index, size_t n, void* d_out) {
  return launch_visibility(c, d_rays, d_index, n, d_out);
}

int32_t ptb_closest_hit_device(ptb_ctx* ctx, const void* d_rays, size_t n, void* d_hits) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n && (!d_rays || !d_hits)) return set_error(c, PTB_ERR_INVALID, "null device buffer");
  return launch_closest_hit(c, d_rays, n, d_hits);
}

int32_t ptb_closest_hit(ptb_ctx* ctx, const ptb_ray* rays, size_t n, ptb_hit* hits) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n == 0) return PTB_OK;
  if (!rays || !hits) return set_error(c, PTB_ERR_INVALID, "null host buffer");
  return staged_batches(c, n, rays, sizeof(ptb_ray), nullptr, 0, hits, sizeof(ptb_hit), closest_hit_batch);
}

int32_t ptb_check_hit_index_device(ptb_ctx* ctx, const void* d_rays, const void* d_index, size_t n, void* d_hits) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n && (!d_rays || !d_index || !d_hits)) return set_error(c, PTB_ERR_INVALID, "null device buffer");
  return launch_visibility(c, d_rays, d_index, n, d_hits);
}

int32_t ptb_check_hit_index(ptb_ctx* ctx, const ptb_ray* rays, const uint32_t* index, size_t n, ptb_hit* hits) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n == 0) return PTB_OK;
  if (!rays || !index || !hits) return set_error(c, PTB_ERR_INVALID, "null host buffer");
  return staged_batches(c, n, rays, sizeof(ptb_ray), index, sizeof(uint32_t), hits, sizeof(ptb_hit), visibility_batch);
}

int32_t ptb_occluded_device(ptb_ctx* ctx, const void* d_rays, size_t n, void* d_occluded) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n && (!d_rays || !d_occluded)) return set_error(c, PTB_ERR_INVALID, "null device buffer");
  return launch_visibility(c, d_rays, nullptr, n, d_occluded);
}

int32_t ptb_occluded(ptb_ctx* ctx, const ptb_occlusion_ray* rays, size_t n, uint8_t* occluded) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (n == 0) return PTB_OK;
  if (!rays || !occluded) return set_error(c, PTB_ERR_INVALID, "null host buffer");
  return staged_batches(c, n, rays, sizeof(ptb_occlusion_ray), nullptr, 0, occluded, 1, visibility_batch);
}

// ---------------------------------------------------------------- render
static int32_t ensure_accum(Ctx* c, uint32_t w, uint32_t h) {
  if (c->accum_w == w && c->accum_h == h && c->d_accum.p) return PTB_OK;
  const size_t bytes = (size_t)w * h * 3 * sizeof(float);
  PTB_CUDA_TRY(c, c->d_accum.alloc(bytes));
  PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_accum.p, 0, bytes, c->stream));
  c->accum_w = w;
  c->accum_h = h;
  c->accum_samples = 0;
  return PTB_OK;
}

// the option checks of every render entry point; `method` is not read by ptb_render_aov
static int32_t check_render_opts(Ctx* c, const ptb_render_opts* opts, bool method) {
  if (!opts) return set_error(c, PTB_ERR_INVALID, "null render opts");
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  if (opts->width < 2 || opts->height < 2) return set_error(c, PTB_ERR_INVALID, "width and height must be >= 2");
  if ((uint64_t)opts->width * opts->height > 0x7FFFFFFFull) return set_error(c, PTB_ERR_INVALID, "image too large");
  if (method && opts->method != PTB_METHOD_NAIVE && opts->method != PTB_METHOD_MIS) return set_error(c, PTB_ERR_INVALID, "unknown method");
  if (opts->row_begin >= opts->height || (uint64_t)opts->row_begin + opts->row_count > opts->height)
    return set_error(c, PTB_ERR_INVALID, "image tile rows [%u, %u) outside the %u rows of the image", opts->row_begin,
                     opts->row_begin + opts->row_count, opts->height);
  return PTB_OK;
}

int32_t ptb_render(ptb_ctx* ctx, const ptb_render_opts* opts, ptb_progress_fn progress, void* user) {
  CTX_OR_FAIL(ctx);
  int32_t rc = check_render_opts(c, opts, true);
  if (rc != PTB_OK) return rc;
  rc = ensure_accum(c, opts->width, opts->height);
  if (rc != PTB_OK) return rc;
  rc = render_wavefront(c, *opts, progress, user);
  if (rc == PTB_ERR_ABORTED) {
    // An aborted call leaves the radiance of the paths that had finished in the accumulator (whole pixels in window
    // mode) without a sample count to divide by: the accumulator is cleared, earlier samples included, exactly as the
    // reference drops its buffers when the closure returns true (random_sampler.rs:84-86).
    cudaMemsetAsync(c->d_accum.p, 0, (size_t)c->accum_w * c->accum_h * 12, c->stream);
    cudaStreamSynchronize(c->stream);
    c->accum_samples = 0;
  }
  return rc;
}

__global__ void k_add_into(const float* __restrict__ src, float* __restrict__ dst, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

int32_t ptb_render_passes(ptb_ctx* ctx, const ptb_render_opts* opts, ptb_pass_fn update, void* user) {
  CTX_OR_FAIL(ctx);
  int32_t rc = check_render_opts(c, opts, true);
  if (rc != PTB_OK) return rc;
  rc = ensure_accum(c, opts->width, opts->height);
  if (rc != PTB_OK) return rc;
  const size_t n = (size_t)opts->width * opts->height * 3;
  PTB_CUDA_TRY(c, c->d_pass.reserve(n * sizeof(float)));
  if (c->h_pass_floats < n) {
    for (float*& h : c->h_pass) {
      if (h) cudaFreeHost(h);
      h = nullptr;
      PTB_CUDA_TRY(c, cudaMallocHost(&h, n * sizeof(float)));
    }
    c->h_pass_floats = n;
  }
  uint64_t rays[2] = {0, 0};
  for (uint32_t k = 0; k < opts->samples_per_pixel; ++k) {
    const int cur = (int)(k & 1u);
    // random_sampler.rs:31-81: render pass k into the `current` buffer
    PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_pass.p, 0, n * sizeof(float), c->stream));
    ptb_render_opts one = *opts;
    one.samples_per_pixel = 1;
    one.sample_offset = opts->sample_offset + k;
    const uint64_t before = c->stats.rays_reference;
    c->accum_target = c->d_pass.as<float>();
    rc = render_wavefront(c, one, nullptr, nullptr);
    c->accum_target = nullptr;
    if (rc != PTB_OK) return rc;
    rays[cur] = c->stats.rays_reference - before;
    k_add_into<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_pass.as<float>(), c->d_accum.as<float>(), n);
    c->stats.kernel_launches += 1;
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->h_pass[cur], c->d_pass.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    // random_sampler.rs:82-88: `previous` (pass k-1) goes to the callback with i = k
    if (k != 0 && update && update(user, c->h_pass[cur ^ 1], n, k, rays[cur ^ 1]))
      return set_error(c, PTB_ERR_ABORTED, "render stopped by the presentation callback after pass %u", k);
  }
  // random_sampler.rs:91-98: the last pass, with i = samples_per_pixel
  if (opts->samples_per_pixel && update) {
    const int last = (int)((opts->samples_per_pixel - 1u) & 1u);
    update(user, c->h_pass[last], n, opts->samples_per_pixel, rays[last]);
  }
  return PTB_OK;
}

int32_t ptb_accum_clear(ptb_ctx* ctx) {
  CTX_OR_FAIL(ctx);
  if (c->d_accum.p) PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_accum.p, 0, (size_t)c->accum_w * c->accum_h * 12, c->stream));
  c->accum_samples = 0;
  return PTB_OK;
}

int32_t ptb_accum_read(ptb_ctx* ctx, float* rgb, size_t n_floats, int32_t normalise) {
  CTX_OR_FAIL(ctx);
  if (!c->d_accum.p) return set_error(c, PTB_ERR_INVALID, "nothing rendered yet");
  const size_t n = (size_t)c->accum_w * c->accum_h * 3;
  if (!rgb || n_floats != n) return set_error(c, PTB_ERR_INVALID, "accum_read expects %zu floats", n);
  if (normalise && c->accum_samples > 0) {
    // running mean of src/main.rs:179-185 == sum / samples; scaled on the device into the staging buffer
    PTB_CUDA_TRY(c, c->d_hits.reserve(n * sizeof(float)));
    k_scale_copy<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_accum.as<float>(), c->d_hits.as<float>(), n,
                                                                     1.0f / (float)c->accum_samples);
    c->stats.kernel_launches += 1;
    PTB_CUDA_TRY(c, cudaMemcpyAsync(rgb, c->d_hits.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  } else {
    PTB_CUDA_TRY(c, cudaMemcpyAsync(rgb, c->d_accum.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  }
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

int32_t ptb_accum_device_ptr(ptb_ctx* ctx, void** d_ptr, size_t* n_floats) {
  CTX_OR_FAIL(ctx);
  if (!c->d_accum.p) return set_error(c, PTB_ERR_INVALID, "nothing rendered yet");
  if (d_ptr) *d_ptr = c->d_accum.p;
  if (n_floats) *n_floats = (size_t)c->accum_w * c->accum_h * 3;
  return PTB_OK;
}

int32_t ptb_accum_set_samples(ptb_ctx* ctx, uint64_t total_samples) {
  CTX_OR_FAIL(ctx);
  c->accum_samples = total_samples;
  return PTB_OK;
}

// ---------------------------------------------------------------- denoiser feature buffers
static int32_t ensure_aov(Ctx* c, uint32_t w, uint32_t h) {
  if (c->aov_w == w && c->aov_h == h && c->d_aov.p) return PTB_OK;
  const size_t bytes = (size_t)w * h * 8 * sizeof(float);
  PTB_CUDA_TRY(c, c->d_aov.alloc(bytes));
  PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_aov.p, 0, bytes, c->stream));
  PTB_CUDA_TRY(c, c->d_motion.alloc(bytes / 2));
  PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_motion.p, 0, bytes / 2, c->stream));
  c->aov_w = w;
  c->aov_h = h;
  c->aov_samples = 0;
  return PTB_OK;
}

int32_t ptb_render_aov(ptb_ctx* ctx, const ptb_render_opts* opts) {
  CTX_OR_FAIL(ctx);
  int32_t rc = check_render_opts(c, opts, false);
  if (rc != PTB_OK) return rc;
  if ((uint64_t)opts->sample_offset + opts->samples_per_pixel > kMaxSampleIndex)
    return set_error(c, PTB_ERR_INVALID, "sample_offset + samples_per_pixel must be <= %u", kMaxSampleIndex);
  rc = ensure_aov(c, opts->width, opts->height);
  if (rc != PTB_OK) return rc;
  rc = launch_aov(c, *opts);
  if (rc != PTB_OK) return rc;
  c->aov_samples += opts->samples_per_pixel;
  return PTB_OK;
}

int32_t ptb_aov_clear(ptb_ctx* ctx) {
  CTX_OR_FAIL(ctx);
  if (c->d_aov.p) PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_aov.p, 0, (size_t)c->aov_w * c->aov_h * 8 * sizeof(float), c->stream));
  if (c->d_motion.p) PTB_CUDA_TRY(c, cudaMemsetAsync(c->d_motion.p, 0, (size_t)c->aov_w * c->aov_h * 4 * sizeof(float), c->stream));
  c->aov_samples = 0;
  return PTB_OK;
}

// one buffer out of the per-pixel records [albedo.rgb | coverage] [normal.xyz | depth]; normalise: albedo, normal and
// coverage over the sample count, depth over the pixel's coverage (0 where nothing was hit)
__global__ void k_aov_read(const float4* __restrict__ sums, float* __restrict__ out, size_t npix, uint32_t aov,
                           int normalise, float samples) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const float4 s0 = sums[2 * i], s1 = sums[2 * i + 1];
  if (aov == PTB_AOV_ALBEDO || aov == PTB_AOV_NORMAL) {
    const float4 s = aov == PTB_AOV_ALBEDO ? s0 : s1;
    out[3 * i + 0] = normalise ? s.x / samples : s.x;
    out[3 * i + 1] = normalise ? s.y / samples : s.y;
    out[3 * i + 2] = normalise ? s.z / samples : s.z;
  } else if (aov == PTB_AOV_DEPTH) {
    out[i] = normalise ? (s0.w > 0.0f ? s1.w / s0.w : 0.0f) : s1.w;
  } else {
    out[i] = normalise ? s0.w / samples : s0.w;
  }
}

int32_t ptb_aov_read(ptb_ctx* ctx, uint32_t aov, float* out, size_t n_floats, int32_t normalise) {
  CTX_OR_FAIL(ctx);
  if (!c->d_aov.p) return set_error(c, PTB_ERR_INVALID, "no AOV rendered yet");
  if (aov > PTB_AOV_COVERAGE) return set_error(c, PTB_ERR_INVALID, "unknown AOV %u", aov);
  const size_t npix = (size_t)c->aov_w * c->aov_h;
  const size_t n = npix * (aov == PTB_AOV_ALBEDO || aov == PTB_AOV_NORMAL ? 3 : 1);
  if (!out || n_floats != n) return set_error(c, PTB_ERR_INVALID, "aov_read expects %zu floats", n);
  PTB_CUDA_TRY(c, c->d_hits.reserve(n * sizeof(float)));
  // with no samples yet there is nothing to divide by: the (zero) sums are returned, as ptb_accum_read does
  const int norm = normalise && c->aov_samples > 0;
  k_aov_read<<<(unsigned)((npix + 255) / 256), 256, 0, c->stream>>>(c->d_aov.as<float4>(), c->d_hits.as<float>(), npix, aov,
                                                                    norm, (float)c->aov_samples);
  c->stats.kernel_launches += 1;
  PTB_CUDA_TRY(c, cudaGetLastError());
  PTB_CUDA_TRY(c, cudaMemcpyAsync(out, c->d_hits.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

// ---------------------------------------------------------------- motion vectors
int32_t ptb_motion_mark(ptb_ctx* ctx) {
  CTX_OR_FAIL(ctx);
  if (!c->committed) return set_error(c, PTB_ERR_INVALID, "scene not committed");
  PTB_CUDA_TRY(c, c->d_mark_spheres.reserve(c->n_spheres * sizeof(ptb_sphere)));
  PTB_CUDA_TRY(c, c->d_mark_tris.reserve(c->n_tris * sizeof(ptb_triangle)));
  if (c->n_spheres)
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_mark_spheres.p, c->d_raw_spheres.p, c->n_spheres * sizeof(ptb_sphere),
                                    cudaMemcpyDeviceToDevice, c->stream));
  if (c->n_tris)
    PTB_CUDA_TRY(c, cudaMemcpyAsync(c->d_mark_tris.p, c->d_raw_tris.p, c->n_tris * sizeof(ptb_triangle), cudaMemcpyDeviceToDevice,
                                    c->stream));
  c->mark_spheres = c->n_spheres;
  c->mark_tris = c->n_tris;
  c->mark_cam[0] = c->dev.cam_origin;
  c->mark_cam[1] = c->dev.cam_lower_left;
  c->mark_cam[2] = c->dev.cam_horizontal;
  c->mark_cam[3] = c->dev.cam_vertical;
  c->have_mark = true;
  return PTB_OK;
}

// mean Δx, Δy, t' over the valid samples of each pixel, 0 where there are none
__global__ void k_motion_read(const float4* __restrict__ sums, float* __restrict__ out, size_t npix) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const float4 s = sums[i];
  const bool any = s.w > 0.0f;
  out[3 * i + 0] = any ? s.x / s.w : 0.0f;
  out[3 * i + 1] = any ? s.y / s.w : 0.0f;
  out[3 * i + 2] = any ? s.z / s.w : 0.0f;
}

int32_t ptb_motion_read(ptb_ctx* ctx, float* out, size_t n_floats) {
  CTX_OR_FAIL(ctx);
  if (!c->d_aov.p) return set_error(c, PTB_ERR_INVALID, "no AOV rendered yet");
  const size_t npix = (size_t)c->aov_w * c->aov_h, n = npix * 3;
  if (!out || n_floats != n) return set_error(c, PTB_ERR_INVALID, "motion_read expects %zu floats", n);
  PTB_CUDA_TRY(c, c->d_hits.reserve(n * sizeof(float)));
  k_motion_read<<<(unsigned)((npix + 255) / 256), 256, 0, c->stream>>>(c->d_motion.as<float4>(), c->d_hits.as<float>(), npix);
  c->stats.kernel_launches += 1;
  PTB_CUDA_TRY(c, cudaGetLastError());
  PTB_CUDA_TRY(c, cudaMemcpyAsync(out, c->d_hits.p, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  PTB_CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return PTB_OK;
}

// ---------------------------------------------------------------- sampler test hook
int32_t ptb_sample_only(ptb_ctx* ctx, const ptb_sampler_query* query, size_t n, float* dirs, float* pdf) {
  CTX_OR_FAIL(ctx);
  if (!query || (n && !dirs)) return set_error(c, PTB_ERR_INVALID, "null argument");
  return sampler_hook(c, *query, n, nullptr, dirs, pdf);
}
int32_t ptb_sampler_pdf(ptb_ctx* ctx, const ptb_sampler_query* query, const float* dirs, size_t n, float* pdf) {
  CTX_OR_FAIL(ctx);
  if (!query || (n && (!dirs || !pdf))) return set_error(c, PTB_ERR_INVALID, "null argument");
  return sampler_hook(c, *query, n, dirs, nullptr, pdf);
}

int32_t ptb_stats_get(ptb_ctx* ctx, ptb_stats* out) {
  CTX_OR_FAIL(ctx);
  if (!out) return PTB_ERR_INVALID;
  *out = c->stats;
  return PTB_OK;
}
int32_t ptb_stats_reset(ptb_ctx* ctx) {
  CTX_OR_FAIL(ctx);
  const double b = c->stats.build_ms;
  c->stats = ptb_stats{};
  c->stats.build_ms = b;
  return PTB_OK;
}

}  // extern "C"
