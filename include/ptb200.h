/*
 * ptb200.h — C ABI of the B200-native path-tracing backend ("ptb200") for
 * nonl4331/raytracing-rust.
 *
 * This header is the drop-in boundary: it is exactly what a Rust `build.rs` +
 * `extern "C"` shim (see ffi/rust/, INTEGRATION.md) binds when the frontend is
 * started with `--backend cuda`.  All citations are file:line into the reference
 * tree (crates/<name>/src/... abbreviated as <name>/...).
 *
 * Conventions
 *   - every entry point returns an int32 status (PTB_OK == 0); no C++ exception
 *     or Rust panic ever crosses the boundary; ptb_last_error() gives the text;
 *   - the caller owns all host buffers; the library copies on upload;
 *   - one ptb_ctx per GPU; a ctx is not thread-safe, distinct ctxs are independent;
 *   - plain pointers and sizes only; every struct below is #[repr(C)]-mirrorable POD;
 *   - primitive ids are indices into the reference's primitive array order:
 *     all spheres first, then all mesh triangles (loader/lib.rs:234-240);
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry
 *     point fails with PTB_ERR_CUDA.
 */
#ifndef PTB200_H
#define PTB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PTB_ABI_VERSION 2u  /* 2: ptb_render_opts gained row_begin / row_count (image-tile axis of the multi-GPU split) */

/* ---------------------------------------------------------------- status -- */
enum {
  PTB_OK = 0,
  PTB_ERR_INVALID = 1,   /* bad argument / bad state (e.g. render before commit)   */
  PTB_ERR_CUDA = 2,      /* CUDA runtime error or no device                          */
  PTB_ERR_OOM = 3,       /* host or device allocation failed                         */
  PTB_ERR_PARSE = 4,     /* .ssml / .obj syntax error     (loader LoadErr::ParseError, lib.rs:180-194) */
  PTB_ERR_IO = 5,        /* file could not be read/written (LoadErr::FileNotRead)    */
  PTB_ERR_MISSING = 6,   /* required key/object missing   (LoadErr::MissingRequired, MissingCamera) */
  PTB_ERR_ABORTED = 7,   /* progress callback asked to stop (random_sampler.rs:84-86) */
  PTB_ERR_UNSUPPORTED = 8
};

/* ------------------------------------------------------------------- POD -- */
/* rt_core/vec.rs:108-114 — `#[repr(C)] struct Vec3 { x, y, z }` with Float = f32 (rt_core/lib.rs:23-29) */
typedef struct ptb_vec3 { float x, y, z; } ptb_vec3;

/* implementations/primitives/sphere.rs:8-13 (material reference -> index into the material array) */
typedef struct ptb_sphere {
  ptb_vec3 center;
  float    radius;
  uint32_t material;
} ptb_sphere;

/* implementations/primitives/triangle.rs:9-14 / :30-36 — Triangle and MeshTriangle both flatten to this:
 * three positions, three vertex normals (MeshData indirection resolved by the host), one material. */
typedef struct ptb_triangle {
  ptb_vec3 p[3];
  ptb_vec3 n[3];
  uint32_t material;
} ptb_triangle;

/* enum order == tag order: implementations/materials/mod.rs:19-25 */
enum {
  PTB_MAT_EMIT = 0,             /* emissive.rs:7-10      param = strength */
  PTB_MAT_LAMBERTIAN = 1,       /* lambertian.rs:6-9     param = albedo   */
  PTB_MAT_TROWBRIDGE_REITZ = 2, /* trowbridge_reitz.rs:6-11  param = alpha (already squared), ior, metallic */
  PTB_MAT_REFLECT = 3,          /* reflect.rs:8-11       param = fuzz     */
  PTB_MAT_REFRACT = 4           /* refract.rs:9-12       param = eta      */
};
typedef struct ptb_material {
  uint32_t kind;
  uint32_t texture;   /* index into the texture array */
  float    param;
  ptb_vec3 ior;       /* TrowbridgeReitz only */
  float    metallic;  /* TrowbridgeReitz only */
} ptb_material;

/* enum order == tag order: implementations/textures/mod.rs:17-24 */
enum {
  PTB_TEX_CHECKERED = 0, /* textures/mod.rs:26-30,61-73   a = colour_one, b = colour_two */
  PTB_TEX_SOLID = 1,     /* textures/mod.rs:182-200       a = colour                     */
  PTB_TEX_IMAGE = 2,     /* textures/mod.rs:202-266       pixels via ptb_scene_set_texture_data  */
  PTB_TEX_LERP = 3,      /* textures/mod.rs:268-291       a = colour_one, b = colour_two */
  PTB_TEX_PERLIN = 4     /* textures/mod.rs:75-180        tables via ptb_scene_set_texture_data  */
};
#define PTB_PERLIN_TABLE_WORDS 1024u /* 256 f32 ran_vecs[i].x (every ran_vec is r*(1,1,1), textures/mod.rs:96-99)
                                        then perm_x, perm_y, perm_z as 3 x 256 uint32 bit patterns */
typedef struct ptb_texture {
  uint32_t kind;
  ptb_vec3 a;
  ptb_vec3 b;
} ptb_texture;

/* implementations/camera.rs:6-17 — only the four vectors get_ray() reads (camera.rs:57-63) */
typedef struct ptb_camera {
  ptb_vec3 origin;
  ptb_vec3 lower_left;
  ptb_vec3 horizontal;
  ptb_vec3 vertical;
} ptb_camera;

/* implementations/sky.rs:12-18 — material is always Emit(texture, 1.0) (loader/misc.rs:26);
 * sampler_res (0,0) disables importance sampling (sky.rs:61-63). The library builds the
 * Distribution2D table itself (sky.rs:20-37, textures/mod.rs:32-50, distributions.rs:82-99). */
typedef struct ptb_sky {
  uint32_t texture;
  uint32_t sampler_res_x;
  uint32_t sampler_res_y;
} ptb_sky;

/* rt_core/ray.rs:4-11 — the caller passes origin + (un-normalised) direction; the library derives
 * direction/|direction|, d_inverse and shear exactly as Ray::new does (ray.rs:13-46). 2 x 16 B. */
typedef struct ptb_ray {
  float ox, oy, oz, _pad0;
  float dx, dy, dz, _pad1;
} ptb_ray;

/* what AccelerationStructure::check_hit returns (implementations/acceleration/mod.rs:265-298), reduced
 * to the comparable part: t, primitive id in the ORIGINAL (pre-BVH) order, barycentrics b1,b2 of
 * triangle.rs:149-151 (0 for spheres). Miss: prim = PTB_MISS, t = 0 (sky.rs:79-91). 16 B. */
#define PTB_MISS 0xFFFFFFFFu
typedef struct ptb_hit {
  float    t;
  uint32_t prim;
  float    u, v;
} ptb_hit;

/* implementations/samplers/mod.rs:43-47 */
enum { PTB_METHOD_NAIVE = 0, PTB_METHOD_MIS = 1 };

/* implementations/samplers/mod.rs:22-29 + the constants of integrators/mod.rs:7-8 made explicit,
 * plus what a deterministic, shardable device renderer needs (seed, sample_offset). */
typedef struct ptb_render_opts {
  uint32_t width;
  uint32_t height;
  uint32_t samples_per_pixel; /* samples rendered by THIS call                                  */
  uint32_t sample_offset;     /* absolute index of the first sample (rank r renders [off, off+spp)) */
  uint32_t method;            /* PTB_METHOD_*; reference default is MIS (parameters.rs:34-35)   */
  uint32_t max_depth;         /* 0 -> 50  (integrators/mod.rs:7)                                */
  uint32_t rr_threshold;      /* 0xFFFFFFFF -> 3 (integrators/mod.rs:8); RR applies when depth > threshold */
  uint32_t flags;             /* reserved, 0                                                    */
  uint64_t seed;              /* counter-based RNG key; same seed + same sample range == same image */
  uint32_t row_begin;         /* image tile: only the pixel rows [row_begin, row_begin + row_count) are rendered;   */
  uint32_t row_count;         /* 0 -> every row from row_begin down. Pixels keep their full-image coordinates (camera,
                                 RNG key, accumulator position), so the tiles of one image add up to the whole image. */
} ptb_render_opts;
#define PTB_RR_DEFAULT 0xFFFFFFFFu

/* BVH2 node as exported for bit-exact tests: both children's boxes live in the parent (64 B).
 * child ref: bit31 set -> leaf, low bits = position in the Morton-sorted primitive order. */
#define PTB_LEAF_BIT 0x80000000u
typedef struct ptb_bvh_node {
  float    lmin[3], lmax[3];
  float    rmin[3], rmax[3];
  uint32_t left, right;
  uint32_t parent;  /* 0xFFFFFFFF for the root */
  uint32_t _pad;
} ptb_bvh_node;

typedef struct ptb_stats {
  uint64_t rays_camera;        /* traversals launched for camera rays                         */
  uint64_t rays_bounce;        /* ... for BSDF-sampled bounce rays                            */
  uint64_t rays_shadow_light;  /* ... for NEE rays towards a light primitive (check_hit_index) */
  uint64_t rays_shadow_sky;    /* ... for NEE rays towards the sky                            */
  uint64_t rays_reference;     /* the reference's own counter: naive = 1 per check_hit (integrators/mod.rs:34),
                                  MIS = 1 per bounce iteration (mis.rs:38)                     */
  uint64_t paths;              /* camera paths finished                                       */
  uint64_t wavefront_iterations;
  uint64_t kernel_launches;    /* kernels of this library launched since the last ptb_stats_reset */
  uint64_t nodes_fetched;      /* PTB_OPT_COUNT_TRAVERSAL: 64-byte BVH nodes fetched by closest-hit traversals */
  uint64_t prims_tested;       /* PTB_OPT_COUNT_TRAVERSAL: primitives tested by closest-hit traversals          */
  uint64_t rays_counted;       /* PTB_OPT_COUNT_TRAVERSAL: closest-hit traversals the two counters cover        */
  uint64_t trace_launches;     /* traversal kernel launches (k_trace / k_closest_hit_api / k_visibility_api)    */
  double   build_ms;           /* last ptb_scene_commit: device LBVH build time (refit time for PTB_BUILD_REFIT) */
  double   render_ms;          /* last ptb_render: device time (CUDA events)                  */
  double   ms_generate;        /* PTB_OPT_TIME_KERNELS: summed CUDA-event time per kernel class */
  double   ms_trace;
  double   ms_shade;
  double   ms_shadow;
  double   ms_tail;            /* fused tail launches (k_tail: closest hit + shade + NEE of a chunk's last paths); they
                                  run on a side stream under the next chunk, so the classes may add up to > render_ms */
} ptb_stats;

typedef struct ptb_ctx ptb_ctx;

/* called between wavefront iterations; return non-zero to abort (random_sampler.rs:82-88 contract,
 * carrying counters only — the per-pass image is replaced by the device accumulator). */
typedef int32_t (*ptb_progress_fn)(void* user, uint64_t samples_completed, uint64_t rays_shot);

/* ------------------------------------------------------------ lifecycle -- */
uint32_t    ptb_abi_version(void);
int32_t     ptb_device_count(int32_t* count);
int32_t     ptb_create(int32_t device, ptb_ctx** out);
int32_t     ptb_destroy(ptb_ctx* ctx);
const char* ptb_last_error(const ptb_ctx* ctx);           /* ctx may be NULL: last error of ptb_create */
int32_t     ptb_set_stream(ptb_ctx* ctx, void* cuda_stream); /* optional: run on the caller's cudaStream_t */
int32_t     ptb_synchronize(ptb_ctx* ctx);
/* Measurement switches (off by default; they add event records / atomic counters to the hot path). */
enum { PTB_OPT_TIME_KERNELS = 1, PTB_OPT_COUNT_TRAVERSAL = 2 };
int32_t     ptb_set_option(ptb_ctx* ctx, uint32_t option, uint32_t value);

/* ---------------------------------------------------------------- scene -- */
/* Replaces what loader::load_file_full returns (loader/lib.rs:196-243) + Bvh::new's input
 * (implementations/acceleration/mod.rs:58-93). Host pointers; copied. n may be 0. */
int32_t ptb_scene_set_spheres(ptb_ctx* ctx, const ptb_sphere* spheres, size_t n);
int32_t ptb_scene_set_triangles(ptb_ctx* ctx, const ptb_triangle* triangles, size_t n);
int32_t ptb_scene_set_materials(ptb_ctx* ctx, const ptb_material* materials, size_t n);
int32_t ptb_scene_set_textures(ptb_ctx* ctx, const ptb_texture* textures, size_t n);
/* Bulk data of one texture (copied). PTB_TEX_IMAGE: ImageTexture.data (textures/mod.rs:202-245) = width*height RGB f32,
 * row-major, n_floats = 3*width*height. PTB_TEX_PERLIN: Perlin's tables (textures/mod.rs:75-112), width = height = 0,
 * n_floats = PTB_PERLIN_TABLE_WORDS. Call after ptb_scene_set_textures; commit fails with PTB_ERR_MISSING without it. */
int32_t ptb_scene_set_texture_data(ptb_ctx* ctx, uint32_t texture, uint32_t width, uint32_t height, const float* data,
                                   size_t n_floats);
int32_t ptb_scene_set_camera(ptb_ctx* ctx, const ptb_camera* camera);
int32_t ptb_scene_set_sky(ptb_ctx* ctx, const ptb_sky* sky);

/* Replaces Bvh::new (acceleration/mod.rs:58-93): builds the acceleration structure on the device — always the LBVH
 * (Morton sort, Karras hierarchy, refit), and on top of it, when the wide tree is selected, its SAH-driven collapse into
 * a compressed 8-wide BVH (quantised 96-byte nodes, leaf groups of up to 3 primitives) which the traversal kernels then
 * walk instead. PTB_BUILD_SAH makes the binary tree with the device's top-down SAH builder instead of the Karras
 * hierarchy (8 bins on each axis of a node's box, exact sweep for subtrees of <= 32 primitives, one primitive per leaf;
 * the replacement for the QUALITY of build_bvh + Split::Sah, acceleration/mod.rs:97-160, split.rs:78-187; CPU definition
 * oracle/sah_ref.hpp; 2..2^24 primitives, otherwise the LBVH is built). Same hits, fewer nodes per ray, a slower commit.
 * PTB_BUILD_DEFAULT follows the environment (PTB_BVH=binary|lbvh|sah|wide) and otherwise the library's default. */
enum { PTB_BUILD_DEFAULT = 0, PTB_BUILD_BINARY = 1, PTB_BUILD_WIDE = 2, PTB_BUILD_SAH = 4, PTB_BUILD_REFIT = 8 };
int32_t ptb_scene_commit(ptb_ctx* ctx, uint32_t build_flags);

/* Dynamic scenes. PTB_BUILD_REFIT commits whatever was set since the last commit but KEEPS the binary tree of the last full
 * commit: its topology (child / parent links) and its primitive slot order stay, and its boxes are refitted bottom-up to
 * the primitives as they are now. Materials, textures, camera, sky table, material-index validation and the light list are
 * redone as in a full commit; Morton codes, sort, hierarchy and SAH build are skipped. Hits do not depend on the tree, so a
 * refitted scene answers every query exactly as a fresh commit of the same primitives does; only the traversal cost
 * changes as the primitives move away from the layout the tree was built for (see ptb_bvh_sah_cost).
 *   - Requirements: the last full commit of this context succeeded (a full commit that fails drops the kept tree), the
 *     numbers of spheres and triangles are those of that commit, and the flag is passed alone. Otherwise the commit fails
 *     with PTB_ERR_INVALID and a message naming the reason; a full commit always works afterwards.
 *   - A scene committed with the compressed 8-wide tree answers PTB_ERR_UNSUPPORTED.
 *   - ptb_bvh_builder keeps reporting the builder that made the topology; ptb_stats.build_ms is the refit's device time;
 *     ptb_bvh_export's morton_sorted keeps the codes of the last full build.
 * Typical animation loop: ptb_scene_update_* -> ptb_scene_commit(PTB_BUILD_REFIT) -> ptb_accum_clear -> ptb_render, with a
 * full commit whenever ptb_bvh_sah_cost has grown too far above the value of a fresh build. */
/* Overwrite primitives [first, first + n) of the current arrays, in original (loader) order, in place; the counts do not
 * change. Like ptb_scene_set_*, they leave the scene uncommitted. first + n beyond the current count (overflow-safe) and a
 * null pointer with n > 0 give PTB_ERR_INVALID; n == 0 is a no-op. The host variants copy before returning. */
int32_t ptb_scene_update_spheres(ptb_ctx* ctx, size_t first, const ptb_sphere* spheres, size_t n);
int32_t ptb_scene_update_triangles(ptb_ctx* ctx, size_t first, const ptb_triangle* triangles, size_t n);
/* Same from device memory: a device-to-device copy enqueued on the context's stream, returning without synchronising. The
 * caller's buffer must be ready when the stream reaches the copy (produce it on the same stream, see ptb_set_stream, or
 * synchronise first) and must stay valid until the next commit or ptb_synchronize. */
int32_t ptb_scene_update_spheres_device(ptb_ctx* ctx, size_t first, const void* d_spheres, size_t n);
int32_t ptb_scene_update_triangles_device(ptb_ctx* ctx, size_t first, const void* d_triangles, size_t n);

/* Indexed triangle meshes. implementations/primitives/triangle.rs:30-36 MeshTriangle: indices into the scene's vertex and
 * normal arrays (the reference's MeshData) plus a material. 28 bytes. */
typedef struct ptb_mesh_triangle {
  uint32_t p[3];     /* vertex indices */
  uint32_t n[3];     /* normal indices */
  uint32_t material;
} ptb_mesh_triangle;
/* The scene's triangles come from one source at a time: the flat array of ptb_scene_set_triangles or an indexed mesh.
 * ptb_scene_set_mesh replaces the triangle array with the mesh (host pointers, copied before returning): triangle id i is
 * mesh triangle i, and primitive ids are still spheres first, then triangles. At commit (full or PTB_BUILD_REFIT) the
 * device expands the mesh into the same ptb_triangle records the flat path uploads, when the mesh changed since the last
 * successful commit; the expansion counts in ptb_stats.build_ms and kernel_launches. A mesh scene therefore builds, traverses
 * and renders bit for bit as the flat scene it expands to. ptb_scene_set_triangles puts the scene back in flat mode and
 * drops the mesh.
 *   - Indices are checked on the device at commit: a vertex index >= n_vertices or a normal index >= n_normals fails the
 *     commit with PTB_ERR_INVALID and a message naming the first such triangle (the expansion never reads out of range).
 *     Fix it with ptb_scene_update_mesh_triangles and commit again.
 *   - More than 2^32 - 1 vertices or normals: PTB_ERR_INVALID.
 *   - PTB_BUILD_REFIT keeps the tree while the sphere and triangle counts are those of the last full commit; the vertex and
 *     normal counts may differ. */
int32_t ptb_scene_set_mesh(ptb_ctx* ctx, const ptb_vec3* vertices, size_t n_vertices, const ptb_vec3* normals, size_t n_normals,
                           const ptb_mesh_triangle* triangles, size_t n_triangles);
/* Overwrite entries [first, first + n) of the mesh's vertex, normal or triangle array in place, with the range and pointer
 * rules of ptb_scene_update_* (host variants copy before returning; _device variants copy device to device on the
 * context's stream without synchronising). They need a mesh scene: on a flat scene they fail with PTB_ERR_INVALID, and so
 * does ptb_scene_update_triangles(_device) on a mesh scene (the next expansion would overwrite it). The usual animation
 * loop moves vertices only: ptb_scene_update_mesh_vertices -> ptb_scene_commit(PTB_BUILD_REFIT). */
int32_t ptb_scene_update_mesh_vertices(ptb_ctx* ctx, size_t first, const ptb_vec3* vertices, size_t n);
int32_t ptb_scene_update_mesh_normals(ptb_ctx* ctx, size_t first, const ptb_vec3* normals, size_t n);
int32_t ptb_scene_update_mesh_triangles(ptb_ctx* ctx, size_t first, const ptb_mesh_triangle* triangles, size_t n);
int32_t ptb_scene_update_mesh_vertices_device(ptb_ctx* ctx, size_t first, const void* d_vertices, size_t n);
int32_t ptb_scene_update_mesh_normals_device(ptb_ctx* ctx, size_t first, const void* d_normals, size_t n);
int32_t ptb_scene_update_mesh_triangles_device(ptb_ctx* ctx, size_t first, const void* d_triangles, size_t n);

/* Mesh instances: placed copies of ranges of the indexed mesh, each under its own transform. One placed copy of mesh
 * triangles [first_triangle, first_triangle + n_triangles). 12 bytes. */
typedef struct ptb_mesh_instance {
  uint32_t first_triangle;
  uint32_t n_triangles;
  uint32_t material;   /* PTB_MISS: every triangle keeps its own material; otherwise all of the instance's triangles get this one */
} ptb_mesh_instance;
/* Object-to-world transform, row-major f32. 84 bytes.
 * position: x' = ((m[0]*x + m[1]*y) + m[2]*z) + m[3], likewise rows 1 and 2 (m[4..7], m[8..11]);
 * normal:   n'.x = (n[0]*nx + n[1]*ny) + n[2]*nz, likewise rows 1 and 2; no translation, no normalisation.
 * Each product and sum is one IEEE f32 operation, with no fused multiply-add (the library is built with -fmad=false). */
typedef struct ptb_instance_xform {
  float m[12];
  float n[9];
} ptb_instance_xform;
/* ptb_scene_set_mesh_instances (host pointers, copied before returning) replaces the triangles of a mesh scene with the
 * concatenation, in instance order, of each instance's range of mesh triangles under that instance's transform: triangle id
 * = the sum of the earlier instances' n_triangles + the position inside the range, and primitive ids are still spheres
 * first, then triangles. Ranges may overlap, repeat or be empty; zero instances means zero triangles. At commit (full or
 * PTB_BUILD_REFIT) the device expands every instance into the ptb_triangle records the flat path uploads, whenever the
 * mesh, the instance list or a transform changed since the last successful commit; the expansion counts in
 * ptb_stats.build_ms and kernel_launches. Nothing after the expansion knows about instances: the device memory of the
 * scene grows with the placed triangles, not with the mesh.
 *   - ptb_scene_set_mesh drops the instance list (the scene's triangles are the mesh's own again); ptb_scene_set_triangles
 *     drops the mesh and the instance list. On a flat scene ptb_scene_set_mesh_instances fails with PTB_ERR_INVALID.
 *   - A range beyond the mesh's triangle count, a total of more than 2^32 - 1 triangles and a null pointer with n > 0 fail
 *     with PTB_ERR_INVALID and a message naming the instance, before anything is allocated.
 *   - ptb_scene_update_mesh_{vertices,normals,triangles}(_device) keep working: their ranges are over the mesh's arrays, and
 *     every instance that places a changed triangle moves with it. Index validation names the mesh triangle, and covers only
 *     the triangles some instance places. ptb_scene_update_triangles(_device) fails, as on every mesh scene.
 *   - A material override goes into each placed triangle's material word and is validated and collected as a light like
 *     any other.
 *   - PTB_BUILD_REFIT keeps the tree while the sphere and total triangle counts are those of the last full commit. */
int32_t ptb_scene_set_mesh_instances(ptb_ctx* ctx, const ptb_mesh_instance* instances, const ptb_instance_xform* xforms, size_t n);
/* Overwrite transforms [first, first + n) of the instance list in place, with the range and pointer rules of
 * ptb_scene_update_* (the host variant copies before returning; the _device variant copies device to device on the
 * context's stream without synchronising). Without an instance list they fail with PTB_ERR_INVALID. Ranges and materials
 * change only through ptb_scene_set_mesh_instances. The rigid animation loop: ptb_scene_update_instance_xforms ->
 * ptb_scene_commit(PTB_BUILD_REFIT), 84 bytes per moving instance. */
int32_t ptb_scene_update_instance_xforms(ptb_ctx* ctx, size_t first, const ptb_instance_xform* xforms, size_t n);
int32_t ptb_scene_update_instance_xforms_device(ptb_ctx* ctx, size_t first, const void* d_xforms, size_t n);
/* SAH cost of the committed binary tree in the reference's cost model (traversal 0.125, intersection 1, split.rs:161-176):
 * (0.125 * sum over inner nodes of SA(node) + sum over leaves of SA(leaf box)) / SA(root), SA = 2 (xy + yz + zx) of the f32
 * box evaluated in f64, root box = union of node 0's two child boxes. 1 primitive: 1.125; 0 primitives or a root of zero
 * area: 0. A device reduction in a fixed order: the same tree gives the same bits on every call. The wide tree answers
 * PTB_ERR_UNSUPPORTED. The signal for refit-or-rebuild: compare with the cost right after the last full commit. */
int32_t ptb_bvh_sah_cost(ptb_ctx* ctx, double* cost);

/* Bit-exact test hooks: n_prims Morton codes and primitive ids in sorted order, n_prims-1 nodes
 * (1 node when n_prims == 1). Any pointer may be NULL. After an SAH build prim_sorted is the SAH tree's own primitive
 * order (what its leaf references index) while morton_sorted still holds the sorted codes of the order it started from.
 * After a PTB_BUILD_REFIT commit morton_sorted and prim_sorted are those of the last full build. */
int32_t ptb_bvh_info(ptb_ctx* ctx, uint64_t* n_prims, uint64_t* n_nodes);
int32_t ptb_bvh_export(ptb_ctx* ctx, uint32_t* morton_sorted, uint32_t* prim_sorted, ptb_bvh_node* nodes);
/* The same binary tree as the traversal kernels read it (bit-exact test hook): 32 bytes per node, both children's boxes
 * snapped outwards onto a 65536^3 grid over the scene box — eight 32-bit words {left box x, y, z, right box x, y, z (each:
 * low half = min, high half = max grid coordinate), left, right}; frame = grid origin xyz, grid step xyz
 * (plane = origin + q * step). nodes32 receives nothing when the committed scene uses the wide tree. CPU definition:
 * oracle/lbvh_ref.hpp. Any pointer may be NULL. The 32-byte nodes are a compile-time option of the library
 * (-DPTB_QNODES=1, DESIGN.md §5): the default build answers PTB_ERR_UNSUPPORTED. */
int32_t ptb_bvh_export_quantised(ptb_ctx* ctx, float frame[6], void* nodes32);

/* The compressed 8-wide tree, for bit-exact tests: *n_nodes = 0 when the committed scene uses the binary tree. Nodes are
 * 96 bytes each (layout: raytracing-rust_b200/csrc/ptb_common.cuh CwNode == oracle/cwbvh_ref.hpp CwNode), slot_prim maps
 * the tree's primitive order to original primitive ids (n_prims entries). Any pointer may be NULL. */
int32_t ptb_bvh_wide_info(ptb_ctx* ctx, uint64_t* n_nodes, uint32_t* max_leaf);
/* Which builder made the committed tree: *builder = PTB_BUILD_BINARY (Karras LBVH), PTB_BUILD_SAH or PTB_BUILD_WIDE;
 * *sah_levels = levels of large tasks the SAH build took (0 otherwise). Either pointer may be NULL. */
int32_t ptb_bvh_builder(ptb_ctx* ctx, uint32_t* builder, uint32_t* sah_levels);
int32_t ptb_bvh_wide_export(ptb_ctx* ctx, void* nodes96, uint32_t* slot_prim);

/* ---------------------------------------------------------- closest hit -- */
/* Replaces AccelerationStructure::check_hit (acceleration/mod.rs:265-298) for a batch of rays.
 * Host buffers; H2D + kernel + D2H. hits[i] answers rays[i]; internally batches of >= 65 536 rays are traced in a
 * spatially sorted order (PTB_HIT_SORT=0 disables), which needs 16 B of device scratch per ray. */
int32_t ptb_closest_hit(ptb_ctx* ctx, const ptb_ray* rays, size_t n, ptb_hit* hits);
/* Same, buffers already resident in device memory (kernel only; used for roofline timing). */
int32_t ptb_closest_hit_device(ptb_ctx* ctx, const void* d_rays, size_t n, void* d_hits);

/* ----------------------------------------------------------- visibility -- */
/* 32 B, two float4 like ptb_ray: origin | tmax, un-normalised direction | excluded primitive (original id, PTB_MISS: none) */
typedef struct ptb_occlusion_ray {
  float ox, oy, oz, tmax;
  float dx, dy, dz;
  uint32_t exclude;
} ptb_occlusion_ray;

/* Batch visibility queries. Rays are handled as in ptb_closest_hit. The direction is normalised as Ray::new does it
 * (make_ray_from_raw), and t is measured along the normalised direction. The primitive's own intersector decides each
 * hit, with the same arithmetic as closest hit.
 *
 * check_hit_index, per acceleration/mod.rs:226-263. The target index[i] is an original primitive id. It is visible when
 * the target's own intersector gives t_target > 0 and no other primitive has 0 < t < t_target. The test is strict: a
 * blocker at exactly t_target does not block. If visible, hits[i] = {t_target, index[i], b1, b2}, the same record
 * ptb_closest_hit reports when that primitive is the closest. Otherwise hits[i] = {0, PTB_MISS, 0, 0}. A target
 * >= n_prims is not visible. It is not an error, because the device variant cannot check without a synchronise. Both
 * variants answer the same way.
 *
 * occluded: occluded[i] = 1 iff some primitive p != exclude has 0 < t_p < tmax, else 0. tmax = +inf asks "does the ray
 * hit anything". tmax <= 0 or NaN gives 0. An exclude of PTB_MISS or out of range excludes nothing.
 *
 * Errors. A call before commit returns PTB_ERR_INVALID. So does a null buffer with n > 0, and more than 0xFFFFFFF0 rays
 * in one device call (the same as ptb_closest_hit_device). n == 0 returns PTB_OK. In an empty scene nothing is occluded
 * and nothing is visible.
 *
 * The host variants stream their buffers like ptb_closest_hit (PTB_HIT_BATCH, PTB_HIT_SORT). The _device variants
 * enqueue on the context's stream and return without synchronising, like ptb_closest_hit_device. Both count in
 * ptb_stats.kernel_launches / trace_launches only, not in the closest-hit traversal counters. */
int32_t ptb_check_hit_index(ptb_ctx* ctx, const ptb_ray* rays, const uint32_t* index, size_t n, ptb_hit* hits);
int32_t ptb_check_hit_index_device(ptb_ctx* ctx, const void* d_rays, const void* d_index, size_t n, void* d_hits);
int32_t ptb_occluded(ptb_ctx* ctx, const ptb_occlusion_ray* rays, size_t n, uint8_t* occluded);
int32_t ptb_occluded_device(ptb_ctx* ctx, const void* d_rays, size_t n, void* d_occluded);

/* --------------------------------------------------------------- render -- */
/* Replaces Sampler::sample_image (samplers/mod.rs:7-20, random_sampler.rs:10-99) + the running mean of
 * src/main.rs:175-191: adds opts->samples_per_pixel samples per pixel into the device accumulator (sums).
 * Device memory: the path state of a call takes at most 8 GiB (PTB_POOL_BYTES=<bytes> changes the budget; 69 B per path,
 * 133 B with MIS), never more than half of the memory that was free at the context's first large render. A call that fits
 * (124 Mi paths, 64 Mi with MIS) runs as one chunk; a larger one runs chunk by chunk in two slots of half the budget each,
 * the wide iterations of chunk k+1 overlapping the latency-bound tail of chunk k. PTB_POOL_PATHS=<paths> sets the slot size directly,
 * PTB_TAIL_PATHS=<paths> the live-path count (default 65 536) below which a chunk is handed to the fused tail kernel (0: never).
 * The image is a pure function of (scene, opts): pool size, chunking and GPU count only change the f32 summation order
 * (finished paths are added with float atomics, so two runs of the same call agree to ~1e-6 relative, not bit for bit).
 * A non-zero return of `progress` stops the call with PTB_ERR_ABORTED and CLEARS the accumulator (samples of earlier
 * calls included): a partially rendered call has no sample count to normalise by. */
int32_t ptb_render(ptb_ctx* ctx, const ptb_render_opts* opts, ptb_progress_fn progress, void* user);
/* The reference's per-pass presentation contract (random_sampler.rs:31-98, SamplerProgress samplers/mod.rs:49-63): one
 * pass = one sample of every pixel. `update` receives the SINGLE-SAMPLE image of a finished pass (row-major, top row
 * first, RGB f32, n_floats = width*height*3; valid only during the call), the 1-based number of that pass and the
 * pass's rays_shot (the reference's own ray counter). As in the reference the image of pass k is handed over after pass
 * k+1 has been rendered, and the last one after the loop; a non-zero return stops the render (PTB_ERR_ABORTED; the
 * reference returns without the final call). Every pass is also added to the device accumulator, so ptb_accum_read
 * afterwards yields the running mean the TUI closure of src/main.rs:175-191 computes. Pass k uses absolute sample index
 * opts->sample_offset + k: the sum of the passes equals one ptb_render call of the same options. */
typedef int32_t (*ptb_pass_fn)(void* user, const float* pass_image, size_t n_floats, uint64_t pass_number, uint64_t rays_shot);
int32_t ptb_render_passes(ptb_ctx* ctx, const ptb_render_opts* opts, ptb_pass_fn update, void* user);
int32_t ptb_accum_clear(ptb_ctx* ctx);
/* Reads back width*height*3 floats, row-major, top row first, RGB (the layout of
 * SamplerProgress.current_image, samplers/mod.rs:49-63). normalise != 0 divides by the samples accumulated. */
int32_t ptb_accum_read(ptb_ctx* ctx, float* rgb, size_t n_floats, int32_t normalise);
/* Device pointer of the width*height*3 float sums (for the NCCL reduce) and its element count. */
int32_t ptb_accum_device_ptr(ptb_ctx* ctx, void** d_ptr, size_t* n_floats);
/* After an external reduce wrote sums of `total_samples` samples into the accumulator. */
int32_t ptb_accum_set_samples(ptb_ctx* ctx, uint64_t total_samples);

/* ------------------------------------------------ denoiser feature buffers -- */
/* The inputs a denoiser (Open Image Denoise, the OptiX denoiser, an SVGF-style filter) reads beside the beauty image,
 * aligned with it sample for sample: ptb_render_aov traces the camera ray of every (pixel, sample) that ptb_render with
 * the same opts traces (width, height, seed, sample_offset, samples_per_pixel, row_begin, row_count: the same jitter, the
 * same ray, bit for bit) and adds per sample, at the ray's closest hit h (wo = the unit camera direction):
 *   albedo   3 floats  LAMBERTIAN: param * texture(wo, h.point); REFLECT, REFRACT, TROWBRIDGE_REITZ: texture(wo, h.point);
 *                      EMIT: the emission the first bounce adds; a miss: the sky's emission. Each channel clamped to [0, 1]
 *                      (a NaN becomes 0).
 *   normal   3 floats  the hit record's normal, as every scatter uses it (not turned towards the camera); 0 on a miss
 *   depth    1 float   t along the unit direction (what ptb_closest_hit reports for that ray); 0 on a miss
 *   coverage 1 float   1 on a hit, 0 on a miss
 * into a separate AOV accumulator. method, max_depth, rr_threshold and flags are not read, so a host passes the opts of
 * its render unchanged; the other checks and messages are ptb_render's. The sums of a pixel are formed in sample order
 * without atomics: the buffers are deterministic, and sample ranges or row tiles of a call add up bit for bit to the one
 * call. The beauty accumulator and its sample count are not touched. Each sample is one traversal launch (counted in
 * ptb_stats.kernel_launches and trace_launches, no ray counters). Enqueues on the context's stream and may return before
 * the work is done; ptb_aov_read synchronises.
 * The first call allocates 8 floats per pixel; a call with another width or height reallocates and resets them. */
enum { PTB_AOV_ALBEDO = 0, PTB_AOV_NORMAL = 1, PTB_AOV_DEPTH = 2, PTB_AOV_COVERAGE = 3 };
int32_t ptb_render_aov(ptb_ctx* ctx, const ptb_render_opts* opts);
/* Zeroes the AOV sums and their sample count. */
int32_t ptb_aov_clear(ptb_ctx* ctx);
/* Reads one buffer (PTB_AOV_*): n_floats = width*height*3 for albedo and normal, width*height for depth and coverage;
 * row-major, top row first, as ptb_accum_read. normalise != 0 divides albedo, normal and coverage by the AOV sample count
 * and depth by the pixel's coverage sum (0 where nothing was hit); the mean normal is not renormalised. Synchronises the
 * stream. A read before any ptb_render_aov, an unknown aov or a wrong n_floats fails with PTB_ERR_INVALID. */
int32_t ptb_aov_read(ptb_ctx* ctx, uint32_t aov, float* out, size_t n_floats, int32_t normalise);

/* ------------------------------------------------------------- denoiser -- */
/* The spatial part of SVGF (Schied et al., "Spatiotemporal Variance-Guided Filtering", HPG 2017, §4.3-4.5): Dammertz et
 * al. 2010's edge-avoiding à-trous wavelet filter with albedo demodulation and variance-guided luminance weights, over the
 * beauty accumulator (sums of S_b = the accumulated sample count) and the AOV sums (S_a samples). All arithmetic is f32,
 * without contraction, in the order written; only exp2f, log2f (and sqrtf, IEEE) are the platform's.
 * Inputs per pixel p:
 *   c = beauty sum * (1/S_b)   (as ptb_accum_read normalises)      a = albedo sum / S_a      α = coverage sum / S_a
 *   n = normal sum / |normal sum|, |v| = sqrtf((v.x*v.x + v.y*v.y) + v.z*v.z); (0,0,0) where that length is 0
 *   z = depth sum / coverage sum, 0 where the coverage sum is 0 (as ptb_aov_read normalises)
 * Prepare:  d = max(a, 1e-3) per channel; irradiance e = c / d per channel; luminance ℓ(e) = (0.2126 e.r + 0.7152 e.g)
 *   + 0.0722 e.b. Depth gradient ∂x z: of the one-sided differences f = z[x+1] - z[x] and b = z[x] - z[x-1], counting only
 *   neighbours inside the image whose coverage sum is > 0: both -> |f| <= |b| ? f : b; one -> that one; none -> 0. ∂y z alike
 *   (y + 1 is the next row down). The sums are finite (the render zeroes non-finite samples); there is no guard.
 * Edge stopping, centre p, tap q at pixel offset Δ = (Δx, Δy):
 *   w_α = 1 - |α_p - α_q|
 *   w_n: both normals zero -> 1; exactly one zero -> 0 (the tap is dropped); otherwise max(0, n_p·n_q)^σ_n,
 *        n_p·n_q = (n_p.x*n_q.x + n_p.y*n_q.y) + n_p.z*n_q.z
 *   D_z = (σ_z * |∂x z_p * Δx + ∂y z_p * Δy| + 1e-3 * z_p) + 1e-6,  t_z = |z_p - z_q| / D_z,  w_z = exp(-t_z)
 *   D_l = σ_l * sqrtf(g_p) + 1e-10,  t_l = |ℓ_p - ℓ_q| / D_l,  w_l = exp(-t_l); g_p = Σ k var / Σ k over the 3x3
 *        neighbours inside the image (row by row), k = 1/4 at the centre, 1/8 beside it, 1/16 at the corners
 *   w_n * w_z (* w_l) is ONE exp2: exp2f(σ_n * log2f(max(0, n_p·n_q)) - (t_z (+ t_l)) * log2(e)) (σ_n * log2f(...) is 0 when
 *   both normals are zero), so the product is w_α * that.
 * Variance (SVGF's spatial estimate): over the 7x7 window inside the image, row by row, w = w_α * exp2f(σ_n log2f(n·n) -
 *   t_z log2(e)) (no w_l; the centre's w is exactly 1): μ1 = Σ w ℓ / Σ w, μ2 = Σ w ℓ² / Σ w, var = max(0, μ2 - μ1*μ1).
 * Level i = 0 .. L-1, step s = 2^i: taps q = p + s*(dx, dy), dx, dy in [-2, 2], inside the image, row by row;
 *   W_q = (h(dx)*h(dy)) * w_α * exp2f(σ_n log2f(n·n) - (t_z + t_l) log2(e)), Δ = s*(dx, dy), h = (3/8, 1/4, 1/16) by |d|;
 *   the centre's W is exactly h(0)² (the sum is never 0). e'_p = Σ W e / Σ W per channel; var'_p = Σ (W*W) var / (ΣW*ΣW).
 * Output: e^(L) * d, RGB, W*H*3 floats in ptb_accum_read's layout.
 * Defaults (0 selects them): L = 5, σ_l = 4, σ_n = 128, σ_z = 1 (SVGF's). Temporal accumulation is not part of this filter.
 *
 * Both accumulators are read and left bit-identical, sums and sample counts. The output is a pure function of them and
 * the options (no atomics: two calls give the same bits). Each launch (one prepare, one variance, one per level) counts in
 * ptb_stats.kernel_launches; none in trace_launches or the ray counters. The scratch (ping-pong irradiance + variance and
 * the guide records, 60 bytes per pixel) belongs to the context: allocated at first use, reallocated on a size change.
 * Errors, PTB_ERR_INVALID before anything is enqueued: null opts; nothing rendered or no AOV rendered yet; beauty and AOV
 * sizes differ; a sample count of 0 (e.g. after a clear); iterations > 10; a negative, NaN or infinite sigma; flags != 0;
 * a null output or n_floats != W*H*3. */
typedef struct ptb_denoise_opts {
  uint32_t iterations;      /* à-trous levels, step 2^i; 0 -> 5; at most 10 */
  float sigma_luminance;    /* 0 -> 4   */
  float sigma_normal;       /* 0 -> 128 */
  float sigma_depth;        /* 0 -> 1   */
  uint32_t flags;           /* reserved, 0 */
} ptb_denoise_opts;
/* Denoises into host memory (W*H*3 floats); synchronises the stream. */
int32_t ptb_denoise(ptb_ctx* ctx, const ptb_denoise_opts* opts, float* rgb, size_t n_floats);
/* Enqueues the same work on the context's stream into a device buffer of W*H*3 floats and returns without waiting. */
int32_t ptb_denoise_device(ptb_ctx* ctx, const ptb_denoise_opts* opts, void* d_rgb);

/* ------------------------------------------------------------ multi-GPU -- */
/* The path shards by samples (independent), scene and BVH replicated per GPU: rank r of `world` renders the absolute
 * samples [first, first + count) of every pixel. */
void    ptb_shard_samples(uint32_t samples_per_pixel, uint32_t sample_offset, int32_t rank, int32_t world,
                          uint32_t* first, uint32_t* count);
/* Second axis, for requests with fewer samples than GPUs: rank r renders every sample of the pixel rows
 * [first, first + count) of the `rows` rows starting at row_begin (bands of whole rows; sizes differ by at most 1). */
void    ptb_shard_rows(uint32_t rows, uint32_t row_begin, int32_t rank, int32_t world, uint32_t* first, uint32_t* count);
/* Scene::render across n GPUs of one box: ctxs[r] (one per GPU, scene already committed on each) renders its share on its
 * own host thread — a sample range of every pixel when samples_per_pixel >= n, else a band of pixel rows at every sample —
 * then ONE ncclReduce(sum) of the accumulators (width*height*3 f32) to ctxs[0] — the path's only collective; the
 * communicators are checked with ncclCommGetAsyncError after the reduce has completed. Afterwards ptb_accum_read(ctxs[0], ..) returns the image of all opts->samples_per_pixel samples. NCCL is
 * bound at run time (libnccl.so.2, or $PTB_NCCL_LIB); n == 1 never touches it. */
int32_t ptb_render_multi(ptb_ctx* const* ctxs, int32_t n, const ptb_render_opts* opts);

/* ----------------------------------------------------- sampler test hook -- */
/* The reference's best-pinned tests are chi-squared tests of its direction samplers against their pdfs
 * (implementations/statistics/spherical_sampling.rs:64-226, bxdfs/lambertian.rs:30-48, bxdfs/trowbridge_reitz_vndf.rs:156-218,
 * sky.rs:43-78). These two entry points run the DEVICE samplers — the same functions the shade kernel calls — outside a
 * render so the same harness can be pointed at them. Host buffers. */
enum {
  PTB_SAMPLER_LAMBERTIAN = 0,     /* lambertian::sample about `normal`                         (bxdfs/lambertian.rs:5-22)   */
  PTB_SAMPLER_TR_VNDF = 1,        /* trowbridge_reitz_vndf::sample(alpha, incoming = aux, normal) (..._vndf.rs:35-52, 84-113) */
  PTB_SAMPLER_SKY = 2,            /* Sky::sample / Sky::pdf of the committed scene             (sky.rs:43-78)               */
  PTB_SAMPLER_LIGHT = 3,          /* sample_visible_from_point / scattering_pdf of light `light_index` seen from the shading
                                     point aux with surface normal `normal`                   (sphere.rs:112-170, triangle.rs:249-280) */
  PTB_SAMPLER_UNIFORM_SPHERE = 4  /* the fixed-budget stand-in for random_unit_vector          (utility/mod.rs:15-25)       */
};
typedef struct ptb_sampler_query {
  uint32_t kind;         /* PTB_SAMPLER_*                                                                           */
  float    alpha;        /* TR_VNDF                                                                                  */
  ptb_vec3 normal;       /* LAMBERTIAN, TR_VNDF: surface normal; LIGHT: normal at the shading point                  */
  ptb_vec3 aux;          /* TR_VNDF: unit direction from the surface towards the viewer; LIGHT: the shading point     */
  uint32_t light_index;  /* LIGHT: index into the scene's light list (original primitive order)                       */
  uint64_t seed;         /* sample k draws from Philox counter (k, 0, test stream), key = seed                        */
} ptb_sampler_query;
/* n sampled directions (3 floats each) and, when pdf != NULL, the sampler's own pdf of each. */
int32_t ptb_sample_only(ptb_ctx* ctx, const ptb_sampler_query* query, size_t n, float* dirs, float* pdf);
/* pdf of n given unit directions under the same sampler. */
int32_t ptb_sampler_pdf(ptb_ctx* ctx, const ptb_sampler_query* query, const float* dirs, size_t n, float* pdf);

int32_t ptb_stats_get(ptb_ctx* ctx, ptb_stats* out);
int32_t ptb_stats_reset(ptb_ctx* ctx);

/* ------------------------------------------------------------- host side -- */
/* C++ restatement of the `loader` crate (loader/lib.rs:196-243, parser.rs:112-197, misc.rs, materials.rs,
 * primitives.rs, meshes.rs, obj.rs, textures.rs): parses a .ssml file (and the OBJ files it names) into the
 * POD arrays above. No GPU needed. */
typedef struct ptb_host_scene ptb_host_scene;
int32_t ptb_ssml_load_file(const char* path, ptb_host_scene** out);
int32_t ptb_ssml_load_str(const char* text, const char* base_dir, ptb_host_scene** out);
void    ptb_host_scene_free(ptb_host_scene* s);
const char* ptb_host_last_error(void);
size_t  ptb_host_scene_spheres(const ptb_host_scene* s, const ptb_sphere** out);
size_t  ptb_host_scene_triangles(const ptb_host_scene* s, const ptb_triangle** out);
size_t  ptb_host_scene_materials(const ptb_host_scene* s, const ptb_material** out);
size_t  ptb_host_scene_textures(const ptb_host_scene* s, const ptb_texture** out);
/* bulk data of texture `texture` (see ptb_scene_set_texture_data); returns n_floats, 0 if the texture has none */
size_t  ptb_host_scene_texture_data(const ptb_host_scene* s, uint32_t texture, uint32_t* width, uint32_t* height,
                                    const float** data);
int32_t ptb_host_scene_camera(const ptb_host_scene* s, ptb_camera* out);
int32_t ptb_host_scene_sky(const ptb_host_scene* s, ptb_sky* out);
/* SimpleCamera::new (camera.rs:20-53); aspect is 16/9 in the loader (loader/misc.rs:15). */
int32_t ptb_camera_make(ptb_vec3 origin, ptb_vec3 lookat, ptb_vec3 vup, float hfov_deg, float aspect,
                        float aperture, float focus_dist, ptb_camera* out);
/* Perlin::new (textures/mod.rs:90-112, 141-159): 256 gen_range(-1..1) scalars + three Fisher-Yates permutations
 * (`target = gen_range(0..i)` for i = 255..1). The reference seeds them from OS entropy (unpinned); here they are a pure
 * function of `seed` (Philox4x32-10). out = PTB_PERLIN_TABLE_WORDS words. */
int32_t ptb_perlin_tables(uint64_t seed, float* out);
/* ImageTexture::new's decode (textures/mod.rs:208-245, `image` crate to_rgb32f): ppm/pgm (P2,P3,P5,P6), pfm, bmp
 * (24/32 bit) and png (8/16 bit, non-interlaced). *rgb = width*height*3 f32, released with ptb_image_free. */
int32_t ptb_image_load(const char* filename, uint32_t* width, uint32_t* height, float** rgb);
void    ptb_image_free(float* rgb);
const char* ptb_image_last_error(void);
/* ptb_scene_set_* for every array of a loaded scene. */
int32_t ptb_scene_upload(ptb_ctx* ctx, const ptb_host_scene* s);

/* output::save_data_to_image (output/lib.rs:74-113): gamma + 8-bit for ppm/bmp/png, linear f32 for pfm. */
int32_t ptb_image_save(const char* filename, uint32_t width, uint32_t height, const float* rgb, float gamma);

#ifdef __cplusplus
}
#endif
#endif /* PTB200_H */
