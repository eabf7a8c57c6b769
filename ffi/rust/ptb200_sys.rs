//! `extern "C"` surface of libptb200.so — mirrors include/ptb200.h one to one (un-compiled here).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub const PTB_OK: i32 = 0;
pub const PTB_MISS: u32 = 0xFFFF_FFFF;
pub const PTB_RR_DEFAULT: u32 = 0xFFFF_FFFF;
pub const PTB_METHOD_NAIVE: u32 = 0;
pub const PTB_METHOD_MIS: u32 = 1;
/// Denoiser feature buffers (ptb_aov_read)
pub const PTB_AOV_ALBEDO: u32 = 0;
pub const PTB_AOV_NORMAL: u32 = 1;
pub const PTB_AOV_DEPTH: u32 = 2;
pub const PTB_AOV_COVERAGE: u32 = 3;

#[repr(C)] #[derive(Clone, Copy, Default)] pub struct ptb_vec3 { pub x: f32, pub y: f32, pub z: f32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_sphere { pub center: ptb_vec3, pub radius: f32, pub material: u32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_triangle { pub p: [ptb_vec3; 3], pub n: [ptb_vec3; 3], pub material: u32 }
/// MeshTriangle (implementations/primitives/triangle.rs:30-36): indices into the scene's vertex / normal arrays (28 B)
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_mesh_triangle { pub p: [u32; 3], pub n: [u32; 3], pub material: u32 }
/// One placed copy of mesh triangles [first_triangle, first_triangle + n_triangles); material PTB_MISS keeps theirs (12 B)
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_mesh_instance { pub first_triangle: u32, pub n_triangles: u32, pub material: u32 }
/// Object-to-world transform, row-major: m = 3x4 position map, n = 3x3 normal map (84 B)
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_instance_xform { pub m: [f32; 12], pub n: [f32; 9] }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_material { pub kind: u32, pub texture: u32, pub param: f32, pub ior: ptb_vec3, pub metallic: f32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_texture { pub kind: u32, pub a: ptb_vec3, pub b: ptb_vec3 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_camera { pub origin: ptb_vec3, pub lower_left: ptb_vec3, pub horizontal: ptb_vec3, pub vertical: ptb_vec3 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_sky { pub texture: u32, pub sampler_res_x: u32, pub sampler_res_y: u32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_ray { pub o: [f32; 3], pub _pad0: f32, pub d: [f32; 3], pub _pad1: f32 }
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_hit { pub t: f32, pub prim: u32, pub u: f32, pub v: f32 }
/// occlusion query (32 B): origin | tmax, un-normalised direction | excluded primitive (original id, PTB_MISS: none)
#[repr(C)] #[derive(Clone, Copy)] pub struct ptb_occlusion_ray { pub o: [f32; 3], pub tmax: f32, pub d: [f32; 3], pub exclude: u32 }
#[repr(C)] #[derive(Clone, Copy)]
pub struct ptb_render_opts {
    pub width: u32, pub height: u32, pub samples_per_pixel: u32, pub sample_offset: u32,
    pub method: u32, pub max_depth: u32, pub rr_threshold: u32, pub flags: u32, pub seed: u64,
    /// image tile (ABI 2): rows [row_begin, row_begin + row_count) only; row_count 0 = to the last row
    pub row_begin: u32, pub row_count: u32,
}
/// denoiser options (ptb_denoise); 0 selects a default: 5 levels, sigma_luminance 4, sigma_normal 128, sigma_depth 1
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct ptb_denoise_opts { pub iterations: u32, pub sigma_luminance: f32, pub sigma_normal: f32, pub sigma_depth: f32, pub flags: u32 }
/// temporal denoiser options (ptb_denoise_temporal); 0 selects a default: alpha_color 0.2, alpha_moments 0.2, max_history 32
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct ptb_temporal_opts { pub spatial: ptb_denoise_opts, pub alpha_color: f32, pub alpha_moments: f32, pub max_history: u32, pub flags: u32 }
#[repr(C)] #[derive(Clone, Copy, Default)]
pub struct ptb_stats {
    pub rays_camera: u64, pub rays_bounce: u64, pub rays_shadow_light: u64, pub rays_shadow_sky: u64,
    pub rays_reference: u64, pub paths: u64, pub wavefront_iterations: u64, pub kernel_launches: u64,
    pub nodes_fetched: u64, pub prims_tested: u64, pub rays_counted: u64, pub trace_launches: u64,
    pub build_ms: f64, pub render_ms: f64, pub ms_generate: f64, pub ms_trace: f64, pub ms_shade: f64, pub ms_shadow: f64, pub ms_tail: f64,
}
/// sampler test hook (chi-squared harness on the device samplers); kind = PTB_SAMPLER_* (0 lambertian, 1 TR VNDF, 2 sky, 3 light, 4 uniform sphere)
#[repr(C)] #[derive(Clone, Copy)]
pub struct ptb_sampler_query { pub kind: u32, pub alpha: f32, pub normal: ptb_vec3, pub aux: ptb_vec3, pub light_index: u32, pub seed: u64 }
#[repr(C)] pub struct ptb_ctx { _private: [u8; 0] }
pub type ptb_progress_fn = Option<unsafe extern "C" fn(user: *mut c_void, samples_completed: u64, rays_shot: u64) -> i32>;
/// per-pass presentation closure (random_sampler.rs:82-98): single-sample image of a finished pass, 1-based pass number
pub type ptb_pass_fn = Option<unsafe extern "C" fn(user: *mut c_void, pass_image: *const f32, n_floats: usize, pass_number: u64, rays_shot: u64) -> i32>;
pub const PTB_PERLIN_TABLE_WORDS: usize = 1024;
// ptb_scene_commit build flags: which builder / tree (PTB_BUILD_DEFAULT: the device SAH builder, or what PTB_BVH says)
pub const PTB_BUILD_DEFAULT: u32 = 0;
pub const PTB_BUILD_BINARY: u32 = 1; // Karras LBVH
pub const PTB_BUILD_WIDE: u32 = 2;   // LBVH collapsed into the compressed 8-wide tree
pub const PTB_BUILD_SAH: u32 = 4;    // top-down SAH builder (Bvh::new with Split::Sah, acceleration/mod.rs:58-160)
pub const PTB_BUILD_REFIT: u32 = 8;  // keep the last full commit's binary tree, refit its boxes (same primitive counts)

extern "C" {
    pub fn ptb_abi_version() -> u32;
    pub fn ptb_create(device: i32, out: *mut *mut ptb_ctx) -> i32;
    pub fn ptb_destroy(ctx: *mut ptb_ctx) -> i32;
    pub fn ptb_last_error(ctx: *const ptb_ctx) -> *const c_char;
    pub fn ptb_scene_set_spheres(ctx: *mut ptb_ctx, p: *const ptb_sphere, n: usize) -> i32;
    pub fn ptb_scene_set_triangles(ctx: *mut ptb_ctx, p: *const ptb_triangle, n: usize) -> i32;
    pub fn ptb_scene_set_materials(ctx: *mut ptb_ctx, p: *const ptb_material, n: usize) -> i32;
    pub fn ptb_scene_set_textures(ctx: *mut ptb_ctx, p: *const ptb_texture, n: usize) -> i32;
    pub fn ptb_scene_set_texture_data(ctx: *mut ptb_ctx, texture: u32, width: u32, height: u32, data: *const f32, n_floats: usize) -> i32;
    pub fn ptb_scene_set_camera(ctx: *mut ptb_ctx, cam: *const ptb_camera) -> i32;
    pub fn ptb_scene_set_sky(ctx: *mut ptb_ctx, sky: *const ptb_sky) -> i32;
    pub fn ptb_scene_update_spheres(ctx: *mut ptb_ctx, first: usize, p: *const ptb_sphere, n: usize) -> i32;
    pub fn ptb_scene_update_triangles(ctx: *mut ptb_ctx, first: usize, p: *const ptb_triangle, n: usize) -> i32;
    pub fn ptb_scene_update_spheres_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_update_triangles_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_set_mesh(ctx: *mut ptb_ctx, vertices: *const ptb_vec3, n_vertices: usize, normals: *const ptb_vec3, n_normals: usize,
                              triangles: *const ptb_mesh_triangle, n_triangles: usize) -> i32;
    pub fn ptb_scene_update_mesh_vertices(ctx: *mut ptb_ctx, first: usize, p: *const ptb_vec3, n: usize) -> i32;
    pub fn ptb_scene_update_mesh_normals(ctx: *mut ptb_ctx, first: usize, p: *const ptb_vec3, n: usize) -> i32;
    pub fn ptb_scene_update_mesh_triangles(ctx: *mut ptb_ctx, first: usize, p: *const ptb_mesh_triangle, n: usize) -> i32;
    pub fn ptb_scene_update_mesh_vertices_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_update_mesh_normals_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_update_mesh_triangles_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_set_mesh_instances(ctx: *mut ptb_ctx, instances: *const ptb_mesh_instance, xforms: *const ptb_instance_xform, n: usize) -> i32;
    pub fn ptb_scene_update_instance_xforms(ctx: *mut ptb_ctx, first: usize, p: *const ptb_instance_xform, n: usize) -> i32;
    pub fn ptb_scene_update_instance_xforms_device(ctx: *mut ptb_ctx, first: usize, d_p: *const c_void, n: usize) -> i32;
    pub fn ptb_scene_commit(ctx: *mut ptb_ctx, build_flags: u32) -> i32;
    pub fn ptb_bvh_sah_cost(ctx: *mut ptb_ctx, cost: *mut f64) -> i32;
    pub fn ptb_bvh_export_quantised(ctx: *mut ptb_ctx, frame: *mut f32, nodes32: *mut c_void) -> i32;
    pub fn ptb_bvh_wide_info(ctx: *mut ptb_ctx, n_nodes: *mut u64, max_leaf: *mut u32) -> i32;
    pub fn ptb_bvh_builder(ctx: *mut ptb_ctx, builder: *mut u32, sah_levels: *mut u32) -> i32;
    pub fn ptb_bvh_wide_export(ctx: *mut ptb_ctx, nodes96: *mut c_void, slot_prim: *mut u32) -> i32;
    pub fn ptb_closest_hit(ctx: *mut ptb_ctx, rays: *const ptb_ray, n: usize, hits: *mut ptb_hit) -> i32;
    pub fn ptb_closest_hit_device(ctx: *mut ptb_ctx, d_rays: *const c_void, n: usize, d_hits: *mut c_void) -> i32;
    pub fn ptb_check_hit_index(ctx: *mut ptb_ctx, rays: *const ptb_ray, index: *const u32, n: usize, hits: *mut ptb_hit) -> i32;
    pub fn ptb_check_hit_index_device(ctx: *mut ptb_ctx, d_rays: *const c_void, d_index: *const c_void, n: usize, d_hits: *mut c_void) -> i32;
    pub fn ptb_occluded(ctx: *mut ptb_ctx, rays: *const ptb_occlusion_ray, n: usize, occluded: *mut u8) -> i32;
    pub fn ptb_occluded_device(ctx: *mut ptb_ctx, d_rays: *const c_void, n: usize, d_occluded: *mut c_void) -> i32;
    pub fn ptb_render(ctx: *mut ptb_ctx, opts: *const ptb_render_opts, progress: ptb_progress_fn, user: *mut c_void) -> i32;
    pub fn ptb_render_passes(ctx: *mut ptb_ctx, opts: *const ptb_render_opts, update: ptb_pass_fn, user: *mut c_void) -> i32;
    pub fn ptb_render_multi(ctxs: *const *mut ptb_ctx, n: i32, opts: *const ptb_render_opts) -> i32;
    pub fn ptb_shard_samples(samples_per_pixel: u32, sample_offset: u32, rank: i32, world: i32, first: *mut u32, count: *mut u32);
    pub fn ptb_shard_rows(rows: u32, row_begin: u32, rank: i32, world: i32, first: *mut u32, count: *mut u32);
    pub fn ptb_accum_clear(ctx: *mut ptb_ctx) -> i32;
    pub fn ptb_accum_read(ctx: *mut ptb_ctx, rgb: *mut f32, n_floats: usize, normalise: i32) -> i32;
    pub fn ptb_accum_device_ptr(ctx: *mut ptb_ctx, d_ptr: *mut *mut c_void, n_floats: *mut usize) -> i32;
    pub fn ptb_render_aov(ctx: *mut ptb_ctx, opts: *const ptb_render_opts) -> i32;
    pub fn ptb_aov_clear(ctx: *mut ptb_ctx) -> i32;
    pub fn ptb_aov_read(ctx: *mut ptb_ctx, aov: u32, out: *mut f32, n_floats: usize, normalise: i32) -> i32;
    pub fn ptb_denoise(ctx: *mut ptb_ctx, opts: *const ptb_denoise_opts, rgb: *mut f32, n_floats: usize) -> i32;
    pub fn ptb_denoise_device(ctx: *mut ptb_ctx, opts: *const ptb_denoise_opts, d_rgb: *mut c_void) -> i32;
    pub fn ptb_motion_mark(ctx: *mut ptb_ctx) -> i32;
    pub fn ptb_motion_read(ctx: *mut ptb_ctx, out: *mut f32, n_floats: usize) -> i32;
    pub fn ptb_denoise_temporal(ctx: *mut ptb_ctx, opts: *const ptb_temporal_opts, rgb: *mut f32, n_floats: usize) -> i32;
    pub fn ptb_denoise_temporal_device(ctx: *mut ptb_ctx, opts: *const ptb_temporal_opts, d_rgb: *mut c_void) -> i32;
    pub fn ptb_denoise_temporal_reset(ctx: *mut ptb_ctx) -> i32;
    pub fn ptb_sample_only(ctx: *mut ptb_ctx, query: *const ptb_sampler_query, n: usize, dirs: *mut f32, pdf: *mut f32) -> i32;
    pub fn ptb_sampler_pdf(ctx: *mut ptb_ctx, query: *const ptb_sampler_query, dirs: *const f32, n: usize, pdf: *mut f32) -> i32;
    pub fn ptb_stats_get(ctx: *mut ptb_ctx, out: *mut ptb_stats) -> i32;
}
