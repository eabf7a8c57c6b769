//! `--backend cuda` for the frontend (un-compiled here). Lives next to src/scene.rs; `Scene::render` dispatches to it.
//! Flattens the concrete types named in src/parameters.rs:7-12 to the POD arrays of include/ptb200.h.
use crate::ptb200_sys::*;
use implementations::{rt_core::*, *};
use std::{collections::HashMap, ffi::CStr, ptr};

type Tex = AllTextures;
type Mat<'a> = AllMaterials<'a, Tex>;
type Prim<'a> = AllPrimitives<'a, Mat<'a>>;

fn v(p: Vec3) -> ptb_vec3 { ptb_vec3 { x: p.x, y: p.y, z: p.z } }

/// `mesh_base`: for a scene made by `new_indexed`, where each interned MeshData starts in the vertex / normal pools.
pub struct CudaScene { ctx: *mut ptb_ctx, mat_ids: HashMap<*const Mat, u32>, mesh_base: HashMap<*const MeshData, (usize, usize)> }

impl CudaScene {
    /// `primitives` in loader order (spheres first, then mesh triangles: loader/src/lib.rs:234-240).
    pub fn new(primitives: &[Prim], camera: &SimpleCamera, sky_tex: &Tex, sampler_res: (usize, usize), device: i32) -> Result<Self, String> {
        Self::create(primitives, camera, sky_tex, sampler_res, device, false)
    }

    /// As `new`, but the triangles go up as an indexed mesh (ptb_scene_set_mesh) and are expanded on the device: every
    /// MeshData is interned by address into one vertex pool and one normal pool (its indices offset by where it starts), a
    /// Prim::Triangle's corners are appended as fresh entries. About half the upload of `new` for grid-like meshes, and
    /// animation can move vertices with `update_mesh_vertices` instead of re-sending whole triangles.
    pub fn new_indexed(primitives: &[Prim], camera: &SimpleCamera, sky_tex: &Tex, sampler_res: (usize, usize), device: i32) -> Result<Self, String> {
        Self::create(primitives, camera, sky_tex, sampler_res, device, true)
    }

    fn create(primitives: &[Prim], camera: &SimpleCamera, sky_tex: &Tex, sampler_res: (usize, usize), device: i32, indexed: bool) -> Result<Self, String> {
        let mut ctx = ptr::null_mut();
        check(ptr::null_mut(), unsafe { ptb_create(device, &mut ctx) })?;
        // intern textures / materials by address: the arena (crates/region) keeps them alive and unique
        let (mut texs, mut mats) = (Vec::<ptb_texture>::new(), Vec::<ptb_material>::new());
        let (mut tex_ids, mut mat_ids) = (HashMap::<*const Tex, u32>::new(), HashMap::<*const Mat, u32>::new());
        let mut tex_data = Vec::<(u32, u32, u32, Vec<f32>)>::new(); // (texture, width, height, words) of image / perlin textures
        let mut tex_id = |t: &Tex| *tex_ids.entry(t as *const _).or_insert_with(|| {
            texs.push(flatten_texture(t));
            let id = texs.len() as u32 - 1;
            if let Some((w, h, words)) = texture_words(t) { tex_data.push((id, w, h, words)); }
            id
        });
        let sky_id = tex_id(sky_tex);
        let (mut spheres, mut tris) = (Vec::new(), Vec::new());
        // indexed: the vertex / normal pools and the mesh triangles that index them
        let (mut verts, mut nrms, mut mtris) = (Vec::<ptb_vec3>::new(), Vec::<ptb_vec3>::new(), Vec::<ptb_mesh_triangle>::new());
        let mut mesh_base = HashMap::<*const MeshData, (usize, usize)>::new();
        for p in primitives {
            let m = match p { Prim::Sphere(s) => s.material, Prim::Triangle(t) => t.material, Prim::MeshTriangle(t) => t.material };
            let mid = *mat_ids.entry(m as *const _).or_insert_with(|| { mats.push(flatten_material(m, &mut tex_id)); mats.len() as u32 - 1 });
            match p {
                Prim::Sphere(s) => spheres.push(ptb_sphere { center: v(s.center), radius: s.radius, material: mid }),
                Prim::Triangle(t) if indexed => {
                    let (bp, bn) = (verts.len() as u32, nrms.len() as u32);
                    verts.extend(t.points.map(v));
                    nrms.extend(t.normals.map(v));
                    mtris.push(ptb_mesh_triangle { p: [bp, bp + 1, bp + 2], n: [bn, bn + 1, bn + 2], material: mid });
                }
                Prim::MeshTriangle(t) if indexed => {
                    let (bp, bn) = *mesh_base.entry(t.mesh as *const _).or_insert_with(|| {
                        let b = (verts.len(), nrms.len());
                        verts.extend(t.mesh.vertices.iter().map(|&p| v(p)));
                        nrms.extend(t.mesh.normals.iter().map(|&p| v(p)));
                        b
                    });
                    mtris.push(ptb_mesh_triangle { p: t.point_indices.map(|i| (bp + i) as u32), n: t.normal_indices.map(|i| (bn + i) as u32), material: mid });
                }
                Prim::Triangle(t) => tris.push(ptb_triangle { p: t.points.map(v), n: t.normals.map(v), material: mid }),
                Prim::MeshTriangle(t) => tris.push(ptb_triangle {
                    p: t.point_indices.map(|i| v(t.mesh.vertices[i])), n: t.normal_indices.map(|i| v(t.mesh.normals[i])), material: mid }),
            }
        }
        if verts.len() > u32::MAX as usize || nrms.len() > u32::MAX as usize { return Err("new_indexed: more than 2^32 - 1 vertices or normals".into()); }
        let cam = ptb_camera { origin: v(camera.origin), lower_left: v(camera.lower_left), horizontal: v(camera.horizontal), vertical: v(camera.vertical) };
        let sky = ptb_sky { texture: sky_id, sampler_res_x: sampler_res.0 as u32, sampler_res_y: sampler_res.1 as u32 };
        unsafe {
            check(ctx, ptb_scene_set_textures(ctx, texs.as_ptr(), texs.len()))?;
            for (id, w, h, words) in &tex_data {
                check(ctx, ptb_scene_set_texture_data(ctx, *id, *w, *h, words.as_ptr(), words.len()))?;
            }
            check(ctx, ptb_scene_set_materials(ctx, mats.as_ptr(), mats.len()))?;
            check(ctx, ptb_scene_set_spheres(ctx, spheres.as_ptr(), spheres.len()))?;
            if indexed {
                check(ctx, ptb_scene_set_mesh(ctx, verts.as_ptr(), verts.len(), nrms.as_ptr(), nrms.len(), mtris.as_ptr(), mtris.len()))?;
            } else {
                check(ctx, ptb_scene_set_triangles(ctx, tris.as_ptr(), tris.len()))?;
            }
            check(ctx, ptb_scene_set_camera(ctx, &cam))?;
            check(ctx, ptb_scene_set_sky(ctx, &sky))?;
            check(ctx, ptb_scene_commit(ctx, 0))?; // Bvh::new
        }
        Ok(Self { ctx, mat_ids, mesh_base })
    }

    /// Scene::render (src/scene.rs:35-42) for the cuda backend: the accumulator comes back as the running-mean image the
    /// TUI closure of src/main.rs:175-191 would hold, ready for output::save_data_to_image.
    pub fn render(&self, opts: RenderOptions, seed: u64) -> Result<(Vec<Float>, u64), String> {
        let o = self.opts(opts, seed);
        let mut image = vec![0.0 as Float; (opts.width * opts.height * 3) as usize];
        let mut st = ptb_stats::default();
        unsafe {
            check(self.ctx, ptb_accum_clear(self.ctx))?;
            check(self.ctx, ptb_render(self.ctx, &o, None, ptr::null_mut()))?;
            check(self.ctx, ptb_accum_read(self.ctx, image.as_mut_ptr(), image.len(), 1))?;
            check(self.ctx, ptb_stats_get(self.ctx, &mut st))?;
        }
        Ok((image, st.rays_reference))
    }

    /// Denoiser feature buffers of the camera rays `render(opts, seed)` traces: (albedo, normal, depth, coverage), each
    /// normalised, row-major with the top row first; albedo and normal hold 3 floats per pixel, depth and coverage one
    /// (depth is the mean t over the samples that hit, 0 where none did). Feed them to the denoiser with the beauty image.
    pub fn render_aov(&self, opts: RenderOptions, seed: u64) -> Result<(Vec<f32>, Vec<f32>, Vec<f32>, Vec<f32>), String> {
        let o = self.opts(opts, seed);
        let n = (opts.width * opts.height) as usize;
        let (mut albedo, mut normal, mut depth, mut coverage) = (vec![0.0f32; 3 * n], vec![0.0f32; 3 * n], vec![0.0f32; n], vec![0.0f32; n]);
        unsafe {
            check(self.ctx, ptb_aov_clear(self.ctx))?;
            check(self.ctx, ptb_render_aov(self.ctx, &o))?;
            for (aov, buf) in [(PTB_AOV_ALBEDO, &mut albedo), (PTB_AOV_NORMAL, &mut normal), (PTB_AOV_DEPTH, &mut depth),
                               (PTB_AOV_COVERAGE, &mut coverage)] {
                check(self.ctx, ptb_aov_read(self.ctx, aov, buf.as_mut_ptr(), buf.len(), 1))?;
            }
        }
        Ok((albedo, normal, depth, coverage))
    }

    /// `render(opts, seed)` denoised on the device: the samples, the feature buffers of the same camera rays, then the
    /// spatial SVGF filter (`denoise`: ptb_denoise_opts, all zeros for the defaults). Same layout as `render`'s image.
    pub fn render_denoised(&self, opts: RenderOptions, seed: u64, denoise: ptb_denoise_opts) -> Result<Vec<Float>, String> {
        let o = self.opts(opts, seed);
        let mut image = vec![0.0 as Float; (opts.width * opts.height * 3) as usize];
        unsafe {
            check(self.ctx, ptb_accum_clear(self.ctx))?;
            check(self.ctx, ptb_render(self.ctx, &o, None, ptr::null_mut()))?;
            check(self.ctx, ptb_aov_clear(self.ctx))?;
            check(self.ctx, ptb_render_aov(self.ctx, &o))?;
            check(self.ctx, ptb_denoise(self.ctx, &denoise, image.as_mut_ptr(), image.len()))?;
        }
        Ok(image)
    }
}

impl CudaScene {
    /// Animation: overwrite triangles [first, first + tris.len()) of the scene (triangle order, i.e. loader order after the
    /// spheres) with new geometry. Their materials must be ones the scene was created with. Call `refit` afterwards.
    pub fn update_triangles(&self, first: usize, tris: &[Prim]) -> Result<(), String> {
        let mut out = Vec::with_capacity(tris.len());
        for p in tris {
            let (pts, nrm, m) = match p {
                Prim::Triangle(t) => (t.points.map(v), t.normals.map(v), t.material),
                Prim::MeshTriangle(t) => (t.point_indices.map(|i| v(t.mesh.vertices[i])), t.normal_indices.map(|i| v(t.mesh.normals[i])), t.material),
                Prim::Sphere(_) => return Err("update_triangles: a sphere in the triangle range".into()),
            };
            let material = *self.mat_ids.get(&(m as *const _)).ok_or("update_triangles: a material the scene does not have")?;
            out.push(ptb_triangle { p: pts, n: nrm, material });
        }
        check(self.ctx, unsafe { ptb_scene_update_triangles(self.ctx, first, out.as_ptr(), out.len()) })
    }

    /// Animation of a scene made by `new_indexed`: overwrite the vertices of `mesh` (one of the scene's MeshData) with
    /// `positions` (as many as the mesh has). Call `refit` afterwards; the device expands the moved mesh at the commit.
    pub fn update_mesh_vertices(&self, mesh: &MeshData, positions: &[Vec3]) -> Result<(), String> {
        let &(base, _) = self.mesh_base.get(&(mesh as *const _)).ok_or("update_mesh_vertices: not a mesh of this indexed scene")?;
        if positions.len() != mesh.vertices.len() { return Err("update_mesh_vertices: one position per vertex of the mesh".into()); }
        let out: Vec<ptb_vec3> = positions.iter().map(|&p| v(p)).collect();
        check(self.ctx, unsafe { ptb_scene_update_mesh_vertices(self.ctx, base, out.as_ptr(), out.len()) })
    }

    /// Place ranges of the indexed mesh (triangle order of `new_indexed`'s mesh) as instances, one transform each: the
    /// scene's triangles become the instances' transformed copies, in order. Call `rebuild` afterwards.
    pub fn set_mesh_instances(&self, instances: &[ptb_mesh_instance], xforms: &[ptb_instance_xform]) -> Result<(), String> {
        if instances.len() != xforms.len() { return Err("set_mesh_instances: one transform per instance".into()); }
        check(self.ctx, unsafe { ptb_scene_set_mesh_instances(self.ctx, instances.as_ptr(), xforms.as_ptr(), instances.len()) })
    }

    /// Rigid animation of an instanced scene: overwrite transforms [first, first + xforms.len()). Call `refit` afterwards;
    /// the device expands the instances again at the commit.
    pub fn update_instance_xforms(&self, first: usize, xforms: &[ptb_instance_xform]) -> Result<(), String> {
        check(self.ctx, unsafe { ptb_scene_update_instance_xforms(self.ctx, first, xforms.as_ptr(), xforms.len()) })
    }

    /// Commit the updates keeping the tree (PTB_BUILD_REFIT); returns the refitted tree's SAH cost, which the caller
    /// compares with the cost after the last full build to decide when to call `rebuild`.
    pub fn refit(&self) -> Result<f64, String> {
        check(self.ctx, unsafe { ptb_scene_commit(self.ctx, PTB_BUILD_REFIT) })?;
        self.sah_cost()
    }

    /// A full commit (Bvh::new's tree for the primitives as they are now); returns its SAH cost.
    pub fn rebuild(&self) -> Result<f64, String> {
        check(self.ctx, unsafe { ptb_scene_commit(self.ctx, PTB_BUILD_DEFAULT) })?;
        self.sah_cost()
    }

    fn sah_cost(&self) -> Result<f64, String> {
        let mut c = 0.0f64;
        check(self.ctx, unsafe { ptb_bvh_sah_cost(self.ctx, &mut c) })?;
        Ok(c)
    }

    /// AccelerationStructure::check_hit_index (acceleration/mod.rs:226-263) for a batch: is primitive `index[i]` (loader
    /// order) the first thing ray i hits? Some((t, b1, b2)) when it is, None when it is blocked, missed or out of range.
    pub fn check_hit_index(&self, rays: &[Ray], index: &[u32]) -> Result<Vec<Option<(Float, Float, Float)>>, String> {
        assert_eq!(rays.len(), index.len());
        let r: Vec<ptb_ray> = rays.iter().map(|r| ptb_ray { o: [r.origin.x, r.origin.y, r.origin.z], _pad0: 0.0,
                                                           d: [r.direction.x, r.direction.y, r.direction.z], _pad1: 0.0 }).collect();
        let mut hits = vec![ptb_hit { t: 0.0, prim: PTB_MISS, u: 0.0, v: 0.0 }; rays.len()];
        check(self.ctx, unsafe { ptb_check_hit_index(self.ctx, r.as_ptr(), index.as_ptr(), r.len(), hits.as_mut_ptr()) })?;
        Ok(hits.iter().map(|h| if h.prim == PTB_MISS { None } else { Some((h.t, h.u, h.v)) }).collect())
    }

    /// Shadow rays: true when a primitive other than `exclude` (loader order; PTB_MISS: none) lies at 0 < t < tmax along
    /// the normalised direction. tmax = Float::INFINITY asks whether the ray hits anything (the sky test, mis.rs:104-115).
    pub fn occluded(&self, rays: &[(Ray, Float, u32)]) -> Result<Vec<bool>, String> {
        let r: Vec<ptb_occlusion_ray> = rays.iter().map(|(r, tmax, exclude)| ptb_occlusion_ray {
            o: [r.origin.x, r.origin.y, r.origin.z], tmax: *tmax, d: [r.direction.x, r.direction.y, r.direction.z], exclude: *exclude,
        }).collect();
        let mut out = vec![0u8; r.len()];
        check(self.ctx, unsafe { ptb_occluded(self.ctx, r.as_ptr(), r.len(), out.as_mut_ptr()) })?;
        Ok(out.iter().map(|&o| o != 0).collect())
    }

    /// The reference's own contract: `presentation_update` sees the single-sample image of every pass
    /// (Sampler::sample_image, samplers/mod.rs:7-20). `f` returns true to stop, like the Rust closure.
    pub fn render_with_update<T, F: Fn(&mut T, &SamplerProgress, u64) -> bool>(&self, opts: RenderOptions, seed: u64, data: &mut T, f: F) -> Result<(), String> {
        struct Thunk<'a, T, F> { data: &'a mut T, f: F, progress: SamplerProgress }
        unsafe extern "C" fn call<T, F: Fn(&mut T, &SamplerProgress, u64) -> bool>(user: *mut std::ffi::c_void, img: *const f32, n: usize, i: u64, rays: u64) -> i32 {
            let t = &mut *(user as *mut Thunk<T, F>);
            t.progress.current_image.copy_from_slice(std::slice::from_raw_parts(img, n));
            t.progress.rays_shot = rays;
            (t.f)(t.data, &t.progress, i) as i32
        }
        let mut thunk = Thunk { data, f, progress: SamplerProgress::new(opts.width * opts.height, 3) };
        let o = self.opts(opts, seed);
        unsafe {
            check(self.ctx, ptb_accum_clear(self.ctx))?;
            match ptb_render_passes(self.ctx, &o, Some(call::<T, F>), &mut thunk as *mut _ as *mut _) {
                7 /* PTB_ERR_ABORTED: the closure asked to stop */ => Ok(()),
                rc => check(self.ctx, rc),
            }
        }
    }
    fn opts(&self, opts: RenderOptions, seed: u64) -> ptb_render_opts {
        ptb_render_opts {
            width: opts.width as u32, height: opts.height as u32, samples_per_pixel: opts.samples_per_pixel as u32, sample_offset: 0,
            method: match opts.render_method { RenderMethod::Naive => PTB_METHOD_NAIVE, RenderMethod::MIS => PTB_METHOD_MIS },
            max_depth: 50, rr_threshold: PTB_RR_DEFAULT, flags: 0, seed, row_begin: 0, row_count: 0,
        }
    }
}

impl Drop for CudaScene { fn drop(&mut self) { unsafe { ptb_destroy(self.ctx); } } }

fn check(ctx: *mut ptb_ctx, rc: i32) -> Result<(), String> {
    if rc == PTB_OK { return Ok(()); }
    Err(unsafe { CStr::from_ptr(ptb_last_error(ctx)) }.to_string_lossy().into_owned())
}

fn flatten_texture(t: &Tex) -> ptb_texture {
    match t { // tag == enum order (textures/mod.rs:17-24)
        AllTextures::CheckeredTexture(c) => ptb_texture { kind: 0, a: v(c.colour_one), b: v(c.colour_two) },
        AllTextures::SolidColour(s) => ptb_texture { kind: 1, a: v(s.colour), b: v(Vec3::zero()) },
        AllTextures::Lerp(l) => ptb_texture { kind: 3, a: v(l.colour_one), b: v(l.colour_two) },
        AllTextures::ImageTexture(_) => ptb_texture { kind: 2, a: v(Vec3::zero()), b: v(Vec3::zero()) }, // pixels: texture_words
        AllTextures::Perlin(_) => ptb_texture { kind: 4, a: v(Vec3::zero()), b: v(Vec3::zero()) },       // tables: texture_words
    }
}

/// Bulk data for ptb_scene_set_texture_data. ImageTexture: `data` as width*height RGB f32 (dim holds width-1, height-1:
/// textures/mod.rs:232). Perlin: 256 ran_vecs[i].x, then perm_x | perm_y | perm_z as u32 bit patterns (needs the four
/// private fields of `Perlin` made pub(crate), textures/mod.rs:76-81).
fn texture_words(t: &Tex) -> Option<(u32, u32, Vec<f32>)> {
    match t {
        AllTextures::ImageTexture(i) => Some((i.dim.0 as u32 + 1, i.dim.1 as u32 + 1, i.data.iter().flat_map(|c| [c.x, c.y, c.z]).collect())),
        AllTextures::Perlin(p) => {
            let mut w: Vec<f32> = p.ran_vecs.iter().map(|r| r.x).collect();
            for perm in [&p.perm_x, &p.perm_y, &p.perm_z] { w.extend(perm.iter().map(|&i| f32::from_bits(i))); }
            Some((0, 0, w))
        }
        _ => None,
    }
}

fn flatten_material(m: &Mat, tex_id: &mut impl FnMut(&Tex) -> u32) -> ptb_material {
    let one = v(Vec3::one());
    match m { // tag == enum order (materials/mod.rs:19-25)
        AllMaterials::Emit(e) => ptb_material { kind: 0, texture: tex_id(e.texture), param: e.strength, ior: one, metallic: 0.0 },
        AllMaterials::Lambertian(l) => ptb_material { kind: 1, texture: tex_id(l.texture), param: l.albedo, ior: one, metallic: 0.0 },
        AllMaterials::TrowbridgeReitz(t) => ptb_material { kind: 2, texture: tex_id(t.texture), param: t.alpha, ior: v(t.ior), metallic: t.metallic },
        AllMaterials::Reflect(r) => ptb_material { kind: 3, texture: tex_id(r.texture), param: r.fuzz, ior: one, metallic: 0.0 },
        AllMaterials::Refract(r) => ptb_material { kind: 4, texture: tex_id(r.texture), param: r.eta, ior: one, metallic: 0.0 },
    }
}
