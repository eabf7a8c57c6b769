"""The `--backend cuda` path as seen from Python: a thin, typed wrapper over the C ABI.

Names follow the reference's interface for this path:
  Bvh            <- implementations::acceleration::Bvh            (acceleration/mod.rs:43-93, check_hit :265-298,
                                                                   check_hit_index :226-263)
  RenderOptions  <- implementations::samplers::RenderOptions       (samplers/mod.rs:22-41)
  RandomSampler  <- implementations::samplers::random_sampler::RandomSampler.sample_image (random_sampler.rs:10-99)
  Scene.render   <- frontend Scene::render                         (src/scene.rs:35-42)
Every compute call goes through libptb200.so; nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L
from .scene import HostScene, IndexedMesh


def _check(ctx_handle, rc: int):
    if rc != L.PTB_OK:
        msg = L.lib.ptb_last_error(ctx_handle)
        raise L.PtbError(rc, msg.decode() if msg else "")


@dataclass
class RenderOptions:
    """samplers/mod.rs:22-41 (defaults identical) + integrator constants + what sharding needs."""
    samples_per_pixel: int = 128
    render_method: int = L.METHOD_MIS
    width: int = 1920
    height: int = 1080
    gamma: float = 2.2
    sample_offset: int = 0
    max_depth: int = 50          # integrators/mod.rs:7
    rr_threshold: int = 3        # integrators/mod.rs:8
    seed: int = 0
    row_begin: int = 0           # image tile (multi-GPU second axis): rows [row_begin, row_begin + row_count); 0 = to the end
    row_count: int = 0

    def to_c(self) -> L.RenderOpts:
        return L.RenderOpts(self.width, self.height, self.samples_per_pixel, self.sample_offset, self.render_method,
                            self.max_depth, self.rr_threshold, 0, self.seed, self.row_begin, self.row_count)


def denoise_opts(iterations: int = 0, sigma_luminance: float = 0.0, sigma_normal: float = 0.0, sigma_depth: float = 0.0,
                 flags: int = 0) -> L.DenoiseOpts:
    """ptb_denoise_opts; 0 selects a default (5 levels, sigma_luminance 4, sigma_normal 128, sigma_depth 1)."""
    return L.DenoiseOpts(iterations, sigma_luminance, sigma_normal, sigma_depth, flags)


class Context:
    """One ptb_ctx == one GPU."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = L.lib.ptb_create(device, C.byref(self._h))
        if rc != L.PTB_OK:
            msg = L.lib.ptb_last_error(None)
            raise L.PtbError(rc, msg.decode() if msg else "ptb_create failed")
        self.device = device
        self._progress_ref = None

    def close(self):
        if self._h:
            L.lib.ptb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- scene
    def set_stream(self, cuda_stream_ptr: int):
        _check(self._h, L.lib.ptb_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def set_option(self, option: int, value: int):
        _check(self._h, L.lib.ptb_set_option(self._h, option, value))

    def synchronize(self):
        _check(self._h, L.lib.ptb_synchronize(self._h))

    def upload(self, s: HostScene, mesh: IndexedMesh | None = None, instances=None):
        """ptb_scene_set_* for every array (host -> library copy). With `mesh`, the scene's triangles are that indexed mesh
        (set_mesh) and s.triangles is not uploaded; with `instances` = (instances, xforms) as well, they are those placed
        copies of the mesh (set_mesh_instances)."""
        h = self._h
        _check(h, L.lib.ptb_scene_set_textures(h, L.ptr(s.textures), len(s.textures)))
        for i, (w, hh, words) in s.texture_data.items():
            _check(h, L.lib.ptb_scene_set_texture_data(h, i, w, hh, L.ptr(words), words.size))
        _check(h, L.lib.ptb_scene_set_materials(h, L.ptr(s.materials), len(s.materials)))
        _check(h, L.lib.ptb_scene_set_spheres(h, L.ptr(s.spheres), len(s.spheres)))
        if mesh is None:
            _check(h, L.lib.ptb_scene_set_triangles(h, L.ptr(s.triangles), len(s.triangles)))
        else:
            self.set_mesh(mesh)
            if instances is not None:
                self.set_mesh_instances(*instances)
        _check(h, L.lib.ptb_scene_set_camera(h, L.ptr(s.camera)))
        _check(h, L.lib.ptb_scene_set_sky(h, L.ptr(s.sky)))

    def commit(self, flags: int = 0):
        """Bvh::new: device build of the acceleration structure. L.BUILD_BINARY: Karras LBVH; L.BUILD_SAH: top-down SAH
        builder (sah_build.cu); L.BUILD_WIDE: the LBVH collapsed into the compressed 8-wide tree; L.BUILD_DEFAULT follows
        PTB_BVH=binary|lbvh|sah|wide, else the library default. L.BUILD_REFIT (alone) keeps the binary tree of the last
        full commit and refits its boxes to the primitives as they are now (see update_triangles)."""
        _check(self._h, L.lib.ptb_scene_commit(self._h, flags))

    # ---- dynamic scenes: overwrite primitives in place, then commit(L.BUILD_REFIT)
    def update_spheres(self, first: int, spheres: np.ndarray):
        """Overwrite spheres [first, first + len(spheres)) (sphere_dtype, original order); the count does not change."""
        a = np.ascontiguousarray(spheres, dtype=L.sphere_dtype)
        _check(self._h, L.lib.ptb_scene_update_spheres(self._h, first, L.ptr(a), len(a)))

    def update_triangles(self, first: int, triangles: np.ndarray):
        """Overwrite triangles [first, first + len(triangles)) (triangle_dtype; triangle ids, not primitive ids)."""
        a = np.ascontiguousarray(triangles, dtype=L.triangle_dtype)
        _check(self._h, L.lib.ptb_scene_update_triangles(self._h, first, L.ptr(a), len(a)))

    def update_spheres_device(self, first: int, d_ptr: int, n: int):
        """Same from device memory (n records of sphere_dtype's layout), enqueued on the context's stream without a
        synchronise: the buffer must be ready when the stream gets there (produce it on that stream, see set_stream)."""
        _check(self._h, L.lib.ptb_scene_update_spheres_device(self._h, first, C.c_void_p(d_ptr), n))

    def update_triangles_device(self, first: int, d_ptr: int, n: int):
        """Same from device memory (n records of triangle_dtype's layout, 76 bytes each)."""
        _check(self._h, L.lib.ptb_scene_update_triangles_device(self._h, first, C.c_void_p(d_ptr), n))

    # ---- indexed meshes: the device expands them into the triangle records at commit
    def set_mesh(self, mesh: IndexedMesh):
        """The scene's triangles become `mesh` (triangle id i = mesh triangle i); set_triangles goes back to flat ones."""
        v, n, t = mesh.vertices, mesh.normals, mesh.triangles
        _check(self._h, L.lib.ptb_scene_set_mesh(self._h, L.ptr(v), len(v), L.ptr(n), len(n), L.ptr(t), len(t)))

    def update_mesh_vertices(self, first: int, vertices: np.ndarray):
        """Overwrite mesh vertices [first, first + len(vertices)) ((k, 3) float32); then commit, e.g. with L.BUILD_REFIT."""
        a = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3)
        _check(self._h, L.lib.ptb_scene_update_mesh_vertices(self._h, first, L.ptr(a), len(a)))

    def update_mesh_normals(self, first: int, normals: np.ndarray):
        a = np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
        _check(self._h, L.lib.ptb_scene_update_mesh_normals(self._h, first, L.ptr(a), len(a)))

    def update_mesh_triangles(self, first: int, triangles: np.ndarray):
        """Overwrite mesh triangles [first, first + len(triangles)) (mesh_triangle_dtype)."""
        a = np.ascontiguousarray(triangles, L.mesh_triangle_dtype)
        _check(self._h, L.lib.ptb_scene_update_mesh_triangles(self._h, first, L.ptr(a), len(a)))

    def update_mesh_vertices_device(self, first: int, d_ptr: int, n: int):
        """Same from device memory (n x 12 bytes), enqueued on the context's stream without a synchronise (as
        update_triangles_device)."""
        _check(self._h, L.lib.ptb_scene_update_mesh_vertices_device(self._h, first, C.c_void_p(d_ptr), n))

    def update_mesh_normals_device(self, first: int, d_ptr: int, n: int):
        _check(self._h, L.lib.ptb_scene_update_mesh_normals_device(self._h, first, C.c_void_p(d_ptr), n))

    def update_mesh_triangles_device(self, first: int, d_ptr: int, n: int):
        """n records of mesh_triangle_dtype's layout (28 bytes each)."""
        _check(self._h, L.lib.ptb_scene_update_mesh_triangles_device(self._h, first, C.c_void_p(d_ptr), n))

    # ---- mesh instances: placed, transformed copies of mesh triangle ranges, expanded on the device at commit
    def set_mesh_instances(self, instances: np.ndarray, xforms: np.ndarray):
        """The scene's triangles become the instances (mesh_instance_dtype) in order, each under its transform
        (instance_xform_dtype); set_mesh drops the list. Needs a mesh scene."""
        i = np.ascontiguousarray(instances, L.mesh_instance_dtype).reshape(-1)
        x = np.ascontiguousarray(xforms, L.instance_xform_dtype).reshape(-1)
        if len(i) != len(x):
            raise ValueError(f"{len(i)} instances but {len(x)} transforms")
        _check(self._h, L.lib.ptb_scene_set_mesh_instances(self._h, L.ptr(i), L.ptr(x), len(i)))

    def update_instance_xforms(self, first: int, xforms: np.ndarray):
        """Overwrite transforms [first, first + len(xforms)) (instance_xform_dtype); then commit, e.g. with L.BUILD_REFIT."""
        x = np.ascontiguousarray(xforms, L.instance_xform_dtype).reshape(-1)
        _check(self._h, L.lib.ptb_scene_update_instance_xforms(self._h, first, L.ptr(x), len(x)))

    def update_instance_xforms_device(self, first: int, d_ptr: int, n: int):
        """Same from device memory (n records of 84 bytes: 21 float32 each), enqueued on the context's stream without a
        synchronise (as update_triangles_device)."""
        _check(self._h, L.lib.ptb_scene_update_instance_xforms_device(self._h, first, C.c_void_p(d_ptr), n))

    def bvh_sah_cost(self) -> float:
        """SAH cost of the committed binary tree (traversal 0.125, intersection 1; normalised by the root's area). Compare
        it with the value right after a full commit to decide when a refitted tree should be rebuilt."""
        v = C.c_double()
        _check(self._h, L.lib.ptb_bvh_sah_cost(self._h, C.byref(v)))
        return v.value

    def bvh_info(self):
        a, b = C.c_uint64(), C.c_uint64()
        _check(self._h, L.lib.ptb_bvh_info(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def bvh_export(self):
        n, m = self.bvh_info()
        morton = np.zeros(n, np.uint32)
        prims = np.zeros(n, np.uint32)
        nodes = np.zeros(m, L.bvh_node_dtype)
        _check(self._h, L.lib.ptb_bvh_export(self._h, L.ptr(morton), L.ptr(prims), L.ptr(nodes)))
        return morton, prims, nodes

    def bvh_export_quantised(self):
        """(frame: grid origin xyz + grid step xyz, nodes (m, 8) uint32: the 32-byte nodes the traversal kernels read)."""
        _, m = self.bvh_info()
        frame = np.zeros(6, np.float32)
        nodes = np.zeros((m, 8), np.uint32)
        _check(self._h, L.lib.ptb_bvh_export_quantised(self._h, L.ptr(frame), L.ptr(nodes)))
        return frame, nodes

    def bvh_builder(self):
        """(L.BUILD_BINARY | L.BUILD_SAH | L.BUILD_WIDE: which builder made the committed tree, levels the SAH build took)."""
        a, b = C.c_uint32(), C.c_uint32()
        _check(self._h, L.lib.ptb_bvh_builder(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def bvh_wide_info(self):
        """(number of 96-byte nodes of the compressed 8-wide tree — 0 when the scene uses the binary tree, max leaf size)."""
        n, m = C.c_uint64(), C.c_uint32()
        _check(self._h, L.lib.ptb_bvh_wide_info(self._h, C.byref(n), C.byref(m)))
        return n.value, m.value

    def bvh_wide_export(self):
        """(nodes (n, 96) uint8, slot_prim: the wide tree's primitive order -> original primitive id)."""
        n, _ = self.bvh_wide_info()
        n_prims, _ = self.bvh_info()
        nodes = np.zeros((n, 96), np.uint8)
        slot_prim = np.zeros(n_prims, np.uint32)
        _check(self._h, L.lib.ptb_bvh_wide_export(self._h, L.ptr(nodes), L.ptr(slot_prim)))
        return nodes, slot_prim

    # ---- closest hit
    def closest_hit(self, rays: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        """AccelerationStructure::check_hit for a batch (host buffers in, host buffers out). `out`: optional caller-owned
        hit buffer (e.g. pinned memory: the library overlaps upload, traversal and read-back of 4 Mi-ray batches)."""
        rays = np.ascontiguousarray(rays, dtype=L.ray_dtype)
        hits = np.zeros(len(rays), L.hit_dtype) if out is None else out
        assert hits.dtype == L.hit_dtype and len(hits) == len(rays) and hits.flags.c_contiguous
        _check(self._h, L.lib.ptb_closest_hit(self._h, L.ptr(rays), len(rays), L.ptr(hits)))
        return hits

    def closest_hit_device(self, d_rays_ptr: int, n: int, d_hits_ptr: int):
        _check(self._h, L.lib.ptb_closest_hit_device(self._h, C.c_void_p(d_rays_ptr), n, C.c_void_p(d_hits_ptr)))

    # ---- visibility
    def check_hit_index(self, rays: np.ndarray, index: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        """AccelerationStructure::check_hit_index per ray: is original primitive index[i] the first thing rays[i] hits?
        Visible: the hit record closest_hit reports for that primitive; otherwise {0, PTB_MISS, 0, 0} (an out-of-range
        target included). `out`: optional caller-owned hit buffer."""
        rays = np.ascontiguousarray(rays, dtype=L.ray_dtype)
        index = np.ascontiguousarray(index, dtype=np.uint32)
        assert index.shape == (len(rays),)
        hits = np.zeros(len(rays), L.hit_dtype) if out is None else out
        assert hits.dtype == L.hit_dtype and len(hits) == len(rays) and hits.flags.c_contiguous
        _check(self._h, L.lib.ptb_check_hit_index(self._h, L.ptr(rays), L.ptr(index), len(rays), L.ptr(hits)))
        return hits

    def check_hit_index_device(self, d_rays_ptr: int, d_index_ptr: int, n: int, d_hits_ptr: int):
        _check(self._h, L.lib.ptb_check_hit_index_device(self._h, C.c_void_p(d_rays_ptr), C.c_void_p(d_index_ptr), n,
                                                          C.c_void_p(d_hits_ptr)))

    def occluded(self, rays: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        """Occlusion per ray (occlusion_ray_dtype, see make_occlusion_rays): True iff a primitive other than `exclude` is
        hit at 0 < t < tmax. `out`: optional caller-owned bool buffer."""
        rays = np.ascontiguousarray(rays, dtype=L.occlusion_ray_dtype)
        occ = np.zeros(len(rays), bool) if out is None else out
        assert occ.dtype == bool and len(occ) == len(rays) and occ.flags.c_contiguous
        _check(self._h, L.lib.ptb_occluded(self._h, L.ptr(rays), len(rays), L.ptr(occ)))
        return occ

    def occluded_device(self, d_rays_ptr: int, n: int, d_occluded_ptr: int):
        """d_occluded: n bytes, 1 = occluded."""
        _check(self._h, L.lib.ptb_occluded_device(self._h, C.c_void_p(d_rays_ptr), n, C.c_void_p(d_occluded_ptr)))

    # ---- render
    def render(self, opts: RenderOptions, progress=None):
        cb = None
        if progress is not None:
            cb = L.PROGRESS_FN(lambda user, samples, rays: 1 if progress(samples, rays) else 0)
        self._progress_ref = cb
        o = opts.to_c()
        rc = L.lib.ptb_render(self._h, C.byref(o), C.cast(cb, C.c_void_p) if cb else None, None)
        self._progress_ref = None
        _check(self._h, rc)

    def render_passes(self, opts: RenderOptions, update):
        """The reference's per-pass contract (random_sampler.rs:31-98): `update(pass_image (H, W, 3), pass_number,
        rays_shot) -> bool` once per pass with that pass's single-sample image; True stops the render."""
        h, w = opts.height, opts.width

        def thunk(user, img, n, i, rays):
            a = np.ctypeslib.as_array(img, shape=(n,)).reshape(h, w, 3)
            return 1 if update(a, int(i), int(rays)) else 0

        cb = L.PASS_FN(thunk)
        o = opts.to_c()
        _check(self._h, L.lib.ptb_render_passes(self._h, C.byref(o), C.cast(cb, C.c_void_p), None))

    def accum_clear(self):
        _check(self._h, L.lib.ptb_accum_clear(self._h))

    def accum_read(self, width: int, height: int, normalise: bool = True, out: np.ndarray | None = None) -> np.ndarray:
        """`out`: optional caller-owned float32 buffer of W*H*3 elements (e.g. pinned memory) to read into."""
        if out is None:
            out = np.empty(width * height * 3, np.float32)
        out = out.reshape(-1)
        _check(self._h, L.lib.ptb_accum_read(self._h, L.ptr(out), out.size, 1 if normalise else 0))
        return out.reshape(height, width, 3)

    def accum_device_ptr(self):
        p, n = C.c_void_p(), C.c_size_t()
        _check(self._h, L.lib.ptb_accum_device_ptr(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def accum_set_samples(self, n: int):
        _check(self._h, L.lib.ptb_accum_set_samples(self._h, n))

    # ---- denoiser feature buffers
    def render_aov(self, opts: RenderOptions):
        """Adds the first-hit albedo, normal, depth and coverage of the camera rays `render(opts)` traces into the AOV
        sums (render_method, max_depth and rr_threshold are not read)."""
        o = opts.to_c()
        _check(self._h, L.lib.ptb_render_aov(self._h, C.byref(o)))

    def aov_clear(self):
        _check(self._h, L.lib.ptb_aov_clear(self._h))

    def aov_read(self, width: int, height: int, aov: int, normalise: bool = True) -> np.ndarray:
        """One AOV buffer (L.PTB_AOV_*): (H, W, 3) float32 for albedo and normal, (H, W) for depth and coverage."""
        c = 3 if aov in (L.PTB_AOV_ALBEDO, L.PTB_AOV_NORMAL) else 1
        out = np.empty(width * height * c, np.float32)
        _check(self._h, L.lib.ptb_aov_read(self._h, aov, L.ptr(out), out.size, 1 if normalise else 0))
        return out.reshape((height, width, 3) if c == 3 else (height, width))

    # ---- denoiser
    def denoise(self, width: int, height: int, **opts) -> np.ndarray:
        """The beauty accumulator filtered by the spatial SVGF filter, guided by the AOV sums: (H, W, 3) float32. Keyword
        options (0 selects the default): iterations (5), sigma_luminance (4), sigma_normal (128), sigma_depth (1)."""
        o = denoise_opts(**opts)
        out = np.empty(width * height * 3, np.float32)
        _check(self._h, L.lib.ptb_denoise(self._h, C.byref(o), L.ptr(out), out.size))
        return out.reshape(height, width, 3)

    def denoise_device(self, d_rgb_ptr: int, **opts):
        """As denoise, into a device buffer of W*H*3 floats; enqueued on the context's stream, not waited for."""
        o = denoise_opts(**opts)
        _check(self._h, L.lib.ptb_denoise_device(self._h, C.byref(o), C.c_void_p(d_rgb_ptr)))

    # ---- sampler test hook (the reference's chi-squared harness pointed at the device samplers)
    @staticmethod
    def _query(kind, alpha, normal, aux, light_index, seed) -> L.SamplerQuery:
        return L.SamplerQuery(kind, float(alpha), L.Vec3(*map(float, normal)), L.Vec3(*map(float, aux)), int(light_index), int(seed))

    def sample_only(self, kind: int, n: int, alpha=0.0, normal=(0, 0, 1), aux=(0, 0, 1), light_index=0, seed=0):
        """n directions from device sampler `kind` (L.SAMPLER_*) and the sampler's pdf of each: (dirs (n, 3), pdf (n,))."""
        q = self._query(kind, alpha, normal, aux, light_index, seed)
        dirs, pdf = np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
        _check(self._h, L.lib.ptb_sample_only(self._h, C.byref(q), n, L.ptr(dirs), L.ptr(pdf)))
        return dirs, pdf

    def sampler_pdf(self, kind: int, dirs: np.ndarray, alpha=0.0, normal=(0, 0, 1), aux=(0, 0, 1), light_index=0):
        q = self._query(kind, alpha, normal, aux, light_index, 0)
        dirs = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        pdf = np.zeros(len(dirs), np.float32)
        _check(self._h, L.lib.ptb_sampler_pdf(self._h, C.byref(q), L.ptr(dirs), len(dirs), L.ptr(pdf)))
        return pdf

    def stats(self) -> L.Stats:
        s = L.Stats()
        _check(self._h, L.lib.ptb_stats_get(self._h, C.byref(s)))
        return s

    def stats_reset(self):
        _check(self._h, L.lib.ptb_stats_reset(self._h))


class Bvh:
    """Device acceleration structure over a host scene (Bvh::new + check_hit)."""

    def __init__(self, ctx: Context, scene: HostScene):
        self.ctx = ctx
        ctx.upload(scene)
        ctx.commit()
        self.n_prims, self.n_nodes = ctx.bvh_info()

    def number_nodes(self) -> int:  # acceleration/mod.rs:94-96
        return self.n_nodes

    def check_hit(self, rays: np.ndarray) -> np.ndarray:
        return self.ctx.closest_hit(rays)

    def check_hit_index(self, rays: np.ndarray, index: np.ndarray) -> np.ndarray:
        return self.ctx.check_hit_index(rays, index)

    def occluded(self, rays: np.ndarray) -> np.ndarray:
        return self.ctx.occluded(rays)


class RandomSampler:
    """RandomSampler::sample_image on the device: `spp` samples of every pixel into the accumulator."""

    def sample_image(self, opts: RenderOptions, bvh: Bvh, update=None, presentation_update=None):
        """`presentation_update(pass_image, i, rays_shot) -> bool`: the reference's per-pass closure; `update(samples,
        rays) -> bool`: counters only (one device accumulator, no per-pass read-back)."""
        if presentation_update is not None:
            bvh.ctx.render_passes(opts, presentation_update)
        else:
            bvh.ctx.render(opts, progress=update)


class Scene:
    """frontend Scene (src/scene.rs:7-43) for `--backend cuda`."""

    def __init__(self, host_scene: HostScene, device: int = 0, ctx: Context | None = None):
        self.ctx = ctx or Context(device)
        self.host = host_scene
        self.acceleration = Bvh(self.ctx, host_scene)

    def render(self, opts: RenderOptions, update=None, presentation_update=None) -> np.ndarray:
        """Returns the running-mean image (H, W, 3) the TUI closure of src/main.rs:175-191 would hold."""
        self.ctx.accum_clear()
        RandomSampler().sample_image(opts, self.acceleration, update, presentation_update)
        return self.ctx.accum_read(opts.width, opts.height, normalise=True)

    def render_aov(self, opts: RenderOptions) -> dict:
        """The denoiser feature buffers of the samples `render(opts)` takes: {"albedo", "normal"} (H, W, 3) and {"depth",
        "coverage"} (H, W), normalised (depth is the mean over the samples that hit)."""
        self.ctx.aov_clear()
        self.ctx.render_aov(opts)
        names = {"albedo": L.PTB_AOV_ALBEDO, "normal": L.PTB_AOV_NORMAL, "depth": L.PTB_AOV_DEPTH, "coverage": L.PTB_AOV_COVERAGE}
        return {k: self.ctx.aov_read(opts.width, opts.height, a) for k, a in names.items()}

    def render_denoised(self, opts: RenderOptions, **denoise) -> np.ndarray:
        """render(opts) and the feature buffers of the same samples, then the denoised image (H, W, 3); `denoise` takes
        Context.denoise's keyword options."""
        self.ctx.accum_clear()
        self.ctx.render(opts)
        self.ctx.aov_clear()
        self.ctx.render_aov(opts)
        return self.ctx.denoise(opts.width, opts.height, **denoise)


def render_multi(contexts, opts: RenderOptions) -> np.ndarray:
    """Scene::render across several GPUs of one box through ptb_render_multi: every context (one per GPU, same scene
    committed on each) renders its share of the samples on its own host thread inside the library, then one
    ncclReduce(sum) to contexts[0]. Returns the mean image."""
    arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    o = opts.to_c()
    _check(contexts[0]._h, L.lib.ptb_render_multi(C.cast(arr, C.c_void_p), len(contexts), C.byref(o)))
    return contexts[0].accum_read(opts.width, opts.height, normalise=True)


def make_rays(origins: np.ndarray, directions: np.ndarray) -> np.ndarray:
    r = np.zeros(len(origins), L.ray_dtype)
    r["o"] = origins
    r["d"] = directions
    return r


def make_occlusion_rays(origins: np.ndarray, directions: np.ndarray, tmax=np.inf, exclude=L.PTB_MISS) -> np.ndarray:
    """Occlusion rays: `tmax` (distance along the normalised direction) and `exclude` (original primitive id that does not
    block, PTB_MISS: none) are scalars or one value per ray."""
    r = np.zeros(len(origins), L.occlusion_ray_dtype)
    r["o"] = origins
    r["d"] = directions
    r["tmax"] = tmax
    r["exclude"] = exclude
    return r
