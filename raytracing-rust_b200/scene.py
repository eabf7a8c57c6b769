"""Host-side scene description (POD arrays) and the .ssml loader binding.

Mirrors what `loader::load_file_full` hands to `Bvh::new` + `Scene::new` in the reference
(crates/loader/src/lib.rs:196-243, src/parameters.rs:45-78): primitives (spheres first, then mesh
triangles), materials, textures, camera, sky. Parsing itself is native (host/ssml_loader.cpp).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L


def _camera_make_native(origin, lookat, vup, hfov_deg, aspect, aperture, focus_dist) -> np.ndarray:
    cam = np.zeros(1, L.camera_dtype)
    rc = L.lib.ptb_camera_make(L.Vec3(*map(float, origin)), L.Vec3(*map(float, lookat)), L.Vec3(*map(float, vup)),
                               float(hfov_deg), float(aspect), float(aperture), float(focus_dist), L.ptr(cam))
    if rc != L.PTB_OK:
        raise L.PtbError(rc, "ptb_camera_make")
    return cam


# SimpleCamera::new. bench.py's `--impl reference` arm swaps in the CPU checker's restatement (bit-equal,
# tests/ pin that) so that its process never maps libptb200.so; nothing in this package does.
CAMERA_MAKE = _camera_make_native


@dataclass
class HostScene:
    spheres: np.ndarray = field(default_factory=lambda: np.zeros(0, L.sphere_dtype))
    triangles: np.ndarray = field(default_factory=lambda: np.zeros(0, L.triangle_dtype))
    materials: np.ndarray = field(default_factory=lambda: np.zeros(0, L.material_dtype))
    textures: np.ndarray = field(default_factory=lambda: np.zeros(0, L.texture_dtype))
    camera: np.ndarray = field(default_factory=lambda: np.zeros(1, L.camera_dtype))
    sky: np.ndarray = field(default_factory=lambda: np.zeros(1, L.sky_dtype))
    # bulk data of ImageTexture / Perlin textures: texture index -> (width, height, float32 words)
    texture_data: dict = field(default_factory=dict)

    @property
    def n_primitives(self) -> int:
        return len(self.spheres) + len(self.triangles)

    def nbytes(self) -> int:
        """Bytes a ptb_scene_upload + commit moves host -> device."""
        return int(self.spheres.nbytes + self.triangles.nbytes + self.materials.nbytes + self.textures.nbytes
                   + self.camera.nbytes + self.sky.nbytes + sum(d.nbytes for _, _, d in self.texture_data.values()))

    # -- builders used by tests / generators ------------------------------------------------------------
    def add_texture(self, kind: int, a=(0, 0, 0), b=(0, 0, 0)) -> int:
        t = np.zeros(1, L.texture_dtype)
        t["kind"], t["a"], t["b"] = kind, a, b
        self.textures = np.concatenate([self.textures, t])
        return len(self.textures) - 1

    def add_image_texture(self, rgb: np.ndarray) -> int:
        """ImageTexture (textures/mod.rs:202-266) from an (H, W, 3) float array."""
        rgb = np.ascontiguousarray(rgb, dtype=np.float32)
        h, w, _ = rgb.shape
        i = self.add_texture(L.TEX_IMAGE)
        self.texture_data[i] = (w, h, rgb.reshape(-1).copy())
        return i

    def add_perlin_texture(self, seed: int = 0) -> int:
        """Perlin (textures/mod.rs:75-180); tables are a pure function of `seed` (the reference uses OS entropy)."""
        i = self.add_texture(L.TEX_PERLIN)
        words = np.zeros(L.PERLIN_TABLE_WORDS, np.float32)
        rc = L.lib.ptb_perlin_tables(seed, L.ptr(words))
        if rc != L.PTB_OK:
            raise L.PtbError(rc, "ptb_perlin_tables")
        self.texture_data[i] = (0, 0, words)
        return i

    def add_material(self, kind: int, texture: int, param: float, ior=(1, 1, 1), metallic: float = 0.0) -> int:
        m = np.zeros(1, L.material_dtype)
        m["kind"], m["texture"], m["param"], m["ior"], m["metallic"] = kind, texture, param, ior, metallic
        self.materials = np.concatenate([self.materials, m])
        return len(self.materials) - 1

    def add_sphere(self, center, radius: float, material: int) -> int:
        s = np.zeros(1, L.sphere_dtype)
        s["center"], s["radius"], s["material"] = center, radius, material
        self.spheres = np.concatenate([self.spheres, s])
        return len(self.spheres) - 1

    def set_camera(self, origin, lookat, vup, hfov_deg, aspect=16.0 / 9.0, aperture=0.0, focus_dist=10.0):
        """SimpleCamera::new (implementations/src/camera.rs:20-53)."""
        self.camera = CAMERA_MAKE(origin, lookat, vup, hfov_deg, aspect, aperture, focus_dist)

    def set_sky(self, texture: int, sampler_res=(100, 100)):
        self.sky = np.zeros(1, L.sky_dtype)
        self.sky["texture"], self.sky["sampler_res_x"], self.sky["sampler_res_y"] = texture, sampler_res[0], sampler_res[1]


@dataclass
class IndexedMesh:
    """The reference's MeshData + MeshTriangle (implementations/primitives/triangle.rs:30-36): vertex and normal arrays and
    triangles that index them (mesh_triangle_dtype). Uploaded with Context.set_mesh; the device expands it into the
    triangle_dtype records expand() returns."""
    vertices: np.ndarray   # (V, 3) float32
    normals: np.ndarray    # (N, 3) float32
    triangles: np.ndarray  # (T,) mesh_triangle_dtype

    def __post_init__(self):
        self.vertices = np.ascontiguousarray(self.vertices, np.float32).reshape(-1, 3)
        self.normals = np.ascontiguousarray(self.normals, np.float32).reshape(-1, 3)
        self.triangles = np.ascontiguousarray(self.triangles, L.mesh_triangle_dtype)

    def expand(self) -> np.ndarray:
        """The flat triangles (triangle_dtype) this mesh stands for: a host-side gather, byte for byte what the device
        expansion writes. An index out of range raises IndexError."""
        tri = np.zeros(len(self.triangles), L.triangle_dtype)
        tri["p"] = self.vertices[self.triangles["p"]]
        tri["n"] = self.normals[self.triangles["n"]]
        tri["material"] = self.triangles["material"]
        return tri

    def expand_instances(self, instances: np.ndarray, xforms: np.ndarray) -> np.ndarray:
        """The flat triangles (triangle_dtype) an instance list over this mesh stands for (Context.set_mesh_instances): for
        each instance in order, mesh triangles [first_triangle, first_triangle + n_triangles) expanded, positions and normals
        transformed in float32 in the header's statement order, and the material replaced unless it is PTB_MISS. Byte for
        byte what the device expansion writes."""
        inst = np.ascontiguousarray(instances, L.mesh_instance_dtype).reshape(-1)
        xf = np.ascontiguousarray(xforms, L.instance_xform_dtype).reshape(-1)
        if len(inst) != len(xf):
            raise ValueError(f"{len(inst)} instances but {len(xf)} transforms")
        count = inst["n_triangles"].astype(np.int64)
        owner = np.repeat(np.arange(len(inst)), count)
        start = np.cumsum(count) - count
        mt = inst["first_triangle"].astype(np.int64)[owner] + (np.arange(len(owner)) - start[owner])
        tri = IndexedMesh(self.vertices, self.normals, self.triangles[mt]).expand()
        m, n = xf["m"][owner], xf["n"][owner]  # (T, 3, 4), (T, 3, 3)
        p, q = tri["p"].copy(), tri["n"].copy()  # (T, 3 corners, 3)
        for r in range(3):
            tri["p"][:, :, r] = ((m[:, r, 0, None] * p[:, :, 0] + m[:, r, 1, None] * p[:, :, 1]) + m[:, r, 2, None] * p[:, :, 2]) \
                + m[:, r, 3, None]
            tri["n"][:, :, r] = (n[:, r, 0, None] * q[:, :, 0] + n[:, r, 1, None] * q[:, :, 1]) + n[:, r, 2, None] * q[:, :, 2]
        over = inst["material"][owner]
        tri["material"] = np.where(over != L.PTB_MISS, over, tri["material"])
        return tri

    def nbytes(self) -> int:
        return int(self.vertices.nbytes + self.normals.nbytes + self.triangles.nbytes)


def instance_xform(rotation=None, scale: float = 1.0, translation=(0.0, 0.0, 0.0)) -> np.ndarray:
    """One instance_xform_dtype record: m = [s R | t], n = R. `rotation` is a 3x3 rotation matrix or a quaternion
    (w, x, y, z), normalised here; None is the identity. With R orthonormal, unit normals stay unit up to rounding. For a
    general affine map build the record yourself with n = the inverse transpose of its linear part: the library does not
    renormalise normals (neither does the reference's interpolated normal)."""
    if rotation is None:
        R = np.eye(3)
    else:
        r = np.asarray(rotation, np.float64)
        if r.shape == (4,):
            w, x, y, z = r / np.linalg.norm(r)
            R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                          [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                          [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        else:
            R = r.reshape(3, 3)
    out = np.zeros(1, L.instance_xform_dtype)
    out["m"][0, :, :3] = (float(scale) * R).astype(np.float32)
    out["m"][0, :, 3] = np.asarray(translation, np.float32)
    out["n"][0] = R.astype(np.float32)
    return out


def _dedup_rows(a: np.ndarray):
    """Distinct float32 3-vectors of `a` (rows compared by their bytes, so -0.0 != 0.0 and NaNs keep their payload) and
    the index of each row among them."""
    rows = np.ascontiguousarray(a, np.float32).reshape(-1, 3)
    keys = rows.view(np.dtype((np.void, 12))).reshape(-1)
    _, first, inverse = np.unique(keys, return_index=True, return_inverse=True)
    return rows[first], inverse.reshape(-1).astype(np.uint32)


def index_triangles(tri: np.ndarray) -> IndexedMesh:
    """Indexed form of a flat triangle array: positions and normals deduplicated by their bytes. expand() of the result
    equals `tri` byte for byte."""
    tri = np.ascontiguousarray(tri, L.triangle_dtype)
    vertices, pi = _dedup_rows(tri["p"])
    normals, ni = _dedup_rows(tri["n"])
    m = np.zeros(len(tri), L.mesh_triangle_dtype)
    m["p"] = pi.reshape(-1, 3)
    m["n"] = ni.reshape(-1, 3)
    m["material"] = tri["material"]
    return IndexedMesh(vertices, normals, m)


def _copy_array(handle, getter, dtype) -> np.ndarray:
    p = C.c_void_p()
    n = getter(handle, C.byref(p))
    if n == 0:
        return np.zeros(0, dtype)
    buf = (C.c_char * (n * dtype.itemsize)).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype, count=n).copy()


def _from_handle(handle) -> HostScene:
    s = HostScene()
    s.spheres = _copy_array(handle, L.lib.ptb_host_scene_spheres, L.sphere_dtype)
    s.triangles = _copy_array(handle, L.lib.ptb_host_scene_triangles, L.triangle_dtype)
    s.materials = _copy_array(handle, L.lib.ptb_host_scene_materials, L.material_dtype)
    s.textures = _copy_array(handle, L.lib.ptb_host_scene_textures, L.texture_dtype)
    for i in range(len(s.textures)):
        w, h, p = C.c_uint32(), C.c_uint32(), C.c_void_p()
        n = L.lib.ptb_host_scene_texture_data(handle, i, C.byref(w), C.byref(h), C.byref(p))
        if n:
            buf = (C.c_float * n).from_address(p.value)
            s.texture_data[i] = (w.value, h.value, np.frombuffer(buf, dtype=np.float32, count=n).copy())
    L.lib.ptb_host_scene_camera(handle, L.ptr(s.camera))
    L.lib.ptb_host_scene_sky(handle, L.ptr(s.sky))
    return s


def load_file(path: str) -> HostScene:
    """loader::load_file_full (crates/loader/src/lib.rs:196-243). Raises PtbError like LoadErr."""
    h = C.c_void_p()
    rc = L.lib.ptb_ssml_load_file(path.encode(), C.byref(h))
    if rc != L.PTB_OK:
        raise L.PtbError(rc, L.lib.ptb_host_last_error().decode())
    try:
        return _from_handle(h)
    finally:
        L.lib.ptb_host_scene_free(h)


def load_str(text: str, base_dir: str = ".") -> HostScene:
    """loader::load_str_full (crates/loader/src/lib.rs:245-288)."""
    h = C.c_void_p()
    rc = L.lib.ptb_ssml_load_str(text.encode(), base_dir.encode(), C.byref(h))
    if rc != L.PTB_OK:
        raise L.PtbError(rc, L.lib.ptb_host_last_error().decode())
    try:
        return _from_handle(h)
    finally:
        L.lib.ptb_host_scene_free(h)


def load_image(filename: str) -> np.ndarray:
    """ImageTexture::new's decode (textures/mod.rs:208-245): (H, W, 3) float32."""
    w, h, p = C.c_uint32(), C.c_uint32(), C.c_void_p()
    rc = L.lib.ptb_image_load(filename.encode(), C.byref(w), C.byref(h), C.byref(p))
    if rc != L.PTB_OK:
        raise L.PtbError(rc, L.lib.ptb_image_last_error().decode())
    try:
        buf = (C.c_float * (w.value * h.value * 3)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.float32).reshape(h.value, w.value, 3).copy()
    finally:
        L.lib.ptb_image_free(p)


def save_image(filename: str, width: int, height: int, rgb: np.ndarray, gamma: float = 2.2):
    """output::save_data_to_image (crates/output/src/lib.rs:74-113)."""
    rgb = np.ascontiguousarray(rgb, dtype=np.float32).reshape(-1)
    assert rgb.size == width * height * 3
    rc = L.lib.ptb_image_save(filename.encode(), width, height, L.ptr(rgb), float(gamma))
    if rc != L.PTB_OK:
        raise L.PtbError(rc, f"ptb_image_save({filename})")
