"""Deterministic synthetic inputs for BASELINE.json's configs (no RNG in the geometry, closed-form heights).

  c3_scene()          1 000 000 triangles: 800 000-triangle Lambertian terrain + 200 000-triangle dielectric UV sphere,
                      Lerp sky as scenes/rtweekend1.ssml, 16:9 camera                         (SURVEY.md §8d "C3")
  c3_deform()         one frame of an animated C3: terrain wave + glass sphere pushed into the terrain (same counts)
  c3_indexed(), heightfield_indexed(), c3_deform_vertices()
                      the same scenes as indexed meshes over their grid points (expand() == the flat triangles)
  c3_instanced(), c3_instanced_frame()
                      c3_indexed's mesh placed as two instances (terrain, glass sphere), and the sphere's transform for
                      c3_deform's motion
  rock(), scatter_instances()
                      a small closed mesh, and many rotated, scaled, translated copies of a mesh over a terrain
  heightfield_scene() R x C quads in [-1,1]^2 x [-0.2,0.2]; 2500 x 2000 -> 10 000 000 triangles      ("C5")
  philox_rays()       incoherent rays from Philox4x32-10 (seed 0x5EED, counter = ray index): origin uniform in the
                      ball of radius 2 about the mesh centre, direction uniform on the sphere
  write_obj()/c3_ssml()  the same C3 mesh as an OBJ (v / vn / usemtl / f v//vn) + .ssml, for the loader path
All arithmetic is float32 numpy; the arrays ARE the input (oracle and device receive identical bytes).
"""
from __future__ import annotations

import copy

import numpy as np

from . import _lib as L
from .scene import HostScene, IndexedMesh, instance_xform

F = np.float32


def _grid_vertices(xs: np.ndarray, ys: np.ndarray, height_fn, normal_fn):
    """Positions and normals at the grid points: (len(xs), len(ys), 3) each."""
    X, Y = np.meshgrid(xs.astype(F), ys.astype(F), indexing="ij")
    Z = height_fn(X, Y).astype(F)
    P = np.stack([X, Y, Z], axis=-1)              # (nx, ny, 3)
    N = normal_fn(X, Y).astype(F)
    return P, N


def _grid_triangles(xs: np.ndarray, ys: np.ndarray, height_fn, normal_fn):
    """(len(xs)-1) x (len(ys)-1) quads -> 2 triangles each; returns positions (T,3,3) and normals (T,3,3)."""
    P, N = _grid_vertices(xs, ys, height_fn, normal_fn)
    p00, p10, p01, p11 = P[:-1, :-1], P[1:, :-1], P[:-1, 1:], P[1:, 1:]
    n00, n10, n01, n11 = N[:-1, :-1], N[1:, :-1], N[:-1, 1:], N[1:, 1:]
    t0 = np.stack([p00, p10, p11], axis=2)         # (nx-1, ny-1, 3, 3)
    t1 = np.stack([p00, p11, p01], axis=2)
    m0 = np.stack([n00, n10, n11], axis=2)
    m1 = np.stack([n00, n11, n01], axis=2)
    pos = np.stack([t0, t1], axis=2).reshape(-1, 3, 3)
    nrm = np.stack([m0, m1], axis=2).reshape(-1, 3, 3)
    return np.ascontiguousarray(pos, F), np.ascontiguousarray(nrm, F)


def _terrain_height(X, Y):
    return F(0.25) * np.sin(F(1.3) * X) * np.cos(F(0.9) * Y) + F(0.1) * np.sin(F(3.1) * X + F(1.7) * Y)


def _terrain_normal(X, Y):
    dzdx = F(0.25) * F(1.3) * np.cos(F(1.3) * X) * np.cos(F(0.9) * Y) + F(0.1) * F(3.1) * np.cos(F(3.1) * X + F(1.7) * Y)
    dzdy = -F(0.25) * F(0.9) * np.sin(F(1.3) * X) * np.sin(F(0.9) * Y) + F(0.1) * F(1.7) * np.cos(F(3.1) * X + F(1.7) * Y)
    n = np.stack([-dzdx, -dzdy, np.ones_like(dzdx)], axis=-1)
    return n / np.linalg.norm(n, axis=-1, keepdims=True)


def _uv_sphere_vertices(center, radius: float, slices: int, stacks: int):
    """Positions and radial normals at the (stacks + 1) x (slices + 1) grid points of the UV sphere."""
    c = np.asarray(center, F)
    theta = (np.arange(stacks + 1, dtype=F) / F(stacks)) * F(np.pi)        # 0 .. pi
    phi = (np.arange(slices + 1, dtype=F) / F(slices)) * F(2 * np.pi)
    st, ct = np.sin(theta), np.cos(theta)
    sp, cp = np.sin(phi), np.cos(phi)
    sp[-1], cp[-1] = sp[0], cp[0]                                           # close the seam exactly
    st[0] = st[-1] = F(0)
    D = np.stack([st[:, None] * cp[None, :], st[:, None] * sp[None, :], np.repeat(ct[:, None], slices + 1, 1)], -1).astype(F)
    P = c + F(radius) * D
    return P, D


def uv_sphere(center, radius: float, slices: int, stacks: int):
    """2 * slices * (stacks - 1) triangles (poles are fans); normals are radial."""
    P, D = _uv_sphere_vertices(center, radius, slices, stacks)
    tris_p, tris_n = [], []
    for k in range(stacks):
        a, b = k, k + 1
        pa0, pa1, pb0, pb1 = P[a, :-1], P[a, 1:], P[b, :-1], P[b, 1:]
        na0, na1, nb0, nb1 = D[a, :-1], D[a, 1:], D[b, :-1], D[b, 1:]
        if k != 0:                # upper triangle degenerates at the north pole
            tris_p.append(np.stack([pa0, pb1, pa1], 1)); tris_n.append(np.stack([na0, nb1, na1], 1))
        if k != stacks - 1:       # lower triangle degenerates at the south pole
            tris_p.append(np.stack([pa0, pb0, pb1], 1)); tris_n.append(np.stack([na0, nb0, nb1], 1))
    return np.ascontiguousarray(np.concatenate(tris_p), F), np.ascontiguousarray(np.concatenate(tris_n), F)


def _base_scene(sky_like_rtweekend: bool = True) -> HostScene:
    s = HostScene()
    sky_tex = s.add_texture(L.TEX_LERP, (0.5, 0.7, 1.0), (1.0, 1.0, 1.0))   # scenes/rtweekend1.ssml:10-14
    grey = s.add_texture(L.TEX_SOLID, (0.5, 0.5, 0.5))
    white = s.add_texture(L.TEX_SOLID, (1.0, 1.0, 1.0))
    s.add_material(L.MAT_LAMBERTIAN, grey, 0.5)      # 0: ground
    s.add_material(L.MAT_REFRACT, white, 1.5)        # 1: glass
    s.set_sky(sky_tex, (100, 100))
    return s


def _grid_indices(nx: int, ny: int) -> np.ndarray:
    """Corner indices (T, 3) into an (nx, ny) grid of points flattened row-major, in _grid_triangles' order."""
    g = np.arange(nx * ny, dtype=np.uint32).reshape(nx, ny)
    i00, i10, i01, i11 = g[:-1, :-1], g[1:, :-1], g[:-1, 1:], g[1:, 1:]
    t0 = np.stack([i00, i10, i11], axis=-1)
    t1 = np.stack([i00, i11, i01], axis=-1)
    return np.stack([t0, t1], axis=2).reshape(-1, 3)


def _uv_sphere_indices(slices: int, stacks: int) -> np.ndarray:
    """Corner indices (T, 3) into the flattened (stacks + 1) x (slices + 1) sphere grid, in uv_sphere's order."""
    g = np.arange((stacks + 1) * (slices + 1), dtype=np.uint32).reshape(stacks + 1, slices + 1)
    out = []
    for k in range(stacks):
        a0, a1, b0, b1 = g[k, :-1], g[k, 1:], g[k + 1, :-1], g[k + 1, 1:]
        if k != 0:
            out.append(np.stack([a0, b1, a1], 1))
        if k != stacks - 1:
            out.append(np.stack([a0, b0, b1], 1))
    return np.concatenate(out)


def _mesh(parts) -> IndexedMesh:
    """One IndexedMesh from (positions grid, normals grid, corner indices (T, 3), material) parts; a triangle's position
    and normal indices are the same grid point."""
    verts, nrms, tris, base = [], [], [], 0
    for P, N, idx, material in parts:
        t = np.zeros(len(idx), L.mesh_triangle_dtype)
        t["p"] = idx + np.uint32(base)
        t["n"] = idx + np.uint32(base)
        t["material"] = material
        verts.append(P.reshape(-1, 3))
        nrms.append(N.reshape(-1, 3))
        tris.append(t)
        base += len(verts[-1])
    return IndexedMesh(np.concatenate(verts), np.concatenate(nrms), np.concatenate(tris))


def _c3_dims(scale: float):
    return (max(2, int(round(1000 * scale))), max(2, int(round(400 * scale))), max(3, int(round(500 * scale))),
            max(3, int(round(201 * scale))))


def _c3_axes(nx: int, ny: int):
    return (np.linspace(-12.5, 12.5, nx + 1, dtype=np.float64).astype(F), np.linspace(0.0, 10.0, ny + 1, dtype=np.float64).astype(F))


C3_CAMERA = ((0.0, -1.5, 1.6), (0.0, 4.0, 0.7), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0)


def c3_scene(scale: float = 1.0) -> HostScene:
    """scale=1 -> exactly 1 000 000 triangles; scale<1 shrinks every grid dimension (tests)."""
    nx, ny, slices, stacks = _c3_dims(scale)
    s = _base_scene()
    xs, ys = _c3_axes(nx, ny)
    tp, tn = _grid_triangles(xs, ys, _terrain_height, _terrain_normal)
    sp_, sn = uv_sphere((0.0, 4.0, 1.0), 0.8, slices, stacks)
    tri = np.zeros(len(tp) + len(sp_), L.triangle_dtype)
    tri["p"][: len(tp)], tri["n"][: len(tp)], tri["material"][: len(tp)] = tp, tn, 0
    tri["p"][len(tp):], tri["n"][len(tp):], tri["material"][len(tp):] = sp_, sn, 1
    s.triangles = tri
    s.set_camera(*C3_CAMERA)
    return s


def c3_indexed(scale: float = 1.0):
    """C3 as an indexed mesh: (scene without triangles, mesh). The vertices are the grid points of the terrain
    ((nx + 1) x (ny + 1)) and of the sphere ((stacks + 1) x (slices + 1)), 502 603 at scale 1; mesh.expand() equals
    c3_scene(scale).triangles byte for byte."""
    nx, ny, slices, stacks = _c3_dims(scale)
    s = _base_scene()
    xs, ys = _c3_axes(nx, ny)
    P, N = _grid_vertices(xs, ys, _terrain_height, _terrain_normal)
    SP, SN = _uv_sphere_vertices((0.0, 4.0, 1.0), 0.8, slices, stacks)
    mesh = _mesh([(P, N, _grid_indices(nx + 1, ny + 1), 0), (SP, SN, _uv_sphere_indices(slices, stacks), 1)])
    s.set_camera(*C3_CAMERA)
    return s, mesh


C3_GLASS_RADIUS = 0.8


def c3_deform(scene: HostScene, wave: float, shift: float) -> HostScene:
    """A frame of an animated C3 (same counts, same order, for PTB_BUILD_REFIT): every terrain vertex's height is scaled by
    1 + wave * sin(0.7 x + 0.4 y), and the glass sphere is moved by `shift` radii along (0.6, 0, -0.8), into the terrain.
    The function of a vertex is a function of its position, so shared vertices stay shared; normals are kept."""
    s = copy.deepcopy(scene)
    tri = s.triangles
    glass = tri["material"] == 1
    p = tri["p"][~glass]
    x, y = p[..., 0], p[..., 1]
    p[..., 2] = p[..., 2] * (F(1) + F(wave) * np.sin(F(0.7) * x + F(0.4) * y))
    tri["p"][~glass] = p
    tri["p"][glass] = tri["p"][glass] + (F(shift) * F(C3_GLASS_RADIUS) * np.array([0.6, 0.0, -0.8], F)).astype(F)
    return s


def c3_deform_vertices(mesh: IndexedMesh, wave: float, shift: float) -> IndexedMesh:
    """c3_deform's motion applied to the vertex array of c3_indexed's mesh (normals and triangles are shared, not copied).
    A vertex belongs to the sphere when a glass triangle uses it. numpy may evaluate sin differently for arrays of other
    shapes, so compare with expand() of the result, not with c3_deform."""
    glass = np.zeros(len(mesh.vertices), bool)
    glass[mesh.triangles["p"][mesh.triangles["material"] == 1].reshape(-1)] = True
    v = mesh.vertices.copy()
    t = v[~glass]
    x, y = t[:, 0], t[:, 1]
    t[:, 2] = t[:, 2] * (F(1) + F(wave) * np.sin(F(0.7) * x + F(0.4) * y))
    v[~glass] = t
    v[glass] = v[glass] + (F(shift) * F(C3_GLASS_RADIUS) * np.array([0.6, 0.0, -0.8], F)).astype(F)
    return IndexedMesh(v, mesh.normals, mesh.triangles)


def _instances(ranges) -> np.ndarray:
    """mesh_instance_dtype records from (first_triangle, n_triangles, material) tuples."""
    inst = np.zeros(len(ranges), L.mesh_instance_dtype)
    for i, (first, n, material) in enumerate(ranges):
        inst[i] = (first, n, material)
    return inst


def c3_instanced(scale: float = 1.0):
    """c3_indexed's mesh placed as two instances, the terrain's triangle range and the glass sphere's, each under an
    identity transform: (scene without triangles, mesh, instances, xforms). Upload with
    Context.upload(scene, mesh=mesh, instances=(instances, xforms)); mesh.expand_instances(instances, xforms) is the flat
    scene (c3_scene's triangles up to the sign of zero coordinates)."""
    s, mesh = c3_indexed(scale)
    n_terrain = int(np.count_nonzero(mesh.triangles["material"] == 0))
    inst = _instances([(0, n_terrain, L.PTB_MISS), (n_terrain, len(mesh.triangles) - n_terrain, L.PTB_MISS)])
    return s, mesh, inst, np.concatenate([instance_xform(), instance_xform()])


def c3_instanced_frame(shift: float) -> np.ndarray:
    """The glass sphere instance's transform (instance 1 of c3_instanced) for c3_deform's motion: a translation by `shift`
    radii along (0.6, 0, -0.8)."""
    return instance_xform(translation=(F(shift) * F(C3_GLASS_RADIUS) * np.array([0.6, 0.0, -0.8], F)).astype(F))


def rock(slices: int = 25, stacks: int = 21) -> IndexedMesh:
    """A small closed mesh about the origin: a unit UV sphere with closed-form bumps on its radius and radial normals,
    2 * slices * (stacks - 1) triangles (1000 by default), material 0."""
    P, D = _uv_sphere_vertices((0.0, 0.0, 0.0), 1.0, slices, stacks)
    bump = F(1) + F(0.15) * np.sin(F(3) * D[..., 0] + F(2) * D[..., 2]) * np.cos(F(4) * D[..., 1])
    return _mesh([((P * bump[..., None]).astype(F), D, _uv_sphere_indices(slices, stacks), 0)])


def scatter_instances(mesh: IndexedMesh, count: int, seed: int = 0, terrain=(200, 80)):
    """`count` copies of `mesh` over a C3-like terrain of 2 * terrain[0] * terrain[1] triangles: (scene without triangles,
    combined mesh, instances, xforms). The combined mesh is the terrain's grid followed by `mesh`; instance 0 places the
    terrain under the identity, instances 1..count place `mesh` with a uniformly random rotation, a scale in [0.05, 0.2]
    and a translation onto the terrain, all drawn from numpy's default_rng(seed)."""
    nx, ny = terrain
    s = _base_scene()
    xs, ys = _c3_axes(nx, ny)
    P, N = _grid_vertices(xs, ys, _terrain_height, _terrain_normal)
    ground = _mesh([(P, N, _grid_indices(nx + 1, ny + 1), 0)])
    t = mesh.triangles.copy()
    t["p"] += np.uint32(len(ground.vertices))
    t["n"] += np.uint32(len(ground.normals))
    combined = IndexedMesh(np.concatenate([ground.vertices, mesh.vertices]), np.concatenate([ground.normals, mesh.normals]),
                           np.concatenate([ground.triangles, t]))
    nt = len(ground.triangles)
    inst = np.zeros(count + 1, L.mesh_instance_dtype)
    inst["first_triangle"][0], inst["n_triangles"][0] = 0, nt
    inst["first_triangle"][1:], inst["n_triangles"][1:] = nt, len(mesh.triangles)
    inst["material"] = L.PTB_MISS
    rng = np.random.default_rng(seed)
    q = rng.normal(size=(count, 4))
    scale = rng.uniform(0.05, 0.2, count)
    x, y = rng.uniform(-12.0, 12.0, count), rng.uniform(0.5, 10.0, count)
    z = _terrain_height(x.astype(F), y.astype(F)).astype(np.float64)
    xf = np.concatenate([instance_xform()] + [instance_xform(q[i], scale[i], (x[i], y[i], z[i])) for i in range(count)])
    s.set_camera(*C3_CAMERA)
    return s, combined, inst, xf


def _hf_height(X, Y):
    return F(0.1) * np.sin(F(9.0) * X) * np.cos(F(7.0) * Y) + F(0.1) * np.sin(F(23.0) * X + F(17.0) * Y)


def _hf_normal(X, Y):
    dx = F(0.9) * np.cos(F(9.0) * X) * np.cos(F(7.0) * Y) + F(2.3) * np.cos(F(23.0) * X + F(17.0) * Y)
    dy = -F(0.7) * np.sin(F(9.0) * X) * np.sin(F(7.0) * Y) + F(1.7) * np.cos(F(23.0) * X + F(17.0) * Y)
    n = np.stack([-dx, -dy, np.ones_like(dx)], -1)
    return n / np.linalg.norm(n, axis=-1, keepdims=True)


def _hf_axes(rows: int, cols: int):
    return (np.linspace(-1.0, 1.0, rows + 1, dtype=np.float64).astype(F), np.linspace(-1.0, 1.0, cols + 1, dtype=np.float64).astype(F))


HF_CAMERA = ((0.0, -3.0, 1.5), (0.0, 0.0, 0.0), (0.0, 0.0, 1.0), 50.0, 16.0 / 9.0, 0.0, 1.0)


def heightfield_scene(rows: int = 2500, cols: int = 2000) -> HostScene:
    """rows x cols quads -> 2*rows*cols triangles in [-1,1]^2 x [-0.2,0.2] (C5: 10 000 000)."""
    s = _base_scene()
    xs, ys = _hf_axes(rows, cols)
    tp, tn = _grid_triangles(xs, ys, _hf_height, _hf_normal)
    tri = np.zeros(len(tp), L.triangle_dtype)
    tri["p"], tri["n"], tri["material"] = tp, tn, 0
    s.triangles = tri
    s.set_camera(*HF_CAMERA)
    return s


def heightfield_indexed(rows: int = 2500, cols: int = 2000):
    """The heightfield as an indexed mesh over its (rows + 1) x (cols + 1) grid points: (scene without triangles, mesh),
    mesh.expand() equal to heightfield_scene(rows, cols).triangles byte for byte."""
    s = _base_scene()
    P, N = _grid_vertices(*_hf_axes(rows, cols), _hf_height, _hf_normal)
    mesh = _mesh([(P, N, _grid_indices(rows + 1, cols + 1), 0)])
    s.set_camera(*HF_CAMERA)
    return s, mesh


# ---- Philox4x32-10 in numpy (vectorised over counters) ---------------------------------------------------------
def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    c0, c1, c2, c3 = (np.asarray(c, np.uint64) & np.uint64(0xFFFFFFFF) for c in (c0, c1, c2, c3))
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    mask = np.uint64(0xFFFFFFFF)
    k0, k1 = np.uint64(k0 & 0xFFFFFFFF), np.uint64(k1 & 0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0 = (k0 + np.uint64(0x9E3779B9)) & mask
        k1 = (k1 + np.uint64(0xBB67AE85)) & mask
    return c0.astype(np.uint32), c1.astype(np.uint32), c2.astype(np.uint32), c3.astype(np.uint32)


def _unit(u32):
    return (u32 >> np.uint32(8)).astype(F) * F(1.0 / 16777216.0)


def philox_rays(n: int, first: int = 0, seed: int = 0x5EED, centre=(0.0, 0.0, 0.0), radius: float = 2.0) -> np.ndarray:
    """Rays [first, first+n) of the C5 stream."""
    idx = np.arange(first, first + n, dtype=np.uint64)
    lo, hi = idx & np.uint64(0xFFFFFFFF), idx >> np.uint64(32)
    zero = np.zeros_like(idx)
    a = philox4x32_10(lo, hi, zero, zero, seed, 0)
    b = philox4x32_10(lo, hi, zero, zero + np.uint64(1), seed, 0)

    def sphere(u, v):
        z = F(1) - F(2) * u
        r = np.sqrt(np.maximum(F(0), F(1) - z * z))
        ph = F(2 * np.pi) * v
        return np.stack([r * np.cos(ph), r * np.sin(ph), z], -1).astype(F)

    od = sphere(_unit(a[0]), _unit(a[1]))
    rad = F(radius) * np.cbrt(_unit(a[2]))
    rays = np.zeros(n, L.ray_dtype)
    rays["o"] = np.asarray(centre, F) + od * rad[:, None]
    rays["d"] = sphere(_unit(b[0]), _unit(b[1]))
    return rays


# ---- OBJ / .ssml export of C3 (exercises the loader path) --------------------------------------------------------
def write_obj(path: str, scene: HostScene, names=("ground", "glass")):
    tri = scene.triangles
    with open(path, "w") as f:
        f.write("# generated by raytracing-rust_b200.meshgen\no mesh\n")
        p = tri["p"].reshape(-1, 3)
        n = tri["n"].reshape(-1, 3)
        for v in p:
            f.write(f"v {float(v[0])!r} {float(v[1])!r} {float(v[2])!r}\n")
        for v in n:
            f.write(f"vn {float(v[0])!r} {float(v[1])!r} {float(v[2])!r}\n")
        cur = None
        for i, m in enumerate(tri["material"]):
            if m != cur:
                f.write(f"usemtl {names[int(m)]}\n")
                cur = m
            a = 3 * i + 1
            f.write(f"f {a}//{a} {a + 1}//{a + 1} {a + 2}//{a + 2}\n")


def c3_ssml(obj_path: str) -> str:
    return f"""camera (
	origin   0 -1.5 1.6
	lookat   0 4 0.7
	vup      0 0 1
	fov      60.0
	aperture 0.0
	focus_dis 1.0
)

texture sky (
	type lerp
	primary 0.5 0.7 1.0
	secondary 1.0
)

sky (
	texture sky
)

texture grey (
	type solid
	colour 0.5
)

texture white (
	type solid
	colour 1.0
)

material ground (
	type lambertian
	texture grey
	albedo 0.5
)

material glass (
	type refract
	texture white
	eta 1.5
)

mesh (
	type mesh
	obj {obj_path}
)
"""
