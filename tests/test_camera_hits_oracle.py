"""CPU: ground truth for the camera-ray tests of tests/test_gpu_camera_hits.py, and the CPU statement of the per-pixel
camera candidate lists (scripts/camcand_ref.cpp) over a sweep of cameras.

- An independent f64 closest hit (numpy, every primitive) on the exact camera rays of a render: wherever its answer has
  a clear margin, the oracle's closest_hit_brute, which the GPU test holds the device to, names the same primitive.
- The lists' CPU statement on every camera of the sweep: list hits equal the ordered walk's, every key is a lower bound.
- A directed check of the frustum predicate: the corner rays of every pixel's jitter square, the extremes the sampler can
  produce, lie inside the pixel's frustum with the box growth switched off. Random jitter almost never comes within the
  error margins (sin_a, the uv margin) of a frustum edge, so this is the check that guards those margins.

The scenes, the id-coded palette, the camera sweep and the vectorised camera rays live here; the GPU test imports them."""
import copy
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scripts"))
import camcand_ref  # noqa: E402

from test_gpu_closest_hit import degenerate  # noqa: E402

F = np.float32
MISS = 0xFFFFFFFF

# ---- id-coded scenes ---------------------------------------------------------------------------------------------
# Every primitive is an emitter of strength 1 whose colour is PALETTE[id % P]; the sky is a colour outside the palette.
# Under the naive integrator a camera sample's radiance is then exactly the colour of its first hit, so a render's
# accumulator is a checksum of the first hits: one wrong sample moves its pixel's sum by PALETTE_STEP or more.
P = 61  # prime: consecutive ids and mesh neighbours (id strides that are no multiple of 61) get different colours
_LEVELS = (0.1, 0.35, 0.6, 0.85)
PALETTE = np.array([(r, g, b) for r in _LEVELS for g in _LEVELS for b in _LEVELS][:P], F)
SKY = np.array((0.0, 0.97, 0.0), F)


def colour_step():
    """Smallest difference, in the channel where they differ most, between two colours a sample can take."""
    c = np.concatenate([PALETTE, SKY[None]]).astype(np.float64)
    d = np.abs(c[:, None, :] - c[None, :, :]).max(axis=2)
    return float(d[~np.eye(len(c), dtype=bool)].min())


PALETTE_STEP = colour_step()


def id_coded(ptb, scene):
    s = copy.deepcopy(scene)
    s.textures = np.zeros(0, s.textures.dtype)
    s.materials = np.zeros(0, s.materials.dtype)
    s.texture_data = {}
    for c in PALETTE:
        s.add_material(ptb.MAT_EMIT, s.add_texture(ptb.TEX_SOLID, tuple(float(v) for v in c)), 1.0)
    s.set_sky(s.add_texture(ptb.TEX_SOLID, tuple(float(v) for v in SKY)), (0, 0))
    ns, nt = len(s.spheres), len(s.triangles)
    s.spheres["material"] = np.arange(ns) % P
    s.triangles["material"] = (ns + np.arange(nt)) % P
    return s


def colours(prims):
    """f64 colour of each first hit (primitive id or MISS)."""
    prims = np.asarray(prims)
    miss = prims == MISS
    out = PALETTE[np.where(miss, 0, prims) % P].astype(np.float64)
    out[miss] = SKY
    return out


def _tri(ptb, p, n=None):
    t = np.zeros(len(p), ptb._lib.triangle_dtype)
    t["p"] = p
    if n is None:
        e = np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]).astype(np.float64)
        ln = np.linalg.norm(e, axis=1, keepdims=True)
        n = np.where(ln > 0, e / np.where(ln > 0, ln, 1), (0, 0, 1))
        n = np.repeat(n[:, None, :], 3, axis=1)
    t["n"] = n
    return t


def c3(ptb, scale):
    return id_coded(ptb, ptb.meshgen.c3_scene(scale))


def moved(ptb, scene, shift, scale):
    """The scene and its camera under p -> p * scale + shift (in f64, rounded once)."""
    s = copy.deepcopy(scene)
    sh = np.asarray(shift, np.float64)
    s.triangles["p"] = (s.triangles["p"].astype(np.float64) * scale + sh).astype(F)
    s.spheres["center"] = (s.spheres["center"].astype(np.float64) * scale + sh).astype(F)
    s.spheres["radius"] = (s.spheres["radius"].astype(np.float64) * scale).astype(F)
    s.place = lambda p: tuple(float(v) for v in np.asarray(p, np.float64) * scale + sh)
    s.scale = scale
    return s


def shell(ptb):
    """(b) A closed, watertight UV-sphere shell of 4096 triangles (shared vertices, closed seam, exact poles) around the
    camera: every camera ray must hit it."""
    s = ptb.HostScene()
    p, n = ptb.meshgen.uv_sphere((0.3, -0.2, 0.1), 4.0, 64, 33)
    s.triangles = _tri(ptb, p, n)
    s.set_camera((0.0, 0.0, 0.0), (1.0, 0.7, 0.4), (0.0, 0.0, 1.0), 120.0, 16.0 / 9.0)
    return id_coded(ptb, s)


def spheres_and_ground(ptb):
    """(c) 2304 spheres of radius 0.08 in a 48 x 48 grid over a ground of 3200 triangles, and a radius-1000 ground
    sphere below it (the shipped scenes' case the cull slack of box_entry is sized for), seen beyond the ground's edge."""
    s = ptb.HostScene()
    g = np.linspace(-6.0, 6.0, 48)
    for x in g:
        for y in g:
            s.add_sphere((float(x), float(y), 0.12 + 0.05 * np.sin(3 * x + 2 * y)), 0.08, 0)
    s.add_sphere((0.0, 0.0, -1000.5), 1000.0, 0)
    xs = np.linspace(-7.0, 7.0, 41, dtype=F)
    X, Y = np.meshgrid(xs, xs, indexing="ij")
    Z = (F(0.03) * np.sin(F(1.7) * X) * np.cos(F(1.3) * Y)).astype(F)
    V = np.stack([X, Y, Z], -1)
    a, b, c, d = V[:-1, :-1], V[1:, :-1], V[1:, 1:], V[:-1, 1:]
    p = np.concatenate([np.stack([a, b, c], -2).reshape(-1, 3, 3), np.stack([a, c, d], -2).reshape(-1, 3, 3)])
    s.triangles = _tri(ptb, p.astype(F))
    s.set_camera((-1.0, -9.0, 2.5), (0.0, 0.0, 0.0), (0.0, 0.0, 1.0), 70.0, 16.0 / 9.0)
    return id_coded(ptb, s)


def hard_geometry(ptb):
    """(e) A base of 1600 triangles (a wavy wall in front of the camera at the origin) plus
    - coincident duplicates of 200 of them under other ids (the tie rule: the lower primitive id wins),
    - 300 zero-area triangles (repeated and collinear corners),
    - 300 slivers, 1e-4 wide, lying in planes through the camera origin or nearly so (seen edge-on),
    - 200 triangles whose planes pass exactly through the camera origin (z = 0, x = y: exact in f32).
    Fewer than 4096 primitives: the GPU test forces the list path."""
    rng = np.random.default_rng(7)
    xs = np.linspace(-3.0, 3.0, 21, dtype=F)
    zs = np.linspace(-2.0, 2.0, 21, dtype=F)
    X, Z = np.meshgrid(xs, zs, indexing="ij")
    Y = (F(4.0) + F(0.4) * np.sin(F(2.1) * X) * np.cos(F(1.7) * Z)).astype(F)
    V = np.stack([X, Y, Z], -1)
    a, b, c, d = V[:-1, :-1], V[1:, :-1], V[1:, 1:], V[:-1, 1:]
    base = np.concatenate([np.stack([a, b, c], -2).reshape(-1, 3, 3), np.stack([a, c, d], -2).reshape(-1, 3, 3)])
    dup = base[rng.choice(len(base), 200, replace=False)]
    z0 = rng.uniform(-2, 2, (150, 3)).astype(F) + np.array([0, 3, 0], F)
    ex = np.array([1, 0, 0], F)
    zero_area = np.concatenate([np.stack([z0, z0, z0 + F(0.3) * ex], 1),                # repeated corner
                                np.stack([z0, z0 + F(0.2) * ex, z0 + F(0.4) * ex], 1)])  # collinear: same y and z
    # slivers: long thin triangles whose plane contains (or nearly contains) the apex at the origin
    dirs = rng.normal(size=(300, 3))
    dirs[:, 1] = np.abs(dirs[:, 1]) + 1.5
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    side = np.cross(dirs, rng.normal(size=(300, 3)))
    side /= np.linalg.norm(side, axis=1, keepdims=True)
    near = rng.uniform(2.0, 3.0, 300)[:, None]
    far = near + 0.3
    sliver = np.stack([dirs * near, dirs * far, dirs * far + 1e-4 * side], 1).astype(F)
    # planes through the origin: z = 0 and x = y, corners exact in f32
    q = rng.uniform(0.5, 3.0, (100, 3, 2)).astype(F)
    in_z0 = np.stack([q[..., 0] - F(1.5), q[..., 1] + F(2.0), np.zeros_like(q[..., 0])], -1)
    in_xy = np.stack([q[..., 0] + F(1.0), q[..., 0] + F(1.0), q[..., 1] - F(1.5)], -1)
    p = np.concatenate([base, dup, zero_area, sliver, in_z0, in_xy]).astype(F)
    s = ptb.HostScene()
    s.triangles = _tri(ptb, p)
    s.set_camera((0.0, 0.0, 0.0), (0.2, 1.0, 0.1), (0.0, 0.0, 1.0), 80.0, 16.0 / 9.0)
    return id_coded(ptb, s)


# ---- the camera sweep --------------------------------------------------------------------------------------------
C3_CAM = ((0.0, -1.5, 1.6), (0.0, 4.0, 0.7), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0)
# C3 coordinates: (origin, lookat, vup, hfov, aspect, aperture, focus_dist). The axis views look exactly along an axis
# with an axis-aligned up vector: on odd image sizes the centre column and row straddle an octant boundary.
C3_SWEEP = {
    "c3": C3_CAM,
    "-z": ((0.0, 4.0, 5.0), (0.0, 4.0, 0.0), (0.0, 1.0, 0.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "-z_up_x": ((0.0, 4.0, 5.0), (0.0, 4.0, 0.0), (1.0, 0.0, 0.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "+z": ((0.0, 4.0, -1.0), (0.0, 4.0, 1.0), (0.0, 1.0, 0.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "+x": ((-5.0, 4.0, 1.0), (0.0, 4.0, 1.0), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "-x": ((5.0, 4.0, 1.0), (0.0, 4.0, 1.0), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "+y": ((0.0, -2.0, 1.0), (0.0, 4.0, 1.0), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "-y": ((0.0, 10.0, 1.2), (0.0, 4.0, 1.2), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0),
    "fov0.5": C3_CAM[:3] + (0.5,) + C3_CAM[4:],
    "fov170": C3_CAM[:3] + (170.0,) + C3_CAM[4:],
    "aspect1": C3_CAM[:4] + (1.0,) + C3_CAM[5:],
    "aperture": C3_CAM[:5] + (0.5, 3.0),  # the device camera is a pinhole: nothing may change
}


def in_leaf_camera(scene):
    """A camera at the centroid of a glass-sphere triangle of C3 (inside that primitive's leaf box), looking outwards."""
    t = scene.triangles[len(scene.triangles) - 137]["p"].astype(np.float64)
    o = t.mean(axis=0)
    return (tuple(o), tuple(o + (o - np.array([0.0, 4.0, 1.0]))), (0.0, 0.0, 1.0), 60.0, 16.0 / 9.0, 0.0, 1.0)


def with_camera(scene, cam):
    """A copy of `scene` under camera `cam` (C3 coordinates for a moved() scene)."""
    s = copy.deepcopy(scene)
    o, at, up, fov, aspect, aperture, focus = cam
    if hasattr(scene, "place"):
        o, at, focus = scene.place(o), scene.place(at), focus * scene.scale
    s.set_camera(o, at, up, fov, aspect, aperture, focus)
    return s


def axis_cameras(origin):
    """Views exactly along +-x, +-y, +-z from `origin`, each with an axis-aligned up vector."""
    o = np.asarray(origin, np.float64)
    out = {}
    for k, name in enumerate("xyz"):
        for sgn in (1.0, -1.0):
            e = np.zeros(3)
            e[k] = sgn
            up = (0.0, 0.0, 1.0) if k != 2 else (0.0, 1.0, 0.0)
            out[("+" if sgn > 0 else "-") + name] = (tuple(o), tuple(o + e), up, 70.0, 16.0 / 9.0, 0.0, 1.0)
    return out


# ---- camera rays, vectorised -------------------------------------------------------------------------------------
def camera_rays_np(ptb, scene, width, height, seed, samples, rows=None):
    """test_aov_oracle.camera_rays for every sample of `samples` at once, in the same f32 arithmetic: ray records
    (ray_dtype, un-normalised directions) of shape (len(rows) * width, len(samples)), pixels row-major."""
    cam = scene.camera[0]
    origin, ll, hor, ver = (np.asarray(cam[k], F) for k in ("origin", "lower_left", "horizontal", "vertical"))
    rows = np.arange(height) if rows is None else np.asarray(rows)
    y, x = np.meshgrid(rows.astype(np.uint64), np.arange(width, dtype=np.uint64), indexing="ij")
    pix = (y * np.uint64(width) + x).reshape(-1, 1)
    smp = np.asarray(samples, np.uint64).reshape(1, -1)
    pix, smp = np.broadcast_arrays(pix, smp)
    zero = np.zeros(pix.shape, np.uint64)
    r0, r1, _, _ = ptb.meshgen.philox4x32_10(pix, smp, zero, zero, seed & 0xFFFFFFFF, seed >> 32)
    xf = x.reshape(-1, 1).astype(F)
    yf = y.reshape(-1, 1).astype(F)
    u = ((r0 >> np.uint32(8)).astype(F) * F(1.0 / 16777216.0) + xf) / F(width - 1)
    v = F(1) - ((r1 >> np.uint32(8)).astype(F) * F(1.0 / 16777216.0) + yf) / F(height - 1)
    d = ll + hor * u[..., None] + ver * v[..., None] - origin
    out = np.zeros(u.shape, ptb.ray_dtype)
    out["o"] = origin
    out["d"] = d
    return out


def normalised(d):
    """Ray::new's f32 normalisation (ray.rs:13-46)."""
    d = np.asarray(d, F)
    return d / np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])[:, None]


def q1_rays(rays):
    """The reference's quirk Q1 (SURVEY.md): y-dominant rays with a vanishing x component (test_gpu_closest_hit)."""
    h = np.zeros(len(rays), [("t", F), ("prim", np.uint32)])
    return degenerate(rays, h, h)  # the same hits twice: no tie is flagged, only Q1


def q1_band(rays):
    """Rays Q1 can still affect: y-dominant with |dx| < 0.05 |dy|. The axis swap divides by dx, and the cancellation it
    causes loses hits well beyond the 1e-3 cut of q1_rays: inside the shell the reference misses y-dominant rays with
    |dx| up to 0.024 |dy| (never any other ray)."""
    d = np.abs(normalised(rays["d"]))
    ydom = ~((d[:, 0] > d[:, 1]) & (d[:, 0] > d[:, 2])) & (d[:, 1] > d[:, 2])
    return ydom & (d[:, 0] < 0.05 * d[:, 1])


# ---- f64 closest hit ---------------------------------------------------------------------------------------------
def closest_hit_f64(scene, rays, chunk=256):
    """Plain f64 closest hit over every primitive (Moller-Trumbore, the sphere quadratic) on the f32 rays (origin and
    f32-normalised direction up-cast). Returns (prim, clear): `clear` where the answer has a margin, i.e. the nearest
    hit lies more than 1e-5 inside every edge (barycentric; for a sphere, inside its silhouette by more than 1e-5 of the
    sphere's distance, the scale of the f32 test's error) and no
    other primitive hits or nearly hits (within 1e-5 outside an edge) within 1e-4 relative of its t. Misses are clear
    when no primitive nearly hits."""
    o_all = rays["o"].astype(np.float64)
    d_all = normalised(rays["d"]).astype(np.float64)
    sp, tr = scene.spheres, scene.triangles
    c, r2 = sp["center"].astype(np.float64), sp["radius"].astype(np.float64) ** 2
    p0, p1, p2 = (tr["p"][:, k].astype(np.float64) for k in range(3))
    e1, e2 = p1 - p0, p2 - p0
    ns = len(sp)
    prim = np.full(len(rays), MISS, np.uint32)
    clear = np.zeros(len(rays), bool)
    for a in range(0, len(rays), chunk):
        o, d = o_all[a:a + chunk, None, :], d_all[a:a + chunk, None, :]
        ts, ms = [], []
        if ns:
            oc = o - c[None]
            b = np.einsum("rnk,rnk->rn", oc, np.broadcast_to(d, oc.shape))
            perp2 = np.einsum("rnk,rnk->rn", oc, oc) - b * b
            ocn = np.sqrt(np.einsum("rnk,rnk->rn", oc, oc))
            m = (np.sqrt(r2)[None] - np.sqrt(np.maximum(perp2, 0.0))) / np.maximum(np.sqrt(r2)[None], ocn)
            sq = np.sqrt(np.maximum(r2[None] - perp2, 0.0))
            t0, t1 = -b - sq, -b + sq
            t = np.where(t0 > 0, t0, np.where(t1 > 0, t1, np.nan))
            ts.append(t)
            ms.append(m)
        if len(tr):
            pv = np.cross(np.broadcast_to(d, (d.shape[0], len(tr), 3)), e2[None])
            det = np.einsum("nk,rnk->rn", e1, pv)
            with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
                inv = 1.0 / det
                tv = o - p0[None]
                u = np.einsum("rnk,rnk->rn", tv, pv) * inv
                qv = np.cross(tv, e1[None])
                v = np.einsum("rnk,rnk->rn", np.broadcast_to(d, qv.shape), qv) * inv
                t = np.einsum("nk,rnk->rn", e2, qv) * inv
            with np.errstate(invalid="ignore"):
                m = np.minimum(np.minimum(u, v), 1.0 - u - v)
            bad = ~np.isfinite(m) | ~np.isfinite(t) | (det == 0)
            ts.append(np.where(bad, np.nan, t))
            ms.append(np.where(bad, -np.inf, m))
        t = np.concatenate(ts, axis=1)
        m = np.concatenate(ms, axis=1)
        cand = (t > 0) & (m > -1e-5)  # hits and near hits
        hit = cand & (m >= 0)
        th = np.where(hit, t, np.inf)
        best = np.argmin(th, axis=1)
        tb = th[np.arange(len(th)), best]
        has = np.isfinite(tb)
        prim[a:a + chunk] = np.where(has, best, MISS)
        tc = np.where(cand, t, np.inf)
        tc[np.arange(len(tc)), best] = np.where(has, np.inf, tc[np.arange(len(tc)), best])
        second = tc.min(axis=1)
        mb = m[np.arange(len(m)), best]
        clear[a:a + chunk] = np.where(has, (mb > 1e-5) & (second > tb * (1 + 1e-4)), ~cand.any(axis=1))
    return prim, clear


# ---- tests -------------------------------------------------------------------------------------------------------
def test_palette_step():
    assert len(PALETTE) == P and PALETTE_STEP >= 0.05


def test_vectorised_camera_rays_equal_camera_rays(ptb, orc):
    from test_aov_oracle import camera_rays
    s = with_camera(c3(ptb, 0.05), C3_SWEEP["fov170"])
    w, h, seed = 37, 23, 0x1234_5678_9ABC
    rows = [0, 7, 11, 22]  # 148 pixels per sample, 3 samples
    for sample in (0, 5, 1000):
        ref = camera_rays(ptb, orc, s, w, h, seed, sample, rows=rows)
        got = camera_rays_np(ptb, s, w, h, seed, [sample], rows=rows)[:, 0]
        assert np.array_equal(ref["o"].view(np.uint32), got["o"].view(np.uint32))
        assert np.array_equal(ref["d"].view(np.uint32), got["d"].view(np.uint32))


def _subsample(rays, n, seed):
    rays = rays.reshape(-1)
    return rays[np.random.default_rng(seed).choice(len(rays), min(n, len(rays)), replace=False)]


@pytest.mark.parametrize("name", ["shell", "spheres_and_ground", "hard_geometry"])
def test_oracle_brute_force_equals_f64_closest_hit(ptb, orc, name):
    """closest_hit_brute (f32, the reference's arithmetic) names the primitive an independent f64 intersector finds,
    wherever that answer has a clear margin, on 20 000 camera rays of the scene under three of its cameras."""
    scene = {"shell": shell, "spheres_and_ground": spheres_and_ground, "hard_geometry": hard_geometry}[name](ptb)
    cams = [None] + list(axis_cameras(scene.camera[0]["origin"]).values())[::2]
    rays = []
    for i, cam in enumerate(cams):
        s = scene if cam is None else with_camera(scene, cam)
        rays.append(_subsample(camera_rays_np(ptb, s, 64, 36, 0xC0FFEE + i, range(8)), 5000, i))
    rays = np.concatenate(rays)
    got = orc.OracleScene(scene).closest_hit_brute(rays)["prim"]
    ref, clear = closest_hit_f64(scene, rays)
    q1, band = q1_rays(rays), q1_band(rays)
    ok = clear & ~band
    bad = np.flatnonzero(ok & (got != ref))
    lost = int((clear & band & (got != ref)).sum())
    print(f"{name}: {len(rays)} rays, {int(ok.sum())} compared, {int(q1.sum())} Q1 rays and {int(band.sum())} in the Q1 "
          f"band excluded ({lost} of these differ from the f64 answer), {int((got != MISS).sum())} hits")
    assert ok.sum() > 0.8 * len(rays)
    assert bad.size == 0, (bad[:10], got[bad[:10]], ref[bad[:10]])
    if name == "shell":
        assert np.all(got[~band] != MISS)  # watertight: only Q1 lets a ray through


@pytest.fixture(scope="module")
def sweep_scenes(ptb):
    base = c3(ptb, 0.05)
    out = [(f"c3/{k}", with_camera(base, cam)) for k, cam in C3_SWEEP.items()]
    out.append(("c3/in_leaf", with_camera(base, in_leaf_camera(base))))
    for shift, scale in (((1e4, -3e3, 5e3), 1.0), ((0.0, 0.0, 0.0), 1e-3), ((0.0, 0.0, 0.0), 1e3)):
        m = moved(ptb, base, shift, scale)
        for k in ("c3", "-z", "+x", "fov0.5"):
            out.append((f"moved{shift}x{scale}/{k}", with_camera(m, C3_SWEEP[k])))
    for name, fn in (("shell", shell), ("spheres_and_ground", spheres_and_ground), ("hard_geometry", hard_geometry)):
        s = fn(ptb)
        out.append((f"{name}/own", s))
        for k, cam in axis_cameras(s.camera[0]["origin"]).items():
            out.append((f"{name}/{k}", with_camera(s, cam)))
    return out


@pytest.mark.parametrize("W,H", [(33, 17), (2, 2)])
def test_camera_sweep_lists_equal_the_ordered_walk(sweep_scenes, W, H):
    """The CPU statement of the lists on every camera of the sweep: list hits equal the ordered walk's bit for bit, no
    list-answered hit lies in a leaf box the walk rejects, and every key bounds its entry's cull key from below."""
    for name, s in sweep_scenes:
        S = camcand_ref.CamCandScene(s)
        L = S.lists(W, H, 16)
        r = S.check(L, spp=32, sample_offset=3, seed=5)
        print(f"{name}: overflow {L.overflowed.mean():.2f}, list rays {r['list_rays']} / {r['rays']}")
        assert r["mismatches"] == 0 and r["box_rejected_hits"] == 0 and r["key_above_tkey"] == 0, (name, r)


# Distances along each corner ray, in units of its distance from the apex to the image plane.
CORNER_DISTANCES = np.array([1.0, 1.5, 4.0, 10.0, 100.0, 1e3, 1e4])


@pytest.mark.parametrize("W,H", [(33, 17), (157, 91), (2, 2)])
def test_frustum_holds_the_corner_rays_of_every_pixel(sweep_scenes, W, H):
    """Argument (b) of ptb_camcand.cuh on its own: the corner rays of each pixel's jitter square, as the device computes
    them, pass the pixel's side planes and lie ahead of the apex at every distance, with no box growth to hide an
    error. Without sin_a (or with a smaller bound) the cameras whose direction sums round coarsely fail here."""
    worst = {}
    for name, s in sweep_scenes:
        r = camcand_ref.CamCandScene(s).frustum_corners(W, H, CORNER_DISTANCES)
        assert r["boxes"] == W * H * 4 * len(CORNER_DISTANCES)
        assert r["side_rejected"] == 0 and r["behind_rejected"] == 0, (name, r)
        worst[name] = r["worst"]
    print({k: round(v, 3) for k, v in worst.items()})
