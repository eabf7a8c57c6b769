"""CPU: the oracle's visibility queries (oracle/visibility_api.cpp: the reference's check_hit_index, acceleration/mod.rs:226-263,
and its blocker scan as an occlusion query), which the device's batch visibility API is compared against, agree with a
brute-force scan and with the oracle's closest hit."""
import copy

import numpy as np

from conftest import random_rays
from visibility_oracle import VisibilityOracle

MISS = 0xFFFFFFFF


def mixed_scene(ptb, base, n_spheres, n_tris, seed):
    """A random scene of spheres and triangles of many sizes, some overlapping, in [-2, 2]^3 (materials of `base`)."""
    rng = np.random.default_rng(seed)
    s = copy.deepcopy(base)
    sp = np.zeros(n_spheres, ptb._lib.sphere_dtype)
    sp["center"] = rng.uniform(-2, 2, (n_spheres, 3))
    sp["radius"] = rng.uniform(0.02, 0.5, n_spheres)
    tr = np.zeros(n_tris, ptb._lib.triangle_dtype)
    c = rng.uniform(-2, 2, (n_tris, 1, 3))
    p = (c + rng.normal(0, 0.3, (n_tris, 3, 3))).astype(np.float32)
    tr["p"] = p
    fn = np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0])
    fn /= np.maximum(np.linalg.norm(fn, axis=1, keepdims=True), 1e-12)
    tr["n"] = fn[:, None, :]
    s.spheres, s.triangles = sp, tr
    return s


def target_points(ptb, scene, ids, rng):
    """A random point on each target primitive (original ids: spheres first, then triangles)."""
    ns = len(scene.spheres)
    pts = np.zeros((len(ids), 3), np.float64)
    sph = ids < ns
    if sph.any():
        s = scene.spheres[ids[sph]]
        u = rng.normal(size=(int(sph.sum()), 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        pts[sph] = s["center"] + s["radius"][:, None] * u
    if (~sph).any():
        t = scene.triangles[ids[~sph] - ns]["p"].astype(np.float64)
        a, b = rng.uniform(size=(2, int((~sph).sum()), 1))
        flip = (a + b) > 1
        a, b = np.where(flip, 1 - a, a), np.where(flip, 1 - b, b)
        pts[~sph] = t[:, 0] + a * (t[:, 1] - t[:, 0]) + b * (t[:, 2] - t[:, 0])
    return pts


def target_rays(ptb, scene, n, seed, centre=(0, 0, 0), radius=3.0):
    """Half of the rays run from random points towards a sampled point on a random target primitive (many are visible),
    half are random rays with a random target (most miss it). Returns (rays, target ids)."""
    rng = np.random.default_rng(seed)
    n_prims = scene.n_primitives
    ids = rng.integers(0, n_prims, n).astype(np.uint32)
    rays = random_rays(ptb, n, seed, centre=centre, radius=radius)
    h = n // 2
    pts = target_points(ptb, scene, ids[:h], rng)
    d = (pts - rays["o"][:h]).astype(np.float32)
    ok = np.linalg.norm(d, axis=1) > 1e-3
    rays["d"][:h][ok] = d[ok]
    return rays, ids


def target_t(ptb, scene, rays, ids):
    """f64 distance along the normalised direction at which each ray meets its own target (nan: it does not). For stating
    how the rays divide into visible / blocked / target missed; never compared bit for bit."""
    o = rays["o"].astype(np.float64)
    d = rays["d"].astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    t = np.full(len(rays), np.nan)
    ns = len(scene.spheres)
    sph = ids < ns
    s = scene.spheres[ids[sph]]
    oc = o[sph] - s["center"]
    b = np.einsum("ij,ij->i", oc, d[sph])
    disc = b * b - (np.einsum("ij,ij->i", oc, oc) - s["radius"].astype(np.float64) ** 2)
    sq = np.sqrt(np.maximum(disc, 0))
    t0, t1 = -b - sq, -b + sq
    ts = np.where(t0 > 0, t0, np.where(t1 > 0, t1, np.nan))
    t[sph] = np.where(disc >= 0, ts, np.nan)
    p = scene.triangles[ids[~sph] - ns]["p"].astype(np.float64)
    e1, e2 = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
    dd, oo = d[~sph], o[~sph]
    pv = np.cross(dd, e2)
    det = np.einsum("ij,ij->i", e1, pv)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = 1.0 / det
        tv = oo - p[:, 0]
        u = np.einsum("ij,ij->i", tv, pv) * inv
        qv = np.cross(tv, e1)
        v = np.einsum("ij,ij->i", dd, qv) * inv
        tt = np.einsum("ij,ij->i", e2, qv) * inv
    hit = (np.abs(det) > 1e-14) & (u >= 0) & (v >= 0) & (u + v <= 1) & (tt > 0)
    t[~sph] = np.where(hit, tt, np.nan)
    return t


def occlusion_rays(ptb, rays, tmax, exclude):
    return ptb.make_occlusion_rays(rays["o"], rays["d"], tmax, exclude)


def test_occluded_matches_brute_force_on_mixed_scenes(ptb, orc, rtweekend1):
    for seed, (ns, nt) in enumerate([(40, 200), (300, 50), (5, 1500)]):
        s = mixed_scene(ptb, rtweekend1, ns, nt, seed)
        o = VisibilityOracle(s)
        rays = random_rays(ptb, 20_000, 100 + seed, radius=3.0)
        c = orc.OracleScene(s).closest_hit(rays)
        rng = np.random.default_rng(seed)
        n = len(rays)
        tmax = np.where(rng.uniform(size=n) < 0.3, np.inf, rng.uniform(0, 6, n)).astype(np.float32)
        exclude = np.where(rng.uniform(size=n) < 0.5, c["prim"], rng.integers(0, s.n_primitives + 5, n)).astype(np.uint32)
        q = occlusion_rays(ptb, rays, tmax, exclude)
        a, b = o.occluded(q), o.occluded(q, brute=True)
        assert np.array_equal(a, b), int((a != b).sum())
        assert 0.1 < a.mean() < 0.9
        # no exclusion, tmax = +inf: "does the ray hit anything" == closest hit found something
        q = occlusion_rays(ptb, rays, np.inf, MISS)
        assert np.array_equal(o.occluded(q), c["prim"] != MISS)
        # tmax <= 0 or NaN: never occluded
        for t in (0.0, -1.0, np.nan):
            assert not o.occluded(occlusion_rays(ptb, rays, t, MISS)).any()


def test_check_hit_index_of_the_closest_primitive_is_the_closest_hit(ptb, orc, rtweekend1, overshadowed):
    for s in (rtweekend1, overshadowed, mixed_scene(ptb, rtweekend1, 50, 400, 7)):
        o = VisibilityOracle(s)
        rays = random_rays(ptb, 20_000, 9, radius=3.0)
        c = orc.OracleScene(s).closest_hit(rays)
        hit = c["prim"] != MISS
        assert hit.mean() > 0.05
        r = o.check_hit_index(rays[hit], c["prim"][hit])
        for f in ("t", "prim", "u", "v"):
            assert np.array_equal(r[f].view(np.uint32), c[f][hit].view(np.uint32)), f


def test_check_hit_index_mix_and_out_of_range_targets(ptb, rtweekend1):
    s = mixed_scene(ptb, rtweekend1, 20, 60, 3)
    o = VisibilityOracle(s)
    rays, ids = target_rays(ptb, s, 20_000, 5)
    r = o.check_hit_index(rays, ids)
    vis = r["prim"] != MISS
    assert np.array_equal(r["prim"][vis], ids[vis]) and np.all(r["t"][vis] > 0)
    assert np.all(r["t"][~vis] == 0) and np.all(r["u"][~vis] == 0) and np.all(r["v"][~vis] == 0)
    tt = target_t(ptb, s, rays, ids)
    missed = np.isnan(tt)
    assert vis.mean() > 0.2 and (~vis & ~missed).mean() > 0.1 and missed.mean() > 0.2
    for bad in (s.n_primitives, s.n_primitives + 1, MISS - 1, MISS):
        out = o.check_hit_index(rays[:1000], np.full(1000, bad, np.uint32))
        assert np.all(out["prim"] == MISS) and np.all(out["t"] == 0)
