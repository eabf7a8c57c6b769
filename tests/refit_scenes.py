"""Moved versions of the test scenes for the refit tests (PTB_BUILD_REFIT): same primitive counts and order, new geometry."""
import copy

import numpy as np

F = np.float32


def move_spheres(scene, seed=1):
    """rtweekend1-style scene: every sphere but the ground (index 0) moved by up to 0.5 and resized by 0.5x..1.5x."""
    s = copy.deepcopy(scene)
    rng = np.random.default_rng(seed)
    sp = s.spheres
    k = np.arange(len(sp)) != 0
    sp["center"][k] += rng.uniform(-0.5, 0.5, (k.sum(), 3)).astype(F)
    sp["radius"][k] *= rng.uniform(0.5, 1.5, k.sum()).astype(F)
    return s


def scatter(scene, seed=2, extent=None):
    """Worst case for a kept tree: every primitive moved by its own random offset across the whole scene box."""
    s = copy.deepcopy(scene)
    rng = np.random.default_rng(seed)
    if extent is None:
        pts = [s.spheres["center"].reshape(-1, 3), s.triangles["p"].reshape(-1, 3)]
        pts = np.concatenate([p for p in pts if len(p)])
        extent = float(np.max(pts.max(0) - pts.min(0))) / 2
    if len(s.spheres):
        s.spheres["center"] += rng.uniform(-extent, extent, (len(s.spheres), 3)).astype(F)
    if len(s.triangles):
        s.triangles["p"] += rng.uniform(-extent, extent, (len(s.triangles), 1, 3)).astype(F)
    return s


def leaf_boxes(scene, prim_ids):
    """f32 boxes of the given original primitive ids, as Prim::aabb / k_prim_bounds compute them."""
    ns = len(scene.spheres)
    mn = np.zeros((len(prim_ids), 3), F)
    mx = np.zeros((len(prim_ids), 3), F)
    sph = prim_ids < ns
    if sph.any():
        sp = scene.spheres[prim_ids[sph]]
        r = sp["radius"][:, None].astype(F)
        mn[sph] = sp["center"] - r * np.ones(3, F)
        mx[sph] = sp["center"] + r * np.ones(3, F)
    if (~sph).any():
        p = scene.triangles["p"][prim_ids[~sph] - ns]
        mn[~sph] = np.minimum(p[:, 0], np.minimum(p[:, 1], p[:, 2]))
        mx[~sph] = np.maximum(p[:, 0], np.maximum(p[:, 1], p[:, 2]))
    return mn, mx


def sah_cost(nodes, n_prims):
    """numpy f64 statement of ptb_bvh_sah_cost over exported nodes."""
    if n_prims == 0:
        return 0.0
    leaf = 0x80000000

    def area(mn, mx):
        d = mx.astype(np.float64) - mn.astype(np.float64)
        return 2.0 * (d[:, 0] * d[:, 1] + d[:, 1] * d[:, 2] + d[:, 2] * d[:, 0])

    umn, umx = np.minimum(nodes["lmin"], nodes["rmin"]), np.maximum(nodes["lmax"], nodes["rmax"])
    total = 0.125 * area(umn, umx).sum()
    total += area(nodes["lmin"], nodes["lmax"])[nodes["left"] >= leaf].sum()
    if n_prims > 1:
        total += area(nodes["rmin"], nodes["rmax"])[nodes["right"] >= leaf].sum()
    root = area(umn[:1], umx[:1])[0]
    return float(total / root) if root > 0 else 0.0
