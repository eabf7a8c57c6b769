"""The CPU statement of PTB_BUILD_REFIT (oracle/refit_api.cpp): a kept binary tree whose boxes are recomputed for moved
primitives.

  * a refit of unchanged primitives reproduces the build's nodes bit for bit, and the tree it starts from is the one the
    LBVH / SAH oracles build;
  * after motion the topology and primitive order are untouched, every leaf box is Prim::aabb of the new primitive and every
    node box is exactly the union of its children's boxes;
  * hits through the refitted tree equal the f32 brute force over every primitive.
"""
import copy

import numpy as np
import pytest

from conftest import random_rays
from refit_scenes import leaf_boxes, move_spheres, scatter

LEAF = 0x80000000
MISS = 0xFFFFFFFF


def small_spheres(ptb, rtweekend1, n, seed=3):
    s = copy.deepcopy(rtweekend1)
    rng = np.random.default_rng(seed)
    sp = np.zeros(n, ptb._lib.sphere_dtype)
    sp["center"] = rng.uniform(-3, 3, (n, 3)).astype(np.float32)
    sp["radius"] = rng.uniform(0.05, 0.4, n).astype(np.float32)
    s.spheres = sp
    return s


def scenes(ptb, rtweekend1, overshadowed):
    return {"rtweekend1": rtweekend1, "overshadowed": overshadowed, "c3": ptb.meshgen.c3_scene(0.05),
            "one": small_spheres(ptb, rtweekend1, 1), "two": small_spheres(ptb, rtweekend1, 2)}


def same_nodes(a, b):
    for f in ("left", "right", "parent"):
        assert np.array_equal(a[f], b[f]), f
    for f in ("lmin", "lmax", "rmin", "rmax"):
        assert np.array_equal(a[f].view(np.uint32), b[f].view(np.uint32)), f


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3", "one", "two"])
def test_refit_of_unchanged_primitives_reproduces_the_build(ptb, orc, rtweekend1, overshadowed, builder, which):
    from refit_oracle import RefitOracle
    scene = scenes(ptb, rtweekend1, overshadowed)[which]
    r = RefitOracle(scene, builder)
    m0, p0, n0 = r.export()
    o = orc.OracleScene(scene, split_type=-1)
    if builder == "sah":
        o.lbvh_sah()
    om, op, on = o.lbvh_export()
    assert np.array_equal(m0, om) and np.array_equal(p0, op)
    same_nodes(n0, on)
    r.refit(scene)
    m1, p1, n1 = r.export()
    assert np.array_equal(m1, m0) and np.array_equal(p1, p0)
    same_nodes(n1, n0)


def check_refitted(scene, prims, nodes, n):
    """Leaf boxes are the new primitives' boxes, node boxes the unions of their children's (bitwise)."""
    u = lambda a: a.view(np.uint32)
    for side, mn, mx in (("left", "lmin", "lmax"), ("right", "rmin", "rmax")):
        ch = nodes[side]
        leaf = ch >= LEAF
        bmn, bmx = leaf_boxes(scene, prims[ch[leaf] & 0x3FFFFFFF].astype(np.int64))
        assert np.array_equal(u(nodes[mn][leaf]), u(bmn)) and np.array_equal(u(nodes[mx][leaf]), u(bmx)), side
        c = nodes[ch[~leaf]]
        assert np.array_equal(u(nodes[mn][~leaf]), u(np.minimum(c["lmin"], c["rmin"]))), side
        assert np.array_equal(u(nodes[mx][~leaf]), u(np.maximum(c["lmax"], c["rmax"]))), side
    assert np.array_equal(np.sort(prims), np.arange(n, dtype=np.uint32))


def moved(ptb, which, scene):
    if which == "c3":
        return ptb.meshgen.c3_deform(scene, 0.5, 1.0)
    if which in ("rtweekend1", "one", "two"):
        return move_spheres(scene)
    return scatter(scene)


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3", "c3_scatter", "one", "two"])
def test_refit_after_motion(ptb, orc, rtweekend1, overshadowed, builder, which):
    from refit_oracle import RefitOracle
    base = scenes(ptb, rtweekend1, overshadowed)["c3" if which == "c3_scatter" else which]
    new = scatter(base) if which == "c3_scatter" else moved(ptb, which, base)
    r = RefitOracle(base, builder)
    m0, p0, n0 = r.export()
    r.refit(new)
    m1, p1, n1 = r.export()
    assert np.array_equal(m1, m0) and np.array_equal(p1, p0)
    for f in ("left", "right", "parent"):
        assert np.array_equal(n1[f], n0[f]), f
    n = base.n_primitives
    check_refitted(new, p1, n1, n)
    # hits through the refitted tree == f32 brute force over every primitive of the moved scene
    centre, radius = {"rtweekend1": ((0, 1, 0), 3.0), "overshadowed": ((-0.3, 0.3, -0.3), 1.5), "one": ((0, 0, 0), 3.0),
                      "two": ((0, 0, 0), 3.0)}.get(which, ((0, 4, 1), 5.0))
    rays = random_rays(ptb, 20_000, 61, centre=centre, radius=radius)
    h, nodes_fetched, prims_tested = r.closest_hit(rays)
    b = orc.OracleScene(new, split_type=-1).closest_hit_brute(rays)
    tie = (h["prim"] != b["prim"]) & (h["t"] == b["t"])
    assert tie.mean() < 1e-3 and np.array_equal(h["prim"][~tie], b["prim"][~tie])
    assert np.array_equal(h["t"].view(np.uint32), b["t"].view(np.uint32))
    assert (h["prim"] != MISS).any() and nodes_fetched > 0 and prims_tested > 0


def test_refit_rejects_other_counts(ptb, rtweekend1):
    from refit_oracle import RefitOracle
    r = RefitOracle(rtweekend1)
    s = copy.deepcopy(rtweekend1)
    s.spheres = s.spheres[:-1]
    with pytest.raises(ValueError):
        r.refit(s)
