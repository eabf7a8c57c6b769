"""Dynamic scenes through the C ABI: ptb_scene_update_* and ptb_scene_commit(PTB_BUILD_REFIT), which keeps the binary tree
of the last full commit and refits its boxes (lbvh_build.cu k_refit_slots), and ptb_bvh_sah_cost.

  * tree: a refit of unchanged primitives changes no bit of the export or the SAH cost; after motion the device tree is the
    CPU refit (oracle/refit_api.cpp) bit for bit, topology and primitive order untouched;
  * hits and queries: closest hit, check_hit_index and occlusion equal a fresh commit of the moved scene bit for bit, and
    the reference-semantics oracle as the SAH tests check it; traversal counts match the CPU walk over the refitted tree;
  * render: after an emitter moves, a primitive turns emissive (or back), or only the camera changes, the image and every
    ray counter equal a fresh commit's;
  * update paths (host, device from a torch tensor, partial ranges), the full-size C3, the SAH cost, and every error.
"""
import copy

import numpy as np
import pytest

from conftest import random_rays
from refit_scenes import move_spheres, sah_cost, scatter

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF
LEAF = 0x80000000
SPHERE_BIT = np.uint32(0x40000000)
BUILDERS = ["lbvh", "sah"]
VIEW = {"rtweekend1": ((0, 1, 0), 3.0), "overshadowed": ((-0.3, 0.3, -0.3), 1.5), "c3": ((0, 4, 1), 5.0),
        "c3_scatter": ((0, 4, 1), 5.0)}


def flag(ptb, builder):
    return {"lbvh": ptb._lib.BUILD_BINARY, "sah": ptb._lib.BUILD_SAH}[builder]


@pytest.fixture()
def ctx2(ptb):
    """A second context: the fresh commit beside the refitted one."""
    c = ptb.Context(0)
    yield c
    c.close()


def base_and_moved(ptb, rtweekend1, overshadowed, which):
    if which == "rtweekend1":
        return rtweekend1, move_spheres(rtweekend1)
    if which == "overshadowed":
        s = copy.deepcopy(overshadowed)
        s.spheres["center"][1] += np.float32([0.2, 0.1, -0.15])           # the emitter
        s.triangles["p"] += np.float32([0.05, 0.02, 0.0])                  # the box
        return overshadowed, s
    base = ptb.meshgen.c3_scene(0.05)
    if which == "c3":
        return base, ptb.meshgen.c3_deform(base, 0.5, 1.0)               # terrain wave, glass sphere pushed into it
    return base, scatter(base)                                          # worst case: every primitive somewhere else


def refit_to(ptb, ctx, base, new, builder):
    """Full commit of `base`, then the camera and primitives of `new` (host update path) and a refit."""
    ctx.upload(base)
    ctx.commit(flag(ptb, builder))
    assert ptb._lib.lib.ptb_scene_set_camera(ctx._h, ptb._lib.ptr(new.camera)) == 0
    if len(new.spheres):
        ctx.update_spheres(0, new.spheres)
    if len(new.triangles):
        ctx.update_triangles(0, new.triangles)
    ctx.commit(ptb._lib.BUILD_REFIT)


def strip(nodes):
    out = nodes.copy()
    for f in ("left", "right"):
        leaf = out[f] >= LEAF
        out[f][leaf] &= ~SPHERE_BIT
    return out


def same_export(a, b):
    (ma, pa, na), (mb, pb, nb) = a, b
    assert np.array_equal(ma, mb) and np.array_equal(pa, pb)
    na, nb = strip(na), strip(nb)
    for f in ("left", "right", "parent"):
        assert np.array_equal(na[f], nb[f]), f
    for f in ("lmin", "lmax", "rmin", "rmax"):
        assert np.array_equal(na[f].view(np.uint32), nb[f].view(np.uint32)), f


def same_hits(a, b):
    for f in ("prim", "t", "u", "v"):
        assert np.array_equal(a[f].view(np.uint32), b[f].view(np.uint32)), f


def check_tree(nodes, prims, n):
    assert np.array_equal(np.sort(prims), np.arange(n, dtype=np.uint32))
    refs = np.concatenate([nodes["left"], nodes["right"]])
    assert np.array_equal(np.sort(refs[refs >= LEAF] & 0x3FFFFFFF), np.arange(n, dtype=np.uint32))
    assert np.array_equal(np.sort(refs[refs < LEAF]), np.arange(1, len(nodes), dtype=np.uint32))
    for side, mn, mx in (("left", "lmin", "lmax"), ("right", "rmin", "rmax")):
        ch = nodes[side]
        m = ch < LEAF
        assert np.array_equal(nodes["parent"][ch[m]], np.nonzero(m)[0].astype(np.uint32))
        c = nodes[ch[m]]
        assert np.array_equal(nodes[mn][m], np.minimum(c["lmin"], c["rmin"])) and np.array_equal(nodes[mx][m], np.maximum(c["lmax"], c["rmax"]))


# ------------------------------------------------------------------------------------------------------------ tree
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3"])
def test_refit_of_unchanged_primitives_changes_nothing(ptb, gpu_ctx, rtweekend1, overshadowed, builder, which):
    base, _ = base_and_moved(ptb, rtweekend1, overshadowed, which)
    gpu_ctx.upload(base)
    gpu_ctx.commit(flag(ptb, builder))
    before, cost = gpu_ctx.bvh_export(), gpu_ctx.bvh_sah_cost()
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx.bvh_export(), before)
    assert gpu_ctx.bvh_sah_cost() == cost
    assert gpu_ctx.bvh_builder()[0] == flag(ptb, builder)


@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3", "c3_scatter"])
def test_refit_matches_the_cpu_refit(ptb, gpu_ctx, rtweekend1, overshadowed, builder, which):
    from refit_oracle import RefitOracle
    base, new = base_and_moved(ptb, rtweekend1, overshadowed, which)
    gpu_ctx.upload(base)
    gpu_ctx.commit(flag(ptb, builder))
    m0, p0, n0 = gpu_ctx.bvh_export()
    refit_to(ptb, gpu_ctx, base, new, builder)
    m1, p1, n1 = gpu_ctx.bvh_export()
    assert np.array_equal(m1, m0) and np.array_equal(p1, p0)
    for f in ("left", "right", "parent"):
        assert np.array_equal(n1[f], n0[f]), f
    r = RefitOracle(base, builder)
    r.refit(new)
    same_export((m1, p1, n1), r.export())
    check_tree(strip(n1), p1, base.n_primitives)


# ------------------------------------------------------------------------------------------------ hits and queries
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3", "c3_scatter"])
def test_refit_queries_equal_a_fresh_commit(ptb, orc, gpu_ctx, ctx2, rtweekend1, overshadowed, builder, which):
    from refit_oracle import RefitOracle
    base, new = base_and_moved(ptb, rtweekend1, overshadowed, which)
    centre, radius = VIEW[which]
    rays = random_rays(ptb, 200_000, 71, centre=centre, radius=radius)
    refit_to(ptb, gpu_ctx, base, new, builder)
    ctx2.upload(new)
    ctx2.commit(flag(ptb, builder))
    gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 1)
    gpu_ctx.stats_reset()
    g = gpu_ctx.closest_hit(rays)
    st = gpu_ctx.stats()
    gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 0)
    same_hits(g, ctx2.closest_hit(rays))
    # the reference's own tree and walk
    r = orc.OracleScene(new).closest_hit(rays)
    tie = (g["prim"] != r["prim"]) & (g["t"] == r["t"])
    assert tie.mean() < 1e-3 and np.array_equal(g["prim"][~tie], r["prim"][~tie])
    assert np.array_equal(g["t"][~tie].view(np.uint32), r["t"][~tie].view(np.uint32))
    # the CPU walk over the same refitted tree: same hits, the device speculates a few percent more
    ro = RefitOracle(base, builder)
    ro.refit(new)
    h, nodes, prims = ro.closest_hit(rays)
    assert np.array_equal(h["prim"], g["prim"])
    assert st.rays_counted == len(rays)
    v_cpu, t_cpu = nodes / len(rays), prims / len(rays)
    v_dev, t_dev = st.nodes_fetched / len(rays), st.prims_tested / len(rays)
    assert v_cpu <= v_dev <= 1.10 * v_cpu + 0.05, (v_dev, v_cpu)
    assert t_cpu <= t_dev <= 1.25 * t_cpu + 0.05, (t_dev, t_cpu)
    # visibility queries
    n = new.n_primitives
    rng = np.random.default_rng(5)
    index = np.where(g["prim"] != MISS, g["prim"], rng.integers(0, n, len(rays))).astype(np.uint32)
    index[::7] = rng.integers(0, n, len(index[::7]))
    same_hits(gpu_ctx.check_hit_index(rays, index), ctx2.check_hit_index(rays, index))
    occ = ptb.make_occlusion_rays(rays["o"], rays["d"], tmax=rng.uniform(0.0, 2 * radius, len(rays)).astype(np.float32),
                                  exclude=np.where(rng.random(len(rays)) < 0.5, index, MISS).astype(np.uint32))
    a, b = gpu_ctx.occluded(occ), ctx2.occluded(occ)
    assert np.array_equal(a, b) and a.any() and not a.all()


# ------------------------------------------------------------------------------------------------------------ render
def render_pair(ptb, ctx_refit, ctx_fresh, base, new, builder, method):
    refit_to(ptb, ctx_refit, base, new, builder)
    ctx_fresh.upload(new)
    ctx_fresh.commit(flag(ptb, builder))
    o = ptb.RenderOptions(samples_per_pixel=16, render_method=method, width=160, height=90, seed=4)
    res = []
    for ctx in (ctx_refit, ctx_fresh):
        ctx.accum_clear()
        ctx.stats_reset()
        ctx.render(o)
        st = ctx.stats()
        res.append((ctx.accum_read(160, 90).copy(),
                    (st.rays_camera, st.rays_bounce, st.rays_shadow_light, st.rays_shadow_sky, st.rays_reference, st.paths)))
    assert np.allclose(res[0][0], res[1][0], rtol=1e-5, atol=1e-5)
    assert res[0][1] == res[1][1]
    return res[0][0]


@pytest.mark.parametrize("method", [0, 1])
@pytest.mark.parametrize("change", ["emitter_moves", "turns_emissive", "camera_only"])
def test_refit_renders_as_a_fresh_commit(ptb, gpu_ctx, ctx2, overshadowed, change, method):
    base = overshadowed
    new = copy.deepcopy(base)
    if change == "emitter_moves":
        new.spheres["center"][1] += np.float32([0.3, 0.2, -0.2])
    elif change == "turns_emissive":                 # one face of the box becomes a light: 1 -> 2 lights
        new.triangles["material"][4] = 1
    else:
        new.set_camera((-4, 4, -2), (0, 0.3, 0), (0, 1, 0), 40.0)
    render_pair(ptb, gpu_ctx, ctx2, base, new, "sah", method)
    if change == "turns_emissive":
        render_pair(ptb, gpu_ctx, ctx2, new, base, "lbvh", method)      # and back


# ------------------------------------------------------------------------------------------------------ update paths
@pytest.mark.parametrize("builder", BUILDERS)
def test_device_update_from_a_torch_tensor(ptb, gpu_ctx, ctx2, builder):
    import torch
    base = ptb.meshgen.c3_scene(0.05)
    new = ptb.meshgen.c3_deform(base, 0.8, 2.0)
    rays = random_rays(ptb, 100_000, 72, centre=(0, 4, 1), radius=5.0)
    refit_to(ptb, ctx2, base, new, builder)
    gpu_ctx.upload(base)
    gpu_ctx.commit(flag(ptb, builder))
    d = torch.from_numpy(np.ascontiguousarray(new.triangles).view(np.uint8)).cuda()
    torch.cuda.synchronize()                        # the tensor is ready before the context's stream copies it
    gpu_ctx.update_triangles_device(0, d.data_ptr(), len(new.triangles))
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx.bvh_export(), ctx2.bvh_export())
    same_hits(gpu_ctx.closest_hit(rays), ctx2.closest_hit(rays))
    # spheres through the device path too
    s0 = copy.deepcopy(base)
    s0.spheres = np.zeros(3, ptb._lib.sphere_dtype)
    s0.spheres["center"] = [[0, 4, 1], [1, 4, 1.5], [-1, 3, 1]]
    s0.spheres["radius"] = 0.3
    s1 = move_spheres(s0)
    refit_to(ptb, ctx2, s0, s1, builder)
    gpu_ctx.upload(s0)
    gpu_ctx.commit(flag(ptb, builder))
    ds = torch.from_numpy(np.ascontiguousarray(s1.spheres).view(np.uint8)).cuda()
    torch.cuda.synchronize()
    gpu_ctx.update_spheres_device(1, ds.data_ptr() + ptb._lib.sphere_dtype.itemsize, 2)
    gpu_ctx.update_spheres(0, s1.spheres[:1])
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx.bvh_export(), ctx2.bvh_export())
    same_hits(gpu_ctx.closest_hit(rays), ctx2.closest_hit(rays))


@pytest.mark.parametrize("builder", BUILDERS)
def test_partial_update_equals_a_full_set(ptb, gpu_ctx, ctx2, builder):
    base = ptb.meshgen.c3_scene(0.05)
    moved = ptb.meshgen.c3_deform(base, 0.3, 0.5)
    glass = np.nonzero(base.triangles["material"] == 1)[0]
    first, last = int(glass[0]) - 100, int(glass[-1]) + 1     # the glass sphere and the 100 triangles before it
    final = copy.deepcopy(base)
    final.triangles[first:last] = moved.triangles[first:last]
    gpu_ctx.upload(base)
    gpu_ctx.commit(flag(ptb, builder))
    gpu_ctx.update_triangles(first, moved.triangles[first:last])
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.upload(base)
    ctx2.commit(flag(ptb, builder))
    ctx2.upload(final)                                       # ptb_scene_set_* of the whole final arrays
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx.bvh_export(), ctx2.bvh_export())
    rays = random_rays(ptb, 100_000, 73, centre=(0, 4, 1), radius=5.0)
    same_hits(gpu_ctx.closest_hit(rays), ctx2.closest_hit(rays))


# ------------------------------------------------------------------------------------------------------------ full size
def test_refit_full_size_c3(ptb, gpu_ctx, ctx2):
    """BASELINE config C3 at 1 M triangles, deformed: tree consistency and 2^19 hits against a fresh commit."""
    base = ptb.meshgen.c3_scene(1.0)
    new = ptb.meshgen.c3_deform(base, 0.6, 2.0)
    refit_to(ptb, gpu_ctx, base, new, "sah")
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)             # second refit: timed without first-use costs
    refit_ms = gpu_ctx.stats().build_ms
    _, gp, gn = gpu_ctx.bvh_export()
    check_tree(strip(gn), gp, 1_000_000)
    ctx2.upload(new)
    ctx2.commit(ptb._lib.BUILD_SAH)
    rays = random_rays(ptb, 1 << 19, 78, centre=(0, 4, 1), radius=6.0)
    same_hits(gpu_ctx.closest_hit(rays), ctx2.closest_hit(rays))
    print(f"refit of 1 M triangles: {refit_ms:.3f} ms (full SAH commit {ctx2.stats().build_ms:.3f} ms)")


# ------------------------------------------------------------------------------------------------------------ SAH cost
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("which", ["rtweekend1", "overshadowed", "c3"])
def test_sah_cost(ptb, gpu_ctx, rtweekend1, overshadowed, builder, which):
    base, _ = base_and_moved(ptb, rtweekend1, overshadowed, which)
    gpu_ctx.upload(base)
    gpu_ctx.commit(flag(ptb, builder))
    cost = gpu_ctx.bvh_sah_cost()
    _, _, nodes = gpu_ctx.bvh_export()
    assert cost == pytest.approx(sah_cost(nodes, base.n_primitives), rel=1e-12)
    assert all(gpu_ctx.bvh_sah_cost() == cost for _ in range(3))
    worse = scatter(base)
    refit_to(ptb, gpu_ctx, base, worse, builder)
    moved_cost = gpu_ctx.bvh_sah_cost()
    _, _, nodes = gpu_ctx.bvh_export()
    assert moved_cost == pytest.approx(sah_cost(nodes, base.n_primitives), rel=1e-12)
    if which == "c3":   # (in overshadowed the moved 1000-radius ground sphere widens the root box more than the children)
        assert moved_cost > cost


def test_sah_cost_small_scenes(ptb, gpu_ctx, rtweekend1):
    s = copy.deepcopy(rtweekend1)
    s.spheres = np.zeros(1, ptb._lib.sphere_dtype)   # one primitive: 0.125 + 1
    s.spheres["center"] = [0.5, 1.0, 2.0]
    s.spheres["radius"] = 0.25
    gpu_ctx.upload(s)
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)
    assert gpu_ctx.bvh_sah_cost() == 1.125
    s.spheres = s.spheres[:0]
    gpu_ctx.upload(s)
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)
    assert gpu_ctx.bvh_sah_cost() == 0.0
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)             # the empty scene refits trivially
    s.spheres = np.zeros(2, ptb._lib.sphere_dtype)   # two points: a root of zero area
    s.spheres["center"] = [[1, 2, 3], [1, 2, 3]]
    gpu_ctx.upload(s)
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)
    assert gpu_ctx.bvh_sah_cost() == 0.0


# ------------------------------------------------------------------------------------------------------------ errors
def expect(ptb, code, fn, *args):
    with pytest.raises(ptb._lib.PtbError) as e:
        fn(*args)
    assert e.value.code == code, str(e.value)
    return str(e.value)


def test_refit_errors(ptb, overshadowed):
    import ctypes as C
    L = ptb._lib
    INVALID, UNSUPPORTED = 1, 8
    s = overshadowed
    with ptb.Context(0) as ctx:
        ctx.upload(s)
        assert "full commit" in expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT)          # nothing to keep yet
        ctx.commit(L.BUILD_BINARY)
        assert "combined" in expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT | L.BUILD_SAH)
        ctx.commit(L.BUILD_REFIT)
        # the counts of the kept tree
        fewer = copy.deepcopy(s)
        fewer.triangles = fewer.triangles[:-2]
        ctx.upload(fewer)
        assert "triangles" in expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT)
        ctx.commit(L.BUILD_SAH)                                                            # a full commit recovers
        ctx.upload(s)
        expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT)
        ctx.commit(L.BUILD_BINARY)
        # a failed full commit drops the kept tree
        bad = copy.deepcopy(s.triangles[:1])
        bad["material"] = 99
        ctx.update_triangles(0, bad)
        expect(ptb, INVALID, ctx.commit, L.BUILD_BINARY)
        ctx.update_triangles(0, s.triangles[:1])
        assert "failed" in expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT)
        ctx.commit(L.BUILD_BINARY)
        # a refit that fails validation keeps the tree: fixing the input is enough
        ctx.update_triangles(0, bad)
        expect(ptb, INVALID, ctx.commit, L.BUILD_REFIT)
        ctx.update_triangles(0, s.triangles[:1])
        ctx.commit(L.BUILD_REFIT)
        # update ranges and pointers
        nt, ns = len(s.triangles), len(s.spheres)
        expect(ptb, INVALID, ctx.update_triangles, nt - 1, s.triangles[:2])
        expect(ptb, INVALID, ctx.update_spheres, ns + 1, s.spheres[:0])
        h = ctx._h
        big = (1 << 64) - 1
        for fn in (L.lib.ptb_scene_update_triangles, L.lib.ptb_scene_update_triangles_device):
            assert fn(h, big, L.ptr(s.triangles), 2) == INVALID                           # first + n wraps around
            assert fn(h, 1, L.ptr(s.triangles), big) == INVALID
            assert fn(h, 0, None, 1) == INVALID
            assert fn(h, nt, None, 0) == 0                                                 # n == 0: a no-op
        for fn in (L.lib.ptb_scene_update_spheres, L.lib.ptb_scene_update_spheres_device):
            assert fn(h, big, L.ptr(s.spheres), 2) == INVALID
            assert fn(h, 0, None, 1) == INVALID
        # the no-op calls left the scene committed; an update does not
        ctx.closest_hit(random_rays(ptb, 10, 1))
        ctx.update_spheres(0, s.spheres[:1])
        rays = random_rays(ptb, 1000, 2)
        expect(ptb, INVALID, ctx.closest_hit, rays)
        expect(ptb, INVALID, ctx.occluded, ptb.make_occlusion_rays(rays["o"], rays["d"]))
        expect(ptb, INVALID, ctx.check_hit_index, rays, np.zeros(len(rays), np.uint32))
        expect(ptb, INVALID, ctx.bvh_sah_cost)
        d = C.c_double()
        assert L.lib.ptb_bvh_sah_cost(h, None) == INVALID and L.lib.ptb_bvh_sah_cost(h, C.byref(d)) == INVALID
        ctx.commit(L.BUILD_REFIT)
        ctx.closest_hit(rays)
        # the wide tree is not refitted
        ctx.commit(L.BUILD_WIDE)
        assert "8-wide" in expect(ptb, UNSUPPORTED, ctx.commit, L.BUILD_REFIT)
        expect(ptb, UNSUPPORTED, ctx.bvh_sah_cost)
        ctx.commit(L.BUILD_BINARY)
        ctx.commit(L.BUILD_REFIT)
        ctx.closest_hit(rays)
