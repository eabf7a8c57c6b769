"""Indexed triangle meshes through the C ABI: ptb_scene_set_mesh, ptb_scene_update_mesh_* and the device expansion
(lbvh_build.cu k_expand_mesh) that runs at commit.

A mesh scene must behave bit for bit as the flat scene its mesh expands to (IndexedMesh.expand()), so every test runs the
indexed scene in one context and the flat scene in a second one and compares them:
  * full commits over the LBVH, SAH and wide builders: tree exports, SAH cost, closest hit, check_hit_index, occlusion;
  * renders (naive and MIS): every ray counter, and the image to the float-atomics tolerance of the render tests;
  * refits after vertex, normal and triangle updates (host, device from a torch tensor, partial ranges);
  * the error rules: index validation at commit, ranges and pointers, the one-source-at-a-time mode rules;
  * build_ms and kernel_launches include the expansion.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import random_rays

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF
INVALID = 1
VIEW = {"overshadowed": ((-0.3, 0.3, -0.3), 1.5), "c3": ((0, 4, 1), 5.0), "rtweekend1": ((0, 1, 0), 3.0)}


def flag(ptb, builder):
    return {"lbvh": ptb._lib.BUILD_BINARY, "sah": ptb._lib.BUILD_SAH, "wide": ptb._lib.BUILD_WIDE}[builder]


@pytest.fixture()
def ctx2(ptb):
    """The flat scene's context, beside the indexed one."""
    c = ptb.Context(0)
    yield c
    c.close()


def flat_of(scene, mesh):
    import copy
    s = copy.copy(scene)
    s.triangles = mesh.expand()
    return s


def indexed(ptb, overshadowed, rtweekend1, which):
    """(scene, mesh): the scene's own triangles are ignored when it is uploaded with the mesh."""
    if which == "overshadowed":
        return overshadowed, ptb.index_triangles(overshadowed.triangles)
    if which == "rtweekend1":  # spheres only: a mesh of 0 triangles
        return rtweekend1, ptb.IndexedMesh(np.zeros((0, 3)), np.zeros((0, 3)), np.zeros(0, ptb.mesh_triangle_dtype))
    return ptb.meshgen.c3_indexed(0.05)


def same_export(ctx_a, ctx_b, builder):
    for x, y in zip(ctx_a.bvh_export(), ctx_b.bvh_export()):
        assert x.tobytes() == y.tobytes()
    if builder == "wide":
        for x, y in zip(ctx_a.bvh_wide_export(), ctx_b.bvh_wide_export()):
            assert x.tobytes() == y.tobytes()
    else:
        assert ctx_a.bvh_sah_cost() == ctx_b.bvh_sah_cost()


def same_hits(a, b):
    assert a.tobytes() == b.tobytes()


def same_queries(ptb, ctx_a, ctx_b, which, n=100_000, seed=31):
    centre, radius = VIEW[which]
    rays = random_rays(ptb, n, seed, centre=centre, radius=radius)
    g = ctx_a.closest_hit(rays)
    same_hits(g, ctx_b.closest_hit(rays))
    n_prims = ctx_a.bvh_info()[0]
    rng = np.random.default_rng(seed)
    index = np.where(g["prim"] != MISS, g["prim"], rng.integers(0, n_prims, len(rays))).astype(np.uint32)
    index[::5] = rng.integers(0, n_prims, len(index[::5]))
    same_hits(ctx_a.check_hit_index(rays, index), ctx_b.check_hit_index(rays, index))
    occ = ptb.make_occlusion_rays(rays["o"], rays["d"], tmax=rng.uniform(0.0, 2 * radius, len(rays)).astype(np.float32),
                                  exclude=np.where(rng.random(len(rays)) < 0.5, index, MISS).astype(np.uint32))
    a = ctx_a.occluded(occ)
    assert np.array_equal(a, ctx_b.occluded(occ)) and a.any()
    return g


# ------------------------------------------------------------------------------------------------------- full commit
@pytest.mark.parametrize("builder", ["lbvh", "sah", "wide"])
@pytest.mark.parametrize("which", ["overshadowed", "c3", "rtweekend1"])
def test_full_commit_equals_the_flat_scene(ptb, gpu_ctx, ctx2, overshadowed, rtweekend1, builder, which):
    scene, mesh = indexed(ptb, overshadowed, rtweekend1, which)
    gpu_ctx.upload(scene, mesh=mesh)
    gpu_ctx.commit(flag(ptb, builder))
    ctx2.upload(flat_of(scene, mesh))
    ctx2.commit(flag(ptb, builder))
    assert gpu_ctx.bvh_info() == ctx2.bvh_info() == (len(scene.spheres) + len(mesh.triangles), gpu_ctx.bvh_info()[1])
    same_export(gpu_ctx, ctx2, builder)
    g = same_queries(ptb, gpu_ctx, ctx2, which)
    assert (g["prim"] != MISS).any()


def test_full_size_c3(ptb, gpu_ctx, ctx2):
    scene, mesh = ptb.meshgen.c3_indexed(1.0)
    gpu_ctx.upload(scene, mesh=mesh)
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    ctx2.upload(ptb.meshgen.c3_scene(1.0))
    ctx2.commit(ptb._lib.BUILD_SAH)
    assert gpu_ctx.bvh_info()[0] == 1_000_000
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "c3", n=400_000)


# ------------------------------------------------------------------------------------------------------------ render
def render_both(ptb, ctx_a, ctx_b, method, seed=4):
    o = ptb.RenderOptions(samples_per_pixel=16, render_method=method, width=160, height=90, seed=seed)
    res = []
    for ctx in (ctx_a, ctx_b):
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
@pytest.mark.parametrize("which", ["overshadowed", "c3"])
def test_render_equals_the_flat_scene(ptb, gpu_ctx, ctx2, overshadowed, rtweekend1, which, method):
    scene, mesh = indexed(ptb, overshadowed, rtweekend1, which)
    gpu_ctx.upload(scene, mesh=mesh)
    gpu_ctx.commit()
    ctx2.upload(flat_of(scene, mesh))
    ctx2.commit()
    img = render_both(ptb, gpu_ctx, ctx2, method)
    assert img.max() > 0


# ------------------------------------------------------------------------------------------------------------- refit
def commit_pair(ptb, ctx_m, ctx_f, scene, mesh, builder):
    ctx_m.upload(scene, mesh=mesh)
    ctx_m.commit(flag(ptb, builder))
    ctx_f.upload(flat_of(scene, mesh))
    ctx_f.commit(flag(ptb, builder))


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
@pytest.mark.parametrize("path", ["host", "device", "partial"])
def test_vertex_update_and_refit_equal_the_flat_update(ptb, gpu_ctx, ctx2, builder, path):
    import torch
    scene, mesh = ptb.meshgen.c3_indexed(0.05)
    moved = ptb.meshgen.c3_deform_vertices(mesh, 0.5, 1.0)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, builder)
    v = moved.vertices
    if path == "host":
        gpu_ctx.update_mesh_vertices(0, v)
    elif path == "device":
        d = torch.from_numpy(v.copy()).cuda()
        torch.cuda.synchronize()  # the tensor is ready before the context's stream copies it
        gpu_ctx.update_mesh_vertices_device(0, d.data_ptr(), len(v))
    else:  # three ranges, host and device mixed; an empty update in between
        a, b = len(v) // 3, 2 * len(v) // 3
        d = torch.from_numpy(v[a:b].copy()).cuda()
        torch.cuda.synchronize()
        gpu_ctx.update_mesh_vertices(b, v[b:])
        gpu_ctx.update_mesh_vertices_device(a, d.data_ptr(), b - a)
        gpu_ctx.update_mesh_vertices(0, v[:0])
        gpu_ctx.update_mesh_vertices(0, v[:a])
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.update_triangles(0, moved.expand())
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, builder)
    # hits of the refitted mesh scene = a fresh commit of the moved flat scene
    ctx2.upload(flat_of(scene, moved))
    ctx2.commit(flag(ptb, builder))
    same_queries(ptb, gpu_ctx, ctx2, "c3", seed=32)


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
def test_normal_update_changes_the_image_as_the_flat_update(ptb, gpu_ctx, ctx2, builder):
    scene, mesh = ptb.meshgen.c3_indexed(0.05)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, builder)
    before = render_both(ptb, gpu_ctx, ctx2, 1)
    k = len(mesh.normals) // 2
    tilted = mesh.normals[k:] + np.float32([0.3, -0.2, 0.0])
    tilted /= np.linalg.norm(tilted, axis=1, keepdims=True)
    gpu_ctx.update_mesh_normals(k, tilted)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    new = ptb.IndexedMesh(mesh.vertices, np.concatenate([mesh.normals[:k], tilted]), mesh.triangles)
    ctx2.update_triangles(0, new.expand())
    ctx2.commit(ptb._lib.BUILD_REFIT)
    after = render_both(ptb, gpu_ctx, ctx2, 1)
    assert not np.allclose(before, after, rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
@pytest.mark.parametrize("method", [0, 1])
def test_triangle_update_turns_emissive_and_back(ptb, gpu_ctx, ctx2, overshadowed, builder, method):
    scene, mesh = overshadowed, ptb.index_triangles(overshadowed.triangles)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, builder)
    for material in (1, int(mesh.triangles["material"][4])):  # one face of the box becomes a light, then not
        t = mesh.triangles[4:5].copy()
        t["material"] = material
        gpu_ctx.update_mesh_triangles(4, t)
        gpu_ctx.commit(ptb._lib.BUILD_REFIT)
        ctx2.update_triangles(4, ptb.IndexedMesh(mesh.vertices, mesh.normals, t).expand())
        ctx2.commit(ptb._lib.BUILD_REFIT)
        render_both(ptb, gpu_ctx, ctx2, method)
        same_queries(ptb, gpu_ctx, ctx2, "overshadowed", n=20_000)


# ------------------------------------------------------------------------------------------------------------ errors
def expect(ptb, fn, *args, match=None):
    with pytest.raises(ptb.PtbError) as e:
        fn(*args)
    assert e.value.code == INVALID
    if match:
        assert match in str(e.value), str(e.value)


@pytest.mark.parametrize("kind", ["p", "n"])
@pytest.mark.parametrize("refit", [False, True])
def test_an_index_out_of_range_fails_the_commit_until_fixed(ptb, gpu_ctx, ctx2, overshadowed, kind, refit):
    scene, mesh = overshadowed, ptb.index_triangles(overshadowed.triangles)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, "sah")
    bad = mesh.triangles[5:8].copy()
    limit = len(mesh.vertices) if kind == "p" else len(mesh.normals)
    bad[kind][1, 2] = limit
    bad[kind][2, 0] = 0xFFFFFFFF
    commit = (lambda: gpu_ctx.commit(ptb._lib.BUILD_REFIT)) if refit else (lambda: gpu_ctx.commit(ptb._lib.BUILD_SAH))
    if refit:
        gpu_ctx.update_mesh_triangles(5, bad)
    else:
        broken = ptb.IndexedMesh(mesh.vertices, mesh.normals, mesh.triangles.copy())
        broken.triangles[5:8] = bad
        gpu_ctx.upload(scene, mesh=broken)
    what = "vertex" if kind == "p" else "normal"
    expect(ptb, commit, match=f"mesh triangle 6: {what} index out of range")
    expect(ptb, commit, match=f"mesh triangle 6: {what} index out of range")  # still broken: nothing was fixed
    gpu_ctx.update_mesh_triangles(5, mesh.triangles[5:8])
    commit()
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "overshadowed", n=20_000)


def test_update_ranges_and_pointers(ptb, gpu_ctx, overshadowed):
    scene, mesh = overshadowed, ptb.index_triangles(overshadowed.triangles)
    gpu_ctx.upload(scene, mesh=mesh)
    gpu_ctx.commit()
    lib, h = ptb._lib.lib, gpu_ctx._h
    nv, nn, nt = len(mesh.vertices), len(mesh.normals), len(mesh.triangles)
    v = np.zeros((2, 3), np.float32)
    t = mesh.triangles[:2].copy()
    big = 2**64 - 1
    for fn, have, rec in ((lib.ptb_scene_update_mesh_vertices, nv, v), (lib.ptb_scene_update_mesh_normals, nn, v),
                          (lib.ptb_scene_update_mesh_triangles, nt, t)):
        p = ptb._lib.ptr(rec)
        assert fn(h, have - 1, p, 2) == INVALID            # one past the end
        assert fn(h, have + 1, p, 0) == INVALID            # first beyond the end, even with n == 0
        assert fn(h, big, p, 2) == INVALID                 # first + n overflows
        assert fn(h, 1, p, big) == INVALID
        assert fn(h, 0, None, 1) == INVALID                # null pointer with n > 0
        assert fn(h, 0, None, 0) == 0 and fn(h, have, p, 0) == 0  # n == 0: no-op
    for fn in (lib.ptb_scene_update_mesh_vertices_device, lib.ptb_scene_update_mesh_normals_device,
               lib.ptb_scene_update_mesh_triangles_device):
        assert fn(h, 0, None, 1) == INVALID and fn(h, big, None, 2) == INVALID and fn(h, 0, None, 0) == 0
    # set_mesh: null arrays and more than 2^32 - 1 vertices or normals are rejected before anything is read
    p = ptb._lib.ptr(mesh.vertices)
    assert lib.ptb_scene_set_mesh(h, None, 1, p, 1, ptb._lib.ptr(t), 0) == INVALID
    assert lib.ptb_scene_set_mesh(h, p, 2**32, p, 1, ptb._lib.ptr(t), 0) == INVALID
    assert lib.ptb_scene_set_mesh(h, p, 1, p, 2**32, ptb._lib.ptr(t), 0) == INVALID
    assert b"2^32" in lib.ptb_last_error(h)


def test_updates_need_the_matching_mode(ptb, gpu_ctx, ctx2, overshadowed):
    import torch
    scene, mesh = overshadowed, ptb.index_triangles(overshadowed.triangles)
    flat = flat_of(scene, mesh)
    d = torch.zeros(76 * 2, dtype=torch.uint8, device="cuda")
    gpu_ctx.upload(scene, mesh=mesh)
    expect(ptb, gpu_ctx.update_triangles, 0, flat.triangles[:1], match="indexed mesh")
    expect(ptb, gpu_ctx.update_triangles_device, 0, d.data_ptr(), 1, match="indexed mesh")
    # back to flat triangles: the mesh is gone, the context is an ordinary flat one
    gpu_ctx.upload(flat)
    for fn, arg in ((gpu_ctx.update_mesh_vertices, mesh.vertices[:1]), (gpu_ctx.update_mesh_normals, mesh.normals[:1]),
                    (gpu_ctx.update_mesh_triangles, mesh.triangles[:1])):
        expect(ptb, fn, 0, arg, match="not an indexed mesh")
    for fn in (gpu_ctx.update_mesh_vertices_device, gpu_ctx.update_mesh_normals_device, gpu_ctx.update_mesh_triangles_device):
        expect(ptb, fn, 0, d.data_ptr(), 1, match="not an indexed mesh")
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    ctx2.upload(flat)
    ctx2.commit(ptb._lib.BUILD_SAH)
    moved = flat.triangles.copy()
    moved["p"] += np.float32([0.05, 0.02, 0.0])
    gpu_ctx.update_triangles(0, moved)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.update_triangles(0, moved)
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "overshadowed", n=20_000)


def test_refit_keeps_triangle_counts_not_vertex_counts(ptb, gpu_ctx, ctx2):
    scene, mesh = ptb.meshgen.c3_indexed(0.05)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, "lbvh")
    # the same triangles over a vertex array with unused entries appended: the refit keeps the tree
    moved = ptb.meshgen.c3_deform_vertices(mesh, 0.3, 0.5)
    extra = ptb.IndexedMesh(np.concatenate([moved.vertices, np.ones((7, 3), np.float32)]), mesh.normals, mesh.triangles)
    gpu_ctx.set_mesh(extra)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.update_triangles(0, moved.expand())
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, "lbvh")
    # a different number of triangles: the refit is refused, a full commit works
    fewer = ptb.IndexedMesh(mesh.vertices, mesh.normals, mesh.triangles[:-1])
    gpu_ctx.set_mesh(fewer)
    expect(ptb, gpu_ctx.commit, ptb._lib.BUILD_REFIT, match="PTB_BUILD_REFIT keeps the tree")
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)
    assert gpu_ctx.bvh_info()[0] == len(mesh.triangles) - 1


# ------------------------------------------------------------------------------------------------------------- stats
def test_build_stats_include_the_expansion(ptb, gpu_ctx, ctx2):
    scene, mesh = ptb.meshgen.c3_indexed(0.05)
    gpu_ctx.upload(scene, mesh=mesh)
    ctx2.upload(flat_of(scene, mesh))

    def launches(ctx, flags):
        ctx.stats_reset()
        ctx.commit(flags)
        st = ctx.stats()
        assert st.build_ms > 0
        return st.kernel_launches

    B, R = ptb._lib.BUILD_BINARY, ptb._lib.BUILD_REFIT
    assert launches(gpu_ctx, B) == launches(ctx2, B) + 1        # the expansion: one kernel
    assert launches(gpu_ctx, B) == launches(ctx2, B)            # unchanged mesh: not expanded again
    assert launches(gpu_ctx, R) == launches(ctx2, R)
    gpu_ctx.update_mesh_vertices(0, mesh.vertices[:3])
    ctx2.update_triangles(0, mesh.expand()[:1])
    assert launches(gpu_ctx, R) == launches(ctx2, R) + 1        # an update makes the next commit expand
